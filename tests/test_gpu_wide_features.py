"""
GPU tests of distance mode 2 for feature vectors wider than 160 (161 <= d <= 1024): the fused kernel with the STREAMED query
operand (fused.cu, gram_select_kernel<KR, NKT_STREAMED>) and the rest of the fused chain at wide d.  The library takes that
path on its own once a stage has WIDE_FUSED_MIN_PAIRS (query, point) pairs, U x n; the tests lower the threshold to 0
(CHB_WIDE_FUSED_MIN_PAIRS) to run it at sizes the sequential oracle checks in seconds.  Bars as everywhere: labels identical to the oracle, kept keys
within their proven slack, pruning never removes a bin that can win.
"""
import os

import numpy as np
import pytest

import chbin_b200
import fused_invariants
import oracle
from chbin_b200 import capi, synth

pytestmark = pytest.mark.gpu

THREADS = os.cpu_count() or 1
DEFAULT_MIN_PAIRS = 250_000  # WIDE_FUSED_MIN_PAIRS, ch-bin_b200/csrc/api.cu


@pytest.fixture
def wide_fused(monkeypatch):
    """Every wide stage takes the fused path, whatever its size."""
    monkeypatch.setenv("CHB_WIDE_FUSED_MIN_PAIRS", "0")


def _features(n, C, d, n_seed, seed, concentration=4000.0):
    """d = k-mer part + coverage samples: 4-mer-like (136) up to d = 296, 5-mer-like (512) beyond."""
    kd = 136 if d <= 296 else 512
    X, bins, truth = synth.make_contig_features(n, C, d - kd, n_seed, seed=seed, concentration=concentration, kmer_dims=kd)
    assert X.shape[1] == d
    return X, bins, truth


def _fit_same_as_oracle(X, C, bins, k, iters, metric="convex", **kw):
    perms = oracle.draw_permutations(bins, iters, seed=0)
    ref, rinfo = oracle.fit_cluster(X, C, bins, None, k, iters, metric=metric, perms=perms, threads=THREADS, return_info=True)
    np.random.seed(0)
    got, info = chbin_b200.fit_cluster(X, C, bins, None, k, iters, metric, return_info=True, **kw)
    assert np.array_equal(got, ref)
    assert info["iterations"] == rinfo["iterations"] and list(info["changed"]) == list(rinfo["changed"])
    return info


def _assert_fused_ran(info, k):
    t = info["timers"]
    assert t["launches_distance"] == 0, "a mode-1 candidate matrix was built"
    if k <= 24:
        assert t["launches_gram"] > 0 and t["gram_tiles"] == t["gram_tiles_planned"] > 0
    else:
        assert t["launches_gram"] == 0  # pruning + exact selection, no Gram kernel (as at d <= 160)


WIDE_CASES = [
    # d, k, metric, n, C
    (161, 5, "convex", 1500, 6),
    (176, 10, "convex", 1500, 6),
    (200, 1, "convex", 1200, 5),
    (200, 16, "affine-qp", 1500, 5),
    (200, 32, "convex", 1500, 4),
    (296, 24, "convex", 1800, 5),
    (296, 5, "affine", 1200, 6),
    (528, 5, "convex", 1500, 6),
    (528, 10, "affine-qp", 1200, 5),
    (528, 32, "convex", 1500, 4),
    (1024, 10, "convex", 1200, 5),
    (1024, 16, "convex", 1500, 4),
    (1024, 24, "affine", 1200, 4),
]


@pytest.mark.parametrize("d,k,metric,n,C", WIDE_CASES)
def test_wide_fused_labels_match_sequential_oracle(wide_fused, d, k, metric, n, C):
    X, bins, _ = _features(n, C, d, 30, seed=d + k, concentration=300.0)
    info = _fit_same_as_oracle(X, C, bins, k, 6, metric=metric)
    _assert_fused_ran(info, k)


@pytest.mark.parametrize("d,k", [(200, 5), (528, 10), (1024, 24)])
def test_wide_fused_duplicates_tiny_bins_and_bins_without_seeds(wide_fused, d, k):
    """Duplicate contigs (more keys inside the slack window than a kept list holds: exact redo), a bin with no seed at
    all, a bin that starts with a single member and bins smaller than k."""
    X, bins, _ = _features(1400, 6, d, 8, seed=d, concentration=400.0)
    X[300:340] = X[300]
    X[700:712] = X[700]
    bins[bins == 2] = -1
    keep = np.where(bins == 4)[0]
    bins[keep[1:]] = -1
    info = _fit_same_as_oracle(X, 6, bins, k, 6)
    _assert_fused_ran(info, k)


@pytest.mark.parametrize("d,k", [(528, 5), (1024, 10)])
def test_wide_fused_keys_within_proven_bound_and_lists_complete(wide_fused, d, k):
    """The kept FP32 keys of the streamed kernel lie within the per-(query, bin) slack of the exact squared distance, the
    kept lists hold every true neighbour, and a pruned bin is never the nearest hull (tests/fused_invariants.py)."""
    C = 5
    X, bins, _ = _features(1300, C, d, 12, seed=29 + d)
    perms = oracle.draw_permutations(bins, 2, seed=0)
    ref = fused_invariants.Reference(X, bins, C, k)
    ctx = capi.Context(0)
    ctx.set_features(X); ctx.set_params(k, "convex"); ctx.set_distance_mode(2); ctx.set_labels(bins, C)
    assert ctx.distance_path() == 2
    ctx.build_distance_matrix(True)
    cur = bins.copy()
    worst = 0.0
    for it in range(2):
        lab, _ = ctx.fit_iteration(perms[it])
        worst = max(worst, fused_invariants.check_iteration(ctx, ref, perms[it], cur, lab, threads=THREADS)["worst"])
        cur = lab
    ctx.close()
    assert worst < 0.5, f"observed error / bound = {worst}: the bound should have a wide margin"


def test_wide_row_bounds_hold_on_large_cancelling_coordinates(wide_fused):
    """d = 1024, features far from the global mean (|x - mu| ~ 1e3) with in-bin offsets ~1e-2: the FP32 differences cancel
    almost completely.  For every row the pruning bounds must still hold against exact FP64 distances to the seeds of the
    guessed bin: ub >= the nearest one, ubk2 >= the k-th smallest squared one (with the rest of tests/fused_invariants.py)."""
    rng = np.random.default_rng(5)
    n, d, C, k, n_seed = 1200, 1024, 4, 5, 40
    truth = np.arange(n) % C
    centres = rng.normal(size=(C, d))
    centres *= 1e3 / np.linalg.norm(centres, axis=1, keepdims=True)
    X = np.ascontiguousarray(centres[truth] + 1e-2 * rng.normal(size=(n, d)))
    bins = np.full(n, -1, dtype=np.int64)
    for c in range(C):
        bins[np.where(truth == c)[0][:n_seed]] = c
    ref = fused_invariants.Reference(X, bins, C, k)
    perm = oracle.draw_permutations(bins, 1, seed=0)[0]
    ctx = capi.Context(0)
    ctx.set_features(X); ctx.set_params(k, "convex"); ctx.set_distance_mode(2); ctx.set_labels(bins, C)
    ctx.build_distance_matrix(True)
    lab, _ = ctx.fit_iteration(perm)
    guess, _, _ = ctx.get_row_bounds(0, len(ref.pts))
    fused_invariants.check_iteration(ctx, ref, perm, bins, lab, threads=THREADS)
    ctx.close()
    assert np.all(guess < C)


@pytest.mark.parametrize("on_device", [False, True])
def test_wide_sharded_contexts_exchange_labels(wide_fused, on_device):
    """Several contexts on one device own slices of the query slots, exchange their guesses and tentative labels by MAX
    (what the NCCL collectives do between ranks); with on_device the permutation is handed over in device memory
    (chb_iteration_begin_dev), the path the driver takes when the library reports the fused path."""
    import torch

    X, bins, _ = _features(2500, 6, 200, 15, seed=23, concentration=120.0)
    perms = oracle.draw_permutations(bins, 3, seed=0)
    U = perms.shape[1]
    edges = [0, int(U * 0.3), int(U * 0.3), U]  # one empty shard
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    ctxs = []
    for u0, u1 in zip(edges[:-1], edges[1:]):
        ctx = capi.Context(0)
        ctx.set_stream(stream.cuda_stream)
        ctx.set_features(X); ctx.set_params(5, "convex"); ctx.set_distance_mode(2)
        ctx.set_labels(bins, 6, u0, u1)
        assert ctx.distance_path() == 2
        ctx.build_distance_matrix(True)
        ctxs.append(ctx)
    cur = bins.copy()
    with torch.cuda.stream(stream):
        gs = [torch.empty(U, dtype=torch.int32, device=dev) for _ in ctxs]
        active = [ctx.guess_export(g.data_ptr()) for ctx, g in zip(ctxs, gs)]
        assert all(active)
        merged_g = torch.stack(gs).max(dim=0).values.contiguous()
        for ctx in ctxs:
            ctx.guess_import(merged_g.data_ptr())
        for it in range(3):
            perm_dev = torch.from_numpy(np.ascontiguousarray(perms[it], dtype=np.int64)).to(dev)
            for ctx in ctxs:
                if on_device:
                    ctx.iteration_begin_dev(perm_dev.data_ptr(), U)
                else:
                    ctx.iteration_begin(perms[it])
            lo = 0
            while lo < U:
                tents = [torch.empty(U - lo, dtype=torch.int32, device=dev) for _ in ctxs]
                for ctx, t in zip(ctxs, tents):
                    ctx.round_run(lo, U, t.data_ptr())
                merged = torch.stack(tents).max(dim=0).values.contiguous()
                firsts = [ctx.round_commit(lo, U, merged.data_ptr()) for ctx in ctxs]
                assert len(set(firsts)) == 1
                lo = U if firsts[0] < 0 else firsts[0] + 1
            changed = [ctx.iteration_end() for ctx in ctxs]
            assert len(set(changed)) == 1
            ref = oracle.fit_cluster(X, 6, cur, None, 5, 1, perms=perms[it:it + 1], threads=THREADS)
            for ctx in ctxs:
                assert np.array_equal(ctx.get_labels(), ref), it
            cur = ref
    for ctx in ctxs:
        ctx.close()


def test_wide_ranks_whose_slices_straddle_the_threshold_take_the_same_path(monkeypatch):
    """The path is chosen from the STAGE's pair count (U x n), latched at chb_set_labels: two ranks whose owned slices fall on
    either side of the threshold (U = 499 split 249 / 250 over n = 1000 contigs, threshold 249 500 owned pairs) must both take
    the fused path, export their guesses (a rank that did not would skip the guess all-reduce the others enter) and produce
    the oracle's labels; changing the variable after chb_set_labels changes nothing for that stage."""
    import torch

    from chbin_b200.clustering import owned_slots

    X, bins, _ = _features(1000, 3, 200, 167, seed=3, concentration=300.0)
    U = int(np.sum(bins == -1))
    assert U == 499
    slices = [owned_slots(U, r, 2) for r in range(2)]
    assert [(u1 - u0) * len(X) for u0, u1 in slices] == [249_000, 250_000]
    monkeypatch.setenv("CHB_WIDE_FUSED_MIN_PAIRS", "249500")
    perms = oracle.draw_permutations(bins, 2, seed=0)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    ctxs = []
    for u0, u1 in slices:
        ctx = capi.Context(0)
        ctx.set_stream(stream.cuda_stream)
        ctx.set_features(X); ctx.set_params(5, "convex"); ctx.set_distance_mode(2)
        ctx.set_labels(bins, 3, u0, u1)
        ctxs.append(ctx)
    monkeypatch.setenv("CHB_WIDE_FUSED_MIN_PAIRS", str(2**62))  # latched: this stage keeps its decision
    assert [ctx.distance_path() for ctx in ctxs] == [2, 2]
    for ctx in ctxs:
        ctx.build_distance_matrix(True)
    cur = bins.copy()
    with torch.cuda.stream(stream):
        gs = [torch.empty(U, dtype=torch.int32, device=dev) for _ in ctxs]
        assert [ctx.guess_export(g.data_ptr()) for ctx, g in zip(ctxs, gs)] == [True, True]
        merged_g = torch.stack(gs).max(dim=0).values.contiguous()
        for ctx in ctxs:
            ctx.guess_import(merged_g.data_ptr())
        for it in range(2):
            for ctx in ctxs:
                ctx.iteration_begin(perms[it])
            lo = 0
            while lo < U:
                tents = [torch.empty(U - lo, dtype=torch.int32, device=dev) for _ in ctxs]
                for ctx, t in zip(ctxs, tents):
                    ctx.round_run(lo, U, t.data_ptr())
                merged = torch.stack(tents).max(dim=0).values.contiguous()
                firsts = [ctx.round_commit(lo, U, merged.data_ptr()) for ctx in ctxs]
                assert len(set(firsts)) == 1
                lo = U if firsts[0] < 0 else firsts[0] + 1
            assert len({ctx.iteration_end() for ctx in ctxs}) == 1
            ref = oracle.fit_cluster(X, 3, cur, None, 5, 1, perms=perms[it:it + 1], threads=THREADS)
            for ctx in ctxs:
                assert np.array_equal(ctx.get_labels(), ref), it
            cur = ref
    for ctx in ctxs:
        ctx.close()
    # below the threshold for the whole stage: every rank takes mode 1
    monkeypatch.setenv("CHB_WIDE_FUSED_MIN_PAIRS", str(U * len(X) + 1))
    for u0, u1 in slices:
        with capi.Context(0) as ctx:
            ctx.set_features(X); ctx.set_params(5, "convex"); ctx.set_distance_mode(2); ctx.set_labels(bins, 3, u0, u1)
            assert ctx.distance_path() == 1


@pytest.mark.parametrize("d", [200, 528])
def test_wide_fused_overlapping_bins_take_row_block_items(wide_fused, monkeypatch, d):
    """Heavily overlapping bins: almost nothing is pruned, the surviving (row, bin) pairs overflow the compact pair-block
    buffer, and the streamed kernel works on (row block, bin) items of the resident-layout operand instead.  That the compact
    buffer overflows is shown by the same stage being refused when the per-(row, bin) lists are forbidden
    (CHB_DENSE_LIST_GB = 0); with them, the labels equal the oracle's."""
    rng = np.random.default_rng(d)
    n, C, n_seed, k = 1200, 8, 30, 5
    truth = np.arange(n) % C
    X = np.ascontiguousarray(0.05 * rng.normal(size=(C, d))[truth] + rng.normal(size=(n, d)))
    bins = np.full(n, -1, dtype=np.int64)
    for c in range(C):
        bins[np.where(truth == c)[0][:n_seed]] = c
    monkeypatch.setenv("CHB_DENSE_LIST_GB", "0")
    with pytest.raises(MemoryError, match="CHB_DENSE_LIST_GB"):
        chbin_b200.fit_cluster(X, C, bins, None, k, 3, reuse_context=False)
    monkeypatch.delenv("CHB_DENSE_LIST_GB")
    info = _fit_same_as_oracle(X, C, bins, k, 3, reuse_context=False)
    _assert_fused_ran(info, k)


def test_wide_routing_follows_the_pair_count(monkeypatch):
    """Without the override: a wide stage just above WIDE_FUSED_MIN_PAIRS stage pairs (U x n) takes the fused path, one just below
    it the matrix path (distance mode 1), d <= 160 is fused at any size and d > 1024 never; labels are the oracle's."""
    monkeypatch.delenv("CHB_WIDE_FUSED_MIN_PAIRS", raising=False)

    def path(X, bins, C, k=5):
        with capi.Context(0) as ctx:
            ctx.set_features(X); ctx.set_labels(bins, C); ctx.set_params(k, "convex"); ctx.set_distance_mode(2)
            return ctx.distance_path()

    def sized(n_own_target, d, C=5, n_seed=20):
        # U x n just above / below the threshold: U = n - C * n_seed
        n = int(np.ceil((C * n_seed + np.sqrt((C * n_seed) ** 2 + 4 * n_own_target)) / 2))
        return _features(n, C, d, n_seed, seed=n)

    X, bins, _ = sized(DEFAULT_MIN_PAIRS, 200)
    n_own = int(np.sum(bins == -1))
    assert n_own * len(X) >= DEFAULT_MIN_PAIRS > (n_own - 1) * (len(X) - 1)
    assert path(X, bins, 5) == 2
    info = _fit_same_as_oracle(X, 5, bins, 5, 2)
    _assert_fused_ran(info, 5)
    Xb, bb, _ = sized(DEFAULT_MIN_PAIRS * 0.9, 200)
    assert path(Xb, bb, 5) == 1
    Xs, bs, _ = synth.make_contig_features(500, 4, 10, 15, seed=8)  # d = 146: always the resident kernel
    assert path(Xs, bs, 4) == 2
    Xw, bw, _ = synth.make_contig_features(600, 4, 600, 15, seed=8, kmer_dims=512)  # d = 1112
    monkeypatch.setenv("CHB_WIDE_FUSED_MIN_PAIRS", "0")
    assert path(Xw, bw, 4) == 1
    assert path(Xb, bb, 5) == 2


def test_wide_at_size_100k_d200_every_position_of_iteration_1():
    """100k contigs x d = 200 (136 4-mers + 64 samples), k = 10: the default routing takes the streamed fused path;
    iteration 1 is checked at every position with the position-parallel oracle."""
    X, bins, _ = synth.make_contig_features(100_000, 100, 64, 50, seed=0)
    C, k = 100, 10
    perms = oracle.draw_permutations(bins, 1, seed=0)
    with capi.Context(0) as ctx:
        ctx.set_features(X); ctx.set_labels(bins, C); ctx.set_params(k, "convex")
        assert ctx.distance_path() == 2
        ctx.build_distance_matrix(False)
        lab, nch = ctx.fit_iteration(perms[0])
        tm = ctx.timers()
    assert tm["launches_distance"] == 0 and tm["launches_gram"] > 0 and tm["gram_tiles"] == tm["gram_tiles_planned"]
    res = oracle.verify_iteration(X, C, bins, lab, perms[0], k, threads=THREADS)
    assert res["mismatches"] == 0, res["mismatches"]
    assert nch == int(np.sum(lab != bins))


def test_wide_at_size_200k_d528_sampled_positions():
    """200k contigs x d = 528 (5-mer-like profiles + 16 samples), k = 5: checked on 3000 sampled positions including the
    first and the last 256."""
    X, bins, _ = synth.make_contig_features(200_000, 100, 16, 50, seed=0, kmer_dims=512)
    C, k = 100, 5
    perms = oracle.draw_permutations(bins, 1, seed=0)
    U = perms.shape[1]
    with capi.Context(0) as ctx:
        ctx.set_features(X); ctx.set_labels(bins, C); ctx.set_params(k, "convex")
        assert ctx.distance_path() == 2
        ctx.build_distance_matrix(False)
        lab, _ = ctx.fit_iteration(perms[0])
        tm = ctx.timers()
    assert tm["launches_distance"] == 0 and tm["launches_gram"] > 0
    rng = np.random.default_rng(1)
    positions = np.unique(np.concatenate([np.arange(256), np.arange(U - 256, U), rng.choice(U, 3000, replace=False)]))
    res = oracle.verify_iteration(X, C, bins, lab, perms[0], k, positions=positions.astype(np.int64), threads=THREADS)
    assert res["mismatches"] == 0, res["mismatches"]
