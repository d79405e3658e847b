"""
GPU parity tests proper: every check goes through the C-ABI (chbin_b200.capi.Context -> libchbin_b200.so) and is
compared with the CPU oracle (oracle/*.c) on the same seeded inputs.  Bars: bit-exact for distances, kNN index
sets and labels; |d_gpu - d_ref| <= 1e-6*d_ref + 1e-12*||x|| for hull distances (BASELINE.md section 4).
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


def _ctx(X, bins, C, k, metric="convex", materialise=True, slots=(0, -1), dist_mode=1, gram_engine=1):
    ctx = capi.Context(0)
    ctx.set_features(X)
    ctx.set_labels(bins, C, *slots)
    ctx.set_params(k, metric)
    ctx.set_distance_mode(dist_mode)
    ctx.set_gram_engine(gram_engine)
    ctx.build_distance_matrix(materialise)
    return ctx


@pytest.mark.parametrize("engine", [0, 1])
@pytest.mark.parametrize("n,S", [(700, 1), (1111, 10), (300, 20)])
def test_candidate_values_within_proven_bound(engine, n, S):
    """|A - d^2| <= eps_rel * (nrm[query] + max nrm) for the FFMA (approx.cu) and tcgen05 (gram_tc.cu) engines."""
    X, bins, _ = synth.make_contig_features(n, 4, S, 10, seed=13)
    X[5] = X[6]
    pts = np.where(bins == -1)[0]
    D = oracle.create_in_mem_distance_matrix(X)[pts]
    with _ctx(X, bins, 4, 5, gram_engine=engine) as ctx:
        A, eps_rel, nrm = ctx.get_candidate_rows(0, len(pts))
    Xc = (X - X.mean(axis=0)).astype(np.float32).astype(np.float64)   # the kernels contract fl32(x - mean)
    nn = np.sum(Xc * Xc, axis=1)
    assert np.all(nrm >= nn * (1 - 1e-6)) and np.all(nrm <= nn * (1 + 1e-5) + 1e-30)
    bound = eps_rel * (nrm[pts].astype(np.float64)[:, None] + float(nrm.max()))
    err = np.abs(A.astype(np.float64) - D * D)
    assert np.all(err <= bound), f"bound violated by {np.max(err / bound):.3f}x"
    assert np.max(err / bound) < 0.5, "the proven bound should hold with margin"


@pytest.mark.parametrize("n,d_extra", [(300, 1), (1000, 10), (257, 3)])
def test_distance_rows_bit_exact(n, d_extra):
    X, bins, _ = synth.make_contig_features(n, 4, d_extra, 10, seed=3)
    D = oracle.create_in_mem_distance_matrix(X)
    pts = np.where(bins == -1)[0]
    for mat in (True, False):
        for mode in (0, 1):
            with _ctx(X, bins, 4, 5, materialise=mat, dist_mode=mode) as ctx:
                rows = ctx.get_distance_rows(0, len(pts))
            assert rows.shape == (len(pts), n)
            assert np.array_equal(rows, D[pts]), "distance rows differ from the scipy-cdist recipe"


@pytest.mark.parametrize("dist_mode", [0, 1])
@pytest.mark.parametrize("k", [1, 3, 5, 10, 32])
def test_knn_per_bin_exact(k, dist_mode):
    n, C = 1500, 7
    X, bins, truth = synth.make_contig_features(n, C, 1, 12, seed=5)
    rng = np.random.default_rng(k)
    labels = truth.copy()
    labels[rng.random(n) < 0.3] = -1            # a mix of assigned / unassigned
    labels[truth == 6] = -1
    labels[np.where(truth == 6)[0][:2]] = 6     # a bin smaller than k
    queries = rng.choice(n, 64, replace=False)
    X[100] = X[101]                              # exact duplicates: ties broken by index
    X[102] = X[101]
    X[200:240] = X[200]                          # 40 identical contigs: more ties than the kept-set reserve
    labels[200:240] = truth[200]
    with _ctx(X, bins, C, k, dist_mode=dist_mode) as ctx:
        idx, m = ctx.knn_per_bin(labels, queries)
    D = oracle.create_in_mem_distance_matrix(X)
    for qi, q in enumerate(queries):
        lab = labels.copy()
        lab[q] = -1                              # algorithm.py:50
        for c in range(C):
            ref = oracle.find_nearest_from_cluster(c, lab, D[q], k)
            got = idx[qi, c, : m[qi, c]]
            assert m[qi, c] == len(ref)
            assert np.array_equal(np.sort(got), np.sort(ref)), (q, c)
            assert np.all(idx[qi, c, m[qi, c]:] == -1)


def _hull_case(X, rng, k, nq, C):
    n = len(X)
    queries = rng.choice(n, nq, replace=False)
    idx = np.full((nq, C, k), -1, dtype=np.int64)
    m = np.zeros((nq, C), dtype=np.int32)
    for qi in range(nq):
        for c in range(C):
            mm = int(rng.integers(0, k + 1)) if c == 0 else k
            m[qi, c] = mm
            cand = np.setdiff1d(np.arange(n), [queries[qi]])
            idx[qi, c, :mm] = rng.choice(cand, mm, replace=False)
    return queries, idx, m


@pytest.mark.parametrize("k", [1, 2, 3, 5, 8, 10, 16, 32])
def test_hull_distance_vs_oracle(k):
    n, C = 800, 6
    X, bins, _ = synth.make_contig_features(n, C, 1 if k <= 5 else 10, 20, seed=11)
    rng = np.random.default_rng(100 + k)
    queries, idx, m = _hull_case(X, rng, k, 48, C)
    with _ctx(X, bins, C, k) as ctx:
        dist, status, alpha = ctx.hull_distance_batch(queries, idx, m, want_alpha=True)
    for qi, q in enumerate(queries):
        for c in range(C):
            mm = m[qi, c]
            if mm == 0:
                assert np.isinf(dist[qi, c]) and status[qi, c] == 3
                continue
            ref = oracle.convex_hull_distance(X[q], X[idx[qi, c, :mm]])
            tol = 1e-6 * ref + 1e-12 * np.linalg.norm(X[q])
            assert abs(dist[qi, c] - ref) <= tol, (q, c, mm, dist[qi, c], ref)
            a = alpha[qi, c, :mm]
            assert abs(a.sum() - 1) < 1e-10 and a.min() >= 0.0


def test_hull_distance_degenerate_duplicates():
    # duplicated neighbour rows and a query identical to a neighbour (SURVEY.md section 7, hard part 3)
    n, C, k = 400, 3, 5
    X, bins, _ = synth.make_contig_features(n, C, 1, 10, seed=2)
    X[10] = X[11]
    X[12] = X[11]
    X[50] = X[51]
    queries = np.array([0, 51], dtype=np.int64)
    idx = np.full((2, C, k), -1, dtype=np.int64)
    m = np.zeros((2, C), dtype=np.int32)
    idx[0, 0] = [10, 11, 12, 13, 14]; m[0, 0] = 5
    idx[0, 1, :3] = [10, 11, 12]; m[0, 1] = 3
    idx[0, 2, :2] = [20, 21]; m[0, 2] = 2
    idx[1, 0] = [50, 60, 61, 62, 63]; m[1, 0] = 5
    idx[1, 1, :1] = [50]; m[1, 1] = 1
    idx[1, 2, :4] = [10, 11, 70, 71]; m[1, 2] = 4
    with _ctx(X, bins, C, k) as ctx:
        dist, status = ctx.hull_distance_batch(queries, idx, m)
    for qi, q in enumerate(queries):
        for c in range(C):
            ref = oracle.convex_hull_distance(X[q], X[idx[qi, c, : m[qi, c]]])
            scale = np.linalg.norm(X[idx[qi, c, : m[qi, c]]] - X[q], axis=1).max() + np.linalg.norm(X[q])
            assert abs(dist[qi, c] - ref) <= 1e-6 * ref + 1e-7 * scale, (qi, c, dist[qi, c], ref)
    assert dist[1, 0] <= 1e-9 and dist[1, 1] <= 1e-12


def test_affine_qp_metric():
    n, C, k = 500, 4, 6
    X, bins, _ = synth.make_contig_features(n, C, 3, 15, seed=4)
    rng = np.random.default_rng(9)
    queries, idx, m = _hull_case(X, rng, k, 24, C)
    m[m == 0] = 1
    for qi in range(len(queries)):
        for c in range(C):
            if idx[qi, c, 0] < 0:
                idx[qi, c, 0] = (queries[qi] + 1) % n
    with _ctx(X, bins, C, k, metric="affine-qp") as ctx:
        dist, status = ctx.hull_distance_batch(queries, idx, m)
    for qi, q in enumerate(queries):
        for c in range(C):
            ref = oracle.affine_hull_distance_qp(X[q], X[idx[qi, c, : m[qi, c]]])
            assert abs(dist[qi, c] - ref) <= 1e-6 * ref + 1e-12, (qi, c)


FIT_CASES = [
    # n, C, S, n_seed, k, concentration, window, materialise, distance path
    (600, 5, 1, 40, 5, 4000.0, 0, True, "filter"),
    (600, 5, 1, 40, 5, 4000.0, 0, True, "exact"),
    (600, 5, 1, 40, 5, 4000.0, 0, True, "fused"),
    (1500, 8, 1, 30, 5, 60.0, 0, True, "filter"),      # hard, overlapping genomes: many repair rounds, 10 iterations
    (1500, 8, 1, 30, 5, 60.0, 0, True, "exact"),
    (1500, 8, 1, 30, 5, 60.0, 0, True, "fused"),
    (1500, 8, 1, 30, 5, 60.0, 97, True, "filter"),     # same with a small window
    (1500, 8, 1, 30, 5, 60.0, 97, True, "fused"),
    (1200, 6, 10, 25, 10, 300.0, 0, False, "filter"),  # k = 10, rows recomputed on demand (InMemDistMatrix = no)
    (1200, 6, 10, 25, 10, 300.0, 0, False, "exact"),
    (1200, 6, 10, 25, 10, 300.0, 0, True, "fused"),
    (900, 4, 3, 3, 7, 500.0, 0, True, "filter"),       # bins smaller than k at the start
    (900, 4, 3, 3, 7, 500.0, 0, True, "fused"),
    (5000, 20, 1, 20, 5, 1000.0, 0, True, "filter"),   # larger: several CTAs per SM, chunked queue
    (5000, 20, 1, 20, 5, 1000.0, 0, True, "fused"),
    (1500, 8, 1, 30, 5, 60.0, 0, True, "filter-ffma"), # distance mode 1 with the FFMA Gram engine
    (1200, 6, 10, 25, 10, 300.0, 0, False, "filter-ffma"),
]
_PATHS = {"exact": (0, 1), "filter": (1, 1), "filter-ffma": (1, 0), "fused": (2, 1)}


@pytest.mark.parametrize("n,C,S,n_seed,k,conc,window,mat,path", FIT_CASES)
def test_fit_cluster_labels_identical(n, C, S, n_seed, k, conc, window, mat, path):
    dmode, engine = _PATHS[path]
    X, bins, _ = synth.make_contig_features(n, C, S, n_seed, seed=7, concentration=conc)
    perms = oracle.draw_permutations(bins, 10, seed=0)
    ref, info = oracle.fit_cluster(X, C, bins, None, k, 10, perms=perms, return_info=True, threads=4)
    np.random.seed(0)
    bins_before = bins.copy()
    got, ginfo = chbin_b200.fit_cluster(X, C, bins, None, k, 10, "convex", "b200", in_mem_dist_matrix=mat,
                                        window=window, return_info=True, distance_mode=dmode, gram_engine=engine)
    assert np.array_equal(bins, bins_before), "inputs must not be mutated (algorithm.py:37)"
    assert got.dtype == np.int64
    assert ginfo["iterations"] == info["iterations"] and ginfo["converged"] == info["converged"]
    assert list(ginfo["changed"]) == list(info["changed"])
    assert np.array_equal(got, ref)


def test_fit_cluster_fused_with_duplicate_contigs():
    # many identical contigs: more candidates inside the filter slack than the kept list holds -> exact-path fallback
    X, bins, _ = synth.make_contig_features(1200, 5, 1, 20, seed=17, concentration=300.0)
    X[300:340] = X[300]
    X[700:712] = X[700]
    perms = oracle.draw_permutations(bins, 10, seed=0)
    ref = oracle.fit_cluster(X, 5, bins, None, 5, 10, perms=perms, threads=4)
    np.random.seed(0)
    got = chbin_b200.fit_cluster(X, 5, bins, None, 5, 10, distance_mode=2)
    assert np.array_equal(got, ref)


@pytest.mark.parametrize("n,C,S,k", [(1500, 6, 1, 5), (2000, 8, 10, 10), (900, 4, 20, 5)])
def test_fused_keys_within_proven_bound_and_lists_complete(n, C, S, k):
    """Distance mode 2 (fused.cu): every FP32 key the fused Gram + selection kernel kept must lie within the per-(query,
    bin) slack of the exact squared distance (per-bin centred operands), and the kept lists must contain every point
    whose exact distance is among the k smallest of its bin -- the two facts the exact re-rank relies on.  Also the rest
    of tests/fused_invariants.py: cached sets and hull distances, pruning, row bounds, guess."""
    X, bins, _ = synth.make_contig_features(n, C, S, 12, seed=29)
    perms = oracle.draw_permutations(bins, 2, seed=0)
    ref = fused_invariants.Reference(X, bins, C, k)
    ctx = capi.Context(0)
    ctx.set_features(X); ctx.set_params(k, "convex"); ctx.set_distance_mode(2); ctx.set_labels(bins, C)
    ctx.build_distance_matrix(True)
    cur = bins.copy()
    worst = 0.0
    for it in range(2):
        lab, _ = ctx.fit_iteration(perms[it])
        worst = max(worst, fused_invariants.check_iteration(ctx, ref, perms[it], cur, lab, threads=THREADS)["worst"])
        cur = lab
    ctx.close()
    assert worst < 0.5, f"observed error / bound = {worst}: the bound should have a wide margin"


@pytest.mark.parametrize("path", ["exact", "filter", "fused"])
def test_cached_neighbour_sets_match_each_querys_view(path):
    """After every iteration, the (query, bin) neighbour sets the rounds left in the cache must equal
    find_nearest_from_cluster evaluated on the labels exactly as the reference's sequential loop showed them to
    that query (earlier positions re-assigned, later positions not yet)."""
    dmode, engine = _PATHS[path]
    X, bins, _ = synth.make_contig_features(1000, 5, 1, 20, seed=17, concentration=300.0)
    X[300:340] = X[300]          # duplicate contigs: ties, candidate-list overflow, exact-path fallback
    X[700:712] = X[700]
    perms = oracle.draw_permutations(bins, 3, seed=0)
    D = oracle.create_in_mem_distance_matrix(X)
    pts = np.where(bins == -1)[0]
    ctx = capi.Context(0)
    ctx.set_features(X); ctx.set_params(5, "convex"); ctx.set_distance_mode(dmode); ctx.set_gram_engine(engine)
    ctx.set_labels(bins, 5); ctx.build_distance_matrix(True)
    cur = bins.copy()
    for it in range(3):
        lab, _ = ctx.fit_iteration(perms[it])
        ref = oracle.fit_cluster(X, 5, cur, None, 5, 1, perms=perms[it:it + 1], threads=4)
        assert np.array_equal(lab, ref)
        idx, cnt, dist = ctx.get_pair_cache(0, len(pts))
        pos = np.full(len(X), -1)
        pos[perms[it]] = np.arange(len(perms[it]))
        for u, j in enumerate(pts[::7]):
            u = u * 7
            eff = np.where(pos < pos[j], lab, cur)
            eff[j] = -1
            drefs, pruned = [], []
            for c in range(5):
                want = np.sort(oracle.find_nearest_from_cluster(c, eff, D[j], 5))
                dref = oracle.convex_hull_distance(X[j], X[want]) if len(want) else np.inf
                drefs.append(dref)
                if cnt[u, c] == 0 and np.isinf(dist[u, c]) and len(want):
                    pruned.append(c)  # distance mode 2 rules bins out by bounds: no neighbour set, distance +inf
                    continue
                got = np.sort(idx[u, c, : cnt[u, c]])
                assert np.array_equal(want, got), (it, j, c)
                assert abs(dist[u, c] - dref) <= 1e-6 * dref + 1e-12
            assert path == "fused" or not pruned
            for c in pruned:
                assert drefs[c] > min(drefs), (it, j, c)  # a pruned bin is never the nearest hull, not even tied
        cur = ref
    ctx.close()


@pytest.mark.parametrize("share_guess", [False, True])
@pytest.mark.parametrize("cuts", [(0.5,), (0.1, 0.1, 0.73)])
def test_sharded_contexts_exchange_labels(cuts, share_guess):
    """The multi-GPU form on one device: several contexts, each owning a slice of the query slots (one of them may be
    empty), run the round protocol of include/chbin_b200.h and exchange tentative labels by element-wise MAX -- what the
    NCCL all-reduce does between ranks.  Labels must equal the sequential oracle after every iteration."""
    import torch

    X, bins, _ = synth.make_contig_features(3000, 7, 3, 15, seed=23, concentration=120.0)
    perms = oracle.draw_permutations(bins, 4, seed=0)
    U = perms.shape[1]
    edges = [0] + [int(U * f) for f in cuts] + [U]   # repeated edges give an empty shard
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    ctxs = []
    for u0, u1 in zip(edges[:-1], edges[1:]):
        ctx = capi.Context(0)
        ctx.set_stream(stream.cuda_stream)
        ctx.set_features(X); ctx.set_params(5, "convex"); ctx.set_distance_mode(2)
        ctx.set_labels(bins, 7, u0, u1); ctx.build_distance_matrix(True)
        ctxs.append(ctx)
    cur = bins.copy()
    with torch.cuda.stream(stream):
        if share_guess:
            # chb_guess_export / chb_guess_import: every context guesses for its own slots, the vectors are merged by MAX
            gs = [torch.empty(U, dtype=torch.int32, device=dev) for _ in ctxs]
            assert all(ctx.guess_export(g.data_ptr()) for ctx, g in zip(ctxs, gs))
            merged_g = torch.stack(gs).max(dim=0).values.contiguous()
            assert int(merged_g.min()) >= 0
            for ctx in ctxs:
                ctx.guess_import(merged_g.data_ptr())
        for it in range(4):
            for ctx in ctxs:
                ctx.iteration_begin(perms[it])
            lo = 0
            while lo < U:
                tents = [torch.empty(U - lo, dtype=torch.int32, device=dev) for _ in ctxs]
                for ctx, t in zip(ctxs, tents):
                    ctx.round_run(lo, U, t.data_ptr())
                merged = torch.stack(tents).max(dim=0).values.contiguous()
                assert int(merged.min()) >= 0, "a position was left un-owned after the exchange"
                firsts = [ctx.round_commit(lo, U, merged.data_ptr()) for ctx in ctxs]
                assert len(set(firsts)) == 1
                lo = U if firsts[0] < 0 else firsts[0] + 1
            changed = [ctx.iteration_end() for ctx in ctxs]
            assert len(set(changed)) == 1
            ref = oracle.fit_cluster(X, 7, cur, None, 5, 1, perms=perms[it:it + 1], threads=4)
            for ctx in ctxs:
                assert np.array_equal(ctx.get_labels(), ref), it
            cur = ref
    for ctx in ctxs:
        ctx.close()


def test_fresh_contexts_back_to_back():
    """Every call builds a NEW library context on recycled device memory: host-to-device set-up copies must be ordered on
    the context's own stream (a synchronous cudaMemcpy from pageable memory only waits for its staging copy)."""
    X, bins, _ = synth.make_contig_features(6000, 12, 10, 20, seed=5, concentration=500.0)
    perms = oracle.draw_permutations(bins, 4, seed=0)
    ref = oracle.fit_cluster(X, 12, bins, None, 10, 4, perms=perms, threads=4)
    for rep in range(4):
        np.random.seed(0)
        got, info = chbin_b200.fit_cluster(X, 12, bins, None, 10, 4, reuse_context=False, return_info=True)
        assert np.array_equal(got, ref), rep
        assert info["timers"]["launches_gram"] > 0


def test_fit_cluster_fortran_order_and_errors():
    X, bins, _ = synth.make_contig_features(400, 3, 1, 20, seed=1)
    perms = oracle.draw_permutations(bins, 10, seed=0)
    ref = oracle.fit_cluster(X, 3, bins, None, 5, 10, perms=perms)
    np.random.seed(0)
    got = chbin_b200.fit_cluster(np.asfortranarray(X), np.int64(3), bins, None, 5, 10)  # DataFrame.values is F-ordered
    assert np.array_equal(got, ref)
    with pytest.raises(NotImplementedError):
        chbin_b200.fit_cluster(X, 3, bins, None, 5, 10, metric="cosine")
    with pytest.raises(NotImplementedError):
        chbin_b200.fit_cluster(X, 3, bins, None, 5, 10, qp_solver="quadprog")
    with pytest.raises(ValueError):
        chbin_b200.fit_cluster(X, 3, bins, None, 64, 10)


def _same_as_oracle(X, C, bins, k, iters, **kw):
    perms = oracle.draw_permutations(bins, iters, seed=0)
    ref = oracle.fit_cluster(X, C, bins, None, k, iters, perms=perms, threads=2) if perms.shape[1] else bins.copy()
    np.random.seed(0)
    got, info = chbin_b200.fit_cluster(X, C, bins, None, k, iters, return_info=True, **kw)
    assert got.dtype == np.int64 and np.array_equal(got, ref)
    return info


def test_edge_nothing_to_assign():
    """Every contig already carries a label: zero query slots, zero QPs, labels returned unchanged (algorithm.py:38-66)."""
    X, bins, truth = synth.make_contig_features(300, 3, 1, 20, seed=2)
    info = _same_as_oracle(X, 3, truth.copy(), 5, 10)
    assert info["iterations"] == 1 and info["converged"]


def test_edge_single_bin_and_single_neighbour():
    X, bins, _ = synth.make_contig_features(500, 1, 2, 30, seed=3)
    _same_as_oracle(X, 1, bins, 5, 4)       # C = 1: nothing to choose, still one hull distance per query
    X, bins, _ = synth.make_contig_features(600, 4, 1, 10, seed=4)
    _same_as_oracle(X, 4, bins, 1, 4)       # k = 1: the hull is a point, the distance is the nearest member's


def test_edge_bins_without_seeds_and_tiny_bins():
    """Bins with no seed contig at all (num_clusters = max label + 1 leaves gaps), a bin with a single seed, and k larger
    than every bin at the start: find_nearest_from_cluster returns all members (distance_matrix.py:58-59)."""
    X, bins, truth = synth.make_contig_features(700, 5, 3, 6, seed=6, concentration=400.0)
    bins[bins == 2] = -1                     # bin 2 has no seeds: it can never win, and has no reference point
    keep = np.where(bins == 4)[0]
    bins[keep[1:]] = -1                      # bin 4 starts with one member
    _same_as_oracle(X, 5, bins, 9, 6)


def test_edge_wide_features_take_the_matrix_path():
    """d > 160 does not fit the resident operand of the fused kernel: the library falls back to distance mode 1 on its
    own (FP32 candidate matrix + scan), still exact."""
    rng = np.random.default_rng(8)
    X, bins, _ = synth.make_contig_features(500, 4, 40, 15, seed=8)     # d = 176
    assert X.shape[1] > 160
    info = _same_as_oracle(X, 4, bins, 5, 5)
    assert info["timers"]["launches_gram"] == 0 and info["timers"]["launches_knn"] > 0
    X2 = np.ascontiguousarray(rng.normal(size=(400, 7)))                # d = 7: tabulated MMA sequence, one operand box
    b2 = np.full(400, -1, dtype=np.int64)
    b2[:30] = np.arange(30) % 3
    _same_as_oracle(X2, 3, b2, 4, 5)


def test_edge_identical_contigs_everywhere():
    """Many exact duplicates (ties at every rank, zero distances, singular Gram matrices)."""
    X, bins, _ = synth.make_contig_features(600, 3, 1, 20, seed=9, concentration=200.0)
    X[100:300] = X[100]
    X[400:420] = X[0]
    _same_as_oracle(X, 3, bins, 5, 5)


def test_abi_argument_validation():
    """Error behaviour at the C-ABI (include/chbin_b200.h): bad arguments come back as CHB_EINVAL -> ValueError with a
    message, never as a crash or a silent wrong answer, and the context stays usable."""
    X, bins, _ = synth.make_contig_features(300, 3, 1, 20, seed=11)
    pts = np.where(bins == -1)[0]
    perm = np.random.default_rng(0).permutation(pts).astype(np.int64)
    ctx = capi.Context(0)
    with pytest.raises(ValueError, match="set_features first"):
        ctx.set_labels(bins, 3)
    ctx.set_features(X)
    with pytest.raises(ValueError, match="outside"):
        ctx.set_labels(np.where(bins == 2, 3, bins), 3)          # label == num_clusters
    with pytest.raises(ValueError, match="same n"):
        ctx.set_labels(bins[:-1], 3)
    with pytest.raises(ValueError, match="num_neighbors"):
        ctx.set_params(0, "convex")
    ctx.set_labels(bins, 3)
    ctx.set_params(5, "convex")
    with pytest.raises(ValueError, match="not set up"):
        ctx.iteration_begin(perm)                                 # distance structure not built yet
    ctx.build_distance_matrix(True)
    with pytest.raises(ValueError, match="permutation length"):
        ctx.iteration_begin(perm[:-1])
    # the entries themselves are validated on the device (distance mode 2): the error surfaces at the first commit that
    # follows, the iteration is abandoned and the labels stay as they were
    def refused(bad, pattern):
        ctx.iteration_begin(bad)
        ctx.round_run(0, len(bad))
        with pytest.raises(ValueError, match=pattern):
            ctx.round_commit(0, len(bad))
        assert np.array_equal(ctx.get_labels(), bins)

    bad = perm.copy(); bad[3] = bad[4]
    refused(bad, "repeats")
    bad = perm.copy(); bad[0] = int(np.where(bins >= 0)[0][0])    # a seed contig is not a query
    refused(bad, "not an un-assigned")
    bad = perm.copy(); bad[0] = len(X)
    refused(bad, "out of range")
    bad = perm.copy(); bad[5] = -7
    with pytest.raises(ValueError, match="out of range"):
        ctx.fit_iteration(bad)
    # distance mode 1 validates on the host, at once
    ctx.set_distance_mode(1); ctx.build_distance_matrix(True)
    bad = perm.copy(); bad[3] = bad[4]
    with pytest.raises(ValueError, match="repeats"):
        ctx.iteration_begin(bad)
    ctx.set_distance_mode(2); ctx.build_distance_matrix(True)
    # the context is still usable after the refused calls
    ref = oracle.fit_cluster(X, 3, bins, None, 5, 1, perms=perm[None, :])
    lab, _ = ctx.fit_iteration(perm)
    assert np.array_equal(lab, ref)
    ctx.close()


@pytest.mark.parametrize("max_iterations", [10, 1, 2])
def test_rng_contract_one_draw_per_executed_iteration(max_iterations):
    """fit_cluster overlaps the NEXT iteration's np.random.permutation with the running round and takes it back when the
    loop stops: afterwards the global legacy RNG must be exactly where the reference leaves it -- one draw per executed
    iteration (algorithm.py:45), whether the loop ends by convergence (:63-66) or by the iteration limit (:74-75)."""
    X, bins, _ = synth.make_contig_features(800, 4, 1, 20, seed=14, concentration=300.0)
    pts = np.where(bins == -1)[0]
    np.random.seed(123)
    got, info = chbin_b200.fit_cluster(X, 4, bins, None, 5, max_iterations, return_info=True)
    after = np.random.random()
    np.random.seed(123)
    perms = np.stack([np.random.permutation(pts) for _ in range(info["iterations"])])
    expect = np.random.random()
    assert after == expect
    ref = oracle.fit_cluster(X, 4, bins, None, 5, info["iterations"], perms=perms.astype(np.int64))
    assert np.array_equal(got, ref)


@pytest.mark.parametrize("k", [13, 14, 15, 16, 17, 20, 24, 25, 32])
def test_large_neighbour_counts(k):
    """BASELINE config #5 sweeps AlgoNumNeighbors up to 32.  The fused kernel keeps 2 x 16 candidates per (query, bin): the
    k + 1 keys the re-rank needs are among them unless one 64-column half holds 16 or more (detected: exact redo of the
    pair) -- the exception up to k = 24 (13..17: lists with little or no spare room; 20, 24: overflowing half-lists are
    common); for k >= 25 distance mode 2 prunes bins and then selects the neighbours of every surviving (query, bin) pair on
    exact distances (exact_group_kernel).  Either way the general QP kernel follows -- same labels as the oracle, in mode 1
    as well."""
    X, bins, _ = synth.make_contig_features(1400, 3, 2, 45, seed=16 + k, concentration=250.0)
    perms = oracle.draw_permutations(bins, 3, seed=0)
    ref = oracle.fit_cluster(X, 3, bins, None, k, 3, perms=perms, threads=4)
    np.random.seed(0)
    got, info = chbin_b200.fit_cluster(X, 3, bins, None, k, 3, return_info=True)
    assert np.array_equal(got, ref)
    assert (info["timers"]["launches_gram"] == 0) == (k > 24) and info["timers"]["launches_distance"] == 0
    np.random.seed(0)
    got1 = chbin_b200.fit_cluster(X, 3, bins, None, k, 3, distance_mode=1)
    assert np.array_equal(got1, ref)


@pytest.mark.parametrize("k,n,C,n_seed", [(16, 7000, 3, 20), (24, 9000, 4, 12), (26, 9000, 4, 12), (32, 5000, 2, 40)])
def test_large_neighbour_counts_big_bins(k, n, C, n_seed):
    """exact_group_kernel beyond one shared-memory pass (1024 members per bin and pass): bins of 2-3 thousand members, bins that
    start with fewer than k members (all-members rule, distance_matrix.py:58-59) and grow through k and through the pass
    size within one iteration, exact duplicates (ties resolved by index)."""
    X, bins, _ = synth.make_contig_features(n, C, 2, n_seed, seed=k, concentration=250.0)
    X[1000:1040] = X[2000:2040]
    X[3000:3003] = X[2000]
    perms = oracle.draw_permutations(bins, 3, seed=0)
    ref = oracle.fit_cluster(X, C, bins, None, k, 3, perms=perms, threads=4)
    np.random.seed(0)
    got, info = chbin_b200.fit_cluster(X, C, bins, None, k, 3, return_info=True)
    assert np.array_equal(got, ref)
    assert (info["timers"]["launches_gram"] == 0) == (k > 24)


def test_uncompacted_items_fallback(monkeypatch):
    """When the surviving (row, bin) pairs would not fit the compact operand buffer, the fused kernel works on (row block,
    bin) items instead (decided on the device).  CHB_FUSED_NO_COMPACT forces that path."""
    monkeypatch.setenv("CHB_FUSED_NO_COMPACT", "1")
    for (n, C, S, n_seed, k, conc) in [(1500, 8, 1, 30, 5, 60.0), (1200, 6, 10, 25, 10, 300.0), (5000, 20, 1, 20, 5, 1000.0)]:
        X, bins, _ = synth.make_contig_features(n, C, S, n_seed, seed=31, concentration=conc)
        perms = oracle.draw_permutations(bins, 4, seed=0)
        ref = oracle.fit_cluster(X, C, bins, None, k, 4, perms=perms, threads=4)
        np.random.seed(0)
        got, info = chbin_b200.fit_cluster(X, C, bins, None, k, 4, return_info=True, reuse_context=False)
        assert np.array_equal(got, ref), (n, C, k)
        assert info["timers"]["launches_gram"] > 0


@pytest.mark.parametrize("seed", [4, 5, 36, 52, 77, 131])
def test_soak_regressions(seed):
    """Cases found by the randomised soak (tests/soak_parity.py).  5: k = 16 with NO pair pruned -- the exact-selection list
    must hold every (row, bin) pair; 4, 36, 52: affine / affine-qp metrics with duplicate contigs among the neighbours
    (affinely dependent vertices: same affine hull without them); 77, 131: two more random draws kept as a canary."""
    from soak_parity import case

    cfg, X, bins = case(seed)
    perms = oracle.draw_permutations(bins, cfg["iters"], seed=0)
    ref = oracle.fit_cluster(X, cfg["C"], bins, None, cfg["k"], cfg["iters"], metric=cfg["metric"], perms=perms, threads=4)
    np.random.seed(0)
    got = chbin_b200.fit_cluster(X, cfg["C"], bins, None, cfg["k"], cfg["iters"], metric=cfg["metric"], distance_mode=cfg["mode"])
    assert np.array_equal(got, ref), cfg


@pytest.mark.parametrize("metric", ["affine-qp", "affine"])
@pytest.mark.parametrize("k", [3, 5])
def test_affine_metrics_never_prune_a_far_bin_whose_flat_passes_the_query(metric, k):
    """The ball bound behind the bin pruning (LB = |x - mu_c| - max|y - mu_c|) holds for CONVEX hulls only: the affine hull
    of k members is unbounded.  Bins 2 and 3 are far from every query (40 cluster radii) and tight, but their members lie
    along a line that runs through one query each: its distance to that affine hull is ~0 while its home bin is at a
    finite distance, so the reference assigns it to the far bin (hull_distance.py:38-87).  Labels must equal the
    oracle's; under the convex metric the same far bins are (rightly) out of reach."""
    X, bins, truth = synth.make_contig_features(900, 4, 1, 25, seed=41, concentration=2000.0)
    rng = np.random.default_rng(41)
    d = X.shape[1]
    targets = []
    for far_bin, home in ((2, 0), (3, 1)):
        tq = np.where((bins == -1) & (truth == home))[0][3]
        members = np.where(truth == far_bin)[0]
        u = rng.normal(size=d)
        u /= np.linalg.norm(u)
        home_pts = X[truth == home]
        spread = np.linalg.norm(home_pts - home_pts.mean(axis=0), axis=1).max()
        t = 40.0 * spread + 2.0 * spread * rng.random(len(members))
        X[members] = X[tq] + t[:, None] * u + 1e-5 * spread * rng.normal(size=(len(members), d))
        targets.append((tq, far_bin))
    perms = oracle.draw_permutations(bins, 3, seed=0)
    ref = oracle.fit_cluster(X, 4, bins, None, k, 3, metric=metric, perms=perms, threads=4)
    assert any(ref[t] == fb for t, fb in targets), "the construction must make a far bin win for its target query"
    for mode in (2, 1):
        np.random.seed(0)
        got = chbin_b200.fit_cluster(X, 4, bins, None, k, 3, metric=metric, distance_mode=mode)
        assert np.array_equal(got, ref), (metric, k, mode)
    refc = oracle.fit_cluster(X, 4, bins, None, k, 3, metric="convex", perms=perms, threads=4)
    np.random.seed(0)
    gotc = chbin_b200.fit_cluster(X, 4, bins, None, k, 3, metric="convex")
    assert np.array_equal(gotc, refc) and not any(refc[t] == fb for t, fb in targets)


def test_query_duplicated_in_two_bins_keeps_the_lower_bin():
    """A query with an exact duplicate among the members of TWO bins is at hull distance 0 from both.  The kernels return
    exactly 0.0 for both (qp_small.cu: a vertex coincides with the query) and the strict '<' of algorithm.py:57 keeps the
    LOWER bin.  (quadprog-style solvers return 0.0 and ~1e-16 of rounding noise and let the noise decide: the reference's
    own answer is not reproducible there, so the pinned behaviour is the deterministic one.)  Every OTHER position must
    still satisfy the sequential equation given these labels (oracle/verify.c)."""
    X, bins, truth = synth.make_contig_features(700, 5, 1, 30, seed=43, concentration=1500.0)
    q = np.where(bins == -1)[0][:6]
    pairs = [(1, 3), (0, 4), (2, 3), (3, 4), (0, 1), (1, 4)]
    for qi, (j, (lo, hi)) in enumerate(zip(q, pairs)):
        X[np.where(bins == lo)[0][qi]] = X[j]
        X[np.where(bins == hi)[0][8 + qi]] = X[j]
    perms = oracle.draw_permutations(bins, 1, seed=0)
    np.random.seed(0)
    got, info = chbin_b200.fit_cluster(X, 5, bins, None, 5, 1, return_info=True)
    for j, (lo, hi) in zip(q, pairs):
        assert got[j] == lo, (j, lo, hi, got[j])
    pos_of = np.full(len(X), -1)
    pos_of[perms[0]] = np.arange(perms.shape[1])
    others = np.setdiff1d(np.arange(perms.shape[1]), pos_of[q])
    res = oracle.verify_iteration(X, 5, bins, got, perms[0], 5, positions=others, threads=4)
    assert res["mismatches"] == 0
    with capi.Context(0) as ctx:
        ctx.set_features(X); ctx.set_labels(bins, 5); ctx.set_params(5, "convex")
        idx = np.full((len(q), 5, 5), -1, dtype=np.int64)
        m = np.zeros((len(q), 5), dtype=np.int32)
        for qi, j in enumerate(q):
            for c in range(5):
                mem = np.where(bins == c)[0]
                near = mem[np.argsort(np.linalg.norm(X[mem] - X[j], axis=1), kind="stable")[:5]]
                idx[qi, c] = near; m[qi, c] = 5
        dist, _ = ctx.hull_distance_batch(q, idx, m)
    assert np.sum(dist == 0.0) == 2 * len(q), "both duplicated bins are at distance exactly 0.0"


def test_candidate_lists_by_compact_pair_id_only(monkeypatch):
    """Beyond a memory budget (CHB_DENSE_LIST_GB; 1M contigs x 500 bins would need 61 GB) the candidate lists exist per
    COMPACT pair id only.  Forced here with a zero budget: binnable data runs compacted rounds and must give the same labels;
    overlapping bins leave more pairs than the compact buffers hold -- that round is refused with MemoryError instead of
    writing outside the lists, and the context is discarded."""
    monkeypatch.setenv("CHB_DENSE_LIST_GB", "0")
    for (n, C, S, n_seed, k, conc) in [(5000, 20, 1, 20, 5, 4000.0), (3000, 12, 10, 25, 10, 4000.0), (2500, 10, 1, 30, 16, 4000.0)]:
        X, bins, _ = synth.make_contig_features(n, C, S, n_seed, seed=33, concentration=conc)
        perms = oracle.draw_permutations(bins, 4, seed=0)
        ref = oracle.fit_cluster(X, C, bins, None, k, 4, perms=perms, threads=4)
        np.random.seed(0)
        got, info = chbin_b200.fit_cluster(X, C, bins, None, k, 4, return_info=True, reuse_context=False)
        assert np.array_equal(got, ref), (n, C, k)
        assert info["timers"]["launches_gram"] > 0
    X, bins, _ = synth.make_contig_features(1500, 8, 1, 30, seed=7, concentration=60.0)
    with pytest.raises(MemoryError, match="CHB_DENSE_LIST_GB"):
        chbin_b200.fit_cluster(X, 8, bins, None, 5, 10, reuse_context=False)


@pytest.mark.parametrize("k", [5, 20])
def test_exact_redo_list_overflow_grows_and_reruns_the_window(monkeypatch, k):
    """More (query, bin) pairs than the exact-redo list holds (forced: CHB_TEST_FB_CAP shrinks the list to 3 entries; many
    identical contigs make the re-rank send pairs there): nothing is committed, the library grows the list to its worst
    case and answers CHB_ROUND_AGAIN, the drivers run the window again -- same labels as with the regular list and as the
    oracle, no error."""
    X, bins, _ = synth.make_contig_features(1200, 5, 1, 20, seed=17, concentration=300.0)
    X[300:340] = X[300]
    X[700:712] = X[700]
    perms = oracle.draw_permutations(bins, 4, seed=0)
    ref = oracle.fit_cluster(X, 5, bins, None, k, 4, perms=perms, threads=4)
    np.random.seed(0)
    regular, rinfo = chbin_b200.fit_cluster(X, 5, bins, None, k, 4, return_info=True, reuse_context=False)
    monkeypatch.setenv("CHB_TEST_FB_CAP", "3")
    np.random.seed(0)
    got, info = chbin_b200.fit_cluster(X, 5, bins, None, k, 4, return_info=True, reuse_context=False)  # Python round loop
    assert np.array_equal(got, regular)
    assert info["iterations"] == rinfo["iterations"] and list(info["changed"]) == list(rinfo["changed"])
    assert np.array_equal(got, ref)
    assert info["timers"]["qp_iter_cap"] == 0
    with capi.Context(0) as ctx:  # chb_fit's own loop
        ctx.set_features(X); ctx.set_labels(bins, 5); ctx.set_params(k, "convex"); ctx.build_distance_matrix(True)
        lab, iters, conv, changed = ctx.fit(perms, 4)
        rounds = ctx.timers()["rounds"]
    assert np.array_equal(lab, regular)
    monkeypatch.delenv("CHB_TEST_FB_CAP")
    with capi.Context(0) as ctx:
        ctx.set_features(X); ctx.set_labels(bins, 5); ctx.set_params(k, "convex"); ctx.build_distance_matrix(True)
        ctx.fit(perms, 4)
        rounds_regular = ctx.timers()["rounds"]
    assert rounds > rounds_regular, "at least one window must have run twice"


def test_prefetched_permutation_is_used_only_when_it_is_the_one_begun():
    """chb_iteration_prefetch uploads the next permutation on the library's side stream while a round runs; the next
    chb_iteration_begin takes that copy only when it is handed the very same host array.  A different array, a prefetch that no
    iteration follows (new label set) and a prefetch in a matrix-backed distance mode (no-op) must all leave the result the
    sequential reference's (algorithm.py:43-72)."""
    X, bins, _ = synth.make_contig_features(3000, 6, 10, 20, seed=21, concentration=80.0)
    perms = oracle.draw_permutations(bins, 4, seed=3)
    U = perms.shape[1]
    ref, info = oracle.fit_cluster(X, 6, bins, None, 5, 4, perms=perms, return_info=True)
    other = np.ascontiguousarray(perms[::-1])  # a decoy: prefetched but never begun

    def iterate(ctx, prefetch):
        for it in range(info["iterations"]):
            ctx.iteration_begin(perms[it])
            lo = 0
            while lo < U:
                ctx.round_run(lo, U)
                if prefetch == "next" and it + 1 < len(perms):
                    ctx.iteration_prefetch(perms[it + 1])
                elif prefetch == "decoy":
                    ctx.iteration_prefetch(other[it])
                first, done, nch = ctx.round_commit_end(lo, U)
                if first == chbin_b200.clustering.ROUND_AGAIN:
                    continue
                lo = U if first < 0 else first + 1
            if not done:
                ctx.iteration_end()
        return ctx.get_labels()

    for mode in (2, 1):
        for prefetch in ("next", "decoy", "none"):
            with _ctx(X, bins, 6, 5, dist_mode=mode) as ctx:
                got = iterate(ctx, prefetch)
                assert np.array_equal(got, ref), (mode, prefetch)
                # a prefetch left pending by the loop above must not leak into the next label set
                ctx.iteration_prefetch(other[0])
                ctx.set_labels(bins, 6, 0, -1)
                ctx.build_distance_matrix(True)
                assert np.array_equal(iterate(ctx, "none"), ref), (mode, prefetch, "second label set")
