"""
The fused path (distance mode 2, csrc/fused.cu) at the shapes that switch its kernels, checked with tests/fused_invariants.py
(keys within their slack, complete kept lists, cached sets and hull distances, pruning, row bounds, guess) besides the labels.
Each case first asserts, from its shape, that it takes the branch it is here for.  The dispatch constants are read from
fused.cu itself (the line is cited beside each), so a change to one of them fails the case instead of silently testing
something else.

    case                 branch
    bin tiles            centroid_terms_kernel past its first CT_N = 64 bins; guess_from_terms_kernel, query_terms_gather_kernel
                         and row_ub_kernel's chunk scan past 32 bins
    seed counts          row_ub_kernel: seed tiles past RU_SEEDS = 32, bins above RU_MAXSEED = 128 (ubk2 = +inf), bins
                         without seeds and below k, at d = 137 (resident kernel) and d = 200 (streamed kernel)
    wide threshold       threshold_kernel<4> (U C >= 2^24) with C % 4 != 0; at C = 2 101 also pairs_plan_kernel's per-bin
                         counts in global memory (C > PLAN_SMEM_BINS = 2048)
    wide column gather   column_gather_wide_kernel (ncol_max >= 2^18)
"""
import os
import re
import time

import numpy as np
import pytest

import fused_invariants
import oracle
from chbin_b200 import capi, synth

pytestmark = pytest.mark.gpu

THREADS = os.cpu_count() or 1
FUSED_CU = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ch-bin_b200", "csrc", "fused.cu")


def _fused_const(pattern):
    with open(FUSED_CU) as f:
        m = re.search(pattern, f.read())
    assert m, f"fused.cu no longer has {pattern!r}: re-derive this case's shape"
    return int(m.group(1))


BN = _fused_const(r"BM = \d+, BN = (\d+),")                         # fused.cu:44, column tile
CT_N = _fused_const(r"CT_M = \d+, CT_N = (\d+),")                   # fused.cu:337, bins per centroid_terms_kernel tile
RU_SEEDS = _fused_const(r"RU_SEEDS = (\d+),")                       # fused.cu:582, seeds per row_ub_kernel tile
RU_MAXSEED = _fused_const(r"RU_MAXSEED = (\d+);")                   # fused.cu:582, above: only the nearest seed
THR_BINS = _fused_const(r"constexpr int THR_BINS = (\d+);")         # fused.cu:1535, bins per threshold_kernel<4> thread
PLAN_SMEM_BINS = _fused_const(r"PLAN_SMEM_BINS = (\d+);")           # fused.cu:965, pairs_plan_kernel shared-memory counts
THR_WIDE_LOG2 = _fused_const(r"nown \* \(int64_t\)C >= \(int64_t\)1 << (\d+);")  # fused.cu:2750, threshold_kernel<4>
GATHER_WIDE_LOG2 = _fused_const(r"if \(ncol_max >= \(int64_t\)1 << (\d+)\)")     # fused.cu:2728, column_gather_wide_kernel


def _ncol_max(n, C):
    return ((2 * n + BN * C + BN - 1) // BN) * BN  # fused.cu:2715


def _context(X, bins, C, k, materialise):
    ctx = capi.Context(0)
    ctx.set_features(X); ctx.set_params(k, "convex"); ctx.set_distance_mode(2); ctx.set_labels(bins, C)
    assert ctx.distance_path() == 2
    ctx.build_distance_matrix(materialise)
    return ctx


def _sample(U, count, seed):
    """first and last 256 slots / positions plus `count` more drawn (seeded) from the rest"""
    assert U > 512 + count
    rest = np.random.default_rng(seed).choice(np.arange(256, U - 256), count, replace=False)
    return np.sort(np.concatenate([np.arange(256), np.arange(U - 256, U), rest])).astype(np.int64)


def _report(name, tot, t0):
    print(f"\n{name}: worst err/slack {tot['worst']:.3g}, keys {tot['keys']}, pruned pairs {tot['pruned']}, "
          f"guess exemptions {tot['exempt']} of {tot['slots']} slots, {time.time() - t0:.1f} s")
    assert tot["worst"] < 0.5, "the key bound should hold with a wide margin"


def _full_check(name, X, bins, C, k, iters, every_seeded_bin_guessed=False):
    """Every slot checked after each iteration; labels equal to the sequential oracle's.  every_seeded_bin_guessed: assert
    that each bin with seeds is the guess of some row, so that row_ub_kernel runs over that bin's seeds."""
    t0 = time.time()
    perms = oracle.draw_permutations(bins, iters, seed=0)
    want = oracle.fit_cluster(X, C, bins, None, k, iters, perms=perms, threads=THREADS)
    ref = fused_invariants.Reference(X, bins, C, k)
    tot = dict(slots=0, worst=0.0, keys=0, pruned=0, exempt=0)
    cur = bins.copy()
    with _context(X, bins, C, k, True) as ctx:
        for it in range(iters):
            lab, _ = ctx.fit_iteration(perms[it])
            if every_seeded_bin_guessed and it == 0:
                guess, _, _ = ctx.get_row_bounds(0, len(ref.pts))
                rows = np.bincount(guess, minlength=C + 1)[:C]
                assert np.all(rows[ref.nseed > 0] > 0), dict(zip(ref.nseed.tolist(), rows.tolist()))
            got = fused_invariants.check_iteration(ctx, ref, perms[it], cur, lab, threads=THREADS)
            tot = {f: max(tot[f], got[f]) if f == "worst" else tot[f] + got[f] for f in tot}
            cur = lab
    assert np.array_equal(cur, want)
    _report(name, tot, t0)
    return tot


# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,k", [(33, 5), (64, 10), (65, 5), (130, 10)])
def test_bin_tiles(C, k):
    X, bins, _ = synth.make_contig_features(6000, C, 1, 20, seed=C + k, concentration=1500.0)
    U = int(np.sum(bins == -1))
    assert X.shape[1] == 137 and 137 % 16 != 0 and U % 128 != 0
    assert C > 32  # warp-wide bin loops: fused.cu:488 (lane loop), :2697 (gridDim.y = ceil(C / 32)), :611 (chunk scan)
    # fused.cu:337: one tile of CT_N bins half full and full, then a second one and a third one, both partial
    assert C in (CT_N // 2 + 1, CT_N, CT_N + 1, 2 * CT_N + 2)
    _full_check(f"bin tiles C={C} k={k}", X, bins, C, k, 2)


def _seed_count_case(d, k):
    counts = [0, 1, k - 1, k, RU_SEEDS - 1, RU_SEEDS, RU_SEEDS + 1, RU_MAXSEED, RU_MAXSEED + 1, 300]
    C = len(counts)
    X, bins, _ = synth.make_contig_features(6000, C, d - 136, 300, seed=d, concentration=600.0)
    for c, ns in enumerate(counts):
        bins[np.where(bins == c)[0][ns:]] = -1
    nseed = np.bincount(bins[bins >= 0], minlength=C)
    assert nseed.tolist() == counts
    # fused.cu:582: several seed tiles of RU_SEEDS, the last one at and one past RU_MAXSEED (ubk2 = +inf beyond)
    assert {RU_SEEDS - 1, RU_SEEDS, RU_SEEDS + 1, RU_MAXSEED, RU_MAXSEED + 1} <= set(counts) and max(counts) > 2 * RU_MAXSEED
    assert 0 in counts and 1 in counts and k - 1 in counts and k in counts
    return X, bins, C


@pytest.mark.parametrize("k", [5, 10])
def test_seed_counts_resident(k):
    X, bins, C = _seed_count_case(137, k)
    _full_check(f"seed counts d=137 k={k}", X, bins, C, k, 2, every_seeded_bin_guessed=True)


def test_seed_counts_streamed(monkeypatch):
    monkeypatch.setenv("CHB_WIDE_FUSED_MIN_PAIRS", "0")  # the streamed kernel at this size (test_gpu_wide_features.py)
    X, bins, C = _seed_count_case(200, 5)
    _full_check("seed counts d=200 k=5", X, bins, C, 5, 2, every_seeded_bin_guessed=True)


# ------------------------------------------------------------------------------------------------------------------
def _sampled_check(name, X, bins, C, k, n_check, n_verify):
    """One iteration: the checker on n_check sampled slots, the labels on n_verify sampled positions (position-parallel
    oracle), each plus the first and the last 256."""
    t0 = time.time()
    perm = oracle.draw_permutations(bins, 1, seed=0)[0]
    U = len(perm)
    ref = fused_invariants.Reference(X, bins, C, k)
    with _context(X, bins, C, k, False) as ctx:
        lab, _ = ctx.fit_iteration(perm)
        tot = fused_invariants.check_iteration(ctx, ref, perm, bins, lab, slots=_sample(U, n_check, 1), threads=THREADS)
    res = oracle.verify_iteration(X, C, bins, lab, perm, k, positions=_sample(U, n_verify, 2), threads=THREADS)
    assert res["mismatches"] == 0, res["mismatches"]
    _report(name, tot, t0)
    return tot


@pytest.mark.parametrize("n,C,n_seed", [(46_003, 411, 10), (16_000, 2101, 3)])
def test_wide_threshold_kernel_with_a_bin_tail(n, C, n_seed):
    X, bins, _ = synth.make_contig_features(n, C, 1, n_seed, seed=C)  # realistic, well separated bins: much pruning
    U = int(np.sum(bins == -1))
    assert U * C >= 2**THR_WIDE_LOG2  # fused.cu:2750: threshold_kernel<4>
    assert C % THR_BINS != 0 and U % 4 != 0  # the cc < C / c >= C tail (fused.cu:1564, :1570) and a partial float4 of rows
    if C > 2048:
        assert C > PLAN_SMEM_BINS  # fused.cu:965, :970: pairs_plan_kernel's per-bin counts in global scratch
        assert n_seed < 5  # every bin below k seeds: ubk2 = +inf everywhere
    _sampled_check(f"wide threshold C={C}", X, bins, C, 5, 1000 - 512, 2000)


@pytest.mark.parametrize("d", [137, 200])
def test_wide_column_gather(d):
    n, C, k = 135_000, 60, 5
    X, bins, _ = synth.make_contig_features(n, C, d - 136, 50, seed=d, concentration=1500.0)
    assert _ncol_max(n, C) >= 2**GATHER_WIDE_LOG2  # fused.cu:2728: column_gather_wide_kernel
    _sampled_check(f"wide column gather d={d}", X, bins, C, k, 1000, 2000)
