"""
The fused-path checker (fused_invariants.py) on the CPU: a state built from the oracle (what a correct distance-mode-2
iteration leaves behind) passes, and each error the checker exists to catch -- applied one at a time -- makes it fail.
"""
import numpy as np
import pytest

import oracle
from chbin_b200 import synth
from fused_invariants import Reference, SliceState, check_slots, nearest_sets

C, K, KR = 6, 5, 8
SEEDS = [129, 3, 10, 10, 10, 0]  # a bin above RU_MAXSEED, one below k, one without any seed


@pytest.fixture(scope="module")
def case():
    X, bins, truth = synth.make_contig_features(1500, C, 1, 140, seed=3, concentration=400.0)
    for c, ns in enumerate(SEEDS):
        members = np.where(bins == c)[0]
        bins[members[ns:]] = -1
    perm = oracle.draw_permutations(bins, 1, seed=0)[0]
    new = oracle.fit_cluster(X, C, bins, None, K, 1, perms=perm[None, :], threads=4)
    ref = Reference(X, bins, C, K)
    slots = np.arange(0, len(ref.pts), 9)
    return ref, perm, bins.copy(), new, slots


def _true_state(ref, perm, old, new, slots):
    """What a correct iteration leaves: kept lists = the k true neighbours plus the next few members of the bin, keys = the
    exact squared distances in FP32, slack = 1e-4 of the row's largest one; pairs whose hull distance is 10 % above the row's
    minimum pruned; tight bounds; the FP64 nearest-centroid guess."""
    X = ref.X
    js = ref.pts[slots]
    S = len(slots)
    pos = np.full(len(X), -1)
    pos[perm] = np.arange(len(perm))
    D = oracle.distance_rows(X, js)
    eff = np.where(pos[None, :] < pos[js][:, None], new[None, :], old[None, :])
    eff[np.arange(S), js] = -1
    wide = nearest_sets(eff, D, C, 2 * KR - 3)
    hd = oracle.verify_iteration(X, C, old, new, perm, K, positions=pos[js], return_distances=True)["distances"]
    pruned = hd > 1.1 * hd.min(axis=1)[:, None]
    idx = np.full((S, C, 2 * KR), -1, dtype=np.int32)
    idx[:, :, : 2 * KR - 3] = wide
    key = np.where(idx >= 0, np.take_along_axis(D, np.maximum(idx, 0).reshape(S, -1), axis=1).reshape(idx.shape) ** 2, np.inf)
    key = key.astype(np.float32)
    slack = np.broadcast_to(1e-4 * (D.max(axis=1) ** 2)[:, None], (S, C)).astype(np.float32).copy()
    pidx = wide[:, :, :K].astype(np.int32)
    pcnt = (pidx >= 0).sum(axis=2).astype(np.int32)
    pdist = hd.copy()
    key[pruned] = np.inf
    idx[pruned] = -1
    pcnt[pruned] = 0
    pdist[pruned] = np.inf
    a = ref.centred(js)
    t = np.sum((a[:, None, :] - ref.mc[None, :, :]) ** 2, axis=2)
    t[:, ref.nseed == 0] = np.inf
    guess = np.argmin(t, axis=1).astype(np.int32)
    ub = np.empty(S, dtype=np.float32)
    ubk2 = np.full(S, np.inf, dtype=np.float32)
    for s in range(S):
        ub[s], ubk2[s] = _bounds(ref, js[s], guess[s])
    return SliceState(np.asarray(slots), key, idx, slack, pidx, pcnt, pdist, guess, ub, ubk2), D, hd, t


def _bounds(ref, j, g):
    """tight (ub, ubk2) of point j against the seeds of bin g, as row_ub_kernel leaves them"""
    dist = np.sort(np.sqrt(np.sum((ref.X[ref.seeds[g]] - ref.X[j]) ** 2, axis=1)))
    kth2 = np.float32((dist[K - 1] * (1 + 1e-5)) ** 2) if K <= len(dist) <= 128 else np.inf
    return np.float32(dist[0] * (1 + 1e-5)), kth2


def test_nearest_sets_match_find_nearest_from_cluster(case):
    ref, perm, old, new, slots = case
    js = ref.pts[slots[:20]]
    D = oracle.distance_rows(ref.X, js)
    eff = np.tile(new, (len(js), 1))
    eff[np.arange(len(js)), js] = -1
    eff[:, ::7] = old[::7]
    X2 = D.copy()
    X2[:, 100:140] = X2[:, 100:101]  # ties: broken by index
    got = nearest_sets(eff, X2, C, K)
    for s in range(len(js)):
        for c in range(C):
            want = oracle.find_nearest_from_cluster(c, eff[s], X2[s], K)
            assert got[s, c, : len(want)].tolist() == want.tolist() and np.all(got[s, c, len(want):] == -1)


def test_correct_state_passes(case):
    ref, perm, old, new, slots = case
    st, _, _, _ = _true_state(ref, perm, old, new, slots)
    assert np.any(st.guess == 0) and st.pcnt.min() == 0, "the case must hold a 129-seed guess and pruned pairs"
    stats = check_slots(ref, st, perm, old, new)
    assert stats["keys"] > 0 and stats["pruned"] > 0 and stats["exempt"] == 0
    assert 0.0 < stats["worst"] < 0.01


def _live(st):
    return np.argwhere(np.isfinite(st.pdist) & (st.pcnt > 0))


def _key_off(st, D, hd, t, ref):
    s, c = _live(st)[0]
    st.key[s, c, 0] = np.float32(D[s, st.idx[s, c, 0]] ** 2 + 2.0 * st.slack[s, c])


def _neighbour_dropped(st, D, hd, t, ref):
    s, c = _live(st)[0]
    e = np.where(st.idx[s, c] == st.pidx[s, c, 0])[0][0]
    st.key[s, c, e] = np.inf
    st.idx[s, c, e] = -1


def _winner_pruned(st, D, hd, t, ref):
    s = 0
    c = int(np.argmin(hd[s]))
    st.key[s, c] = np.inf
    st.idx[s, c] = -1
    st.pcnt[s, c] = 0
    st.pdist[s, c] = np.inf


def _ub_low(st, D, hd, t, ref):
    st.ub[3] *= np.float32(0.99)


def _ubk2_finite_above_maxseed(st, D, hd, t, ref):
    s = int(np.where(st.guess == 0)[0][0])
    js = ref.pts[st.slots[s]]
    dist = np.sort(np.sum((ref.X[ref.seeds[0]] - ref.X[js]) ** 2, axis=1))
    st.ubk2[s] = np.float32(dist[K - 1] * 1.01)


def _guess_second(st, D, hd, t, ref):
    srt = np.sort(t, axis=1)
    margin = (srt[:, 1] - srt[:, 0]) / srt[:, 0]
    s = int(np.argmax(margin))
    assert margin[s] > 1e-3
    g = int(np.argsort(t[s])[1])
    st.guess[s] = g
    st.ub[s], st.ubk2[s] = _bounds(ref, ref.pts[st.slots[s]], g)  # a wrong guess comes with bounds for that bin


def _slack_nan(st, D, hd, t, ref):
    s, c = _live(st)[0]
    st.slack[s, c] = np.nan


def _pair_distance_off(st, D, hd, t, ref):
    s, c = _live(st)[0]
    st.pdist[s, c] *= 1 + 1e-5


@pytest.mark.parametrize("mutate,caught_by", [
    (_key_off, "key outside its slack"),
    (_slack_nan, "key outside its slack"),
    (_neighbour_dropped, "missing from its kept list"),
    (_winner_pruned, "is the row minimum"),
    (_ub_low, "ub below the nearest seed"),
    (_ubk2_finite_above_maxseed, "ubk2 finite"),
    (_guess_second, "guess is not the nearest seed centroid"),
    (_pair_distance_off, "hull distance of point"),
])
def test_each_error_is_caught(case, mutate, caught_by):
    ref, perm, old, new, slots = case
    st, D, hd, t = _true_state(ref, perm, old, new, slots)
    mutate(st, D, hd, t, ref)
    with pytest.raises(AssertionError, match=caught_by):
        check_slots(ref, st, perm, old, new)
