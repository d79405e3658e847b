"""
TEST INFRASTRUCTURE: the facts the default distance path (distance mode 2, csrc/fused.cu) relies on, checked for a set of
query slots of an open context after chb_fit_iteration against FP64 references:

  keys       every kept FP32 key of a (slot, bin) pair the bounds did not rule out lies within the pair's slack of the exact
             squared distance (oracle.distance_rows, the cdist recipe);
  lists      the kept lists hold every true neighbour: find_nearest_from_cluster on the labels as this query saw them (new
             labels for earlier positions, old ones for later positions, the query itself excluded);
  pair cache the cached neighbour set of a surviving pair is exactly the oracle's and its hull distance is within
             1e-6 ref + 1e-12 |x| of the oracle's (oracle.verify_iteration); a pruned pair (no neighbours, distance +inf)
             has an oracle hull distance strictly above the row's minimum;
  row bounds ub / ubk2 bound the exact distances to the seeds of the guessed bin (nearest / k-th nearest squared), ub is
             tight, ubk2 is +inf exactly when that bin has fewer than k or more than RU_MAXSEED seeds;
  guess      the speculation start is the nearest seed centroid, recomputed in FP64 (tolerance derived in _guess_tolerance).

check_iteration() fetches the device tables in slot slices (a single fetch of every slot is gigabytes at C = 2 101) and
checks each slice with check_slots(), which takes plain arrays so that the checker itself can be tested without a GPU.
"""
from dataclasses import dataclass

import numpy as np

import oracle

SLICE = 256
RU_MAXSEED = 128  # row_ub_kernel: only the minimum is kept for a bin with more seeds (ubk2 = +inf), csrc/fused.cu


@dataclass
class SliceState:
    """Device tables of the query slots `slots`, as the test aids of the C-ABI return them."""
    slots: np.ndarray  # (S,) slot indices
    key: np.ndarray    # (S, C, 2 KR) float32, +inf = empty
    idx: np.ndarray    # (S, C, 2 KR) int32
    slack: np.ndarray  # (S, C) float32
    pidx: np.ndarray   # (S, C, k) cached neighbour sets
    pcnt: np.ndarray   # (S, C)
    pdist: np.ndarray  # (S, C) cached hull distances
    guess: np.ndarray  # (S,) guessed bin (C = none)
    ub: np.ndarray     # (S,) float32
    ubk2: np.ndarray   # (S,) float32


class Reference:
    """What does not change between slices: the features, the seeds, the FP64 bin reference points."""

    def __init__(self, X, bins, C, k):
        self.X = np.ascontiguousarray(X, dtype=np.float64)
        self.bins = np.asarray(bins, dtype=np.int64)
        self.C, self.k = int(C), int(k)
        self.pts = np.where(self.bins == -1)[0]
        self.nseed = np.bincount(self.bins[self.bins >= 0], minlength=self.C)[: self.C]
        self.seeds = [np.where(self.bins == c)[0] for c in range(self.C)]
        # centring as the kernels do it: a = fl32(x - mu), m_c = (mean of the bin's seeds) - mu, zero without seeds
        self.mu = self.X.mean(axis=0)
        self.mc = np.zeros((self.C, self.X.shape[1]))
        for c in np.where(self.nseed > 0)[0]:
            self.mc[c] = self.X[self.seeds[c]].mean(axis=0) - self.mu
        self.mc2 = np.sum(self.mc * self.mc, axis=1)

    def centred(self, rows):
        return (self.X[rows] - self.mu).astype(np.float32).astype(np.float64)


def _guess_tolerance(t_g, t_b, anorm, mdiff):
    """How far above the FP64 minimum t_b the term t_g of the bin the kernels guessed may lie.  The kernels compute
    t_c = |a - m_c|^2 in FP64 from their own a' = fl32(x - mu') and round it to FP32 (centroid_terms_kernel), then take the
    lowest bin of minimum FP32 value (guess_from_terms_kernel).  So they can prefer g over b when
        t_g - t_b <= 2^-24 (t_g + t_b)                 (one FP32 rounding of each term)
                   + 2 |a' - a| |m_g - m_b|              (t_g - t_b = |m_g|^2 - |m_b|^2 - 2 a.(m_g - m_b) moves by 2 (a' - a).(m_b - m_g))
    with |a' - a| <= 2^-23 |a|: mu' is summed in another order than here, which can move fl32(x - mu) by one ulp per
    coordinate.  The FP64 evaluation adds ~d 2^-53 (|a|^2 + |m|^2), covered by the last term."""
    return 2.0**-24 * (t_g + t_b) * 1.001 + 2.0**-22 * anorm * mdiff + 1e-12 * (anorm * anorm + t_g + t_b)


def nearest_sets(eff, drows, C, k):
    """find_nearest_from_cluster(c, eff[s], drows[s], k) for every slot s and bin c at once: (S, C, k), -1 padded.  The
    canonical (distance, index) order of the oracle: a stable sort by distance, then a stable one by label."""
    S, n = drows.shape
    out = np.full((S, C, k), -1, dtype=np.int64)
    ar = np.arange(k)
    for s in range(S):
        o1 = np.argsort(drows[s], kind="stable")
        lab = eff[s][o1]
        o2 = np.argsort(lab, kind="stable")
        order, lab = o1[o2], lab[o2]
        beg = np.searchsorted(lab, np.arange(C), side="left")
        end = np.searchsorted(lab, np.arange(C), side="right")
        take = ar[None, :] < np.minimum(end - beg, k)[:, None]
        pos = np.minimum(beg[:, None] + ar[None, :], n - 1)
        out[s] = np.where(take, order[pos], -1)
    return out


def check_slots(ref, st, perm, old, new, threads=0):
    """Every invariant of the module docstring for the slots of one slice; returns the slice's statistics."""
    X, C, k = ref.X, ref.C, ref.k
    S = len(st.slots)
    js = ref.pts[st.slots]
    pos = np.full(len(X), -1, dtype=np.int64)
    pos[perm] = np.arange(len(perm))
    stats = dict(slots=S, worst=0.0, keys=0, pruned=0, exempt=0)

    # ---- keys: |key - D^2| <= slack on every pair the bounds kept
    D = oracle.distance_rows(X, js)
    pruned = (st.pcnt == 0) & np.isinf(st.pdist)
    fin = np.isfinite(st.key) & ~pruned[:, :, None]
    assert np.all(st.idx[fin] >= 0), "a finite key without a point"
    d2 = np.take_along_axis(D[:, None, :], np.where(fin, st.idx, 0).reshape(S, 1, -1), axis=2).reshape(st.key.shape) ** 2
    err = np.where(fin, np.abs(st.key.astype(np.float64) - d2), 0.0)
    # the slack of a pruned pair is never written: whatever bits it holds are not looked at
    sl = np.broadcast_to(np.where(pruned, np.float32(1), st.slack).astype(np.float64)[:, :, None], err.shape)
    bad = fin & ~(err <= sl)  # a NaN key or slack fails as well
    if bad.any():
        s, c, e = np.argwhere(bad)[0]
        raise AssertionError(f"key outside its slack: slot {st.slots[s]} point {js[s]} bin {c}: key {st.key[s, c, e]} "
                             f"exact {d2[s, c, e]} err {err[s, c, e]:.3e} slack {sl[s, c, e]:.3e}")
    if fin.any():
        stats["worst"] = float(np.max(err[fin] / sl[fin]))
        stats["keys"] = int(fin.sum())
        assert np.isfinite(stats["worst"]), ("key outside its slack: err / slack is not finite", stats["worst"])

    # ---- lists and pair cache against the labels as each query saw them
    eff = np.where(pos[None, :] < pos[js][:, None], new[None, :], old[None, :])
    eff[np.arange(S), js] = -1
    want = nearest_sets(eff, D, C, k)
    wcnt = (want >= 0).sum(axis=2)
    kept = np.where(np.isfinite(st.key), st.idx, -2)
    missing = (want >= 0) & ~(want[:, :, :, None] == kept[:, :, None, :]).any(axis=3)
    missing &= ~pruned[:, :, None]
    if missing.any():
        s, c, e = np.argwhere(missing)[0]
        raise AssertionError(f"true neighbour {want[s, c, e]} of point {js[s]} (slot {st.slots[s]}) in bin {c} missing from "
                             f"its kept list")
    big = np.iinfo(np.int64).max
    got = np.sort(np.where(np.arange(k)[None, None, :] < st.pcnt[:, :, None], st.pidx.astype(np.int64), big), axis=2)
    exp = np.sort(np.where(want >= 0, want, big), axis=2)
    wrong = ~pruned & ((st.pcnt != wcnt) | (got != exp).any(axis=2))
    if wrong.any():
        s, c = np.argwhere(wrong)[0]
        raise AssertionError(f"cached neighbour set of point {js[s]} bin {c}: {got[s, c, : st.pcnt[s, c]]} != oracle "
                             f"{exp[s, c, : wcnt[s, c]]}")
    res = oracle.verify_iteration(X, C, old, new, perm, k, positions=pos[js], threads=threads, return_distances=True)
    hd = res["distances"]
    tol = 1e-6 * hd + 1e-12 * np.linalg.norm(X[js], axis=1)[:, None]
    live = ~pruned & np.isfinite(hd)
    off = live & ~(np.abs(np.subtract(st.pdist, hd, out=np.zeros_like(hd), where=live)) <= tol)
    off |= ~pruned & ~np.isfinite(hd) & np.isfinite(st.pdist)
    if off.any():
        s, c = np.argwhere(off)[0]
        raise AssertionError(f"hull distance of point {js[s]} bin {c}: {st.pdist[s, c]!r} != oracle {hd[s, c]!r}")
    rowmin = hd.min(axis=1)
    lost = pruned & ~(hd > rowmin[:, None])
    if lost.any():
        s, c = np.argwhere(lost)[0]
        raise AssertionError(f"bin {c} pruned for point {js[s]} but its hull distance {hd[s, c]!r} is the row minimum")
    stats["pruned"] = int((pruned & np.isfinite(hd)).sum())

    # ---- row bounds against the exact distances to the guessed bin's seeds
    for s in range(S):
        g = int(st.guess[s])
        if g == C:
            assert np.isinf(st.ub[s]) and np.isinf(st.ubk2[s]), (js[s], "no guessed bin: no bound")
            continue
        dist = np.sqrt(np.sum((X[ref.seeds[g]] - X[js[s]]) ** 2, axis=1))
        dmin = dist.min()
        assert float(st.ub[s]) >= dmin, ("ub below the nearest seed", js[s], g, float(st.ub[s]), dmin)
        assert float(st.ub[s]) <= dmin * (1 + 1e-3) + 1e-3, ("ub not tight", js[s], g, float(st.ub[s]), dmin)
        ns = len(dist)
        if ns < k or ns > RU_MAXSEED:
            assert np.isinf(st.ubk2[s]), ("ubk2 finite", js[s], g, ns, float(st.ubk2[s]))
        else:
            kth = np.sort(dist)[k - 1]
            assert float(st.ubk2[s]) >= kth * kth, ("ubk2 below the k-th seed", js[s], g, float(st.ubk2[s]), kth * kth)
            assert np.sqrt(float(st.ubk2[s])) <= kth * (1 + 1e-3) + 1e-3, ("ubk2 not tight", js[s], g, float(st.ubk2[s]), kth)

    # ---- guess: nearest seed centroid in FP64
    has = ref.nseed > 0
    if not has.any():
        assert np.all(st.guess == C), "a guess without any seeded bin"
    else:
        a = ref.centred(js)
        t = np.sum(a * a, axis=1)[:, None] - 2.0 * (a @ ref.mc.T) + ref.mc2[None, :]
        t = np.where(has[None, :], np.maximum(t, 0.0), np.inf)
        b = np.argmin(t, axis=1)  # lowest bin of minimum value
        for s in np.where(st.guess != b)[0]:
            g = int(st.guess[s])
            assert 0 <= g < C and has[g], ("guess is not a seeded bin", js[s], g)
            tg, tb = t[s, g], t[s, b[s]]
            lim = _guess_tolerance(tg, tb, np.linalg.norm(a[s]), np.linalg.norm(ref.mc[g] - ref.mc[b[s]]))
            assert tg - tb <= lim, ("guess is not the nearest seed centroid", js[s], g, int(b[s]), tg, tb, lim)
            stats["exempt"] += 1
    return stats


def fetch(ctx, slot0, nslots):
    key, idx, slack = ctx.get_fused_candidates(slot0, nslots)
    pidx, pcnt, pdist = ctx.get_pair_cache(slot0, nslots)
    guess, ub, ubk2 = ctx.get_row_bounds(slot0, nslots)
    return SliceState(np.arange(slot0, slot0 + nslots), key, idx, slack, pidx, pcnt, pdist, guess, ub, ubk2)


def _concat(states):
    return SliceState(*(np.concatenate([getattr(st, f) for st in states]) for f in SliceState.__dataclass_fields__))


def _runs(slots, width):
    """maximal runs of consecutive slots, cut every `width`"""
    slots = np.unique(np.asarray(slots, dtype=np.int64))
    if len(slots) == 0:
        return
    cuts = np.where(np.diff(slots) != 1)[0] + 1
    for run in np.split(slots, cuts):
        for i in range(0, len(run), width):
            yield int(run[i]), int(min(width, len(run) - i))


def check_iteration(ctx, ref, perm, old, new, slots=None, threads=0):
    """check_slots() over `slots` (all owned slots if None) of an open mode-2 context right after chb_fit_iteration with
    `perm`, `old` = the labels before it, `new` = after.  Returns the totals: worst err / slack, keys checked, pruned pairs
    checked, guess exemptions."""
    if slots is None:
        slots = np.arange(len(ref.pts))
    old = np.asarray(old, dtype=np.int64)
    new = np.asarray(new, dtype=np.int64)
    tot = dict(slots=0, worst=0.0, keys=0, pruned=0, exempt=0)

    def check(states):
        st = check_slots(ref, _concat(states), perm, old, new, threads=threads)
        tot["worst"] = max(tot["worst"], st["worst"])
        for f in ("slots", "keys", "pruned", "exempt"):
            tot[f] += st[f]

    # runs are fetched one by one (sampled slots are mostly runs of one) and checked SLICE slots at a time, so that the
    # position-parallel oracle gets enough positions to spread over its threads
    pending, npend = [], 0
    for s0, m in _runs(slots, SLICE):
        pending.append(fetch(ctx, s0, m))
        npend += m
        if npend >= SLICE:
            check(pending)
            pending, npend = [], 0
    if pending:
        check(pending)
    assert tot["keys"] > 0, "no key was checked"
    # exemptions need a near tie of two centroid distances at the level of FP32 rounding
    assert tot["exempt"] <= 1 + tot["slots"] // 1000, f"{tot['exempt']} of {tot['slots']} guesses are not the nearest centroid"
    return tot
