"""
ctypes binding of libchbin_b200.so (include/chbin_b200.h).  No torch, no numpy types cross the ABI: only raw
pointers and sizes.  The library is hand-written sm_100a CUDA; there is NO CPU fallback -- `load()` raises if the
shared object is missing and `Context()` raises if no B200-class device is usable.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import numpy as np

from . import build as _build

CHB_OK, CHB_EINVAL, CHB_ENODEV, CHB_ECUDA, CHB_ENOMEM, CHB_ENOTIMPL, CHB_EUNASSIGNED = range(7)
METRICS = {"convex": 0, "affine-qp": 1, "affine": 2}
UNOWNED = -(2**31)
OWN_STREAM = 2**64 - 1  # CHB_OWN_STREAM: (void*)-1

EXPORTED_SYMBOLS = [
    "chb_abi_version", "chb_create", "chb_destroy", "chb_last_error", "chb_set_stream", "chb_synchronize",
    "chb_get_timers", "chb_reset_timers", "chb_enable_timers", "chb_set_features", "chb_set_features_dev", "chb_set_features_dev_async", "chb_features_buffer", "chb_features_commit",
    "chb_set_labels", "chb_set_params", "chb_build_distance_matrix", "chb_get_distance_rows", "chb_knn_per_bin",
    "chb_hull_distance_batch", "chb_fit_iteration", "chb_fit", "chb_get_labels", "chb_iteration_begin", "chb_iteration_begin_dev", "chb_iteration_prefetch",
    "chb_round_run", "chb_round_commit", "chb_round_commit_end", "chb_iteration_end", "chb_set_window", "chb_get_window",
    "chb_measure_fp64_tflops", "chb_measure_l2_gbs", "chb_guess_export", "chb_guess_import", "chb_set_distance_mode", "chb_get_distance_path", "chb_set_gram_engine", "chb_get_candidate_rows", "chb_get_pair_cache",
    "chb_get_fused_candidates", "chb_get_row_bounds", "chb_set_features_async", "chb_set_features_colmajor", "chb_set_features_merged", "chb_get_features",
    "chb_group_create", "chb_group_destroy", "chb_group_buffer", "chb_group_all_max", "chb_group_replicate_features",
]


class Timers(ctypes.Structure):
    _fields_ = [
        ("ms_distance", ctypes.c_double), ("ms_knn", ctypes.c_double), ("ms_qp", ctypes.c_double),
        ("ms_commit", ctypes.c_double),
        ("launches_distance", ctypes.c_int64), ("launches_knn", ctypes.c_int64), ("launches_qp", ctypes.c_int64),
        ("launches_commit", ctypes.c_int64), ("launches_other", ctypes.c_int64),
        ("qps_solved", ctypes.c_int64), ("qps_reference", ctypes.c_int64), ("rounds", ctypes.c_int64),
        ("rows_scanned", ctypes.c_int64),
        ("ms_gram", ctypes.c_double), ("launches_gram", ctypes.c_int64), ("gram_tiles", ctypes.c_int64),
        ("gram_tiles_planned", ctypes.c_int64), ("qp_iter_cap", ctypes.c_int64),
    ]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


_lib: Optional[ctypes.CDLL] = None
_vp, _i64, _i32, _dbl = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_double


def library_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True) -> ctypes.CDLL:
    """dlopen libchbin_b200.so (building it with nvcc first if the in-tree .so is missing or stale)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if build_if_missing and (not os.path.exists(path) or (_build.is_stale() and _nvcc_available())):
        _build.build_library()
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} not found: the CUDA extension of chbin_b200 is not built and there is no CPU fallback. "
            "Run `python -c 'import __graft_entry__ as g; g.build()'`."
        )
    L = ctypes.CDLL(path)
    L.chb_abi_version.restype = ctypes.c_int
    L.chb_last_error.restype = ctypes.c_char_p
    L.chb_last_error.argtypes = [_vp]
    L.chb_create.argtypes = [ctypes.POINTER(_vp), ctypes.c_int]
    L.chb_destroy.argtypes = [_vp]
    L.chb_set_stream.argtypes = [_vp, _vp]
    L.chb_synchronize.argtypes = [_vp]
    L.chb_get_timers.argtypes = [_vp, ctypes.POINTER(Timers)]
    L.chb_reset_timers.argtypes = [_vp]
    L.chb_enable_timers.argtypes = [_vp, ctypes.c_int]
    L.chb_set_features.argtypes = [_vp, _vp, _i64, _i32]
    L.chb_set_features_dev.argtypes = [_vp, _vp, _i64, _i32]
    L.chb_set_features_dev_async.argtypes = [_vp, _vp, _i64, _i32]
    L.chb_features_buffer.argtypes = [_vp, _i64, _i32, ctypes.POINTER(_vp), ctypes.POINTER(_i64)]
    L.chb_features_commit.argtypes = [_vp, ctypes.c_int]
    L.chb_set_features_async.argtypes = [_vp, _vp, _i64, _i32]
    L.chb_set_features_colmajor.argtypes = [_vp, _vp, _i64, _i32, ctypes.c_int]
    L.chb_set_features_merged.argtypes = [_vp, _vp, _i64, _i32, _vp, _i64, _i32, _vp, _vp]
    L.chb_get_features.argtypes = [_vp, _vp]
    L.chb_set_labels.argtypes = [_vp, _vp, _i64, _i32, _i64, _i64]
    L.chb_set_params.argtypes = [_vp, _i32, _i32]
    L.chb_build_distance_matrix.argtypes = [_vp, ctypes.c_int]
    L.chb_set_distance_mode.argtypes = [_vp, ctypes.c_int]
    L.chb_set_gram_engine.argtypes = [_vp, ctypes.c_int]
    L.chb_get_pair_cache.argtypes = [_vp, _i64, _i64, _vp, _vp, _vp]
    L.chb_get_fused_candidates.argtypes = [_vp, _i64, _i64, _vp, _vp, _vp, ctypes.POINTER(_i32)]
    L.chb_get_candidate_rows.argtypes = [_vp, _i64, _i64, _vp, ctypes.POINTER(_dbl), _vp]
    L.chb_get_distance_rows.argtypes = [_vp, _i64, _i64, _vp]
    L.chb_knn_per_bin.argtypes = [_vp, _vp, _vp, _i64, _vp, _vp]
    L.chb_hull_distance_batch.argtypes = [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp]
    L.chb_fit_iteration.argtypes = [_vp, _vp, _i64, _vp, ctypes.POINTER(_i64)]
    L.chb_fit.argtypes = [_vp, _vp, _i64, _i32, _vp, ctypes.POINTER(_i32), ctypes.POINTER(_i32), _vp]
    L.chb_get_labels.argtypes = [_vp, _vp]
    L.chb_iteration_begin.argtypes = [_vp, _vp, _i64]
    L.chb_iteration_begin_dev.argtypes = [_vp, _vp, _i64]
    L.chb_iteration_prefetch.argtypes = [_vp, _vp, _i64]
    L.chb_round_run.argtypes = [_vp, _i64, _i64, _vp]
    L.chb_round_commit.argtypes = [_vp, _i64, _i64, _vp, ctypes.POINTER(_i64)]
    L.chb_iteration_end.argtypes = [_vp, ctypes.POINTER(_i64)]
    L.chb_round_commit_end.argtypes = [_vp, _i64, _i64, _vp, ctypes.POINTER(_i64), ctypes.POINTER(_i64), ctypes.POINTER(_i32)]
    L.chb_set_window.argtypes = [_vp, _i64]
    L.chb_get_window.argtypes = [_vp]
    L.chb_get_window.restype = _i64
    L.chb_measure_fp64_tflops.argtypes = [_vp, ctypes.POINTER(_dbl)]
    L.chb_measure_l2_gbs.argtypes = [_vp, ctypes.POINTER(_dbl)]
    L.chb_guess_export.argtypes = [_vp, _vp, ctypes.POINTER(_i32)]
    L.chb_guess_import.argtypes = [_vp, _vp]
    L.chb_get_distance_path.argtypes = [_vp, ctypes.POINTER(_i32)]
    L.chb_get_row_bounds.argtypes = [_vp, _i64, _i64, _vp, _vp, _vp]
    L.chb_group_create.argtypes = [ctypes.POINTER(_vp), ctypes.POINTER(_vp), _i32]
    L.chb_group_destroy.argtypes = [_vp]
    L.chb_group_buffer.argtypes = [_vp, _i32, _i64, ctypes.POINTER(_vp)]
    L.chb_group_all_max.argtypes = [_vp, _i64]
    L.chb_group_replicate_features.argtypes = [_vp, _i32]
    for name in EXPORTED_SYMBOLS:
        fn = getattr(L, name)
        if name not in ("chb_last_error", "chb_get_window"):
            fn.restype = ctypes.c_int
    _lib = L
    return L


def _nvcc_available() -> bool:
    try:
        _build.find_nvcc()
        return True
    except RuntimeError:
        return False


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data


class Context:
    """One libchbin_b200 context = one GPU.  Error codes become the exceptions the reference raises."""

    def __init__(self, device: int = 0):
        self._lib = load()
        self._h = _vp()
        rc = self._lib.chb_create(ctypes.byref(self._h), int(device))
        if rc != CHB_OK:
            msg = self._lib.chb_last_error(None).decode()
            self._h = None
            raise RuntimeError(f"chb_create failed ({rc}): {msg}")
        self.device = int(device)

    # -- plumbing
    def _check(self, rc: int):
        if rc == CHB_OK:
            return
        msg = self._lib.chb_last_error(self._h).decode()
        if rc in (CHB_EINVAL, CHB_EUNASSIGNED):
            raise ValueError(msg)
        if rc == CHB_ENOTIMPL:
            raise NotImplementedError(msg)
        if rc == CHB_ENOMEM:
            raise MemoryError(msg)
        raise RuntimeError(f"libchbin_b200 error {rc}: {msg}")

    def close(self):
        if getattr(self, "_h", None):
            self._lib.chb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_stream(self, cuda_stream_ptr: int):
        self._check(self._lib.chb_set_stream(self._h, _vp(cuda_stream_ptr)))

    def synchronize(self):
        self._check(self._lib.chb_synchronize(self._h))

    def timers(self) -> dict:
        t = Timers()
        self._check(self._lib.chb_get_timers(self._h, ctypes.byref(t)))
        return t.as_dict()

    def reset_timers(self):
        self._check(self._lib.chb_reset_timers(self._h))

    def enable_timers(self, on: bool):
        self._check(self._lib.chb_enable_timers(self._h, int(bool(on))))

    # -- set-up
    def set_features(self, samples: np.ndarray, asynchronous: bool = False):
        """asynchronous=True: returns once the upload is enqueued; the array is kept alive (and must stay unchanged) until
        build_distance_matrix() / synchronize().  An F-ordered float64 array -- what DataFrame.values hands over at
        cli/clustering.py:53 -- is uploaded as it lies in memory and transposed on the device (chb_set_features_colmajor);
        anything else goes through one C-contiguous float64 copy (a no-op for an array that already is one)."""
        a = np.asarray(samples)
        if a.ndim != 2:
            raise ValueError("samples must be a 2-D array")
        self.n, self.d = a.shape
        if a.dtype == np.float64 and a.flags.f_contiguous and not a.flags.c_contiguous:
            if asynchronous:
                self._pending_features = a
            self._check(self._lib.chb_set_features_colmajor(self._h, _ptr(a), a.shape[0], a.shape[1], int(bool(asynchronous))))
            return
        x = np.ascontiguousarray(a, dtype=np.float64)
        if asynchronous:
            self._pending_features = x
            self._check(self._lib.chb_set_features_async(self._h, _ptr(x), x.shape[0], x.shape[1]))
        else:
            self._check(self._lib.chb_set_features(self._h, _ptr(x), x.shape[0], x.shape[1]))

    def set_features_merged(self, kmer: Optional[np.ndarray], cov_raw: np.ndarray, parent: np.ndarray,
                            want_coverages: bool = False):
        """chb_set_features_merged: samples = [kmer | normalised coverage of the parent contig], built on the device
        (coverage.py:35-41 + cli/features.py:106-109).  Returns the normalised (P, S) coverages when asked."""
        cov = np.ascontiguousarray(cov_raw, dtype=np.float64)
        if cov.ndim != 2:
            raise ValueError("coverages must be a 2-D (P, S) array")
        par = np.ascontiguousarray(parent, dtype=np.int64)
        if par.ndim != 1:
            raise ValueError("parent must be a 1-D index array")
        if kmer is None:
            km = np.zeros((par.shape[0], 0), dtype=np.float64)
        else:
            km = np.ascontiguousarray(kmer, dtype=np.float64)
        if km.ndim != 2 or km.shape[0] != par.shape[0]:
            raise ValueError("kmer must be (n, dk) with one row per entry of parent")
        out = np.empty_like(cov) if want_coverages else None
        self._check(self._lib.chb_set_features_merged(self._h, _ptr(km) if km.shape[1] else None, km.shape[0], km.shape[1],
                                                      _ptr(cov), cov.shape[0], cov.shape[1], _ptr(par), _ptr(out)))
        self.n, self.d = km.shape[0], km.shape[1] + cov.shape[1]
        return out

    def get_features(self) -> np.ndarray:
        out = np.empty((self.n, self.d), dtype=np.float64)
        self._check(self._lib.chb_get_features(self._h, _ptr(out)))
        return out

    def set_features_dev(self, dev_ptr: int, n: int, d: int, asynchronous: bool = False):
        self.n, self.d = int(n), int(d)
        fn = self._lib.chb_set_features_dev_async if asynchronous else self._lib.chb_set_features_dev
        self._check(fn(self._h, _vp(dev_ptr), n, d))

    def features_buffer(self, n: int, d: int):
        """(device address, number of float64 elements) of the context's feature matrix, allocated for (n, d)."""
        ptr, cnt = _vp(), _i64(0)
        self._check(self._lib.chb_features_buffer(self._h, int(n), int(d), ctypes.byref(ptr), ctypes.byref(cnt)))
        self.n, self.d = int(n), int(d)
        return int(ptr.value), int(cnt.value)

    def features_commit(self, asynchronous: bool = False):
        self._check(self._lib.chb_features_commit(self._h, int(bool(asynchronous))))

    def set_labels(self, initial_bins: np.ndarray, num_clusters: int, slot_begin: int = 0, slot_end: int = -1):
        b = np.ascontiguousarray(initial_bins, dtype=np.int64)
        self.C = int(num_clusters)
        self.U = int(np.sum(b == -1))
        self._check(self._lib.chb_set_labels(self._h, _ptr(b), len(b), int(num_clusters), int(slot_begin), int(slot_end)))

    def set_params(self, num_neighbors: int, metric: str = "convex"):
        if metric not in METRICS:
            raise NotImplementedError(f"Metric {metric} not implemented")
        self.k = int(num_neighbors)
        self._check(self._lib.chb_set_params(self._h, int(num_neighbors), METRICS[metric]))

    def set_distance_mode(self, mode: int):
        """1 = FP32 candidate filter + exact FP64 re-rank (default), 0 = exact FP64 rows."""
        self._check(self._lib.chb_set_distance_mode(self._h, int(mode)))

    def distance_path(self) -> int:
        """The distance mode the rounds will run for the current features, labels, parameters and mode: 2 = fused path,
        1 = FP32 candidate filter, 0 = exact rows (mode 2 falls back to 1 where the fused path does not serve)."""
        out = _i32(0)
        self._check(self._lib.chb_get_distance_path(self._h, ctypes.byref(out)))
        return int(out.value)

    def set_gram_engine(self, engine: int):
        """1 = tcgen05 TF32x3 tensor-core Gram (default), 0 = FFMA Gram."""
        self._check(self._lib.chb_set_gram_engine(self._h, int(engine)))

    def get_candidate_rows(self, slot0: int, nrows: int):
        out = np.empty((nrows, self.n), dtype=np.float32)
        nrm = np.empty(self.n, dtype=np.float32)
        eps = _dbl(0.0)
        self._check(self._lib.chb_get_candidate_rows(self._h, slot0, nrows, _ptr(out), ctypes.byref(eps), _ptr(nrm)))
        return out, float(eps.value), nrm

    def get_fused_candidates(self, slot0: int, nslots: int):
        """(keys, idx) of shape (nslots, C, 2*KR) and slack (nslots, C): test aid of distance mode 2."""
        key = np.empty((nslots, self.C, 32), dtype=np.float32)
        idx = np.empty((nslots, self.C, 32), dtype=np.int32)
        slack = np.empty((self.C, nslots), dtype=np.float32)
        kr = _i32(0)
        self._check(self._lib.chb_get_fused_candidates(self._h, slot0, nslots, _ptr(key), _ptr(idx), _ptr(slack), ctypes.byref(kr)))
        m = nslots * self.C * 2 * kr.value
        key = key.reshape(-1)[:m].reshape(nslots, self.C, 2 * kr.value)
        idx = idx.reshape(-1)[:m].reshape(nslots, self.C, 2 * kr.value)
        return key, idx, np.ascontiguousarray(slack.T)

    def get_row_bounds(self, slot0: int, nslots: int):
        """Test aid (fused path): (guessed bin, ub, ubk2) of each owned slot -- the bin-pruning bounds."""
        guess = np.empty(nslots, dtype=np.int32)
        ub = np.empty(nslots, dtype=np.float32)
        ubk2 = np.empty(nslots, dtype=np.float32)
        self._check(self._lib.chb_get_row_bounds(self._h, slot0, nslots, _ptr(guess), _ptr(ub), _ptr(ubk2)))
        return guess, ub, ubk2

    def get_pair_cache(self, slot0: int, nslots: int):
        idx = np.empty((nslots, self.C, self.k), dtype=np.int32)
        cnt = np.empty((nslots, self.C), dtype=np.int32)
        dist = np.empty((nslots, self.C))
        self._check(self._lib.chb_get_pair_cache(self._h, slot0, nslots, _ptr(idx), _ptr(cnt), _ptr(dist)))
        return idx, cnt, dist

    def build_distance_matrix(self, materialise: bool = True):
        self._check(self._lib.chb_build_distance_matrix(self._h, int(bool(materialise))))

    def get_distance_rows(self, slot0: int, nrows: int) -> np.ndarray:
        out = np.empty((nrows, self.n))
        self._check(self._lib.chb_get_distance_rows(self._h, slot0, nrows, _ptr(out)))
        return out

    # -- building blocks
    def knn_per_bin(self, labels: np.ndarray, queries: np.ndarray):
        labels = np.ascontiguousarray(labels, dtype=np.int64)
        queries = np.ascontiguousarray(queries, dtype=np.int64)
        nq = len(queries)
        idx = np.empty((nq, self.C, self.k), dtype=np.int64)
        m = np.empty((nq, self.C), dtype=np.int32)
        self._check(self._lib.chb_knn_per_bin(self._h, _ptr(labels), _ptr(queries), nq, _ptr(idx), _ptr(m)))
        return idx, m

    def hull_distance_batch(self, queries: np.ndarray, idx: np.ndarray, m: np.ndarray, want_alpha: bool = False):
        queries = np.ascontiguousarray(queries, dtype=np.int64)
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        m = np.ascontiguousarray(m, dtype=np.int32)
        nq = len(queries)
        dist = np.empty((nq, self.C))
        status = np.empty((nq, self.C), dtype=np.int32)
        alpha = np.empty((nq, self.C, self.k)) if want_alpha else None
        self._check(self._lib.chb_hull_distance_batch(self._h, _ptr(queries), nq, _ptr(idx), _ptr(m), _ptr(dist),
                                                      _ptr(status), _ptr(alpha)))
        return (dist, status, alpha) if want_alpha else (dist, status)

    # -- assignment loop
    def set_window(self, window: int):
        self._check(self._lib.chb_set_window(self._h, int(window)))

    def get_window(self) -> int:
        return int(self._lib.chb_get_window(self._h))

    def fit_iteration(self, perm: np.ndarray, want_labels: bool = True):
        perm = np.ascontiguousarray(perm, dtype=np.int64)
        labels = np.empty(self.n, dtype=np.int64) if want_labels else None
        nch = _i64(0)
        self._check(self._lib.chb_fit_iteration(self._h, _ptr(perm), len(perm), _ptr(labels), ctypes.byref(nch)))
        return labels, int(nch.value)

    def fit(self, perms: np.ndarray, max_iterations: int):
        perms = np.ascontiguousarray(perms, dtype=np.int64)
        U = perms.shape[1] if perms.ndim == 2 else 0
        labels = np.empty(self.n, dtype=np.int64)
        iters, conv = _i32(0), _i32(0)
        changed = np.zeros(max(int(max_iterations), 1), dtype=np.int64)
        self._check(self._lib.chb_fit(self._h, _ptr(perms), U, int(max_iterations), _ptr(labels), ctypes.byref(iters),
                                      ctypes.byref(conv), _ptr(changed)))
        return labels, int(iters.value), bool(conv.value), changed[: iters.value].copy()

    def get_labels(self) -> np.ndarray:
        labels = np.empty(self.n, dtype=np.int64)
        self._check(self._lib.chb_get_labels(self._h, _ptr(labels)))
        return labels

    def iteration_begin(self, perm: np.ndarray):
        perm = np.ascontiguousarray(perm, dtype=np.int64)
        self._check(self._lib.chb_iteration_begin(self._h, _ptr(perm), len(perm)))

    def iteration_prefetch(self, perm: np.ndarray):
        """chb_iteration_prefetch: uploads the NEXT iteration's permutation while the current rounds run; `perm` must be the
        very array (int64, contiguous) later handed to iteration_begin."""
        if perm.dtype != np.int64 or not perm.flags.c_contiguous:
            return  # iteration_begin would convert it into a temporary: nothing to match the prefetched copy with
        self._check(self._lib.chb_iteration_prefetch(self._h, _ptr(perm), len(perm)))

    def guess_export(self, guess_dev_ptr: int) -> bool:
        """chb_guess_export: the owned slots' speculation start into a device buffer of U int32; False = nothing to exchange."""
        active = _i32(0)
        self._check(self._lib.chb_guess_export(self._h, _vp(guess_dev_ptr), ctypes.byref(active)))
        return bool(active.value)

    def guess_import(self, guess_dev_ptr: int):
        self._check(self._lib.chb_guess_import(self._h, _vp(guess_dev_ptr)))

    def iteration_begin_dev(self, perm_dev_ptr: int, U: int):
        """chb_iteration_begin_dev: the permutation (int64, U entries) already lies in device memory."""
        self._check(self._lib.chb_iteration_begin_dev(self._h, _vp(perm_dev_ptr), int(U)))

    def round_run(self, lo: int, hi: int, tent_dev_ptr: Optional[int] = None):
        """Enqueues one speculate round (asynchronous).  tent_dev_ptr None: the library's own tentative buffer."""
        self._check(self._lib.chb_round_run(self._h, lo, hi, _vp(tent_dev_ptr)))

    def round_commit(self, lo: int, hi: int, tent_dev_ptr: Optional[int] = None) -> int:
        first = _i64(-1)
        self._check(self._lib.chb_round_commit(self._h, lo, hi, _vp(tent_dev_ptr), ctypes.byref(first)))
        return int(first.value)

    def round_commit_end(self, lo: int, hi: int, tent_dev_ptr: Optional[int] = None):
        """chb_round_commit_end: (first_changed, iteration_done, n_changed) -- one synchronisation for the commit and, when
        the round settled the iteration, its end."""
        first, nch, done = _i64(-1), _i64(0), _i32(0)
        self._check(self._lib.chb_round_commit_end(self._h, lo, hi, _vp(tent_dev_ptr), ctypes.byref(first), ctypes.byref(nch),
                                                   ctypes.byref(done)))
        return int(first.value), bool(done.value), int(nch.value)

    def measure_fp64_tflops(self) -> float:
        v = _dbl(0.0)
        self._check(self._lib.chb_measure_fp64_tflops(self._h, ctypes.byref(v)))
        return float(v.value)

    def measure_l2_gbs(self) -> float:
        v = _dbl(0.0)
        self._check(self._lib.chb_measure_l2_gbs(self._h, ctypes.byref(v)))
        return float(v.value)

    def iteration_end(self) -> int:
        nch = _i64(0)
        self._check(self._lib.chb_iteration_end(self._h, ctypes.byref(nch)))
        return int(nch.value)


class Group:
    """A device group (chb_group_*): N distinct contexts driven from this thread, exchanging int32 label windows on the
    devices.  Holds its member Contexts; close the group before any of them."""

    def __init__(self, members):
        self._lib = load()
        self.members = list(members)
        if not self.members or any(getattr(m, "_h", None) is None for m in self.members):
            raise ValueError("a device group needs at least one open context")
        self._h = _vp()
        arr = (_vp * len(self.members))(*[m._h for m in self.members])
        self._check(self._lib.chb_group_create(ctypes.byref(self._h), arr, len(self.members)))
        self._bufs = [None] * len(self.members)  # (device address, entries) per member

    def _check(self, rc: int):
        if rc == CHB_OK:
            return
        msg = self._lib.chb_last_error(None).decode()
        if rc == CHB_EINVAL:
            raise ValueError(msg)
        if rc == CHB_ENOMEM:
            raise MemoryError(msg)
        raise RuntimeError(f"libchbin_b200 error {rc}: {msg}")

    def close(self):
        if getattr(self, "_h", None):
            self._lib.chb_group_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def buffer(self, m: int, count: int) -> int:
        """Device address of member m's group buffer, grown to at least `count` int32 entries."""
        cur = self._bufs[m]
        if cur is None or cur[1] < count:
            ptr = _vp()
            self._check(self._lib.chb_group_buffer(self._h, int(m), int(count), ctypes.byref(ptr)))
            cur = self._bufs[m] = (int(ptr.value), int(count))
        return cur[0]

    def all_max(self, count: int):
        """Element-wise MAX of the members' buffers [0, count), into every member's buffer (enqueued only)."""
        self._check(self._lib.chb_group_all_max(self._h, int(count)))

    def replicate_features(self, root: int = 0):
        """Member `root`'s feature matrix into every other member (enqueued; each receiver derives its own FP32 copy)."""
        self._check(self._lib.chb_group_replicate_features(self._h, int(root)))
        r = self.members[root]
        for m in self.members:
            m.n, m.d = r.n, r.d
