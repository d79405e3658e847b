"""
Host-side mirror of the reference's clustering interface for the B200 path.

    fit_cluster(...)           <- /root/reference/ch_bin/core/clustering/algorithm.py:12-76   (same names, same
                                  argument meaning, same RNG draws, same log lines, same return value)
    perform_clustering(...)    <- /root/reference/ch_bin/cli/clustering.py:19-99 steps 01-04 (CSV in, CSV out)
    install(ref_module)        <- adds the `AlgoQpSolver = b200` branch to the reference's own
                                  ch_bin.cli.clustering module (see INTEGRATION.md)

All arithmetic of the hot path (distance rows, per-bin kNN, hull-distance QPs, ordered assignment) runs in
libchbin_b200.so (hand-written sm_100a CUDA) behind the C-ABI of include/chbin_b200.h.  This module only owns
what the reference keeps in Python: the permutation draws on numpy's global legacy RNG, the early-stop rule,
logging, and -- when torch.distributed is initialised with more than one rank -- the per-round label exchange (a device
group of fit_cluster(devices=...) exchanges the labels inside the library instead).
There is no CPU fallback.
"""
from __future__ import annotations

import logging
import os
import shutil
import time
from pathlib import Path
from typing import Optional, Sequence, Tuple

import numpy as np

from . import capi, distance_cache

logger = logging.getLogger(__name__)

B200_SOLVER = "b200"
ROUND_AGAIN = -2  # CHB_ROUND_AGAIN (include/chbin_b200.h)

# One library context per device is kept alive between fit_cluster calls of a process (like a BLAS handle): creating
# a context, its stream and its multi-GB device buffers costs ~10 ms, comparable to the whole 20k-contig stage.
_CTX_CACHE = {}
# ... and one torch stream per device for the sharded path: torch's caching allocator keeps its pools per stream, so a fresh
# stream per call would turn every torch.empty into a cudaMalloc (tens of milliseconds)
_STREAM_CACHE = {}
# Device groups of fit_cluster(devices=...), by device tuple, with their member contexts.  Member 0 is the device's ordinary
# cached context; member i > 0 has a context of its own under (device, i), so that a device may appear more than once.
_GROUP_CACHE = {}


def _get_context(device: int, reuse: bool, member: int = 0) -> "capi.Context":
    if not reuse:
        return capi.Context(device)
    key = device if member == 0 else (device, member)
    ctx = _CTX_CACHE.get(key)
    if ctx is None or getattr(ctx, "_h", None) is None:
        ctx = capi.Context(device)
        _CTX_CACHE[key] = ctx
    return ctx


def _get_group(devices, members, reuse: bool) -> "capi.Group":
    if not reuse:
        return capi.Group(members)
    key = tuple(devices)
    g = _GROUP_CACHE.get(key)
    if g is None or g._h is None or any(a is not b for a, b in zip(g.members, members)):
        g = _GROUP_CACHE[key] = capi.Group(members)
    return g


def _drop(ctxs) -> None:
    """Closes these contexts and every cached group that holds one of them (groups first: they refer to their members)."""
    for key, g in list(_GROUP_CACHE.items()):
        if any(m is c for m in g.members for c in ctxs):
            g.close()
            del _GROUP_CACHE[key]
    for key, c in list(_CTX_CACHE.items()):
        if any(c is x for x in ctxs):
            del _CTX_CACHE[key]
    for c in ctxs:
        c.close()


def shutdown() -> None:
    """Destroys the cached device groups and per-device contexts (frees all device memory held by the library)."""
    for g in list(_GROUP_CACHE.values()):
        g.close()
    _GROUP_CACHE.clear()
    for ctx in list(_CTX_CACHE.values()):
        ctx.close()
    _CTX_CACHE.clear()


# ----------------------------------------------------------------------------------------------------------
# round driver (shared by the single- and multi-GPU paths; engine-agnostic so the host logic is testable)
# ----------------------------------------------------------------------------------------------------------
def owned_slots(U: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous slice of query slots (= points_to_assign in ascending order) a rank owns."""
    return (U * rank) // world, (U * (rank + 1)) // world


# Below this many (query, bin) pairs per stage the ranks do not shard: a stage is then a ~1 ms chain of short kernels, and every
# collective of the sharded protocol (feature broadcast, guess exchange, one label all-reduce per round, the permutation
# broadcast) costs 30-100 us of launch latency and host time -- measured at 20k contigs x 50 bins (875k pairs): 0.97 ms on one GPU,
# 0.92-1.06 ms sharded over 2-8, and end to end 1.65 ms against 2.1-2.9 ms.  Every rank then runs the whole (deterministic, exact)
# stage on its own GPU with no communication at all and returns the same labels.  Ranks must share the RNG state, as they do under
# the reference's CLI (np.random.seed(0) in every process, ch_bin/ch_bin.py:22).  100k contigs x 100 bins (9.5 M pairs) shards.
SHARD_MIN_PAIRS = int(os.environ.get("CHB_SHARD_MIN_PAIRS", 2_000_000))


def sharding_pays(num_points_to_assign: int, num_clusters: int, world: int) -> bool:
    """True when `world` ranks should shard the query slots of a stage (see SHARD_MIN_PAIRS)."""
    return world > 1 and int(num_points_to_assign) * int(num_clusters) >= SHARD_MIN_PAIRS


def run_iteration(engine, perm, comm=None, next_perm=None) -> Tuple[int, int]:
    """One iteration of algorithm.py:43-72 as speculate/repair rounds (csrc/api.cu header).

    next_perm: the permutation of the iteration after this one, if the caller already has it (host array): engines with a
    prefetch() upload it while this iteration's first round runs on the device.

    engine: iteration_begin(perm), round_run(lo, hi) -> tent, round_commit(lo, hi, tent) -> first_changed (-1 = none),
            iteration_end() -> n_changed, window() -> int; optionally round_commit_end(lo, hi, tent) ->
            (first_changed, iteration_done, n_changed), which ends the iteration in the same call when the round settled it.
    comm:   None, or an object with all_reduce_max(tent) -> tent merging the ranks' tentative labels.
    Returns (n_changed, rounds)."""
    U = len(perm)
    engine.iteration_begin(perm)
    W = engine.window() or U
    merged = getattr(engine, "round_commit_end", None)
    lo, rounds = 0, 0
    while lo < U:
        hi = min(U, lo + W)
        tent = engine.round_run(lo, hi)
        if comm is not None:
            tent = comm.all_reduce_max(tent)
        if next_perm is not None and hasattr(engine, "prefetch"):
            engine.prefetch(next_perm)
            next_perm = None
        if merged is not None:
            first, done, n_changed = merged(lo, hi, tent)
            rounds += 1
            if done:
                return n_changed, rounds
        else:
            first = engine.round_commit(lo, hi, tent)
            rounds += 1
        if first == ROUND_AGAIN:
            continue  # the library enlarged its exact-redo list: the same window runs again
        lo = hi if first < 0 else first + 1
    return engine.iteration_end(), rounds


class GpuEngine:
    """Engine over one libchbin_b200 context; tentative labels live in a torch int32 device tensor so that
    torch.distributed (NCCL) can all-reduce them in place between chb_round_run and chb_round_commit."""

    def __init__(self, ctx: capi.Context, device_index: int, stream=None):
        import torch

        self.ctx = ctx
        self.torch = torch
        self.device = torch.device("cuda", device_index)
        self._tent = None
        # one dedicated stream shared by the library's kernels and torch.distributed's collectives: the all-reduce
        # of the tentative labels must be ordered between chb_round_run and chb_round_commit
        self.stream = stream if stream is not None else torch.cuda.Stream(self.device)
        ctx.set_stream(self.stream.cuda_stream)

    def stream_context(self):
        return self.torch.cuda.stream(self.stream)

    def window(self) -> int:
        return self.ctx.get_window()

    def iteration_begin(self, perm):
        if isinstance(perm, self.torch.Tensor):  # rank 0's draw, broadcast over NCCL: stays on the device
            try:
                self.ctx.iteration_begin_dev(perm.data_ptr(), perm.numel())
                return
            except ValueError:  # not distance mode 2 (wide features, ...): the library wants the permutation on the host
                perm = perm.cpu().numpy()
        self.ctx.iteration_begin(perm)

    def round_commit_end(self, lo, hi, tent):
        return self.ctx.round_commit_end(lo, hi, tent.data_ptr())

    def prefetch(self, perm):
        if isinstance(perm, np.ndarray):  # a host permutation: uploaded on the library's side stream while a round runs
            self.ctx.iteration_prefetch(perm)

    def guess_export(self, U):
        g = self.torch.empty(max(U, 1), dtype=self.torch.int32, device=self.device)[:U]
        return g if self.ctx.guess_export(g.data_ptr()) else None

    def guess_import(self, g):
        self.ctx.guess_import(g.data_ptr())

    def round_run(self, lo, hi):
        n = hi - lo
        if self._tent is None or self._tent.numel() < n:
            self._tent = self.torch.empty(max(n, self.ctx.get_window()), dtype=self.torch.int32, device=self.device)
        t = self._tent[:n]
        self.ctx.round_run(lo, hi, t.data_ptr())
        return t

    def round_commit(self, lo, hi, tent):
        return self.ctx.round_commit(lo, hi, tent.data_ptr())

    def iteration_end(self):
        return self.ctx.iteration_end()


class _ContextEngine:
    """The round interface over a context that owns every query slot (no exchange: the library keeps the tentative labels
    itself, nothing of torch is touched)."""

    def __init__(self, ctx: capi.Context):
        self.ctx = ctx

    def window(self):
        return self.ctx.get_window()

    def iteration_begin(self, perm):
        self.ctx.iteration_begin(perm)

    def prefetch(self, perm):
        self.ctx.iteration_prefetch(perm)

    def round_run(self, lo, hi):
        self.ctx.round_run(lo, hi)
        return None

    def round_commit_end(self, lo, hi, tent):
        return self.ctx.round_commit_end(lo, hi)

    def iteration_end(self):
        return self.ctx.iteration_end()


class GroupEngine:
    """The round interface over a device group (capi.Group) in one process: every member runs the round of its owned slots
    into its group buffer, then chb_group_all_max merges the windows by element-wise MAX on the devices -- what the NCCL
    all-reduce does between ranks, without torch.  The members commit the same merged labels and must agree on the result."""

    def __init__(self, group: "capi.Group", U: int):
        self.group = group
        self.members = group.members
        self.bufs = [group.buffer(m, max(U, 1)) for m in range(len(self.members))]

    def stream_context(self):
        import contextlib

        return contextlib.nullcontext()  # every member runs on its own stream

    def window(self):
        return self.members[0].get_window()

    def iteration_begin(self, perm):
        for m in self.members:
            m.iteration_begin(perm)

    def prefetch(self, perm):
        for m in self.members:
            m.iteration_prefetch(perm)

    def round_run(self, lo, hi):
        for m, b in zip(self.members, self.bufs):
            m.round_run(lo, hi, b)
        self.group.all_max(hi - lo)
        return None

    def _agree(self, results, what):
        if any(r != results[0] for r in results):
            raise RuntimeError(f"the members of the device group disagree on {what}: {results}")
        return results[0]

    def round_commit_end(self, lo, hi, tent):
        return self._agree([m.round_commit_end(lo, hi, b) for m, b in zip(self.members, self.bufs)],
                           "(first_changed, done, n_changed)")

    def iteration_end(self):
        return self._agree([m.iteration_end() for m in self.members], "n_changed")

    def guess_export(self, U):
        active = [m.guess_export(b) for m, b in zip(self.members, self.bufs)]
        return U if self._agree(active, "the guess exchange") else None

    def all_reduce_max(self, count):
        """The guess exchange of exchange_guess: the same MAX over the members' buffers."""
        self.group.all_max(count)
        return count

    def guess_import(self, g):
        for m, b in zip(self.members, self.bufs):
            m.guess_import(b)


class TorchComm:
    """Label exchange between ranks: one all-reduce(MAX) of a window of int32 labels per round (un-owned
    positions hold INT32_MIN).  NCCL over NVLink on the GPU box, gloo in the CPU tests."""

    def __init__(self, group=None):
        import torch.distributed as dist

        self.dist = dist
        self.group = group

    def all_reduce_max(self, tent):
        self.dist.all_reduce(tent, op=self.dist.ReduceOp.MAX, group=self.group)
        return tent


class _CudaArray:
    """Minimal __cuda_array_interface__ carrier: lets torch wrap device memory the library owns (no copy, no ownership)."""

    def __init__(self, ptr: int, count: int):
        self.__cuda_array_interface__ = {"shape": (count,), "typestr": "<f8", "data": (ptr, False), "version": 3}


def _device_view(torch, ptr: int, count: int, device):
    return torch.as_tensor(_CudaArray(ptr, count), device=device)


def exchange_guess(engine, comm, U: int, mark=None) -> bool:
    """Sharded contexts: every rank computes the first iteration's speculation start (nearest seed centroid) for its OWN query
    slots and the ranks merge them with one all-reduce(MAX) of U int32 labels (un-owned entries are INT32_MIN) -- instead of
    every rank repeating the U x C x d contraction.  No-op for engines without the export/import pair."""
    if not hasattr(engine, "guess_export"):
        return False
    mark = mark or (lambda label: None)
    with engine.stream_context():
        g = engine.guess_export(U)
        mark("  guess exported")
        if g is None:
            return False
        g = comm.all_reduce_max(g)
        mark("  guess all-reduced")
        engine.guess_import(g)
    return True


def _dist_state():
    try:
        import torch.distributed as dist
    except Exception:  # torch missing: single process
        return None, 0, 1
    if dist.is_available() and dist.is_initialized():
        return dist, dist.get_rank(), dist.get_world_size()
    return None, 0, 1


def draw_permutations(initial_bins: np.ndarray, max_iterations: int, seed: Optional[int] = 0) -> np.ndarray:
    """The permutations fit_cluster would draw (algorithm.py:45) for up to `max_iterations` iterations, as one
    (max_iterations, U) int64 array: np.random.seed(seed) as in ch_bin/ch_bin.py:22, then one
    np.random.permutation(points_to_assign) per iteration on the global legacy RNG.  For callers that drive the C-ABI
    themselves (chb_fit, benchmarks)."""
    pts = np.where(np.asarray(initial_bins) == -1)[0]
    if seed is not None:
        np.random.seed(seed)
    return np.stack([np.random.permutation(pts) for _ in range(max_iterations)]).astype(np.int64).reshape(max_iterations, len(pts))


def _draw_permutation(points_to_assign: np.ndarray, dist_mod, device_index: int, keep_on_device: bool = False):
    """algorithm.py:45.  Every rank draws from its own global RNG (so the stream advances exactly as in the
    reference); rank 0's draw is authoritative and broadcast so that differently-seeded ranks cannot diverge.  With NCCL
    and keep_on_device the broadcast permutation is returned as a device tensor (it goes straight into
    chb_iteration_begin_dev: no device -> host -> device round trip); otherwise as a numpy array."""
    perm = np.random.permutation(points_to_assign).astype(np.int64)
    if dist_mod is not None and dist_mod.get_world_size() > 1:
        import torch

        nccl = dist_mod.get_backend() == "nccl"
        dev = torch.device("cuda", device_index) if nccl else torch.device("cpu")
        if nccl and dist_mod.get_rank() != 0:
            t = torch.empty(len(perm), dtype=torch.int64, device=dev)  # the receivers need no upload of their own draw
        else:
            t = torch.from_numpy(perm).to(dev)
        dist_mod.broadcast(t, src=0)
        if nccl and keep_on_device:
            return t
        perm = t.cpu().numpy()
    return perm


# ----------------------------------------------------------------------------------------------------------
# fit_cluster
# ----------------------------------------------------------------------------------------------------------
def fit_cluster(
    samples: np.ndarray,
    num_clusters: int,
    initial_bins: np.ndarray,
    distance_matrix: Optional[np.ndarray] = None,
    num_neighbors: int = 15,
    max_iterations: int = 10,
    metric: str = "convex",
    qp_solver: str = B200_SOLVER,
    in_mem_dist_matrix: bool = True,
    device: Optional[int] = None,
    window: int = 0,
    return_info: bool = False,
    distance_mode: int = 2,
    reuse_context: bool = True,
    gram_engine: int = 1,
    devices: Optional[Sequence[int]] = None,
):
    """
    Cevikalp et al. 2019 convex-hull binning specialised for metagenomic binning, on B200.

    Drop-in for algorithm.py:12-21 (`fit_cluster`).  `distance_matrix` is accepted for signature compatibility
    and ignored: distances are the same doubles (scipy-cdist recipe, bit-exact), produced on the device --
    materialised in HBM when `in_mem_dist_matrix` (InMemDistMatrix=yes) and recomputed on demand otherwise.
    `qp_solver` must be "b200": quadprog / cvxopt belong to the reference's CPU path (solve_qp.py:125-132).

    :param samples: Dataset points (n, d) float64.
    :param num_clusters: Number of clusters.
    :param initial_bins: Initial bin vector. Use -1 for un-binned.
    :param num_neighbors: Number of neighbors to consider for polytope.
    :param max_iterations: Number of maximum iterations to perform.
    :param metric: Polytope distance metric (convex/affine/affine-qp).
    :param devices: CUDA ordinals of this process to run the stage on (None: `device`, today's single-GPU path).  With two
        or more entries and a stage large enough to pay for the exchange (sharding_pays), the query slots are sharded over
        them as a device group (one context per entry; an ordinal may repeat) that merges the labels on the devices,
        without torch.distributed; a smaller stage runs whole on devices[0].  Same labels and RNG draws either way.
    :return: Final binning result (int64, n).
    """
    if qp_solver != B200_SOLVER:
        raise NotImplementedError(f"Unknown solver {qp_solver}")  # solve_qp.py:132
    if metric not in capi.METRICS:
        raise NotImplementedError(f"Metric {metric} not implemented")  # hull_distance.py:108

    dist_mod, rank, world = _dist_state()
    if devices is not None:
        devices = [int(dv) for dv in devices]
        if not devices:
            raise ValueError("devices must name at least one CUDA device")
        if world > 1:
            raise ValueError(f"devices={devices} shards the stage inside this process, but torch.distributed already runs it "
                             f"on {world} ranks: use one of the two")
        if device is not None:
            raise ValueError("pass either device or devices")
        device = devices[0]
    if device is None:
        device = 0
        if world > 1:
            import torch

            device = torch.cuda.current_device()

    initial_bins = np.asarray(initial_bins)
    curr = initial_bins.astype(np.int64, copy=True)  # algorithm.py:37 -- inputs are never mutated
    points_to_assign = np.where(curr == -1)[0]  # algorithm.py:38
    num_points_to_assign = len(points_to_assign)
    logger.debug("Assigning %s points.", num_points_to_assign)
    job_rank, job_world = rank, world
    if world > 1 and not sharding_pays(num_points_to_assign, num_clusters, world):
        dist_mod, rank, world = None, 0, 1  # too small to pay for the collectives: every rank runs the whole stage (SHARD_MIN_PAIRS)

    marks = [] if os.environ.get("CHB_PROFILE_FIT") else None  # wall-clock marks of the host driver (tools/e2e_multi.py)

    def mark(label):
        if marks is not None:
            marks.append((label, time.perf_counter()))

    mark("start")
    ctxs = [_get_context(dv, reuse_context, i) for i, dv in enumerate(devices or [device])]  # every ordinal is checked
    ctx = ctxs[0]
    group = None
    try:
        if len(ctxs) > 1 and sharding_pays(num_points_to_assign, num_clusters, len(ctxs)):
            group = _get_group(devices, ctxs, reuse_context)
        members = group.members if group is not None else [ctx]
        for m in members:
            m.set_stream(capi.OWN_STREAM)
            m.reset_timers()
        engine = comm = None
        u0, u1 = owned_slots(num_points_to_assign, rank, world)
        if world > 1:
            import torch

            stream = _STREAM_CACHE.get(device)
            if stream is None:
                stream = _STREAM_CACHE[device] = torch.cuda.Stream(torch.device("cuda", device))
            engine = GpuEngine(ctx, device, stream)
            comm = TorchComm()
        if world > 1 and dist_mod.get_backend() == "nccl":
            # SURVEY 8(e): the (small) feature matrix is replicated with ONE NCCL broadcast over NVLink -- rank 0 uploads its
            # host array once, the other ranks receive it device to device instead of pushing the same bytes over PCIe
            import torch

            with engine.stream_context():
                n_, d_ = np.shape(samples)
                if rank == 0:  # exactly the single-GPU upload: pinned or pageable, C- or F-ordered (transposed on the device)
                    ctx.set_features(samples, asynchronous=True)
                ptr, count = ctx.features_buffer(n_, d_)
                Xd = _device_view(torch, ptr, count, engine.device)  # the library's own matrix: no copy on either side
                mark("X upload enqueued")
                dist_mod.broadcast(Xd, src=0)
                mark("broadcast X enqueued")
                if rank != 0:
                    ctx.features_commit(asynchronous=True)
            del Xd
            mark("features set")
        else:
            ctx.set_features(samples, asynchronous=True)  # the upload overlaps the label set-up and the first permutation draw
            if group is not None:
                group.replicate_features(0)  # device to device, as the NCCL broadcast does between ranks
        for i, m in enumerate(members):
            if group is not None:
                u0, u1 = owned_slots(num_points_to_assign, i, len(members))
            m.set_labels(curr, int(num_clusters), u0, u1)
            m.set_params(int(num_neighbors), metric)
            m.set_window(int(window))
            m.set_distance_mode(int(distance_mode))
            m.set_gram_engine(int(gram_engine))
        spec_perm = spec_state = None  # a permutation drawn ahead of the iteration that will use it
        # the permutation stays on the device when the library's fused path serves the stage (chb_get_distance_path)
        on_device = world > 1 and dist_mod.get_backend() == "nccl" and ctx.distance_path() == 2
        if max_iterations > 0:  # iteration 1 always executes: its permutation is drawn while the features are still in flight
            if world > 1:
                with engine.stream_context():
                    spec_perm = _draw_permutation(points_to_assign, dist_mod, device, keep_on_device=on_device)
            else:
                spec_perm = _draw_permutation(points_to_assign, dist_mod, device)
        mark("labels/params set")
        for m in members:
            m.build_distance_matrix(bool(in_mem_dist_matrix))
        ctx._pending_features = None
        mark("distance structure")
        if group is not None:
            engine = GroupEngine(group, num_points_to_assign)
            if num_points_to_assign > 0 and max_iterations > 0:
                exchange_guess(engine, engine, num_points_to_assign, mark)  # the group's MAX serves as the collective
                mark("guess exchanged")
        if world > 1 and num_points_to_assign > 0 and max_iterations > 0:
            exchange_guess(engine, comm, num_points_to_assign, mark)
            mark("guess exchanged")

        iterations, converged, rounds_total, changed = 0, False, 0, []
        # One loop for one context and for sharded contexts.  chb_round_run only enqueues, the commit synchronises: the NEXT
        # iteration's np.random.permutation (algorithm.py:45) is drawn -- and, between ranks, broadcast -- while the first
        # round runs on the device; if the loop then stops (algorithm.py:63-66, or the iteration limit) the global RNG is put
        # back, so that exactly one draw per EXECUTED iteration remains visible: the reference's RNG contract.
        import contextlib

        eng = engine if engine is not None else _ContextEngine(ctx)
        stream_ctx = engine.stream_context() if world > 1 else contextlib.nullcontext()
        with stream_ctx:
            if spec_perm is None and max_iterations > 0:
                spec_perm = _draw_permutation(points_to_assign, dist_mod, device, keep_on_device=on_device)
            for i_iter in range(max_iterations):
                sample_perm, spec_perm, spec_state = spec_perm, None, None
                U = num_points_to_assign
                eng.iteration_begin(sample_perm)
                mark(f"it{i_iter + 1} begun")
                W = eng.window() or U
                lo = rounds = 0
                done, change_count = False, 0
                while lo < U:
                    hi = min(U, lo + W)
                    tent = eng.round_run(lo, hi)
                    if comm is not None:
                        tent = comm.all_reduce_max(tent)
                    if spec_state is None and i_iter + 1 < max_iterations:
                        spec_state = np.random.get_state()
                        spec_perm = _draw_permutation(points_to_assign, dist_mod, device, keep_on_device=on_device)
                        if isinstance(spec_perm, np.ndarray) and hasattr(eng, "prefetch"):
                            eng.prefetch(spec_perm)  # uploaded on a side stream while this round runs on the device
                    first, done, change_count = eng.round_commit_end(lo, hi, tent)
                    rounds += 1
                    if first == ROUND_AGAIN:
                        continue  # the library enlarged its exact-redo list: the same window runs again
                    lo = hi if first < 0 else first + 1
                if not done:
                    change_count = eng.iteration_end()
                mark(f"it{i_iter + 1} rounds done ({rounds})")
                stop = change_count == 0 or i_iter + 1 == max_iterations
                if stop and spec_state is not None:
                    np.random.set_state(spec_state)  # the speculative draw never happened
                    spec_perm = spec_state = None
                rounds_total += rounds
                iterations += 1
                changed.append(change_count)
                # If the assignments did not change, break  (algorithm.py:63-66)
                if change_count == 0:
                    logger.info("Iteration %s: No changes with previous iteration... Stopping...", i_iter + 1)
                    converged = True
                    break
                change_avg = change_count / len(curr)
                logger.info("Iteration %s: Points changed clusters. avg=%s, count=%s", i_iter + 1, change_avg, change_count)
                if spec_perm is None and not stop:
                    spec_perm = _draw_permutation(points_to_assign, dist_mod, device, keep_on_device=on_device)
            else:
                logger.info("Exit due to max iteration limit.")
        labels = ctx.get_labels()
        mark("labels read back")
        tm_end = ctx.timers()
        if tm_end.get("qp_iter_cap", 0):
            logger.warning("%s hull-distance QPs stopped on the iteration cap of the active-set method (feasible, possibly not "
                           "optimal); the reference would have fallen back to cvxopt there.", tm_end["qp_iter_cap"])
        info = dict(iterations=iterations, converged=converged, changed=changed, timers=tm_end, rank=job_rank,
                    world=job_world, owned_slots=(u0, u1), replicated=job_world > 1 and world == 1)
        if devices is not None:
            # the device group: member i owns owned_slots(U, i, len(devices)); a stage too small to shard ran whole on devices[0]
            info.update(world=len(devices), devices=devices, sharded=group is not None,
                        owned_slots=[owned_slots(num_points_to_assign, i, len(members)) for i in range(len(members))])
        if marks is not None:
            info["marks_ms"] = [(lab, (t - marks[0][1]) * 1e3) for lab, t in marks]
    except BaseException:
        if group is not None:
            group.close()
        _drop(ctxs)  # never reuse a context (or a group holding it) after a failure
        raise
    finally:
        if not reuse_context:
            if group is not None:
                group.close()
            for c in ctxs:
                c.close()
    if return_info:
        return labels, info
    return labels


# ----------------------------------------------------------------------------------------------------------
# perform_clustering (steps 01-04 of cli/clustering.py) and the plug-in hook
# ----------------------------------------------------------------------------------------------------------
def perform_clustering(
    contig_fasta: Optional[Path],
    features_csv: Path,
    operating_dir: Path,
    num_neighbors: int = 15,
    max_iterations: int = 10,
    metric: str = "convex",
    qp_solver: str = B200_SOLVER,
    in_mem_dist_matrix: bool = True,
    devices: Optional[Sequence[int]] = None,
) -> Path:
    """cli/clustering.py:19-99 with steps 02-03 on the GPU.  Step 05 (FASTA dump, needs Biopython) is the
    reference's own `dump_bins` and is only invoked when this function is installed into the reference.
    devices: as for fit_cluster (None: one GPU; several: one stage sharded over them from this process)."""
    import pandas as pd

    operating_dir = Path(operating_dir)
    dist_bin_csv = operating_dir / "binning-assignment.csv"
    operating_dir.mkdir(parents=True, exist_ok=True)

    logger.info(">> Reading feature CSV...")
    samples = None
    if distance_cache.sidecar_path(features_csv).exists():
        # binary side-car of the samples block (distance_cache.write_features_sidecar): only the three label columns are
        # parsed from the CSV text
        df_features = pd.read_csv(features_csv, usecols=distance_cache.META_COLUMNS)
        samples = distance_cache.load_samples(features_csv, len(df_features))
    if samples is None:
        df_features = pd.read_csv(features_csv)
        samples = df_features.drop(distance_cache.META_COLUMNS, axis=1).values
    num_clusters = int(df_features.CLUSTER.max() + 1)
    initial_bins = df_features.CLUSTER.values.copy()
    num_samples = len(samples)

    if not in_mem_dist_matrix:
        # cli/clustering.py:60-63: the on-disk matrix is produced (or found) exactly where the reference keeps it, so that a
        # later reference run can reuse it; the assignment rounds below regenerate distances on the device and never read
        # it back.  The file is 8 n^2 bytes (320 GB at 200k contigs): beyond CHB_DISTANCE_MATRIX_MAX_GB (default 64) or
        # the free space of the volume it is skipped -- InMemDistMatrix = no exists for inputs whose matrix does not fit,
        # and this path does not need the matrix at all.
        need = 8 * num_samples * num_samples
        limit = float(os.environ.get("CHB_DISTANCE_MATRIX_MAX_GB", "64")) * (1 << 30)
        existing = operating_dir / distance_cache.DISTANCE_MATRIX_NAME
        if existing.exists():
            logger.info("Reusing already existing distance matrix at %s.", existing)
            if not distance_cache.validate_distance_matrix(existing, samples):
                logger.warning("%s does not hold the distances of these features (stale cache); the b200 solver does not "
                               "read it, a later reference run would.", existing)
        elif need > limit or need > shutil.disk_usage(operating_dir).free:
            logger.info(">> Skipping the in-disk distance matrix of %s (%.1f GB): not needed by the %s solver.",
                        (num_samples, num_samples), need / (1 << 30), qp_solver)
        else:
            logger.info(">> Creating a distance matrix of %s in-disk...", (num_samples, num_samples))
            distance_cache.create_distance_matrix(samples, operating_dir)

    logger.info(">> Performing binning using %s solver...", qp_solver)
    multi = {} if devices is None else dict(devices=devices)  # the default call is exactly the single-GPU one
    convex_labels = fit_cluster(
        samples=samples, num_clusters=num_clusters, initial_bins=initial_bins, num_neighbors=num_neighbors,
        max_iterations=max_iterations, metric=metric, qp_solver=qp_solver, in_mem_dist_matrix=in_mem_dist_matrix,
        **multi,
    )
    if np.any(convex_labels < 0):
        raise ValueError("There were some un-clustered points left... Aborting.")  # cli/clustering.py:79-80

    logger.info(">> Assigning bins...")
    df_combined = pd.concat([df_features[["PARENT_NAME"]], pd.DataFrame({"BIN": convex_labels})], axis=1)
    parent_groups = df_combined[["PARENT_NAME", "BIN"]].groupby("PARENT_NAME")
    df_dist_bin = parent_groups.BIN.apply(lambda x: np.bincount(x).argmax()).reset_index()
    df_dist_bin.rename(columns={"PARENT_NAME": "CONTIG_NAME"}, inplace=True)
    df_dist_bin.to_csv(dist_bin_csv, index=False)
    logger.info("Dumped binning assignment CSV at %s...", dist_bin_csv)
    return dist_bin_csv


def install(ref_cli_clustering_module, devices: Optional[Sequence[int]] = None) -> None:
    """Adds the `AlgoQpSolver = b200` branch to the reference's own `ch_bin.cli.clustering` module, in place:
    `perform_clustering(..., qp_solver="b200")` then runs steps 01-04 here (distance structure + fit_cluster on
    the GPU) and hands step 05 (FASTA dump) back to the reference's `dump_bins`; any other solver value goes
    to the untouched original.  `run_perform_clustering` (cli/clustering.py:102-127) needs no change: it looks
    `perform_clustering` up in the module at call time.  devices: the CUDA ordinals every b200 stage runs on (None: one
    GPU), so that the reference's single-process CLI can use several GPUs (fit_cluster's `devices`)."""
    mod = ref_cli_clustering_module
    orig_perform = mod.perform_clustering

    def perform_dispatch(contig_fasta, features_csv, operating_dir, num_neighbors=15, max_iterations=10,
                         metric="convex", qp_solver="quadprog", in_mem_dist_matrix=True):
        if qp_solver != B200_SOLVER:
            return orig_perform(contig_fasta, features_csv, operating_dir, num_neighbors, max_iterations, metric,
                                qp_solver, in_mem_dist_matrix)
        import pandas as pd

        multi = {} if devices is None else dict(devices=devices)
        csv = perform_clustering(contig_fasta, features_csv, operating_dir, num_neighbors, max_iterations, metric,
                                 qp_solver, in_mem_dist_matrix, **multi)
        bin_dump_dir = Path(operating_dir) / "bins"
        bin_dump_dir.mkdir(parents=True, exist_ok=True)
        logger.info(">> Writing binned FASTA files...")
        mod.dump_bins(pd.read_csv(csv), contig_fasta, bin_dump_dir)  # cli/clustering.py:94-97
        return csv

    perform_dispatch.__wrapped__ = orig_perform
    mod.perform_clustering = perform_dispatch
