#!/usr/bin/env python
"""
bench.py -- headline benchmark of the B200 clustering hot path (BASELINE.json: "point-to-hull QP distances/sec
(k=5, d~137) and clustering-stage wall time").

A STEP is one complete clustering stage on one synthetic contig set: distance structure build + every assignment
iteration until the reference's stop rule fires (cli/clustering.py:56-76 of the reference).  Work is counted in
REFERENCE-EQUIVALENT QPs: sum over executed iterations of U*C (one (query, bin) pair = kNN gather + QP + residual
norm).  Speculative re-solves the GPU path performs on top of that are NOT counted.

  value : QPs/s with the feature matrix already resident in HBM when the timed region starts.
  e2e   : the same metric through the public API chbin_b200.fit_cluster() with HOST (pinned) buffers -- H2D of the
          features / labels / permutations and D2H of the final labels all inside the timed region (the library context
          of the device is created once per process and reused, like a BLAS handle).  `e2e_pageable_f_order` repeats
          it from the reference's own boundary layout: a pageable, F-ordered `samples` array.
  roofline     : the dominant kernel of the timed region, timed live with CUDA events on the launch stream.
  cpu_baseline : the oracle port (oracle/*.c) on the host cores, bounded sample, rank 0 at N=1 only.

`--impl reference` times the reference's CPU algorithm (the oracle port: /root/reference is pure Python + two
absent third-party solvers and cannot travel to the GPU box) on all host threads, on a bounded sample.

`--dump-outputs DIR` writes what the timed path returned in its last step, the final labels, as DIR/labels.npy (float64).
The workload and the permutations are seeded, so two builds run with the same arguments can be compared label for label.

N > 1 (torchrun): queries are sharded over ranks, the per-round label exchange is an NCCL all-reduce; the workload is
the same total problem (strong scaling).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MAX_ITERATIONS = 10


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="20k")
    ap.add_argument("--n", type=int, default=None, help="override the number of contigs of the workload")
    ap.add_argument("--window", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-qp-isolated", action="store_true")
    ap.add_argument("--scale-workloads", default="100k,1m",
                    help="other BASELINE workloads timed briefly at this N (stage ms in `scale_workloads`); '' to skip")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the labels of the last timed step as DIR/labels.npy (float64) to compare two builds")
    return ap.parse_args()


def workload(args):
    from chbin_b200 import synth

    X, bins, truth, cfg = synth.make_config(args.workload, seed=0, n=args.n)
    U = int(np.sum(bins == -1))
    return X, bins, cfg, U


def flops_per_qp(k, d):
    return k * (k + 1) * d + 4 * k * d + 3 * d + 2 * k ** 3  # SURVEY.md 8(d) F(k,d)


def bytes_per_qp(k, d, C):
    return 8 * k * d + 4 * k + 8 + 8 * d / C  # SURVEY.md 8(d) B(k,d)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe).  The timed region of this
    benchmark is short (tens of milliseconds), so the primary sampler polls NVML in-process every few milliseconds;
    `nvidia-smi --query-gpu=... -lms` is the fallback when the NVML bindings are missing."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0, period_s=0.004):
        self.rows, self.proc, self.gpu, self.period = [], None, gpu_index, period_s
        self.nv, self.handle, self.thread, self.stop_flag = None, None, None, threading.Event()
        self.sm, self.mx, self.reasons = [], [], set()

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.gpu
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu])
                except Exception:
                    idx = self.gpu
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            try:
                self.mx.append(float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)))
            except Exception:
                pass
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        nv = self.nv
        bits = {}
        for nm, attr in (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
                         ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap")):
            v = getattr(nv, attr, None)
            if v is None:
                v = getattr(nv, attr.replace("ClocksEventReason", "ClocksThrottleReason"), None)
            if v is not None:
                bits[nm] = int(v)
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                if get_reasons is not None:
                    r = int(get_reasons(self.handle))
                    for nm, b in bits.items():
                        if r & b:
                            self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(self.period)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nv is not None:
            self.stop_flag.set()
            self.thread.join(timeout=1.0)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                    "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for nm, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


# ----------------------------------------------------------------------------------------------------------
def cpu_sample(X, bins, cfg, seconds, threads, return_labels=False):
    """Oracle port on `threads` host threads over a bounded prefix of iteration 1 (rows computed on the fly)."""
    import oracle

    C, k = cfg["C"], cfg["k"]
    perms = oracle.draw_permutations(bins, 1, seed=0)
    U = perms.shape[1]
    probe = min(U, 256)
    t0 = time.perf_counter()
    oracle.fit_cluster(X, C, bins, None, k, 1, perms=perms, threads=threads, max_steps=probe)
    per_step = (time.perf_counter() - t0) / probe
    steps = int(max(probe, min(U, seconds / max(per_step, 1e-9))))
    t0 = time.perf_counter()
    labels, info = oracle.fit_cluster(X, C, bins, None, k, 1, perms=perms, threads=threads, max_steps=steps, return_info=True)
    dt = time.perf_counter() - t0
    if return_labels:
        return info["qps"] / dt, steps, dt, labels, perms[0]
    return info["qps"] / dt, steps, dt


def cpu_extras(X, bins, cfg, seconds=3.0):
    """BASELINE.md section 3 beside the all-threads port: the port on ONE thread (QP/s per core), scipy's cdist (B3) on a
    bounded block of rows, and what the image offers of the reference's own solvers."""
    out = {}
    try:
        v, steps, dt = cpu_sample(X, bins, cfg, seconds, 1)
        out["single_thread"] = {"value": v, "unit": "QP/s", "cores": 1, "kind": "port",
                                "sample": f"first {steps} sequential steps of iteration 1 ({dt:.1f} s)"}
    except Exception as e:  # noqa: BLE001
        out["single_thread"] = {"error": repr(e)}
    try:
        from scipy.spatial.distance import cdist

        rows = max(64, min(len(X), int(2.5e8 / (len(X) * X.shape[1]))))
        t0 = time.perf_counter()
        cdist(X[:rows], X, "euclidean")
        dt = time.perf_counter() - t0
        out["b3_cdist"] = {"value": rows * len(X) / dt, "unit": "pairs/s", "cores": 1, "kind": "reference (scipy)",
                           "sample": f"cdist of the first {rows} rows against all {len(X)} (distance_matrix.py:41), {dt:.2f} s"}
    except Exception as e:  # noqa: BLE001
        out["b3_cdist"] = {"error": repr(e)}
    for mod in ("quadprog", "cvxopt"):
        try:
            __import__(mod)
            out[mod] = "importable (not timed: the reference flow around it needs /root/reference)"
        except Exception:
            out[mod] = "unavailable in image"
    p = os.path.join(ROOT, "profiles", "r2_baseline_b1_b3_container.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            out["b1_reference_verbatim"] = dict(j["b1_reference_verbatim"], where="build container (the reference tree does not "
                                                "travel to the GPU box), oracle/baseline_b1.py", solver=j.get("quadprog"), file="profiles/r2_baseline_b1_b3_container.json")
        except Exception:
            pass
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    X, bins, cfg, U = workload(args)
    threads = os.cpu_count() or 1
    per_step_seconds = max(2.0, min(args.cpu_seconds, 150.0 / max(args.steps + args.warmup, 1)))
    vals, steps_used = [], 0
    for i in range(args.warmup + args.steps):
        v, steps_used, dt, labels, _ = cpu_sample(X, bins, cfg, per_step_seconds, threads, return_labels=True)
        if i >= args.warmup:
            vals.append((v, dt))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, labels=labels)
    qps = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([dt for _, dt in vals]) * 1e3)
    sample = (f"first {steps_used} sequential steps of iteration 1 ({steps_used * cfg['C']} QPs) of the {args.workload} workload, "
              f"distance rows recomputed on the fly, OpenMP over rows/bins")
    line = {
        "impl": "reference", "metric": "point-to-hull QP distances/sec", "value": qps, "unit": "QP/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(args, cfg, U),
        "cpu_baseline": {"value": qps, "unit": "QP/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": qps, "unit": "QP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference = CPU oracle port (GI restatement); quadprog/cvxopt and the Python reference are not installable offline",
    }
    _emit(line)


def config_dict(args, cfg, U):
    return {"workload": f"synthetic {args.workload}: n={cfg['n']} contigs, d={136 + cfg['S']} (136-dim 4-mer + {cfg['S']} coverage), "
                        f"C={cfg['C']} bins, n_seed={cfg['n_seed']}, k={cfg['k']}, U={U}, max_iterations={MAX_ITERATIONS}",
            "n": cfg["n"], "d": 136 + cfg["S"], "C": cfg["C"], "k": cfg["k"], "U": U,
            "in_mem_dist_matrix": True, "l2_policy": "L2 flushed between steps (256 MB memset outside the timed brackets)",
            "window": args.window}


# ----------------------------------------------------------------------------------------------------------
class StageRunner:
    """One resident feature matrix in one library context; run() = one clustering stage (label set-up, distance structure,
    every iteration to the reference's stop rule) -- through chb_fit on one GPU, through the round protocol + NCCL
    all-reduce when the query slots are sharded over ranks."""

    def __init__(self, torch, dist, rank, world, local_rank, stream, X, bins, cfg, window):
        from chbin_b200 import capi, clustering

        self.torch, self.dist, self.rank, self.world, self.clustering = torch, dist, rank, world, clustering
        self.bins, self.C, self.k = bins, cfg["C"], cfg["k"]
        self.U = int(np.sum(bins == -1))
        self.perms = clustering.draw_permutations(bins, MAX_ITERATIONS, seed=0)  # the host RNG contract (algorithm.py:45)
        self.ctx = capi.Context(local_rank)
        self.ctx.set_stream(stream.cuda_stream)
        dev = torch.device("cuda", local_rank)
        n, d = X.shape
        # the library's own rule (clustering.SHARD_MIN_PAIRS): a stage too small to pay for the collectives is not sharded --
        # every rank runs all of it (identical labels, no communication); `value` is then the N = 1 figure at every N
        self.replicated = world > 1 and not clustering.sharding_pays(self.U, self.C, world)
        if self.replicated:
            world = 1
        if world > 1:
            # SURVEY 8(e): the feature matrix is uploaded by rank 0 only and replicated with ONE NCCL broadcast over NVLink
            Xd = torch.empty((n, d), dtype=torch.float64, device=dev)
            if rank == 0:
                Xd.copy_(torch.from_numpy(X))
            dist.broadcast(Xd, src=0)
        else:
            Xd = torch.from_numpy(X).to(dev)
        self.ctx.set_features_dev(Xd.data_ptr(), n, d)
        del Xd
        self.ctx.set_params(self.k, "convex")
        self.ctx.set_window(window)
        self.u0, self.u1 = clustering.owned_slots(self.U, rank if world > 1 else 0, world)
        self.world = world
        self.engine = self.comm = None
        self.local_rank, self.stream = local_rank, stream

    def run(self):
        ctx = self.ctx
        ctx.set_labels(self.bins, self.C, self.u0, self.u1)
        ctx.build_distance_matrix(True)
        if self.world == 1:
            labels, iters, conv, changed = ctx.fit(self.perms, MAX_ITERATIONS)
            return labels, iters
        if self.engine is None:
            self.engine = self.clustering.GpuEngine(ctx, self.local_rank, self.stream)
            self.comm = self.clustering.TorchComm()
        self.clustering.exchange_guess(self.engine, self.comm, self.U)  # every rank guesses for its own slots only (enqueued)
        ctx.iteration_prefetch(self.perms[0])  # side stream; the host-side staging of the upload overlaps the set-up kernels
        iters = 0
        with self.engine.stream_context():
            for it in range(MAX_ITERATIONS):
                nxt = self.perms[it + 1] if it + 1 < MAX_ITERATIONS else None
                nch, _ = self.clustering.run_iteration(self.engine, self.perms[it], self.comm, next_perm=nxt)
                iters += 1
                if nch == 0:
                    break
        return ctx.get_labels(), iters

    def timed(self, steps, flush, barrier, stream):
        """K stages, each bracketed by CUDA events on the launch stream, L2 flushed in between; returns total ms (max over
        ranks), iterations executed and the labels of the last stage."""
        torch = self.torch
        events, total_iters, labels = [], 0, None
        barrier()
        for _ in range(steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            labels, iters = self.run()
            e1.record(stream)
            events.append((e0, e1))
            total_iters += iters
        barrier()
        ms = float(sum(a.elapsed_time(b) for a, b in events))
        t = torch.tensor([ms], dtype=torch.float64, device=flush.device)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item()), total_iters, labels

    def close(self):
        self.ctx.close()


def run_b200(args):
    import torch

    import chbin_b200
    from chbin_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout to the one JSON line
        import datetime

        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=300))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(dev)  # the library's kernels, torch events and NCCL collectives all run on this stream
    torch.cuda.set_stream(stream)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    X, bins, cfg, U = workload(args)
    n, d = X.shape
    C, k = cfg["C"], cfg["k"]
    # L2 policy: a 256 MB memset (2x the 126 MB L2) runs between steps, outside the per-step event brackets, so that no
    # step starts with the previous step's feature rows or candidate lists in cache
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    # ---------------- value arm: features resident in HBM, one context reused ----------------
    R = StageRunner(torch, dist, rank, world, local_rank, stream, X, bins, cfg, args.window)
    ctx = R.ctx
    for _ in range(args.warmup):
        R.run()
    # pass A (the headline): per-kernel event timers OFF, nothing but the stage itself between the step's two events
    ctx.enable_timers(False)
    ctx.reset_timers()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    elapsed_ms, total_iters, labels_v = R.timed(args.steps, flush, barrier, stream)
    clocks = sampler.stop() if rank == 0 else None
    tmA = ctx.timers()
    # pass B (explains it): the same K steps again with a CUDA-event pair around every timed kernel launch -> live durations
    # for the roofline records; its own step time is reported next to the headline
    ctx.enable_timers(True)
    ctx.reset_timers()
    elapsed_ms_b, _, _ = R.timed(args.steps, flush, barrier, stream)
    tm = ctx.timers()
    qps_ref_total = total_iters * U * C
    value = qps_ref_total / (elapsed_ms * 1e-3)

    # iteration-1 labels of the device, for the oracle check below
    lab1 = None
    if world == 1:
        ctx.set_labels(bins, C, 0, -1)
        ctx.build_distance_matrix(True)
        lab1, _ = ctx.fit_iteration(R.perms[0])
    fp64_peak = ctx.measure_fp64_tflops() if rank == 0 else 0.0
    l2_gbs = ctx.measure_l2_gbs() if rank == 0 else 0.0
    qp_iso = qp_isolated(ctx, X, bins, cfg) if (rank == 0 and world == 1 and not args.no_qp_isolated) else None
    R.close()  # the end-to-end arm below builds its own context through the public API: release this one's HBM first

    # ---------------- e2e arm: public API, host buffers, H2D of features/labels and D2H of the labels inside ----------------
    def e2e_arm(Xh, bh, steps):
        iters = 0
        for _ in range(max(1, min(args.warmup, 2))):
            np.random.seed(0)
            chbin_b200.fit_cluster(Xh, C, bh, None, k, MAX_ITERATIONS, device=local_rank, window=args.window)
        barrier()
        secs, lab = 0.0, None
        for _ in range(steps):
            flush.zero_()
            torch.cuda.synchronize(dev)
            np.random.seed(0)
            t0 = time.perf_counter()
            lab, info = chbin_b200.fit_cluster(Xh, C, bh, None, k, MAX_ITERATIONS, device=local_rank, window=args.window,
                                               return_info=True)
            secs += time.perf_counter() - t0
            iters += info["iterations"]
        barrier()
        t = torch.tensor([secs], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), iters, lab

    Xp = torch.empty((n, d), dtype=torch.float64, pin_memory=True)
    Xp.copy_(torch.from_numpy(X))
    bp = torch.empty((n,), dtype=torch.int64, pin_memory=True)
    bp.copy_(torch.from_numpy(bins))
    e2e_s, e2e_iters, lab_e = e2e_arm(Xp.numpy(), bp.numpy(), args.steps)
    e2e_value = e2e_iters * U * C / e2e_s
    same = bool(np.array_equal(lab_e, labels_v))
    # the reference's own boundary (SURVEY 8b): `samples` is DataFrame.values of one float block -- a PAGEABLE, F-ORDERED
    # (n, d) array -- and `initial_bins` a pageable int64 copy
    Xf = np.asfortranarray(X)
    pg_s, pg_iters, lab_pg = e2e_arm(Xf, bins.copy(), args.steps)
    e2e_pageable = {"value": pg_iters * U * C / pg_s, "unit": "QP/s", "ms_per_step": pg_s * 1e3 / args.steps,
                    "buffers": "pageable, F-ordered float64 samples (DataFrame.values, cli/clustering.py:53) + pageable int64 bins; "
                               "transposed on the device",
                    "labels_equal_value_arm": bool(np.array_equal(lab_pg, labels_v))}
    del Xp, Xf

    # ---------------- the other BASELINE workloads, one short measurement each (scaling record) ----------------
    scale = {}
    for name in [w for w in args.scale_workloads.split(",") if w and w != args.workload]:
        try:
            scale[name] = scale_workload(torch, dist, rank, world, local_rank, stream, flush, barrier, name, args.window)
        except Exception as e:  # noqa: BLE001
            scale[name] = {"error": repr(e)[:300]}

    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, labels=labels_v)
        line = report(args, cfg, X, bins, U, world, elapsed_ms, elapsed_ms_b, total_iters, tmA, tm, fp64_peak, l2_gbs, clocks, value,
                      qps_ref_total, e2e_value, e2e_s, e2e_iters, same, e2e_pageable, scale, lab1, labels_v, R.perms, qp_iso, torch)
        _emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def scale_workload(torch, dist, rank, world, local_rank, stream, flush, barrier, name, window, steps=2, warmup=1):
    """Stage time of another BASELINE workload (config #3: 100k / k = 10, config #4: 1M / C = 500) at this N, features
    resident, so that every `--gpus N` line carries the sizes BASELINE.json asks to scale beside the 20k headline."""
    from chbin_b200 import synth

    X, bins, truth, cfg = synth.make_config(name, seed=0)
    R = StageRunner(torch, dist, rank, world, local_rank, stream, X, bins, cfg, window)
    try:
        for _ in range(warmup):
            R.run()
        R.ctx.enable_timers(False)
        R.ctx.reset_timers()
        ms, iters, labels = R.timed(steps, flush, barrier, stream)
        tm = R.ctx.timers()
        U = R.U
        out = {"n": cfg["n"], "d": X.shape[1], "C": cfg["C"], "k": cfg["k"], "U": U, "steps": steps,
               "stage_ms": ms / steps, "iterations_per_stage": iters / steps,
               "value_qps": iters * U * cfg["C"] / (ms * 1e-3), "qps_solved_per_stage_this_rank": tm["qps_solved"] / steps,
               "rounds_per_stage": tm["rounds"] / steps, "labels_equal_ground_truth": bool(np.array_equal(labels, truth))}
        if rank == 0:
            try:  # a seeded sample of positions of iteration-1-equivalent state against the position-parallel oracle
                import oracle

                if iters / steps == 2:  # converged after one changing iteration: the final labels ARE iteration 1's result
                    pos = np.sort(np.random.default_rng(5).choice(U, min(U, 1024), replace=False)).astype(np.int64)
                    res = oracle.verify_iteration(X, cfg["C"], bins, labels, R.perms[0], cfg["k"], positions=pos, threads=os.cpu_count() or 1)
                    out["oracle_sampled_positions"] = int(len(pos))
                    out["oracle_mismatches"] = int(res["mismatches"])
            except Exception as e:  # noqa: BLE001
                out["oracle_error"] = repr(e)[:200]
        return out
    finally:
        R.close()


def qp_isolated(ctx, X, bins, cfg):
    """The QP kernel on a FULL batch, isolated (north_star: 'QP kernel as a fraction of the FP64 roofline'): every
    (query, bin) pair of the workload with fixed, precomputed neighbour lists (chb_knn_per_bin on the generator's labels),
    timed by the library's CUDA-event pair around the kernel launch."""
    from chbin_b200 import synth

    C, k = cfg["C"], cfg["k"]
    _, _, truth = synth.make_contig_features(cfg["n"], C, cfg["S"], cfg["n_seed"], seed=0)
    queries = np.where(bins == -1)[0][:20000].astype(np.int64)
    ctx.set_labels(bins, C, 0, -1)
    ctx.build_distance_matrix(True)
    idx, m = ctx.knn_per_bin(truth, queries)
    best = None
    for _ in range(3):
        ctx.reset_timers()
        dist, status = ctx.hull_distance_batch(queries, idx, m)
        t = ctx.timers()
        if best is None or t["ms_qp"] < best:
            best = t["ms_qp"]
    return {"pairs": int(dist.size), "ms": best, "qps_per_s": dist.size / (best * 1e-3)}


def report(args, cfg, X, bins, U, world, elapsed_ms, elapsed_ms_b, total_iters, tmA, tm, fp64_peak, l2_gbs, clocks, value,
           qps_ref_total, e2e_value, e2e_s, e2e_iters, same, e2e_pageable, scale, lab1, labels_v, perms, qp_iso, torch):
    n, d = X.shape
    C, k = cfg["C"], cfg["k"]
    hbm_peak, hbm_src = measured_peaks()
    l2_bytes = int(torch.cuda.get_device_properties(0).L2_cache_size)
    ms = {"distance": tm["ms_distance"], "gram": tm["ms_gram"], "knn": tm["ms_knn"], "qp": tm["ms_qp"], "commit": tm["ms_commit"]}
    ln = {"distance": tm["launches_distance"], "gram": tm["launches_gram"], "knn": tm["launches_knn"],
          "qp": tm["launches_qp"], "commit": tm["launches_commit"]}
    traffic_all = {}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            traffic_all = json.load(open(tp))
        except Exception:
            traffic_all = {}
    try:
        tf32_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"]) / 2.0
        tf32_src = "MEASURED_PEAKS.json bf16_tflops / 2 (TF32 runs at half the bf16 rate)"
    except Exception:
        tf32_peak, tf32_src = 1590.0 / 2.0, "fallback (B200_PROFILING.md bf16 figure / 2)"
    # L2 -> SM fabric ceiling: the documented LTS throughput cap (B300_MICROARCH.md: ~6300 B/cycle full chip, same L2 design)
    # at the SM clock sampled during the run; the live gather microbenchmark (chb_measure_l2_gbs) is reported beside it -- it
    # is a LOWER bound of the ceiling (the QP kernel itself gathers faster than it)
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    l2_cap_gbs = max(6300.0 * sm_mhz * 1e6 / 1e9, l2_gbs)
    x_bytes = n * ((d + 1) // 2 * 2) * 8
    x_in_l2 = x_bytes < 0.5 * l2_bytes
    ai = flops_per_qp(k, d) / bytes_per_qp(k, d, C)

    def qp_ceilings():
        """min over the ceilings that APPLY (SURVEY 8d): the FP64 pipe always; the neighbour-row gather through the L2 fabric
        while the feature matrix is L2-resident, through HBM once it is not."""
        c = {"fp64": fp64_peak}
        if x_in_l2:
            c["l2_gather"] = ai * l2_cap_gbs / 1e3
        else:
            c["hbm"] = ai * hbm_peak / 1e3
        bind = min(c, key=lambda kk: c[kk])
        return c, bind

    stages = {}
    if ln["gram"]:
        # fused tcgen05 Gram + per-bin selection (distance mode 2): TF32 3-term split, K = 3 * dp8 per 128x128 tile; tiles are
        # counted by the MMA-issuing warps (gram_tiles) and must equal the planner's count (gram_tiles_planned)
        dp8 = (d + 7) // 8 * 8
        fl = tm["gram_tiles"] * 2.0 * 128 * 128 * 3 * dp8
        fl_alg = tm["gram_tiles"] * 2.0 * 128 * 128 * d
        t = ms["gram"] * 1e-3
        stages["gram"] = {"kernel": "gram_select_kernel", "bound": "tensor", "achieved": fl / t / 1e12, "peak": tf32_peak,
                          "unit": "TFLOP/s", "ms_total": ms["gram"], "launches": ln["gram"], "flops_per_launch": fl / ln["gram"],
                          "tiles_128x128": tm["gram_tiles"], "tiles_planned": tm["gram_tiles_planned"], "peak_source": tf32_src,
                          "achieved_algorithmic": fl_alg / t / 1e12, "frac_algorithmic": fl_alg / t / 1e12 / tf32_peak,
                          "note": "achieved/frac count the executed MMA work (3-term TF32 split, d padded to a multiple of 8); "
                                  "*_algorithmic count SURVEY 8(d)'s 2*d flop per (query, column)"}
    if ln["knn"]:
        if ln["gram"]:
            # re-rank: per surviving (query, bin) pair reads the two kept half-lists (keys + indices) and writes k indices;
            # algorithmic bytes against the L2 gather bandwidth (the lists were just written by the fused kernel)
            KR = 8 if k + 3 <= 8 else 16
            b = tm["qps_solved"] * (2 * KR * 8 + 4 * k + 8.0)
            stages["knn"] = {"kernel": "rerank_kernel", "bound": "l2", "achieved": b / (ms["knn"] * 1e-3) / 1e9, "peak": l2_cap_gbs,
                             "unit": "GB/s", "ms_total": ms["knn"], "launches": ln["knn"], "bytes_per_launch": b / ln["knn"],
                             "peak_source": "LTS throughput cap 6300 B/cycle x sampled SM clock (B300_MICROARCH.md)",
                             "note": "latency/issue-bound bookkeeping kernel: a few KB per surviving pair; bytes counted for the pairs "
                                     "whose neighbour set changed (a lower bound of the pairs re-ranked)"}
        else:
            b = tm["rows_scanned"] * n * 4.0  # kNN scan: one row of FP32 candidate values (4n bytes) per item
            stages["knn"] = {"kernel": "knn_scan_kernel", "bound": "hbm", "achieved": b / (ms["knn"] * 1e-3) / 1e9, "peak": hbm_peak,
                             "unit": "GB/s", "ms_total": ms["knn"], "launches": ln["knn"], "bytes_per_launch": b / ln["knn"],
                             "peak_source": hbm_src}
    qp_name = ("qp_small_kernel" if k <= 5 else "qp_mid_kernel" if k <= 10 else
               "gram_dmma_kernel + qp_lane_solve_kernel" if k <= 24 else "qp_kernel")
    ceil, bind = qp_ceilings()
    if ln["qp"]:
        f = tm["qps_solved"] * flops_per_qp(k, d)
        ach = f / (ms["qp"] * 1e-3) / 1e12
        stages["qp"] = {"kernel": qp_name, "bound": bind, "achieved": ach, "peak": ceil[bind], "unit": "TFLOP/s",
                        "ms_total": ms["qp"], "launches": ln["qp"], "flops_per_launch": f / ln["qp"],
                        "qps_solved": tm["qps_solved"], "qps_per_s": tm["qps_solved"] / (ms["qp"] * 1e-3),
                        "ceilings_tflops": ceil, "fp64_frac": ach / fp64_peak if fp64_peak else None,
                        "features_l2_resident": x_in_l2, "peak_source": "fp64: chb_measure_fp64_tflops (live DFMA microbenchmark); l2_gather: AI x LTS cap 6300 B/cycle x "
                        "sampled SM clock (B300_MICROARCH.md); hbm: " + hbm_src,
                        "note": "algorithmic flops F(k,d) per QP (SURVEY 8d) over the small post-pruning batches of this workload "
                                "(launch-latency dominated); the full-batch rate is in qp_isolated"}
    if ln["distance"]:
        stages["distance"] = {"kernel": "gram_tc_kernel", "bound": "tensor", "achieved": None, "peak": tf32_peak,
                              "unit": "TFLOP/s", "ms_total": ms["distance"], "launches": ln["distance"], "peak_source": tf32_src}
    for s in stages.values():
        s["frac"] = (s["achieved"] / s["peak"]) if (s["peak"] and s["achieved"] is not None) else None
        s["share_of_step"] = s["ms_total"] / elapsed_ms_b
        s["avg_launch_ms"] = s["ms_total"] / max(s["launches"], 1)
    dom = max(stages, key=lambda s: ms[s])  # the longest-running timed kernel family of the step
    roof = dict(stages[dom])
    roof["traffic"] = traffic_all.get(roof["kernel"])
    if qp_iso:
        f = qp_iso["pairs"] * flops_per_qp(k, d)
        ach = f / (qp_iso["ms"] * 1e-3) / 1e12
        qp_iso.update({"kernel": qp_name, "achieved": ach, "unit": "TFLOP/s", "ceilings_tflops": ceil, "bound": bind, "peak": ceil[bind],
                       "frac": ach / ceil[bind], "fp64_frac": ach / fp64_peak if fp64_peak else None,
                       "l2_cap_gbs": l2_cap_gbs, "l2_gather_microbench_gbs": l2_gbs, "gathered_gbs": qp_iso["pairs"] * bytes_per_qp(k, d, C) / (qp_iso["ms"] * 1e-3) / 1e9})

    cpu = oracle_check = None
    if not args.no_cpu_baseline:
        import oracle

        threads = os.cpu_count() or 1
        if world == 1:
            v, steps_used, dt, seq_labels, perm0 = cpu_sample(X, bins, cfg, args.cpu_seconds, threads, return_labels=True)
            cpu = {"value": v, "unit": "QP/s", "cores": threads, "kind": "port",
                   "sample": f"oracle port, first {steps_used} sequential steps of iteration 1 ({steps_used * C} QPs, {dt:.1f} s), "
                             f"rows recomputed on the fly"}
            cpu.update(cpu_extras(X, bins, cfg))
            head = perm0[:steps_used]
            oracle_check = {"kind": "sequential oracle, iteration 1", "positions": int(steps_used), "of": int(U),
                            "equal": bool(np.array_equal(seq_labels[head], lab1[head]))}
        # any N: the final labels against the position-parallel oracle on a seeded sample (valid when the run converged after
        # one changing iteration, i.e. the final labels are iteration 1's result)
        if total_iters / args.steps == 2:
            pos = np.sort(np.random.default_rng(11).choice(U, min(U, 2048), replace=False)).astype(np.int64)
            res = oracle.verify_iteration(X, C, bins, labels_v, perms[0], k, positions=pos, threads=threads)
            oracle_check = dict(oracle_check or {}, sampled_positions=int(len(pos)), sampled_mismatches=int(res["mismatches"]))
    labels_equal_oracle = None
    if oracle_check is not None:
        labels_equal_oracle = bool(oracle_check.get("equal", True) and oracle_check.get("sampled_mismatches", 0) == 0)

    kernel_ms = sum(ms.values())
    from chbin_b200 import clustering as _cl

    sharded = _cl.sharding_pays(U, cfg["C"], world)
    parallelism = {"parallelism": "1 GPU" if world == 1 else
                   (f"query slots sharded over {world} ranks (one label all-reduce per round)" if sharded else
                    f"{world} ranks, NOT sharded: {U * cfg['C']} (query, bin) pairs per stage is below the library's shard threshold "
                    f"({_cl.SHARD_MIN_PAIRS}); every rank runs the whole stage with no communication and returns identical labels -- "
                    "the sharded path at this N is measured in scale_workloads")}
    launches_step = (sum(tmA[f] for f in ("launches_distance", "launches_gram", "launches_knn", "launches_qp", "launches_commit",
                                           "launches_other"))) / args.steps
    return {
        "metric": "point-to-hull QP distances/sec", "value": value, "unit": "QP/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": dict(config_dict(args, cfg, U), **parallelism),
        "clustering_stage_ms": elapsed_ms / args.steps, "iterations_per_step": total_iters / args.steps,
        "qps_reference_per_step": qps_ref_total / args.steps,
        "qps_solved_per_step": tmA["qps_solved"] / args.steps, "rounds_per_step": tmA["rounds"] / args.steps,
        "labels_equal_oracle": labels_equal_oracle, "oracle_check": oracle_check,
        "roofline": roof, "stages": stages, "qp_isolated": qp_iso,
        "latency": {"ms_per_step": elapsed_ms / args.steps, "ms_per_step_with_stage_timers": elapsed_ms_b / args.steps,
                    "timed_kernels_ms_per_step": kernel_ms / args.steps, "launches_per_step": launches_step,
                    "launch_chain": "programmatic dependent launch (griddepcontrol) through the stage's kernels, no copy / memset "
                                    "nodes inside a round, row_ub on a side stream, next permutation prefetched"
                                    + (" [CHB_NO_PDL set: plain launches]" if os.environ.get("CHB_NO_PDL") else ""),
                    "note": "timed kernels = gram_select, rerank (+exact redo), QP, argmin/commit; the rest of the step is the "
                            "per-label-set and per-round set-up kernels and host round trips; the pass with stage timers records an "
                            "event pair around each timed kernel, which also breaks the programmatic launch chain there"},
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": "QP/s", "h2d_bytes_per_step": int(n * d * 8 + n * 8 + e2e_iters / args.steps * U * 8),
                "d2h_bytes_per_step": int(n * 8), "ms_per_step": e2e_s * 1e3 / args.steps,
                "buffers": "pinned, C-contiguous", "labels_equal_value_arm": same},
        "e2e_pageable_f_order": e2e_pageable,
        "scale_workloads": scale,
        "gpu_launches": int(launches_step * args.steps),
        "launches_by_stage": {"distance": tmA["launches_distance"], "gram": tmA["launches_gram"], "knn": tmA["launches_knn"],
                              "qp": tmA["launches_qp"], "commit": tmA["launches_commit"], "other": tmA["launches_other"]},
        "peaks": {"fp64_tflops": fp64_peak, "l2_cap_gbs": l2_cap_gbs, "l2_gather_microbench_gbs": l2_gbs, "hbm_gbs": hbm_peak, "tf32_tflops": tf32_peak, "l2_bytes": l2_bytes},
        "clocks": clocks,
    }


DUMP_MAX_ELEMENTS = 3_000_000  # per dump: values and their positions, 8 bytes each, stay below 64 MB


def dump_outputs(out_dir, **arrays):
    """Writes each array as out_dir/<name>.npy in float64 (exact for labels).  An array longer than its share of
    DUMP_MAX_ELEMENTS is replaced by a fixed, seeded sample of its elements in position order; the positions go to
    out_dir/<name>_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_MAX_ELEMENTS // len(arrays)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64).ravel()
        if a.size > cap:
            idx = np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))
            np.save(os.path.join(out_dir, f"{name}_index.npy"), idx.astype(np.float64))
            a = a[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def _emit(line: dict):
    """The ONE JSON line goes to the real stdout; everything else written to fd 1 meanwhile (NCCL's version banner,
    library chatter) was diverted to stderr by main()."""
    line["bench_wall_s"] = round(time.perf_counter() - _T_START, 1)  # this process, argument parsing to the line (all legs)
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1
_T_START = time.perf_counter()


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
