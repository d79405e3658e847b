"""Stage times of distance mode 2 for feature vectors wider than 160, on both sides of WIDE_FUSED_MIN_PAIRS (api.cu).

For every workload the features are uploaded once (resident); each timed stage is set_labels + build_distance_matrix +
`--iterations` iterations (chb_fit_iteration), bracketed by CUDA events after a synchronise, with the L2 overwritten (a
256 MB write) before every repetition.  Paths: "fused" = the streamed fused kernel (CHB_WIDE_FUSED_MIN_PAIRS=0), "matrix" =
distance mode 1 (threshold above the stage's pair count) where its FP32 candidate matrix fits the device; each path runs in
a context of its own.  Also recorded: the device memory that context holds after the stage (cudaMemGetInfo before the
context was created and after the last repetition: features, operands, caches and scratch), the library's timers, and the
labels of iteration 1
checked against the position-parallel oracle (oracle/verify.c) on sampled positions, the first and last 256 included.
One JSON per run under --out (default profiles/), with the card name and power limit read in the same process.

usage: python tools/wide_features.py [--workloads crossover,20k,100k,200k,1m] [--out profiles]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

from chbin_b200 import capi, synth

# name: (n, C, S, kmer_dims, n_seed, k) -- d = kmer_dims + S
WORKLOADS = {
    "20k": (20_000, 50, 64, 136, 50, 5),
    "100k": (100_000, 100, 64, 136, 50, 10),
    "200k": (200_000, 100, 16, 512, 50, 5),
    "1m": (1_000_000, 500, 64, 136, 100, 5),
}
CROSSOVER_N = [300, 500, 700, 1_000, 1_500, 2_500, 4_000, 9_000]  # d = 200, k = 5; C = 4 below 1 500 contigs, 20 from there


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return {"query": q, "value": out or "nvidia-smi unavailable"}


def stage(torch, X, bins, C, k, perms, iterations, path, reps, flush):
    """(median ms over reps, device bytes the path's context holds, timers, labels after iteration 1) of one path."""
    os.environ["CHB_WIDE_FUSED_MIN_PAIRS"] = "0" if path == "fused" else str(2**62)
    torch.cuda.synchronize()
    free_base = torch.cuda.mem_get_info()[0]
    ctx = capi.Context(0)
    ctx.enable_timers(True)
    ctx.set_features(X)
    ctx.set_params(k, "convex")
    times, used, lab1, tm = [], 0, None, None
    for r in range(reps + 1):  # repetition 0 warms every shape up and is not timed
        ctx.set_distance_mode(2)
        ctx.synchronize()
        flush.zero_()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.reset_timers()
        e0.record()
        ctx.set_labels(bins, C)
        assert ctx.distance_path() == (2 if path == "fused" else 1)
        ctx.build_distance_matrix(path == "matrix")
        for it in range(iterations):
            lab, _ = ctx.fit_iteration(perms[it], want_labels=it == 0)
            if it == 0:
                lab1 = lab
        ctx.synchronize()
        e1.record()
        torch.cuda.synchronize()
        if r > 0:
            times.append(e0.elapsed_time(e1))
        used = max(used, free_base - torch.cuda.mem_get_info()[0])
        tm = ctx.timers()
    ctx.close()
    return float(np.median(times)), int(used), tm, lab1


def verify(X, C, bins, lab, perm, k, count, seed):
    import oracle

    U = len(perm)
    rng = np.random.default_rng(seed)
    pos = np.unique(np.concatenate([np.arange(min(256, U)), np.arange(max(U - 256, 0), U), rng.choice(U, min(count, U), replace=False)]))
    t0 = time.perf_counter()
    res = oracle.verify_iteration(X, C, bins, lab, perm, k, positions=pos.astype(np.int64), threads=os.cpu_count() or 1)
    return {"positions": int(len(pos)), "mismatches": int(res["mismatches"]), "seconds": round(time.perf_counter() - t0, 1)}


def run(torch, name, n, C, S, kd, n_seed, k, paths, iterations, reps, flush, check, out_dir, info):
    X, bins, _ = synth.make_contig_features(n, C, S, n_seed, seed=0, kmer_dims=kd)
    pts = np.where(bins == -1)[0]
    rng = np.random.default_rng(0)
    perms = np.stack([rng.permutation(pts) for _ in range(iterations)]).astype(np.int64)
    rec = dict(workload=name, n=n, d=int(X.shape[1]), C=C, k=k, n_own=int(len(pts)), owned_pairs=int(len(pts)) * n,
               iterations=iterations, repetitions=reps, l2="overwritten (256 MB) before every repetition", card=info, paths={})
    for path in paths:
        if path == "matrix" and 4.0 * len(pts) * ((n + 3) // 4 * 4) > 0.8 * torch.cuda.mem_get_info()[0]:
            rec["paths"][path] = "not measured: the FP32 candidate matrix does not fit the device"
            continue
        ms, used, tm, lab1 = stage(torch, X, bins, C, k, perms, iterations, path, reps, flush)
        entry = dict(stage_ms=round(ms, 3), ms_per_iteration=round(ms / iterations, 3), device_bytes_held_by_context=used,
                     timers={kk: (round(v, 3) if isinstance(v, float) else v) for kk, v in tm.items()})
        if check:
            entry["verify_iteration_1"] = verify(X, C, bins, lab1, perms[0], k, 2000, 1)
        rec["paths"][path] = entry
        print(name, path, json.dumps(entry), flush=True)
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, f"wide_features_{name}.json"), "w") as f:
        json.dump(rec, f, indent=1)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="crossover,20k,100k,200k,1m")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--iterations", type=int, default=2)
    ap.add_argument("--reps", type=int, default=2)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: these are GPU measurements")
    info = card()
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
    for w in args.workloads.split(","):
        if w == "crossover":
            for n in CROSSOVER_N:
                C, n_seed = (20, 20) if n >= 1_500 else (4, 15)
                run(torch, f"crossover_n{n}", n, C, 64, 136, n_seed, 5, ["fused", "matrix"], args.iterations, max(args.reps, 3),
                    flush, False, args.out, info)
        else:
            n, C, S, kd, n_seed, k = WORKLOADS[w]
            paths = ["fused"] if w == "1m" else ["fused", "matrix"]
            run(torch, w, n, C, S, kd, n_seed, k, paths, args.iterations, args.reps, flush, True, args.out, info)


if __name__ == "__main__":
    main()
