"""Stage times of one clustering stage sharded over N members of a device group (chb_group_*) in ONE process.

For every workload (BASELINE configs #3 = 100k / C = 100 / k = 10 and #4 = 1M / C = 500 / k = 5, as in bench.py's
`scale_workloads`) and every N:
  * stage_ms: the stage of bench.py's scale_workloads -- features resident (uploaded once and replicated to the members with
    chb_group_replicate_features), each stage = set_labels + build_distance_matrix on every member + the guess exchange + the
    iterations to convergence (GroupEngine, comm=None); N = 1 is one context running chb_fit.  The L2 is overwritten (a
    256 MB write on every device) before each repetition; host clock around a stage that ends in device synchronisations;
    median of --reps repetitions after one warm-up;
  * all_max_ms: chb_group_all_max over one whole-iteration window (U labels) from CUDA events on every member's stream,
    averaged over 50 back-to-back calls (the max over members);
  * e2e_ms: fit_cluster(devices=...) end to end from pinned host buffers (N = 1: devices=None), median of --reps after a
    warm-up -- feature upload and replication, label set-up, permutation draws, label read-back included;
  * the labels of every N against N = 1 (and the stage's labels against the end-to-end call's).
Members are devices 0..N-1; with --same-device every member runs on device 0 (the protocol's overhead without the extra
GPUs, for machines with one GPU).  N larger than the number of visible GPUs is skipped otherwise.  One JSON per workload
under --out (default profiles/), with the card name and power limit read in the same process.

usage: python tools/device_group.py [--workloads 100k,1m] [--members 1,2,4,8] [--same-device] [--reps 3] [--out profiles]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

from chbin_b200 import capi, clustering, synth

MAX_ITERATIONS = 10


def card():
    q = "index,name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return {"query": q, "value": out or "nvidia-smi unavailable"}


class GroupStage:
    """The stage of bench.py's scale_workloads over N members (N = 1: one context, chb_fit)."""

    def __init__(self, X, bins, C, k, devices):
        self.bins, self.C, self.k = bins, C, k
        self.U = int(np.sum(bins == -1))
        self.perms = clustering.draw_permutations(bins, MAX_ITERATIONS, seed=0)
        self.ctxs = [capi.Context(dv) for dv in devices]
        self.group = capi.Group(self.ctxs) if len(devices) > 1 else None
        self.ctxs[0].set_features(X)
        if self.group is not None:
            self.group.replicate_features(0)
        for c in self.ctxs:
            c.set_params(k, "convex")
            c.synchronize()

    def run(self):
        n = len(self.ctxs)
        for i, c in enumerate(self.ctxs):
            u0, u1 = clustering.owned_slots(self.U, i, n)
            c.set_labels(self.bins, self.C, u0, u1)
            c.build_distance_matrix(True)
        if self.group is None:
            labels, iters, _, _ = self.ctxs[0].fit(self.perms, MAX_ITERATIONS)
            return labels, iters
        eng = clustering.GroupEngine(self.group, self.U)
        clustering.exchange_guess(eng, eng, self.U)
        iters = 0
        for it in range(MAX_ITERATIONS):
            nxt = self.perms[it + 1] if it + 1 < MAX_ITERATIONS else None
            nch, _ = clustering.run_iteration(eng, self.perms[it], None, next_perm=nxt)
            iters += 1
            if nch == 0:
                break
        return self.ctxs[0].get_labels(), iters

    def all_max_ms(self, torch, calls=50):
        """Mean time of one chb_group_all_max over U labels, CUDA events on every member's stream (max over members)."""
        streams = [torch.cuda.Stream(device=c.device) for c in self.ctxs]
        for c, s in zip(self.ctxs, streams):
            c.set_stream(s.cuda_stream)
        for m in range(len(self.ctxs)):
            self.group.buffer(m, self.U)
        self.group.all_max(self.U)  # warm-up
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in streams]
        for (e0, _), s in zip(ev, streams):
            e0.record(s)
        for _ in range(calls):
            self.group.all_max(self.U)
        for (_, e1), s in zip(ev, streams):
            e1.record(s)
        for s in streams:
            s.synchronize()
        for c in self.ctxs:
            c.set_stream(capi.OWN_STREAM)
        return max(e0.elapsed_time(e1) for e0, e1 in ev) / calls

    def close(self):
        if self.group is not None:
            self.group.close()
        for c in self.ctxs:
            c.close()


def measure(torch, name, members, same_device, reps):
    X, bins, truth, cfg = synth.make_config(name, seed=0)
    C, k = cfg["C"], cfg["k"]
    U = int(np.sum(bins == -1))
    ngpu = torch.cuda.device_count()
    flush = [torch.empty(64 << 20, dtype=torch.float32, device=f"cuda:{i}") for i in range(ngpu)]  # 256 MB per device
    Xp = torch.from_numpy(X).pin_memory().numpy()  # page-locked host features for the end-to-end calls
    out = {"workload": name, "n": cfg["n"], "d": X.shape[1], "C": C, "k": k, "U": U, "reps": reps,
           "members_on_device_0": same_device, "visible_gpus": ngpu, "shard_min_pairs": clustering.SHARD_MIN_PAIRS,
           "l2_policy": "256 MB written on every device before each repetition, outside the timed stage", "by_members": {}}
    ref_labels = None
    for N in members:
        if not same_device and N > ngpu:
            out["by_members"][str(N)] = {"skipped": f"{ngpu} GPU(s) visible"}
            continue
        devices = [0] * N if same_device else list(range(N))
        row = {"devices": devices}
        S = GroupStage(X, bins, C, k, devices)
        try:
            S.run()  # warm-up: every shape of the stage
            times = []
            for _ in range(reps):
                for f in flush:
                    f.zero_()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                labels, iters = S.run()
                times.append((time.perf_counter() - t0) * 1e3)
            row.update(stage_ms=statistics.median(times), stage_ms_all=times, iterations=iters,
                       labels_equal_ground_truth=bool(np.array_equal(labels, truth)))
            if S.group is not None:
                row["all_max_ms_per_call_U_labels"] = S.all_max_ms(torch)
        finally:
            S.close()
        if ref_labels is None:
            ref_labels = labels
        row["labels_equal_n1"] = bool(np.array_equal(labels, ref_labels))
        e2e = []
        for r in range(reps + 1):
            np.random.seed(0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            got, info = clustering.fit_cluster(Xp, C, bins, None, k, MAX_ITERATIONS, return_info=True,
                                               devices=devices if N > 1 else None)
            if r:
                e2e.append((time.perf_counter() - t0) * 1e3)
        row.update(e2e_ms=statistics.median(e2e), e2e_ms_all=e2e, e2e_sharded=bool(info.get("sharded", False)),
                   e2e_labels_equal_stage=bool(np.array_equal(got, labels)))
        clustering.shutdown()
        out["by_members"][str(N)] = row
        print(json.dumps({name: {N: {k_: v for k_, v in row.items() if not k_.endswith("_all")}}}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default="100k,1m")
    ap.add_argument("--members", default="1,2,4,8")
    ap.add_argument("--same-device", action="store_true")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    os.makedirs(args.out, exist_ok=True)
    members = [int(m) for m in args.members.split(",") if m]
    for name in [w for w in args.workloads.split(",") if w]:
        res = measure(torch, name, members, args.same_device, args.reps)
        res["card"] = card()
        tag = "_same_device" if args.same_device else ""
        path = os.path.join(args.out, f"device_group_{name}{tag}.json")
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
        print(f"wrote {path}", flush=True)


if __name__ == "__main__":
    main()
