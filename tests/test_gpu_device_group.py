"""
GPU tests of the device group (include/chbin_b200.h, chb_group_*; clustering.GroupEngine): one process shards a stage over
several contexts with fit_cluster(devices=...) and merges their tentative labels with chb_group_all_max.  A device may appear
more than once (every member has a context of its own), so everything but the last test runs on one GPU.  Bars as
everywhere: labels, iteration counts and change counts identical to the sequential oracle, and the reference's RNG contract.
"""
import os

import numpy as np
import pytest

import chbin_b200
import oracle
from chbin_b200 import capi, clustering, synth

pytestmark = pytest.mark.gpu

THREADS = os.cpu_count() or 1


@pytest.fixture
def always_shard(monkeypatch):
    """Every stage with two or more devices is sharded, whatever its size."""
    monkeypatch.setattr(clustering, "SHARD_MIN_PAIRS", 0)


def _fit_same_as_oracle(X, C, bins, k, iters, devices, metric="convex", **kw):
    perms = oracle.draw_permutations(bins, iters, seed=0)
    ref, rinfo = oracle.fit_cluster(X, C, bins, None, k, iters, metric=metric, perms=perms, threads=THREADS, return_info=True)
    np.random.seed(0)
    got, info = chbin_b200.fit_cluster(X, C, bins, None, k, iters, metric, return_info=True, devices=devices, **kw)
    assert np.array_equal(got, ref)
    assert info["iterations"] == rinfo["iterations"] and list(info["changed"]) == list(rinfo["changed"])
    assert info["world"] == len(devices) and info["devices"] == list(devices)
    return info


class _Int32View:
    """__cuda_array_interface__ over a group buffer: lets torch fill and read device memory the library owns."""

    def __init__(self, ptr, count):
        self.__cuda_array_interface__ = {"shape": (count,), "typestr": "<i4", "data": (ptr, False), "version": 3}


@pytest.mark.parametrize("n_members", [2, 3])
@pytest.mark.parametrize("count", [3, 1001, 65536])
def test_all_max_merges_every_members_buffer(n_members, count):
    """chb_group_all_max: every member's buffer ends as the element-wise MAX of all of them, INT32_MIN (an un-owned
    position) included, for counts with and without a tail beyond the int4 loads."""
    import torch

    ctxs = [capi.Context(0) for _ in range(n_members)]
    g = capi.Group(ctxs)
    try:
        rng = np.random.default_rng(count + n_members)
        vals = rng.integers(-(2**31), 2**31 - 1, size=(n_members, count), dtype=np.int64).astype(np.int32)
        vals[:, ::5] = capi.UNOWNED
        views = [torch.as_tensor(_Int32View(g.buffer(m, count), count), device="cuda:0") for m in range(n_members)]
        for v, row in zip(views, vals):
            v.copy_(torch.from_numpy(row))
        torch.cuda.synchronize()
        g.all_max(count)
        for c in ctxs:
            c.synchronize()
        want = vals.max(axis=0)
        for v in views:
            assert np.array_equal(v.cpu().numpy(), want)
    finally:
        g.close()
        for c in ctxs:
            c.close()


def test_replicate_features_and_group_errors():
    """chb_group_replicate_features copies the root's matrix into every member; bad arguments are ValueErrors."""
    X, _, _ = synth.make_contig_features(500, 3, 4, 20, seed=2)
    ctxs = [capi.Context(0) for _ in range(3)]
    g = capi.Group(ctxs)
    try:
        ctxs[1].set_features(X)
        g.replicate_features(1)
        for c in ctxs:
            assert np.array_equal(c.get_features(), X)
        with pytest.raises(ValueError, match="out of range"):
            g.replicate_features(3)
        with pytest.raises(ValueError, match="no group buffer"):
            g.all_max(10)
        with pytest.raises(ValueError, match="same context"):
            capi.Group([ctxs[0], ctxs[0]])
    finally:
        g.close()
        for c in ctxs:
            c.close()


@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]])
def test_group_on_one_device_matches_sequential_oracle(always_shard, devices):
    """Overlapping bins (several repair rounds per iteration), sharded over members on one GPU: labels, iteration count and
    change counts == the oracle, and the global RNG ends where the reference leaves it (one draw per executed iteration)."""
    # genomes overlap (low Dirichlet concentration): all 10 iterations change labels, ~7 rounds each
    X, bins, _ = synth.make_contig_features(3000, 7, 1, 15, seed=5, concentration=60.0)
    info = _fit_same_as_oracle(X, 7, bins, 5, 10, devices)
    assert info["sharded"] and info["timers"]["rounds"] >= 3 * info["iterations"]
    U = int(np.sum(bins == -1))
    assert info["owned_slots"] == [clustering.owned_slots(U, i, len(devices)) for i in range(len(devices))]

    pts = np.where(bins == -1)[0]
    for max_iterations in (10, 2):
        np.random.seed(123)
        _, info = chbin_b200.fit_cluster(X, 7, bins, None, 5, max_iterations, return_info=True, devices=devices)
        after = np.random.random()
        np.random.seed(123)
        for _ in range(info["iterations"]):
            np.random.permutation(pts)
        assert after == np.random.random()


def test_group_with_fewer_queries_than_members(always_shard):
    """Two queries over three members: the first member owns no slot at all."""
    X, bins, _ = synth.make_contig_features(400, 3, 1, 20, seed=4, concentration=200.0)
    bins = np.where(bins == -1, np.arange(len(bins)) % 3, bins)
    bins[[7, 311]] = -1
    info = _fit_same_as_oracle(X, 3, bins, 5, 5, [0, 0, 0])
    assert info["sharded"] and info["owned_slots"][0] == (0, 0)


GROUP_PATHS = [
    # id, (n, C, S, n_seed, concentration), k, metric, env -- one per distance path the rounds can take
    ("resident-k5", (2500, 6, 1, 30, 300.0), 5, "convex", {}),
    ("resident-k10", (2500, 6, 1, 30, 300.0), 10, "convex", {}),
    ("streamed-wide", (1500, 6, 64, 30, 300.0), 5, "convex", {"CHB_WIDE_FUSED_MIN_PAIRS": "0"}),
    ("exact-k32", (1500, 4, 1, 45, 250.0), 32, "convex", {}),
    ("mode1-d1112", (1200, 5, 600, 30, 300.0), 5, "convex", {}),
    ("affine", (2000, 6, 1, 30, 300.0), 5, "affine", {}),
]


@pytest.mark.parametrize("case", GROUP_PATHS, ids=[c[0] for c in GROUP_PATHS])
def test_group_runs_every_distance_path(always_shard, monkeypatch, case):
    name, (n, C, S, n_seed, conc), k, metric, env = case
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    kd = 512 if name == "mode1-d1112" else 136
    X, bins, _ = synth.make_contig_features(n, C, S, n_seed, seed=31 + k, concentration=conc, kmer_dims=kd)
    info = _fit_same_as_oracle(X, C, bins, k, 5, [0, 0], metric=metric)
    assert info["sharded"]
    t = info["timers"]
    if name == "mode1-d1112":
        assert X.shape[1] == 1112 and t["launches_gram"] == 0 and t["launches_knn"] > 0
    elif k <= 24:
        assert t["launches_gram"] > 0 and t["launches_distance"] == 0
    else:
        assert t["launches_gram"] == 0 and t["launches_distance"] == 0


def test_small_stage_runs_whole_on_the_first_device():
    """Below SHARD_MIN_PAIRS (20k contigs x 50 bins) the stage is not sharded: it runs whole on devices[0]."""
    X, bins, _, cfg = synth.make_config("20k")
    assert not clustering.sharding_pays(int(np.sum(bins == -1)), cfg["C"], 2)
    info = _fit_same_as_oracle(X, cfg["C"], bins, cfg["k"], 10, [0, 0])
    assert not info["sharded"]
    assert info["owned_slots"] == [(0, int(np.sum(bins == -1)))]


def test_devices_errors_leave_the_default_path_working(always_shard, monkeypatch):
    X, bins, _ = synth.make_contig_features(800, 4, 1, 20, seed=14, concentration=300.0)
    perms = oracle.draw_permutations(bins, 5, seed=0)
    ref = oracle.fit_cluster(X, 4, bins, None, 5, 5, perms=perms)

    def default_path_still_works():
        np.random.seed(0)
        assert np.array_equal(chbin_b200.fit_cluster(X, 4, bins, None, 5, 5), ref)

    with monkeypatch.context() as mp:  # a torch.distributed job of two ranks is already sharding the stage
        mp.setattr(clustering, "_dist_state", lambda: (object(), 0, 2))
        with pytest.raises(ValueError, match="torch.distributed"):
            chbin_b200.fit_cluster(X, 4, bins, None, 5, 5, devices=[0, 0])
    default_path_still_works()
    with pytest.raises(RuntimeError, match="out of range"):
        chbin_b200.fit_cluster(X, 4, bins, None, 5, 5, devices=[0, 1 << 20])
    default_path_still_works()
    np.random.seed(0)
    assert np.array_equal(chbin_b200.fit_cluster(X, 4, bins, None, 5, 5, devices=[0, 0]), ref)


# ------------------------------------------------------------------------------------------------------------------
def _all_devices():
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip(f"needs two or more GPUs, this machine has {n}")
    return list(range(n))


def _sample_positions(U, count, seed):
    rng = np.random.default_rng(seed)
    edge = np.concatenate([np.arange(min(256, U)), np.arange(max(U - 256, 0), U)])
    return np.unique(np.concatenate([edge, rng.choice(U, min(count, U), replace=False)])).astype(np.int64)


def _verify_first_iteration(name, devices, positions_count=None):
    X, bins, _, cfg = synth.make_config(name)
    C, k = cfg["C"], cfg["k"]
    perms = oracle.draw_permutations(bins, 1, seed=0)
    U = perms.shape[1]
    np.random.seed(0)
    lab1, info = chbin_b200.fit_cluster(X, C, bins, None, k, 1, return_info=True, devices=devices)
    assert info["sharded"]
    pos = None if positions_count is None else _sample_positions(U, positions_count, 7)
    res = oracle.verify_iteration(X, C, bins, lab1, perms[0], k, positions=pos, threads=THREADS)
    assert res["mismatches"] == 0, f"{name}: {res['mismatches']} positions differ from the oracle"
    return X, bins, C, k


def test_real_gpus_config3_and_config4(tmp_path):
    """Every GPU of the machine: config #3 iteration 1 at every position and the final labels of a single-GPU run; config #4
    on sampled positions; perform_clustering writes the same binning-assignment.csv bytes as on one GPU."""
    import pandas as pd

    devices = _all_devices()
    X, bins, C, k = _verify_first_iteration("100k", devices)
    np.random.seed(0)
    one = chbin_b200.fit_cluster(X, C, bins, None, k, 10)
    np.random.seed(0)
    assert np.array_equal(chbin_b200.fit_cluster(X, C, bins, None, k, 10, devices=devices), one)

    csv = tmp_path / "features.csv"
    df = pd.DataFrame(X)
    df.insert(0, "CLUSTER", bins)
    df.insert(0, "PARENT_NAME", [f"contig_{i // 3}" for i in range(len(X))])
    df.insert(0, "CONTIG_NAME", [f"sub_{i}" for i in range(len(X))])
    df.to_csv(csv, index=False)
    np.random.seed(0)
    single = chbin_b200.perform_clustering(None, csv, tmp_path / "one", k, 10).read_bytes()
    np.random.seed(0)
    multi = chbin_b200.perform_clustering(None, csv, tmp_path / "all", k, 10, devices=devices).read_bytes()
    assert multi == single

    _verify_first_iteration("1m", devices, positions_count=1500)
