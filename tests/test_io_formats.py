"""
CPU tests of the data formats either side of the hot path (SURVEY.md 8(f) rows 2-3) and of the caller's host logic
(cli/clustering.py:47-92): features.csv ingest, the binary side-car of the samples block, majority vote and the
binning-assignment.csv writer -- pinned against the reference's own perform_clustering output (tests/golden/make_golden.py
section 5).  fit_cluster is replaced by the CPU oracle here; the GPU run of the same file is tests/test_gpu_io.py.
"""
import os
import time
import types

import numpy as np
import pandas as pd
import pytest

import chbin_b200
import oracle
from chbin_b200 import clustering, distance_cache


@pytest.fixture(scope="module")
def G(golden_dir):
    return np.load(os.path.join(golden_dir, "reference_golden.npz"))


def _oracle_fit(samples, num_clusters, initial_bins, num_neighbors, max_iterations, metric, qp_solver, in_mem_dist_matrix):
    perms = oracle.draw_permutations(initial_bins, max_iterations, seed=None)  # consumes the global RNG like the reference
    return oracle.fit_cluster(np.ascontiguousarray(samples), int(num_clusters), initial_bins, None, num_neighbors, max_iterations,
                              metric=metric, perms=perms)


@pytest.fixture
def features_csv(G, tmp_path):
    p = tmp_path / "features.csv"
    p.write_bytes(G["pc_features_csv"].tobytes())
    return p


def test_sidecar_round_trip_and_staleness(features_csv):
    ref = pd.read_csv(features_csv).drop(distance_cache.META_COLUMNS, axis=1).values
    assert distance_cache.load_samples(features_csv) is None
    sc = distance_cache.write_features_sidecar(features_csv)
    assert sc.name == "features.csv.samples.npy"
    got = distance_cache.load_samples(features_csv, len(ref))
    assert got.dtype == np.float64 and np.array_equal(got, ref)  # bit-identical to the pandas parse
    assert distance_cache.load_samples(features_csv, len(ref) + 1) is None  # row-count mismatch: ignored
    os.utime(features_csv, (time.time() + 10, time.time() + 10))  # CSV newer than the side-car: ignored
    assert distance_cache.load_samples(features_csv, len(ref)) is None


@pytest.mark.parametrize("sidecar", [False, True])
def test_perform_clustering_host_logic_matches_reference_output(G, features_csv, tmp_path, monkeypatch, sidecar):
    k, iters = (int(v) for v in G["pc_params"])
    monkeypatch.setattr(clustering, "fit_cluster",
                        lambda samples, num_clusters, initial_bins, num_neighbors, max_iterations, metric, qp_solver,
                        in_mem_dist_matrix: _oracle_fit(samples, num_clusters, initial_bins, num_neighbors, max_iterations,
                                                        metric, qp_solver, in_mem_dist_matrix))
    if sidecar:
        distance_cache.write_features_sidecar(features_csv)
    np.random.seed(0)
    out = clustering.perform_clustering(None, features_csv, tmp_path / "out", k, iters, "convex", "b200", True)
    assert out.name == "binning-assignment.csv"
    assert out.read_bytes() == G["pc_assignment_csv"].tobytes()


def test_perform_clustering_rejects_unassigned(G, features_csv, tmp_path, monkeypatch):
    monkeypatch.setattr(clustering, "fit_cluster", lambda **kw: np.asarray(kw["initial_bins"]))  # leaves -1 labels behind
    with pytest.raises(ValueError, match="un-clustered"):  # cli/clustering.py:79-80
        clustering.perform_clustering(None, features_csv, tmp_path / "out", 5, 2)


def test_install_dispatches_on_solver(tmp_path, monkeypatch):
    calls = []
    fake = types.SimpleNamespace(
        perform_clustering=lambda *a, **k: calls.append(("reference", a[6] if len(a) > 6 else k.get("qp_solver"))) or "ref.csv",
        dump_bins=lambda df, fasta, d: calls.append(("dump_bins", str(d))))
    csv = tmp_path / "binning-assignment.csv"
    pd.DataFrame({"CONTIG_NAME": ["a"], "BIN": [0]}).to_csv(csv, index=False)
    monkeypatch.setattr(clustering, "perform_clustering", lambda *a, **k: calls.append(("b200", a[6])) or csv)
    clustering.install(fake)
    assert fake.perform_clustering("c.fa", "f.csv", tmp_path, 5, 2, "convex", "quadprog", True) == "ref.csv"
    assert fake.perform_clustering("c.fa", "f.csv", tmp_path, 5, 2, "convex", "b200", True) == csv
    assert calls == [("reference", "quadprog"), ("b200", "b200"), ("dump_bins", str(tmp_path / "bins"))]


def test_install_on_the_real_reference_module_through_the_ini_route(G, features_csv, tmp_path, monkeypatch):
    """install() applied to the reference's OWN ch_bin.cli.clustering (imported unmodified from /root/reference; Biopython
    and the two solver packages are stand-ins, oracle/ref_shim.py) and driven the way ch_bin/ch_bin.py:30 drives it:
    run_perform_clustering(contigs, features.csv, dir, USER_CONFIG["PARAMETERS"]) (cli/clustering.py:102-127) with
    `AlgoQpSolver = b200` in the INI.  The engine behind fit_cluster is the CPU oracle here (no GPU in this container); what
    is under test is the dispatch: the b200 value reaches this package, every other value reaches the untouched original,
    and both write the same binning-assignment.csv bytes as the reference's own run (tests/golden, section 5)."""
    from configparser import ConfigParser

    from oracle import ref_shim

    if not ref_shim.available():
        pytest.skip(f"no reference project tree at {ref_shim.REFERENCE_ROOT} (CHB_REFERENCE_ROOT)")
    mod = ref_shim.load_cli_clustering()
    original = mod.perform_clustering
    seen = []

    def oracle_fit(**kw):
        seen.append(kw["qp_solver"])
        return _oracle_fit(kw["samples"], kw["num_clusters"], kw["initial_bins"], kw["num_neighbors"], kw["max_iterations"],
                           kw["metric"], kw["qp_solver"], kw["in_mem_dist_matrix"])

    monkeypatch.setattr(clustering, "fit_cluster", oracle_fit)
    k, iters = (int(v) for v in G["pc_params"])
    cfg = ConfigParser()
    cfg.read(os.path.join(ref_shim.REFERENCE_ROOT, "config", "default.ini"))
    cfg["PARAMETERS"]["AlgoNumNeighbors"] = str(k)
    cfg["PARAMETERS"]["AlgoMaxIterations"] = str(iters)
    try:
        clustering.install(mod)
        assert mod.perform_clustering is not original and mod.perform_clustering.__wrapped__ is original
        cfg["PARAMETERS"]["AlgoQpSolver"] = "b200"
        np.random.seed(0)  # ch_bin/ch_bin.py:22
        out = mod.run_perform_clustering(tmp_path / "contigs.fasta", features_csv, tmp_path / "b200", cfg["PARAMETERS"])
        assert seen == ["b200"]
        assert out == tmp_path / "b200" / "binning-assignment.csv"
        assert out.read_bytes() == G["pc_assignment_csv"].tobytes()
        assert (tmp_path / "b200" / "bins").is_dir()  # step 05 was handed back to the reference's dump_bins
        # any other solver value: the reference's own perform_clustering, untouched (quadprog stand-in behind it)
        cfg["PARAMETERS"]["AlgoQpSolver"] = "quadprog"
        np.random.seed(0)
        out2 = mod.run_perform_clustering(tmp_path / "contigs.fasta", features_csv, tmp_path / "ref", cfg["PARAMETERS"])
        assert seen == ["b200"]
        assert out2.read_bytes() == G["pc_assignment_csv"].tobytes()
        with pytest.raises(NotImplementedError):  # solve_qp.py:132 still answers for unknown values
            cfg["PARAMETERS"]["AlgoQpSolver"] = "gurobi"
            mod.run_perform_clustering(tmp_path / "contigs.fasta", features_csv, tmp_path / "bad", cfg["PARAMETERS"])
    finally:
        mod.perform_clustering = original
