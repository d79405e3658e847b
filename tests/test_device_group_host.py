"""CPU: the device group's host-side rules -- argument checks of fit_cluster(devices=...) that come before any device work,
the ctypes binding of the chb_group_* entry points, and the group's MAX kernel in the built library."""
import subprocess

import numpy as np
import pytest

import chbin_b200
from chbin_b200 import capi, clustering, synth


@pytest.fixture(scope="module")
def stage():
    X, bins, _ = synth.make_contig_features(100, 2, 1, 5)
    return X, bins


def test_devices_must_name_a_device(stage):
    X, bins = stage
    with pytest.raises(ValueError, match="at least one"):
        chbin_b200.fit_cluster(X, 2, bins, None, 5, 2, devices=[])


def test_devices_and_device_are_exclusive(stage):
    X, bins = stage
    with pytest.raises(ValueError, match="either device or devices"):
        chbin_b200.fit_cluster(X, 2, bins, None, 5, 2, device=0, devices=[0, 0])


def test_devices_refused_under_torch_distributed(stage, monkeypatch):
    X, bins = stage
    monkeypatch.setattr(clustering, "_dist_state", lambda: (object(), 1, 4))
    with pytest.raises(ValueError, match="torch.distributed"):
        chbin_b200.fit_cluster(X, 2, bins, None, 5, 2, devices=[0, 1])


def test_install_passes_devices_through(tmp_path, monkeypatch):
    """install(module, devices=...) hands the device list to every b200 stage of the reference's CLI module; the default
    leaves the call exactly as before."""
    import types

    calls = []

    def fake_perform(*args, **kw):
        calls.append(kw)
        csv = tmp_path / "binning-assignment.csv"
        csv.write_text("CONTIG_NAME,BIN\n")
        return csv

    monkeypatch.setattr(clustering, "perform_clustering", fake_perform)
    for devices, want in ((None, {}), ([0, 1], {"devices": [0, 1]})):
        mod = types.SimpleNamespace(perform_clustering=lambda *a, **k: None, dump_bins=lambda *a: None)
        chbin_b200.install(mod, devices=devices)
        mod.perform_clustering(None, tmp_path / "f.csv", tmp_path, qp_solver="b200")
        assert calls[-1] == want


def test_group_entry_points_bound():
    lib = capi.load()
    for name in ("chb_group_create", "chb_group_destroy", "chb_group_buffer", "chb_group_all_max", "chb_group_replicate_features"):
        assert name in capi.EXPORTED_SYMBOLS and getattr(lib, name).argtypes is not None


def test_group_max_kernel_in_library():
    out = subprocess.run(["cuobjdump", "-sass", capi.library_path()], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    assert "group_max_kernel" in out.stdout
