"""
chbin_b200 -- B200-native (sm_100a) implementation of CH-Bin's clustering hot path.

The directory is named `ch-bin_b200` (not importable as written); `import chbin_b200` works through the loader
`chbin_b200.py` at the repository root, which registers this directory as the package `chbin_b200`.

Public surface (mirrors /root/reference/ch_bin/core/clustering/algorithm.py and ch_bin/cli/clustering.py):
    fit_cluster, perform_clustering, install, B200_SOLVER
    capi.Context        thin ctypes wrapper over the C-ABI (include/chbin_b200.h)
    distance_cache      on-disk distance matrix (.npy, reference format) and the features.csv side-car
    features            coverage normalisation + [k-mer | coverage] merge on the device (coverage.py, cli/features.py)
    synth               synthetic contig feature sets of the BASELINE configs
"""
from . import build, capi, distance_cache, features, synth  # noqa: F401
from .clustering import (  # noqa: F401
    B200_SOLVER,
    GpuEngine,
    GroupEngine,
    TorchComm,
    draw_permutations,
    exchange_guess,
    fit_cluster,
    install,
    owned_slots,
    perform_clustering,
    run_iteration,
    shutdown,
)

__all__ = [
    "B200_SOLVER", "GpuEngine", "GroupEngine", "TorchComm", "draw_permutations", "exchange_guess", "fit_cluster", "install", "owned_slots", "perform_clustering",
    "run_iteration", "shutdown", "build", "capi", "distance_cache", "features", "synth",
]
