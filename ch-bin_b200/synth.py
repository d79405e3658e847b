"""
Synthetic contig feature sets with the shape of CH-Bin's `features.csv` (SURVEY.md 8(d)).

k-mer part: normalised 4-mer profile, 136 canonical dims, Dirichlet around a per-genome centroid
(what seq2vec emits, /root/reference/ch_bin/core/features/kmer_count.py:65-107).
coverage part: per-sample abundance with the reference's normalisation
(/root/reference/ch_bin/core/features/coverage.py:36-40): every column divided by its sum, then -- only when
there is more than one sample -- every row divided by its row sum.
Seeds: the first `n_seed` contigs of every genome carry that genome's bin id (a long single-copy-marker contig
split into 10 kb pieces, /root/reference/ch_bin/core/features/preprocess.py:38-67); all others are -1.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np

KMER_DIMS = 136


def normalise_coverages(cov: np.ndarray) -> np.ndarray:
    """coverage.py:36-40 on a dense (n, S) array."""
    cov = np.asarray(cov, dtype=np.float64)
    cov = cov / cov.sum(axis=0, keepdims=True)
    if cov.shape[1] > 1:
        cov = cov / cov.sum(axis=1, keepdims=True)
    return cov


def make_contig_features(
    n: int,
    num_genomes: int,
    num_cov_samples: int = 1,
    n_seed: int = 50,
    seed: int = 0,
    concentration: float = 4000.0,
    coverage_column: Optional[np.ndarray] = None,
    kmer_dims: int = KMER_DIMS,
) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Returns (samples (n, kmer_dims+S) float64 C-contiguous, initial_bins (n,) int64 with -1 = unassigned,
    true_genome (n,) int64).  kmer_dims: width of the k-mer profile, 136 canonical 4-mers by default; 512 gives
    5-mer-like profiles."""
    rng = np.random.default_rng(seed)
    C, S = int(num_genomes), int(num_cov_samples)
    centroids = rng.dirichlet(np.full(int(kmer_dims), 8.0), size=C)
    truth = rng.integers(0, C, size=n)
    # every genome needs at least n_seed members
    need = np.repeat(np.arange(C), n_seed)
    if len(need) > n:
        raise ValueError("n too small for num_genomes * n_seed")
    truth[: len(need)] = need
    rng.shuffle(truth)
    kmers = np.empty((n, int(kmer_dims)))
    for c in range(C):
        idx = np.where(truth == c)[0]
        if len(idx):
            kmers[idx] = rng.dirichlet(concentration * centroids[c], size=len(idx))
    abundance = rng.lognormal(3.0, 1.0, size=(C, S))
    cov = abundance[truth] * np.abs(1.0 + 0.05 * rng.standard_normal((n, S)))
    if coverage_column is not None:
        col = np.asarray(coverage_column, dtype=np.float64).reshape(-1)
        cov[:, 0] = col[:n] if len(col) >= n else np.resize(col, n)
    cov = normalise_coverages(cov)
    samples = np.ascontiguousarray(np.concatenate([kmers, cov], axis=1))
    bins = np.full(n, -1, dtype=np.int64)
    for c in range(C):
        idx = np.where(truth == c)[0][:n_seed]
        bins[idx] = c
    return samples, bins, truth.astype(np.int64)


CONFIGS = {
    # name: (n, C, S, n_seed, k)  -- SURVEY.md 8(d) "Config -> concrete inputs"
    "five-genomes-like": dict(n=735, C=5, S=1, n_seed=98, k=5),
    "20k": dict(n=20_000, C=50, S=1, n_seed=50, k=5),
    "100k": dict(n=100_000, C=100, S=10, n_seed=50, k=10),
    "200k": dict(n=200_000, C=100, S=1, n_seed=50, k=5),
    "1m": dict(n=1_000_000, C=500, S=20, n_seed=100, k=5),
}


def make_config(name: str, seed: int = 0, n: Optional[int] = None):
    cfg = dict(CONFIGS[name])
    if n is not None:
        cfg["n"] = int(n)
    samples, bins, truth = make_contig_features(cfg["n"], cfg["C"], cfg["S"], cfg["n_seed"], seed=seed)
    return samples, bins, truth, cfg
