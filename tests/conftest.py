import hashlib
import os
import sys

import numpy as np
import torch
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def c1():
    """C1 fixture: the reference's bundled peptide test (164 x 54) + its golden artefacts."""
    return dict(np.load(os.path.join(GOLDEN, "peptide_c1.npz"), allow_pickle=False))


KMEANS_CASES = {
    # name: (n, d, k, rounded to the 1e-4 CSV grid?)
    "blobs_d2_k5": (3000, 2, 5, False),
    "blobs_d4_k10_grid": (5000, 4, 10, True),
    "blobs_d10_k40": (20000, 10, 40, False),
    "uniform_d3_k7_grid": (4000, 3, 7, True),
}


def kmeans_inputs():
    """The seeded inputs the reference clustered for kmeans_ref.npz: ``{name}_X`` and ``{name}_init``
    (its first k rows) for every case of KMEANS_CASES, then ``opt_X`` for the k-means++ and k-search
    cases, all drawn in this order from one generator."""
    rng = np.random.default_rng(7)
    out = {}
    for name, (n, d, k, grid) in KMEANS_CASES.items():
        if name.startswith("blobs"):
            cent = rng.uniform(-0.9, 0.9, size=(k, d))
            X = cent[rng.integers(0, k, size=n)] + 0.08 * rng.standard_normal((n, d))
        else:
            X = rng.uniform(-1, 1, size=(n, d))
        if grid:
            X = np.round(X, 4)
        X = np.ascontiguousarray(X, dtype=np.float64)
        out[f"{name}_X"], out[f"{name}_init"] = X, X[:k].copy()
    cent = rng.uniform(-0.8, 0.8, size=(5, 3))
    out["opt_X"] = np.ascontiguousarray(
        np.round(cent[rng.integers(0, 5, size=6000)] + 0.09 * rng.standard_normal((6000, 3)), 4))
    return out


def sha256(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="session")
def kmeans_ref():
    """The reference's KMeans outputs (kmeans_ref.npz) with the inputs they were computed from.
    The inputs are regenerated from their seed rather than stored (the largest is 1.6 MB of
    incompressible float64); the file keeps each input's SHA-256, so inputs that differ from the
    ones the reference saw fail here instead of being compared with its outputs."""
    ref = dict(np.load(os.path.join(GOLDEN, "kmeans_ref.npz"), allow_pickle=False))
    for key, a in kmeans_inputs().items():
        if key.endswith("_X"):
            assert sha256(a) == str(ref[f"{key}_sha256"]), f"regenerated {key} differs from the reference's input"
        ref[key] = a
    return ref


def synth_features(n, f, seed=0, n_slow=6, dtype=np.float32):
    """Small CPU twin of the benchmark generator (SURVEY 8d): AR(1) slow modes mixed
    into F features with per-feature scale/offset (|mean| >> std)."""
    rng = np.random.default_rng(seed)
    T = 400.0 * 2.0 ** (-np.arange(n_slow))
    rho = np.exp(-1.0 / T)
    z = np.empty((n, n_slow))
    z[0] = rng.standard_normal(n_slow)
    eps = rng.standard_normal((n, n_slow))
    for t in range(1, n):
        z[t] = rho * z[t - 1] + np.sqrt(1 - rho ** 2) * eps[t]
    A = np.random.default_rng(seed + 1).standard_normal((n_slow, f))
    s = rng.uniform(0.05, 0.5, size=f)
    m = rng.uniform(0.5, 3.0, size=f)
    X = (z @ A + 0.5 * rng.standard_normal((n, f))) * s + m
    return np.ascontiguousarray(X.astype(dtype))


# ---- CPU stand-ins for the DeepTICA kernels (host-logic and gloo tests) -------------------------
def cpu_ticacov_sums(f, g, w=None, wl=None):
    """CPU stand-in for ops.ticacov_sums (the kernel's output layout, dcg.h)."""
    f64, g64 = f.double(), g.double()
    B, d = f.shape
    w64 = torch.ones(B, dtype=torch.float64) if w is None else w.double()
    wl64 = torch.ones(B, dtype=torch.float64) if wl is None else wl.double()
    out = torch.cat([w64.sum().reshape(1), wl64.sum().reshape(1), (w64[:, None] * f64).sum(0),
                     ((w64[:, None] * f64).T @ f64).reshape(-1), ((wl64[:, None] * f64).T @ g64).reshape(-1),
                     (wl64[:, None] * f64).sum(0), (wl64[:, None] * g64).sum(0)])
    o = 2 + d
    return {"flat": out, "sw": out[0], "swl": out[1], "swf": out[2:o],
            "sff": out[o:o + d * d].view(d, d), "sfg": out[o + d * d:o + 2 * d * d].view(d, d),
            "slf": out[o + 2 * d * d:o + 2 * d * d + d], "slg": out[o + 2 * d * d + d:]}


def cpu_ticaloss(sums, d, reg, n_eig=0):
    """CPU stand-in for ops.ticaloss (dcg_ticaloss_f64): loss, eigenvalues and the gradients with
    respect to the symmetric C0 / C_tau from the raw sums."""
    sw, swl = sums[0], sums[1]
    o = 2 + d
    swf = sums[2:o]; sff = sums[o:o + d * d].view(d, d); sfg = sums[o + d * d:o + 2 * d * d].view(d, d)
    slf = sums[o + 2 * d * d:o + 2 * d * d + d]; slg = sums[o + 2 * d * d + d:]
    mu, nu, xi = swf / sw, slg / swl, slf / swl
    C0 = sff / sw - torch.outer(mu, mu); C0 = 0.5 * (C0 + C0.T)
    Ct = sfg / swl - torch.outer(mu, nu) - torch.outer(xi, mu) + torch.outer(mu, mu); Ct = 0.5 * (Ct + Ct.T)
    L = torch.linalg.cholesky(C0 + reg * torch.eye(d, dtype=torch.float64))
    Li = torch.linalg.inv(L)
    A = Li @ Ct @ Li.T
    ev, U = torch.linalg.eigh(0.5 * (A + A.T))
    ev, U = ev.flip(0), U.flip(1)
    W = Li.T @ U
    used = n_eig if 0 < n_eig < d else d
    G0 = sum(2.0 * ev[r] ** 2 * torch.outer(W[:, r], W[:, r]) for r in range(used))
    Gt = sum(-2.0 * ev[r] * torch.outer(W[:, r], W[:, r]) for r in range(used))
    return {"loss": -(ev[:used] ** 2).sum(), "status": torch.zeros(()), "sw": sw, "swl": swl, "evals": ev,
            "mu": mu, "G0": G0, "Gt": Gt}


