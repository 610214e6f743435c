"""The block-diagonal hTICA path (C3: 4950 features, 10 subspaces of 495 -> 5 each -> d = 10) on one GPU,
stage by stage and end to end, against float64.

Part A calls the eigen stage of ``linalg`` directly at the sizes hTICA gives it: the padded triangular inverse
against a long-double forward substitution, and the batched shift-and-invert solve (its cached CUDA graph of
round 0, the graph cache's eviction and the re-shift branches) on pencils whose spectra are known.
Part B runs ``HTICACalculator.compute_cv`` on the block path (block sums on the covariance engine, batched
level 1, block projection or its per-chunk fallback, level-2 sums, level-2 TICA) and checks every stage
against ``oracle.float64_device`` run with the calculator's own (mean, range).

Tolerances.  u = 2^-53.
  * Triangular inverse (Higham, Accuracy and Stability, 2nd ed., section 14.2): forward substitution gives
    |X L - I| <= gamma_F |X| |L|, so ||X - L^-1|| / ||L^-1|| <= gamma_F kappa(L); the block assembly adds
    products of the same kind once more: 2 F u kappa_inf(L).
  * Known pencils B = V^-T V^-1, C = V^-T diag(lam) V^-1 (cond V = 100, kappa(B) = 10^4).  Forming B and C
    rounds them by F u relative; through a definite pencil that moves an eigenvalue by at most
    (||dC|| + |lam| ||dB||) / lambda_min(B) <= 2 F u kappa(B) and a B-normalised eigenvector by that over the
    gap.  The solver stops when ||C x - theta B x|| <= 1e-12 ||C||_F ||x||; in the coordinates y = V^-1 x
    (where the pencil is diag(lam)) that is a residual of at most r = kappa(V)^2 1e-12 ||lam||_2, which bounds
    a Ritz value's error by r^2 / gap and the eigenvector's angle by r / gap, times kappa(V) back in x.
    The eigenvalue bound is the sum of the rounding and the quadratic term (~1e-9); the eigenvector bound is
    the sum of both linear terms (~1e-3 at F = 1000: the acceptance test, not the arithmetic, dominates).
  * Block sums: the exact engine rounds each value once, to the grid 2^-e of its column
    (test_cov_i8_exact.prep), where the float64 checker rounds fl32((x - c) / r); per value
    |z_dev - z_ref| <= delta_j = 2^-(e_j+1) / r_j + 2^-24 max|z_j|.  With the omitted d0 d0 digit product
    (|d0| <= 128) and the FP64 adds (test_cov_i8_exact.tau_factor) the entrywise bound is
        delta_i sum|z_j| + delta_j sum|z_i| + M delta_i delta_j + M 128^2 s_i s_j + tau M qmax_i qmax_j s_i s_j.
    The float engine (FP32 tensor-core accumulation) is held to the suite's 1e-5 of max |S|.
  * Level 1 and the weights: pushing a perturbation through an eigenproblem multiplies it, to first order and
    in the worst case, by kappa(C0) / gap.  For level 1 that is ~10^3 / 2.5e-3 on these blocks; for level 2,
    whose inputs are fifty projections of the same fourteen slow modes, kappa(C0_2) ~ 1e4 and the smallest gap
    among the d + 1 leading eigenvalues is ~4e-4 at C3, so the FP32 rounding of T1 (2^-24) plus the split-TF32
    projection (2^-22) alone allow 2 (2^-24 + 2^-22) kappa(C0_2) / gap_2 ~ 40: no bound on the columns of W
    follows from the arithmetic, and the single columns do move by ~1e-3 (also against the full-Gram path,
    whose level 2 is T1^T S T1 in FP64).  What is held to an eigenvalue tolerance is the lag-tau
    autocorrelation each column realises on the float64 data (``autocorrelations``): the eigenvalue is
    stationary in its eigenvector, so it moves only to second order, and a rotation inside a group of nearly
    equal eigenvalues leaves it alone.  The column errors are printed beside it.  The exact engine is held to
    the north-star 1e-5 of the largest.  The float engine's sums carry up to 1e-5 relative error themselves
    (a hundred times the exact engine's quantisation), which reaches the eigenvalues of both levels at the
    same order; it gets the 5e-5 the suite already gives this engine on centred features
    (test_gpu_parity.test_normalisation_modes_through_the_fused_kernels).
  * Normalised projections: the calculator's weights through the float64 projection, 1e-4 (north star).
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U53 = 2.0 ** -53


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from deep_cartograph_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


# ================================================================================================
# A. the eigen stage at the sizes hTICA uses
# ================================================================================================
TRI_FMAX = 1030


@pytest.fixture(scope="module")
def tri_ref():
    """L: Cholesky factor of a C0-like matrix (eigenvalues 1 .. 1e-4, kappa(L) ~ 1e4 in the inf-norm) and
    L^-1 by forward substitution in long double.  A leading F x F block of L is the Cholesky factor of the
    leading block of C, and its inverse is the leading block of L^-1: one reference serves every size."""
    g = np.random.default_rng(495)
    Q, _ = np.linalg.qr(g.standard_normal((TRI_FMAX, TRI_FMAX)))
    C = (Q * np.logspace(0, -4, TRI_FMAX)) @ Q.T
    L = np.linalg.cholesky(0.5 * (C + C.T))
    Ll = L.astype(np.longdouble)
    Xi = np.zeros((TRI_FMAX, TRI_FMAX), dtype=np.longdouble)
    for i in range(TRI_FMAX):                      # row i of L^-1 from the rows above it, all columns at once
        r = -(Ll[i, :i] @ Xi[:i, :i + 1])
        r[i] += 1
        Xi[i, :i + 1] = r / Ll[i, i]
    return L, Xi


@pytest.mark.parametrize("nb", [1, 3, 10])
@pytest.mark.parametrize("F", [256, 495, 496, 511, 512, 1000, 1001, 1023, 1030])
def test_tri_inv_lower_against_long_double(dev, tri_ref, F, nb):
    """4 vs 8 diagonal blocks, padded (495, 511, 1001, 1023, 1030) vs not, blocks of <= 128 rows on the
    hand-written kernel vs 129 (1030) on solve_triangular.  Batch member k is D_k L E_k with power-of-two
    diagonal scalings, so its inverse E_k^-1 L^-1 D_k^-1 is known exactly and members that were swapped or
    mixed would differ by the scalings."""
    from deep_cartograph_b200 import linalg
    L0, Xi = tri_ref
    L0 = L0[:F, :F]
    Li0 = Xi[:F, :F].astype(np.float64)
    g = np.random.default_rng(F * 10 + nb)
    Ls, refs = [], []
    for k in range(nb):
        dr = np.ldexp(1.0, g.integers(-2, 3, F)) if k else np.ones(F)
        dc = np.ldexp(1.0, g.integers(-2, 3, F)) if k else np.ones(F)
        Ls.append(dr[:, None] * L0 * dc[None, :])
        refs.append(Li0 / dc[:, None] / dr[None, :])
    R = linalg._tri_inv_lower(torch.from_numpy(np.stack(Ls)).to(dev))
    torch.cuda.synchronize()
    assert R.shape == (nb, F, F)
    assert bool((torch.triu(R, 1) == 0).all()), "strict upper triangle is not exactly zero"
    nblk = 8 if F >= 512 else 4
    Fp = -(-F // nblk) * nblk
    if Fp != F:
        # the assembly multiplies through the pad: it must be the inverse of an identity block, not inf / NaN
        # that only stays out of the F x F corner because 0 * finite = 0 in the products that touch it
        full = R._base
        assert full is not None and full.shape == (nb, Fp, Fp)
        assert bool(torch.isfinite(full).all())
        assert torch.equal(full[:, F:, F:], torch.eye(Fp - F, dtype=full.dtype, device=dev).expand(nb, -1, -1))
        assert bool((full[:, F:, :F] == 0).all())
    got = R.cpu().numpy()
    for k in range(nb):
        kappa = np.abs(Ls[k]).sum(1).max() * np.abs(refs[k]).sum(1).max()
        err = np.abs(got[k] - refs[k]).sum(1).max() / np.abs(refs[k]).sum(1).max()
        bound = 2 * F * U53 * kappa
        print(f"tri_inv F={F} nb={nb} k={k}: err {err:.2e} bound {bound:.2e}")
        assert err <= bound, (F, nb, k, err, bound)


def known_pencil(F, lead, g, bulk=(-0.2, 0.8), cond=100.0):
    """B = V^-T V^-1, C = V^-T diag(lam) V^-1 with cond(V) = ``cond``: C v = lam B v for every column v of V.
    lam = ``lead`` followed by F - len(lead) values uniform in ``bulk``."""
    Uo, _ = np.linalg.qr(g.standard_normal((F, F)))
    Wo, _ = np.linalg.qr(g.standard_normal((F, F)))
    s = np.logspace(0, -math.log10(cond), F)
    V = (Uo * s) @ Wo.T
    Vi = (Wo / s) @ Uo.T
    lam = np.concatenate([np.asarray(lead, dtype=np.float64), g.uniform(bulk[0], bulk[1], F - len(lead))])
    B = Vi.T @ Vi
    C = (Vi.T * lam) @ Vi
    return 0.5 * (B + B.T), 0.5 * (C + C.T), lam, V


def normalised(V):
    """Unit columns, first row non-negative (the rule _cholesky_eigh applies)."""
    V = V / np.linalg.norm(V, axis=0, keepdims=True)
    return V * np.where(V[0:1] < 0, -1.0, 1.0)


def pencil_bounds(F, lam, out, cond=100.0):
    """(eigenvalue bound, eigenvector bound) of the module docstring for the leading ``out`` pairs."""
    srt = np.sort(lam)[::-1]
    gap = min(np.min(-np.diff(srt[:out + 1])), 1.0)
    kB = cond ** 2
    r = kB * 1e-12 * np.linalg.norm(lam)
    return 2 * F * U53 * kB + r * r / gap, (2 * F * U53 * kB + r * cond) / gap


def check_pencils(ev, V, pencils, out, what):
    ev, V = ev.cpu().numpy(), V.cpu().numpy()
    if ev.ndim == 1:
        ev, V = ev[None], V[None]
    for k, (B, C, lam, Vt) in enumerate(pencils):
        F = B.shape[0]
        evb, vb = pencil_bounds(F, lam, out)
        ref = normalised(Vt[:, :out])
        e_ev = np.abs(ev[k] - lam[:out]).max()
        got = normalised(V[k])
        e_v = np.linalg.norm(got * np.sign((got * ref).sum(0)) - ref, axis=0).max()
        # the solver's own promise, in float64 here: every accepted pair has a residual <= 1e-12 ||C||_F ||x||
        res = np.linalg.norm(C @ got - (B @ got) * ev[k][None, :], axis=0).max() / np.linalg.norm(C)
        print(f"{what} pencil {k} F={F}: eigenvalues {e_ev:.2e} (bound {evb:.2e}), eigenvectors {e_v:.2e} "
              f"(bound {vb:.2e}), residual {res:.2e}")
        assert e_ev <= evb, (what, k, e_ev, evb)
        assert e_v <= vb, (what, k, e_v, vb)
        assert res <= 1e-12 + 4 * F * U53, (what, k, res)


LEAD5 = np.linspace(0.99, 0.9, 5)                 # gaps 2.25e-2
LEAD10 = np.linspace(0.99, 0.9, 10)               # gaps 1e-2


@pytest.mark.parametrize("graph", ["1", "0"])
@pytest.mark.parametrize("nb,F,out", [(10, 495, 5), (1, 1000, 10)])
def test_batched_shift_invert_on_known_pencils(dev, monkeypatch, graph, nb, F, out):
    """hTICA level 1 at C3 (10 blocks of 495 -> 5) and one pencil of F = 1000, with the round-0 CUDA graph
    and without it: both meet the same bounds, and the fast route answers."""
    from deep_cartograph_b200 import linalg
    monkeypatch.setenv("DCG_EIG_GRAPH", graph)
    g = np.random.default_rng(F + nb)
    pencils = [known_pencil(F, LEAD5 if out == 5 else LEAD10, g) for _ in range(nb)]
    B = torch.from_numpy(np.stack([p[0] for p in pencils])).to(dev)
    C = torch.from_numpy(np.stack([p[1] for p in pencils])).to(dev)
    if nb == 1:
        B, C = B[0], C[0]
    fast, dense = linalg.EIG_STATS["fast"], linalg.EIG_STATS["dense"]
    ev, V = linalg._cholesky_eigh(B, C, 0.0, out)
    assert linalg.EIG_STATS["fast"] == fast + nb and linalg.EIG_STATS["dense"] == dense, "the fast route did not run"
    if graph == "1":
        key = (nb, F, out, min(F, out + 8), dev.index, torch.float64)
        ent = linalg._ROUND0_GRAPHS.get(key)
        assert ent is not None and not ent["failed"] and "graph" in ent, "round 0 was not captured as a graph"
    check_pencils(ev, V, pencils, out, f"graph={graph}")


def test_round0_graph_replays_on_its_inputs_and_survives_eviction(dev, monkeypatch):
    """Two calls of one shape with different pencils each give their own answer, and the first call's results
    are not overwritten by the second replay.  Then more than _ROUND0_GRAPHS_MAX shapes evict the first
    graph; coming back to it captures it again and is still right."""
    from deep_cartograph_b200 import linalg
    monkeypatch.setenv("DCG_EIG_GRAPH", "1")
    out, F, nb = 5, 495, 10
    g = np.random.default_rng(7)

    def solve(pencils):
        B = torch.from_numpy(np.stack([p[0] for p in pencils])).to(dev)
        C = torch.from_numpy(np.stack([p[1] for p in pencils])).to(dev)
        got = linalg._shift_invert_topk(B, C, out)
        assert got is not None
        return got

    p1 = [known_pencil(F, LEAD5, g) for _ in range(nb)]
    p2 = [known_pencil(F, LEAD5 - 0.005, g) for _ in range(nb)]
    ev1, V1 = solve(p1)
    keep = (ev1.clone(), V1.clone())
    ev2, V2 = solve(p2)
    torch.cuda.synchronize()
    assert torch.equal(ev1, keep[0]) and torch.equal(V1, keep[1]), "the second replay changed the first results"
    check_pencils(ev1, V1, p1, out, "first call")
    check_pencils(ev2, V2, p2, out, "second call")

    # eviction: nine more shapes (F = 200, nb = 1..9), then the first shape again
    first = (nb, F, out, out + 8, dev.index, torch.float64)
    assert first in linalg._ROUND0_GRAPHS
    for k in range(1, 10):
        ps = [known_pencil(200, LEAD5, g, bulk=(-0.2, 0.6)) for _ in range(k)]
        check_pencils(*solve(ps), ps, out, f"eviction nb={k}")
        assert len(linalg._ROUND0_GRAPHS) <= linalg._ROUND0_GRAPHS_MAX
    assert first not in linalg._ROUND0_GRAPHS, "the oldest graph was not evicted"
    p3 = [known_pencil(F, LEAD5 + 0.003, g) for _ in range(nb)]
    check_pencils(*solve(p3), p3, out, "after eviction")
    assert not linalg._ROUND0_GRAPHS[first]["failed"]


def _record_factors(monkeypatch):
    """The shifts of the checked factorisations (the re-shift branches; round 0 uses an unchecked one)."""
    from deep_cartograph_b200 import linalg
    seen = []
    real = linalg._factor

    def spy(B, Ct, sig, check=True):
        if check:
            seen.append(sig.reshape(-1).tolist())
        return real(B, Ct, sig, check)
    monkeypatch.setattr(linalg, "_factor", spy)
    return seen


@pytest.mark.parametrize("graph", ["1", "0"])
def test_shift_doubles_when_the_spectrum_reaches_above_sigma(dev, monkeypatch, graph):
    """lam_max = 1.5 > 1.05: the unchecked first factorisation of 1.05 B - C fails, sigma doubles to 2.1."""
    from deep_cartograph_b200 import linalg
    monkeypatch.setenv("DCG_EIG_GRAPH", graph)
    seen = _record_factors(monkeypatch)
    g = np.random.default_rng(15)
    out, nb, F = 5, 3, 495
    pencils = [known_pencil(F, np.linspace(1.5, 1.3, 5), g, bulk=(-0.2, 0.2)) for _ in range(nb)]
    B = torch.from_numpy(np.stack([p[0] for p in pencils])).to(dev)
    C = torch.from_numpy(np.stack([p[1] for p in pencils])).to(dev)
    fast, dense = linalg.EIG_STATS["fast"], linalg.EIG_STATS["dense"]
    ev, V = linalg._cholesky_eigh(B, C, 0.0, out)
    assert any(all(abs(s - 2.1) < 1e-12 for s in sig) for sig in seen), seen
    assert linalg.EIG_STATS["fast"] - fast + linalg.EIG_STATS["dense"] - dense == nb
    check_pencils(ev, V, pencils, out, f"sigma doubled graph={graph}")


@pytest.mark.parametrize("graph", ["1", "0"])
def test_slow_rate_moves_the_shift_to_the_top_ritz_value(dev, monkeypatch, graph):
    """lam_out = 0.95 with the bulk reaching 0.9: the predicted rate (1.05 - 0.95) / (1.05 - 0.9) > 0.25,
    so every shift moves just above its top Ritz value and K is refactorised (a checked factorisation with
    sigma < 1.05)."""
    from deep_cartograph_b200 import linalg
    monkeypatch.setenv("DCG_EIG_GRAPH", graph)
    seen = _record_factors(monkeypatch)
    g = np.random.default_rng(16)
    out, nb, F = 5, 4, 495
    pencils = [known_pencil(F, np.linspace(0.99, 0.95, 5), g, bulk=(-0.2, 0.9)) for _ in range(nb)]
    B = torch.from_numpy(np.stack([p[0] for p in pencils])).to(dev)
    C = torch.from_numpy(np.stack([p[1] for p in pencils])).to(dev)
    fast, dense = linalg.EIG_STATS["fast"], linalg.EIG_STATS["dense"]
    ev, V = linalg._cholesky_eigh(B, C, 0.0, out)
    assert any(max(sig) < 1.05 for sig in seen), seen
    assert linalg.EIG_STATS["fast"] - fast + linalg.EIG_STATS["dense"] - dense == nb
    print("slow-rate re-shift: fast", linalg.EIG_STATS["fast"] - fast, "dense", linalg.EIG_STATS["dense"] - dense)
    check_pencils(ev, V, pencils, out, f"re-shifted graph={graph}")


def test_flat_spectrum_goes_to_the_dense_route(dev):
    """The fifth wanted eigenvalue sits on a plateau of 491 within 1e-6: no shift converges in time, the
    iteration returns None and _cholesky_eigh solves the pencils densely.  The four separated pairs are
    still right."""
    from deep_cartograph_b200 import linalg
    g = np.random.default_rng(17)
    out, nb, F = 5, 2, 495
    pencils = [known_pencil(F, [0.99, 0.98, 0.97, 0.96], g, bulk=(0.5, 0.5 + 1e-6)) for _ in range(nb)]
    B = torch.from_numpy(np.stack([p[0] for p in pencils])).to(dev)
    C = torch.from_numpy(np.stack([p[1] for p in pencils])).to(dev)
    assert linalg._shift_invert_topk(B, C, out) is None
    fast, dense = linalg.EIG_STATS["fast"], linalg.EIG_STATS["dense"]
    ev, V = linalg._cholesky_eigh(B, C, 0.0, out)
    assert linalg.EIG_STATS["dense"] == dense + nb and linalg.EIG_STATS["fast"] == fast
    check_pencils(ev[:, :4], V[..., :4], pencils, 4, "dense after None")
    top = np.array([np.sort(p[2])[::-1][4] for p in pencils])
    assert np.abs(ev[:, 4].cpu().numpy() - top).max() <= 2 * F * U53 * 1e4 + 1e-6


# ================================================================================================
# B. HTICACalculator's block path against float64
# ================================================================================================
# name: (frames, features, row stride, subspaces, subspace dim, d, lag, htica_full_gram_max_features, column offset)
CASES = {
    "c3_geometry": (200_000, 4950, 4952, 10, 5, 10, 10, None, 0),     # 10 x 495, project_blocks
    "ragged_1003": (40_000, 1003, 1004, 10, 5, 10, 10, 0, 0),         # 10 x 100 + a 3-wide last chunk
    "by_size_2100": (30_000, 2100, 2100, 7, 5, 10, 10, None, 0),      # block mode chosen by size, 300 wide
    "sd20_fallback": (30_000, 600, 600, 6, 20, 10, 10, 0, 0),         # per-chunk fallback (sd > 16)
    "wide_1050": (30_000, 2100, 2100, 2, 5, 10, 10, 0, 0),            # blocks > 1018: fallback, ranges in project
    "misaligned": (30_000, 990, 996, 10, 5, 10, 10, 0, 1),           # data_ptr % 16 == 4: register-tile kernel
}
STREAMED = ("c3_geometry", "ragged_1003")
ENGINES = ["tc_i8x3", "tc_3xtf32"]
# eigenvalue tolerance per engine (module docstring)
EV_TOL = {"tc_i8x3": 1e-5, "tc_3xtf32": 5e-5}
_REF = {}


def case_matrix(name, dev):
    n, f, ld, ns, sd, d, lag, full_max, off = CASES[name]
    from deep_cartograph_b200.synthetic import feature_matrix
    buf = torch.empty((n, ld), dtype=torch.float32, device=dev)
    X = buf[:, off:off + f]
    feature_matrix(n, f, 0, n, dev, seed=f + ns, n_slow=14, out=X)
    return X


def make_calc(name, engine, tmp_path, X, extra=None):
    from deep_cartograph_b200.modules.cv_learning.cv_calculator import HTICACalculator
    n, f, ld, ns, sd, d, lag, full_max, off = CASES[name]
    backend = {"cov_engine": engine}
    if full_max is not None:
        backend["htica_full_gram_max_features"] = full_max
    backend.update(extra or {})
    cfg = {"dimension": d, "lag_time": lag, "features_normalization": "mean_std", "num_subspaces": ns,
           "subspaces_dimension": sd, "backend": backend}
    calc = HTICACalculator(configuration=cfg, output_path=str(tmp_path))
    calc.load_training_tensor(X)
    if X.is_cuda and X.data_ptr() % 16:
        # load_training_tensor copies a misaligned matrix into an aligned buffer; hand the view back so the
        # sums and the projections run on it (the alignment test of _htica_level2 takes the fallback)
        assert torch.equal(calc.training_data, X)
        calc.training_data = X
    calc.cv_dimension = d
    return calc


def reference(name, X, mean, rng):
    """float64 checker of one case (engine-independent; computed once): per-block sums, W, T1, V2, and the
    condition / gaps of the level-2 problem for its tolerance."""
    from oracle import float64_device as f64
    if name in _REF:
        r = _REF[name]
        assert torch.equal(r["mean"], mean) and torch.equal(r["rng"], rng)
        return r
    n, f, ld, ns, sd, d, lag, full_max, off = CASES[name]
    chunks = f64.htica_chunks(f, ns)
    blocks = [f64.lagged_sums(X, lag, mean, rng, cols=c) for c in chunks]
    W, T1, V2 = f64.htica(X, lag, mean, rng, ns, sd, d)
    P = torch.cat([f64.standardize_f32(X[s:s + 100_000], mean, rng).double() @ T1 for s in range(0, n, 100_000)])
    s2 = f64.lagged_sums(P, lag)
    S1 = T1.shape[1]
    ev2, _ = f64.tica_from_sums(s2["S0"], s2["St"], s2["a"], s2["b"], s2["M"], S1)
    mu = s2["a"] / s2["M"]
    C02 = s2["S0"] / s2["M"] - torch.outer(mu, mu)
    B2 = 0.5 * (C02 + C02.T) + 1e-6 * torch.eye(S1, dtype=torch.float64, device=X.device)
    e = torch.linalg.eigvalsh(B2)
    kappa2 = float(e[-1] / e[0])
    gap2 = float((ev2[:d + 1] if S1 > d else torch.cat([ev2, ev2[-1:] - 1])).diff().abs().min())
    _REF[name] = r = {"mean": mean, "rng": rng, "chunks": chunks, "blocks": blocks, "W": W, "T1": T1,
                      "kappa2": kappa2, "gap2": gap2, "rho": autocorrelations(X, mean, rng, W, lag),
                      "rho1": level1_autocorrelations(X, mean, rng, T1, chunks, sd, lag)}
    return r


def autocorrelations(X, mean, rng, W, lag):
    """float64 lag-``lag`` autocorrelations of the CVs z W (z the float32-standardised rows), with TICA's
    centring: the eigenvalue each column of W realises.  An eigenvalue is stationary in its eigenvector, so this
    is second order in a column's error, and unlike the column it is not spread by a rotation inside a group of
    nearly equal eigenvalues."""
    from oracle import float64_device as f64
    W = W.double()
    P = torch.cat([f64.standardize_f32(X[s:s + 100_000], mean, rng).double() @ W for s in range(0, X.shape[0], 100_000)])
    s = f64.lagged_sums(P, lag)
    mu, nu = s["a"] / s["M"], s["b"] / s["M"]
    C0 = torch.diagonal(s["S0"]) / s["M"] - mu * mu
    Ct = torch.diagonal(s["St"]) / s["M"] - mu * nu
    return Ct / C0


def level1_autocorrelations(X, mean, rng, T1, chunks, sd, lag):
    out, c = [], 0
    for (s0, e0) in chunks:
        w = min(sd, e0 - s0)
        out.append(autocorrelations(X[:, s0:e0], mean[s0:e0], rng[s0:e0], T1[s0:e0, c:c + w], lag))
        c += w
    return torch.cat(out)


def i8_block_bound(X, mean, rng, xmin, xmax, c, M):
    """Entrywise bound on |S_dev - S_ref| of one diagonal block for the exact engine (module docstring), and
    the bound M delta on its column sums."""
    from test_cov_i8_exact import prep, tau_factor
    sl = slice(c[0], c[1])
    mb, rb = mean[sl], rng[sl]
    _, _, e, s = prep(mb.cpu().numpy(), rb.cpu().numpy(), xmin[sl].cpu().numpy(), xmax[sl].cpu().numpy())
    Z = ((X[:, sl] - mb) / rb).double()
    zabs = Z.abs().sum(0)
    zmax = Z.abs().max(0).values
    delta = torch.from_numpy(np.ldexp(1.0, -(e + 1)) / rb.double().cpu().numpy()).to(X.device) + 2.0 ** -24 * zmax
    s = torch.from_numpy(s).to(X.device)
    qs = zmax + s                                   # |q| s <= max|z| + one grid step
    # St's finish sums three Grams (G of q_t + q_t+lag, S0 twice), hence the factors 2 and 4
    bound = (delta[:, None] * zabs[None, :] + zabs[:, None] * delta[None, :] + M * delta[:, None] * delta[None, :]
             + 2 * M * 128.0 ** 2 * s[:, None] * s[None, :] + 4 * tau_factor(M) * M * qs[:, None] * qs[None, :])
    return bound, M * delta


def check_block_sums(calc, name, engine, X, mean, rng, ref):
    """Every diagonal block of the calculator's block-mode sums against the float64 sums of its columns;
    returns level 1 (T1) computed from them."""
    from deep_cartograph_b200 import linalg
    n, f, ld, ns, sd, d, lag, full_max, off = CASES[name]
    width = f // ns
    s = calc._lagged_sums(lag, block=width)
    M = n - lag
    assert s["M"] == M
    xmin, xmax = calc._bounds_on_device()
    worst = 0.0
    for c, r in zip(ref["chunks"], ref["blocks"]):
        sl = slice(c[0], c[1])
        if engine == "tc_i8x3":
            bound, bnd_a = i8_block_bound(X, mean, rng, xmin, xmax, c, M)
        for k in ("S0", "St"):
            got, want = s[k][sl, sl], r[k]
            if k == "St" and engine == "tc_i8x3":
                want = 0.5 * (want + want.T)           # the exact engine returns the symmetric part of St
            err = (got - want).abs()
            if engine == "tc_i8x3":
                worst = max(worst, float((err / bound).max()))
                assert bool((err <= bound).all()), (name, k, c, float((err / bound).max()))
            else:
                rel = float(err.max() / want.abs().max())
                worst = max(worst, rel / 1e-5)
                assert rel <= 1e-5, (name, k, c, rel)
        for k in ("a", "b"):
            err = (s[k][sl] - r[k]).abs()
            if engine == "tc_i8x3":
                assert bool((err <= bnd_a + 1e-12 * M).all()), (name, k, c)
            else:
                assert bool((err <= 1e-6 * r[k].abs() + 1e-6 * M ** 0.5 + 1e-4).all()), (name, k, c)
    print(f"{name} {engine}: block sums at {worst:.2f} of their bound")
    return linalg.htica_level1(s["S0"], s["St"], s["a"], s["b"], s["M"], linalg.htica_chunks(f, ns), sd)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", list(CASES))
def test_block_path_against_float64(dev, tmp_path, monkeypatch, name, engine):
    """Block sums, level 1, the weights, the full-Gram path's weights and the normalised projections.  The
    block-mode sums leave the entries outside their diagonal blocks unwritten: here they are NaN, and no
    consumer may read them."""
    from deep_cartograph_b200 import linalg, ops
    from oracle import float64_device as f64
    n, f, ld, ns, sd, d, lag, full_max, off = CASES[name]
    real = ops.lagged_covariance

    def poisoned(X, lag, *a, block=0, **k):
        s = real(X, lag, *a, block=block, **k)
        if block:
            idx = torch.arange(X.shape[1], device=X.device) // block
            outside = idx[:, None] != idx[None, :]
            for key in ("S0", "St"):
                if s.get(key) is not None:
                    s[key].masked_fill_(outside, float("nan"))
        return s
    monkeypatch.setattr(ops, "lagged_covariance", poisoned)

    X = case_matrix(name, dev)
    calc = make_calc(name, engine, tmp_path / "block", X)
    assert calc._sums_plan()[1] == f // ns, "the block path was not chosen"
    mean, rng = calc._norm_on_device()
    ref = reference(name, X, mean, rng)

    # stages 1 and 2: block sums and level 1 on them
    T1 = check_block_sums(calc, name, engine, X, mean, rng, ref)
    e1 = 0.0
    c = 0
    for (s0, e0) in ref["chunks"]:
        w = min(sd, e0 - s0)
        e1 = max(e1, f64.eigvec_error(T1[s0:e0, c:c + w], ref["T1"][s0:e0, c:c + w]))
        assert bool((T1[s0:e0, :c] == 0).all()) and bool((T1[s0:e0, c + w:] == 0).all())
        c += w
    assert c == T1.shape[1] == ref["T1"].shape[1]
    r1 = level1_autocorrelations(X, mean, rng, T1, ref["chunks"], sd, lag)
    d1 = float((r1 - ref["rho1"]).abs().max() / ref["rho1"].abs().max())

    # stage 3: the whole calculator
    calc.create_output_folders()
    calc.compute_cv()
    assert calc.cv is not None, "compute_cv failed (see the log)"
    W = torch.from_numpy(calc.cv).to(dev)
    ew = f64.eigvec_error(W, ref["W"])
    rho = autocorrelations(X, mean, rng, W, lag)
    dw = float((rho - ref["rho"]).abs().max() / ref["rho"].abs().max())
    P = calc.normalize_cv()
    Pn, _, _ = f64.project_normalized(calc.training_data, mean, rng, W)
    ep = float((P.double() - Pn).abs().max())

    # one layer more: the full-Gram path on the same data
    monkeypatch.setattr(ops, "lagged_covariance", real)
    full = make_calc(name, engine, tmp_path / "full", X, {"htica_full_gram_max_features": 1 << 20})
    full.compute_cv()
    assert full.cv is not None
    Wf = torch.from_numpy(full.cv).to(dev)
    ef = f64.eigvec_error(W, Wf)
    df = float((rho - autocorrelations(X, mean, rng, Wf, lag)).abs().max() / ref["rho"].abs().max())
    print(f"{name} {engine}: level 1 eigenvalues {d1:.2e}, eigenvectors {e1:.2e}; W eigenvalues {dw:.2e}, "
          f"eigenvectors {ew:.2e} (kappa2 {ref['kappa2']:.2e}, gap2 {ref['gap2']:.2e}, first order "
          f"{2 * (2.0 ** -24 + 2.0 ** -22) * ref['kappa2'] / ref['gap2']:.2e}); vs full-Gram eigenvalues {df:.2e}, "
          f"eigenvectors {ef:.2e}; projections {ep:.2e}")
    tol = EV_TOL[engine]
    assert d1 <= tol, (name, engine, d1)
    assert dw <= tol, (name, engine, dw)
    assert df <= 2 * tol, (name, engine, df)
    assert ep <= 1e-4, (name, engine, ep)

    if name in STREAMED:
        # from pinned host memory in small chunks: the speculative block sums are taken during the copy under
        # provisional statistics, then restandardised; the weights equal the resident path's
        monkeypatch.setattr(ops, "lagged_covariance", poisoned)
        Xh = X.cpu().contiguous().pin_memory()
        st = make_calc(name, engine, tmp_path / "streamed", Xh, {"h2d_chunk_bytes": 4 * f * 8192})
        assert st._spec is not None and st._spec["rows_done"] == n
        assert st._spec["plan"] == (lag, f // ns, True)
        # the chunked statistics are merged, so the last bit of a mean or range may differ
        np.testing.assert_allclose(st.features_norm_mean, calc.features_norm_mean, rtol=2.5e-7)
        np.testing.assert_allclose(st.features_norm_range, calc.features_norm_range, rtol=2.5e-7)
        st.compute_cv()
        assert st._spec is None, "the speculative sums were not consumed"
        assert st.cv is not None
        Ws = torch.from_numpy(st.cv).to(dev)
        ms, rs = st._norm_on_device()
        ds = float((autocorrelations(X, ms, rs, Ws, lag) - rho).abs().max() / ref["rho"].abs().max())
        print(f"{name} {engine}: streamed vs resident W eigenvalues {ds:.2e}, eigenvectors "
              f"{f64.eigvec_error(Ws, W):.2e}")
        assert ds <= 2 * tol, (name, engine, ds)
