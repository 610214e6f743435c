"""The DeepTICA minibatch loss (A11): ``dcg_ticacov_f32`` (raw weighted sums), ``dcg_ticaloss_f64`` (the d x d
eigen-loss and its gradient), ``dcg_gen_eig_small_f64`` on a poisoned batch, and the autograd backward of
``_TicaCov`` / ``_TicaLoss``, against exact and high-precision references.  Every test keeps the instant
weights ``w`` and the lagged weights ``wl`` different, so a kernel or backward that swaps them fails.

Tolerances.  u = 2^-53.
  * Sums, exact model (section A).  f, g integers in [-16, 16], w, wl integers in [0, 4], stored as float32.
    Every product w f_i f_j is an integer below 2^10 and every partial or total sum is an integer below
    2^53 (B <= 2^21: 2^21 * 4 * 256 = 2^31), so every FP32 or FP64 add is exact in any order: all seven
    segments must equal the int64 sums bit for bit.
  * Sums, real data (section B).  The kernel forms (double)w * f_i exactly (two 24-bit significands), then
    one FMA per row in FP64 (its product with f_j is exact inside the FMA), over R = min(B, 128) rows of a
    tile; CTA k adds its T = ceil(tiles / G) tiles in turn, and a second launch adds the G = min(tiles, 1024)
    CTA sums.  Recursive summation (Higham, Accuracy and Stability, 2nd ed., section 4.2) of R terms, then
    of T, then of G partial sums gives
        |S_dev - S| <= gamma_{R + T + G} sum_n |w_n f_ni f_nj|,   gamma_n = n u / (1 - n u),
    entry by entry and for the vector and weight sums alike.  Both stages run in a fixed order, so the sums
    are also bitwise the same from call to call.  The reference is a long-double sum, whose own
    error gamma_B(eps_ld) sum|.| is added to the bound (it is ~2^11 times smaller on x86).  The centred
    C0 / C_tau (``tica_covariances``) are held to the north star, 1e-5 of the largest entry of the float64
    oracle, at outputs whose mean is 0 to 1000 standard deviations from zero: with the bound above the
    cancellation in sff / sw - mu mu^T costs gamma_{R+T+G} (1 + |mu|^2 / var) ~ 1e-7 at 1000 spreads.
  * Eigen-loss (section C).  The input sums are chosen doubles; the reference (mpmath, 120 bits) recomputes
    C0, C_tau from the same doubles, so it sees exactly the kernel's input.  The kernel's Cholesky, triangular
    inverse, reduction and Jacobi are backward stable: they solve a pencil (B + dB, C_tau + dC) with
    ||dB|| <= c (d + 1) u ||B||, ||dC|| <= c (d + 1) u ||C_tau|| (the inverse's row-wise backward error is
    carried into both).  Through a definite pencil an eigenvalue then moves by at most
    (||dC|| + |lam| ||dB||) / lambda_min(B) <= 2 c (d + 1) u kappa(B) max|lam| (||B|| >= ||C_tau|| / max|lam|).
    The tolerance is that with c = 8.  The loss moves by at most 2 d max|lam| times it.  For n_eig <= 0 or
    >= d the gradients are the matrix functions G0 = 2 B^-1 Ct B^-1 Ct B^-1, Gt = -2 B^-1 Ct B^-1, whose
    first-order relative change under (dB, dC) is at most 5 kappa(B) times theirs; in the max-entry norm
    (||G||_2 <= d max|G_ij|) that is 16 (d + 1) d u kappa(B) max|G|.  For a cut 0 < n_eig < d each partial
    projector also turns by the eigenvalue tolerance over the gap at the cut, which multiplies the gradient
    tolerance by (1 + 2 max|lam| / gap).  mu = sum w f / sum w is one IEEE division: bitwise.
  * Backward (section D).  The kernel's G0 / Gt and the float64 chain rule are cast to float32 at the end:
    2e-6 of the largest gradient entry (the suite's existing gradient tolerance) covers the 2^-24 cast and
    the section-C error at these well-conditioned batches.
"""
import math

import numpy as np
import pytest
import torch

U53 = 2.0 ** -53
ROWS = 128                                      # kTcRowsPerCta (ticacov.cu)
MAX_CTAS = 1024                                 # kTcMaxCtas (ticacov.cu)
SEGMENTS = ("sw", "swl", "swf", "sff", "sfg", "slf", "slg")


def _gamma(n, u=U53):
    return n * u / (1.0 - n * u)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from deep_cartograph_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


# ================================================================================================
# host-side references
# ================================================================================================
def exact_sums(f, g, w, wl):
    """The seven segments of dcg_ticacov_f32 in int64 from integer-valued f, g, w, wl (None = 1)."""
    fi, gi = f.astype(np.int64), g.astype(np.int64)
    B = fi.shape[0]
    wi = np.ones(B, np.int64) if w is None else w.astype(np.int64)
    li = np.ones(B, np.int64) if wl is None else wl.astype(np.int64)
    return {"sw": wi.sum(), "swl": li.sum(), "swf": (wi[:, None] * fi).sum(0), "sff": (wi[:, None] * fi).T @ fi,
            "sfg": (li[:, None] * fi).T @ gi, "slf": (li[:, None] * fi).sum(0), "slg": (li[:, None] * gi).sum(0)}


def sums_with_abs(f, g, w, wl):
    """(long-double sums, float64 sums of |terms|) of the seven segments."""
    ld = np.longdouble
    F, G = f.astype(ld), g.astype(ld)
    W, L = w.astype(ld), wl.astype(ld)
    ref = {"sw": W.sum(), "swl": L.sum(), "swf": (W[:, None] * F).sum(0), "sff": (W[:, None] * F).T @ F,
           "sfg": (L[:, None] * F).T @ G, "slf": (L[:, None] * F).sum(0), "slg": (L[:, None] * G).sum(0)}
    af, ag, aw, al = np.abs(f.astype(np.float64)), np.abs(g.astype(np.float64)), np.abs(w.astype(np.float64)), \
        np.abs(wl.astype(np.float64))
    mag = {"sw": aw.sum(), "swl": al.sum(), "swf": (aw[:, None] * af).sum(0), "sff": (aw[:, None] * af).T @ af,
           "sfg": (al[:, None] * af).T @ ag, "slf": (al[:, None] * af).sum(0), "slg": (al[:, None] * ag).sum(0)}
    return ref, mag


def sums_vector(sw, swl, mu, nu, xi, C0, Ct):
    """Raw sums (the dcg_ticacov_f32 layout) whose means are mu (sum w f / sum w), nu (sum wl g / sum wl),
    xi (sum wl f / sum wl) and whose centred C0 / C_tau are C0, Ct, rounded to float64."""
    mm = np.outer(mu, mu)
    return np.concatenate([[sw, swl], sw * mu, (sw * (C0 + mm)).ravel(),
                           (swl * (Ct + np.outer(mu, nu) + np.outer(xi, mu) - mm)).ravel(), swl * xi, swl * nu])


def mp_loss_reference(sums, d, reg, prec=120):
    """Everything dcg_ticaloss_f64 returns, from the same doubles, in mpmath: the eigenpairs of the reduced
    pencil (``eigsy``) and the n_eig = 0 closed forms loss = -tr((B^-1 Ct)^2), G0 = 2 B^-1 Ct B^-1 Ct B^-1,
    Gt = -2 B^-1 Ct B^-1 (W L W^k W^T = (B^-1 Ct)^k B^-1 with W^T B W = I)."""
    import mpmath as mp
    with mp.workprec(prec):
        v = [mp.mpf(float(x)) for x in sums]
        dd = d * d
        sw, swl = v[0], v[1]
        swf, sff = v[2:2 + d], v[2 + d:2 + d + dd]
        sfg = v[2 + d + dd:2 + d + 2 * dd]
        slf, slg = v[2 + d + 2 * dd:2 + 2 * d + 2 * dd], v[2 + 2 * d + 2 * dd:]
        mu = [x / sw for x in swf]
        nu = [x / swl for x in slg]
        xi = [x / swl for x in slf]
        C0r = mp.matrix(d, d)
        Ctr = mp.matrix(d, d)
        for i in range(d):
            for j in range(d):
                C0r[i, j] = sff[i * d + j] / sw - mu[i] * mu[j]
                Ctr[i, j] = sfg[i * d + j] / swl - mu[i] * nu[j] - xi[i] * mu[j] + mu[i] * mu[j]
        C0 = (C0r + C0r.T) / 2
        Ct = (Ctr + Ctr.T) / 2
        Bm = C0 + mp.mpf(reg) * mp.eye(d)
        Li = mp.inverse(mp.cholesky(Bm))
        A = Li * Ct * Li.T
        E, U = mp.eigsy((A + A.T) / 2)
        order = sorted(range(d), key=lambda k: -E[k])
        ev = [E[k] for k in order]
        W = Li.T * U
        W = mp.matrix([[W[i, k] for k in order] for i in range(d)])
        Bi = mp.inverse(Bm)
        M = Bi * Ct
        P = M * Bi
        M2 = M * M
        out = {"ev": np.array([float(x) for x in ev]), "mu": np.array([float(x) for x in mu]),
               "loss_cf": -float(sum(M2[i, i] for i in range(d))), "G0_cf": _np(2 * P * Ct * Bi),
               "Gt_cf": _np(-2 * P), "_ev": ev, "_W": W}
        Bf = _np(Bm)
    lam_b = np.linalg.eigvalsh(0.5 * (Bf + Bf.T))
    out["kappa"] = float(lam_b[-1] / lam_b[0]) if lam_b[0] > 0 else math.inf
    return out


def _np(M):
    return np.array([[float(M[i, j]) for j in range(M.cols)] for i in range(M.rows)])


def mp_partial(ref, d, n_eig):
    """loss, G0, Gt of the first ``used`` eigenpairs (used = n_eig if 0 < n_eig < d else d)."""
    import mpmath as mp
    used = n_eig if 0 < n_eig < d else d
    with mp.workprec(120):
        ev, W = ref["_ev"], ref["_W"]
        G0 = mp.matrix(d, d)
        Gt = mp.matrix(d, d)
        for r in range(used):
            for i in range(d):
                for j in range(d):
                    vv = W[i, r] * W[j, r]
                    G0[i, j] += 2 * ev[r] ** 2 * vv
                    Gt[i, j] -= 2 * ev[r] * vv
        loss = -float(sum(ev[r] ** 2 for r in range(used)))
    return loss, _np(G0), _np(Gt)


def pencil_sums(d, lam, kappa, seed, reg=1e-6, sw=37.5, swl=12.3):
    """Sums of a pencil with eigenvalues ``lam``: X with singular values 1 .. kappa^-1/2, B = X X^T (so
    kappa(B) = kappa, ||B|| = 1), C_tau = X diag(lam) X^T, C0 = B - reg I; sw != swl and mu, nu, xi
    distinct and O(1)."""
    rng = np.random.default_rng(seed)
    lam = np.asarray(lam, dtype=np.float64)
    Q1, _ = np.linalg.qr(rng.standard_normal((d, d)))
    Q2, _ = np.linalg.qr(rng.standard_normal((d, d)))
    s = np.logspace(0.0, -0.5 * math.log10(kappa), d) if d > 1 else np.ones(1)
    X = (Q1 * s) @ Q2
    Bm = X @ X.T
    Ct = (X * lam) @ X.T
    mu, nu, xi = (rng.uniform(-0.5, 0.5, d) for _ in range(3))
    return sums_vector(sw, swl, mu, nu, xi, 0.5 * (Bm + Bm.T) - reg * np.eye(d), 0.5 * (Ct + Ct.T))


def rank_old(keys):
    """ticaloss_kernel's eigenvalue rank before the fix, restated: lane i's slot."""
    d = len(keys)
    return [sum((keys[j] > keys[i]) or (keys[j] == keys[i] and j < i) for j in range(d)) for i in range(d)]


def rank_new(keys):
    """The rank of ticaloss_kernel and gen_eig_small_kernel: NaN keys rank as -inf."""
    k = [(-math.inf if x != x else x) for x in keys]
    d = len(k)
    return [sum((k[j] > k[i]) or (k[j] == k[i] and j < i) for j in range(d)) for i in range(d)]


# ================================================================================================
# E. host checks (no GPU)
# ================================================================================================
def test_rank_rule_old_collides_on_nan_new_is_a_permutation():
    """The old rule gives every NaN key rank 0 (NaN compares false), so ranks collide and slots of order[]
    stay unwritten; the new one is a permutation for any keys and keeps the descending order of the rest."""
    nan, inf = math.nan, math.inf
    assert sorted(rank_old([nan] * 5)) != list(range(5))
    assert sorted(rank_old([0.5, nan, -0.2, nan])) != list(range(4))
    rng = np.random.default_rng(0)
    pool = [nan, inf, -inf, 0.0, -0.0, 1.0, 1.0, -3.5, 2.0]
    for d in range(1, 33):
        for _ in range(20):
            keys = list(rng.choice(pool, size=d)) if rng.random() < 0.7 else list(rng.standard_normal(d))
            r = rank_new(keys)
            assert sorted(r) == list(range(d)), keys
            slot = [None] * d
            for i, ri in enumerate(r):
                slot[ri] = keys[i]
            key = [(-math.inf if x != x else x) for x in slot]
            assert key == sorted(key, reverse=True)                  # descending, NaN among the -inf at the end
            if not any(x != x for x in keys):
                assert r == rank_old(keys)                           # unchanged where the old rule was right


@pytest.mark.parametrize("d", [1, 5, 17, 32])
def test_closed_forms_agree_with_the_eigen_decomposition(d):
    """The n_eig = 0 closed forms (mpmath) against the eigenpair sums (mpmath eigsy) and against
    ``conftest.cpu_ticaloss`` (torch float64 eigh), so the section-C references check each other."""
    from conftest import cpu_ticaloss
    lam = np.linspace(0.9, -0.97, d) if d > 1 else np.array([-0.6])
    sums = pencil_sums(d, lam, 1e3, seed=d)
    ref = mp_loss_reference(sums, d, 1e-6)
    loss, G0, Gt = mp_partial(ref, d, 0)
    assert abs(loss - ref["loss_cf"]) <= 4 * U53 * abs(loss)
    np.testing.assert_allclose(G0, ref["G0_cf"], rtol=0, atol=1e-13 * np.abs(G0).max())
    np.testing.assert_allclose(Gt, ref["Gt_cf"], rtol=0, atol=1e-13 * np.abs(Gt).max())
    np.testing.assert_allclose(ref["ev"], np.sort(lam)[::-1], atol=1e-12)
    c = cpu_ticaloss(torch.from_numpy(sums), d, 1e-6)
    assert abs(c["loss"].item() - loss) <= 1e-9 * abs(loss)
    np.testing.assert_allclose(c["G0"].numpy(), G0, rtol=0, atol=1e-9 * np.abs(G0).max())
    np.testing.assert_allclose(c["Gt"].numpy(), Gt, rtol=0, atol=1e-9 * np.abs(Gt).max())


def test_ticacov_sums_rejects_mismatched_shapes():
    """g must have f's shape and w / wl B elements: the kernel would read past a shorter tensor's end."""
    from deep_cartograph_b200 import ops
    f = torch.zeros((300, 4))
    with pytest.raises(ValueError, match="one shape"):
        ops.ticacov_sums(f, torch.zeros((299, 4)))
    with pytest.raises(ValueError, match="one shape"):
        ops.ticacov_sums(f, torch.zeros((300, 3)))
    with pytest.raises(ValueError, match="one shape"):
        ops.ticacov_sums(torch.zeros(300), torch.zeros(300))
    for kw in ({"w": torch.ones(299)}, {"wl": torch.ones(301)}, {"w": torch.ones((300, 1))},
               {"w": torch.ones(300), "wl": torch.ones(150)}):
        with pytest.raises(ValueError, match="tensor on"):
            ops.ticacov_sums(f, f, **kw)
    with pytest.raises(RuntimeError, match="CUDA tensor"):              # right shapes reach the device check
        ops.ticacov_sums(f, f, torch.ones(300), torch.ones(300))


def test_ticacov_workspace_size():
    """One column of output doubles per CTA, min(ceil(B / 128), 1024) CTAs; 0 for arguments out of range."""
    from deep_cartograph_b200 import _lib
    lib = _lib.load()
    for B, d in ((1, 1), (128, 4), (129, 4), (65536, 10), (ROWS * MAX_CTAS, 32), (ROWS * MAX_CTAS + 1, 32), (2 ** 31, 3)):
        G = min(-(-B // ROWS), MAX_CTAS)
        assert lib.dcg_ticacov_workspace_bytes(B, d) == 8 * G * lib.dcg_ticacov_out_doubles(d)
    assert lib.dcg_ticacov_workspace_bytes(0, 4) == 0 and lib.dcg_ticacov_workspace_bytes(10, 33) == 0


@pytest.mark.gpu
def test_ticacov_sums_rejects_mismatched_shapes_on_device(dev):
    from deep_cartograph_b200 import ops
    f = torch.zeros((300, 4), device=dev)
    with pytest.raises(ValueError):
        ops.ticacov_sums(f, torch.zeros((299, 4), device=dev))
    with pytest.raises(ValueError):
        ops.ticacov_sums(f, f, torch.ones(299, device=dev))
    with pytest.raises(ValueError):
        ops.ticacov_sums(f, f, None, torch.ones(300))                  # host weights with device outputs


# ================================================================================================
# A. sums: exact integer model
# ================================================================================================
def _int_data(B, d, seed):
    rng = np.random.default_rng(seed)
    f = rng.integers(-16, 17, (B, d)).astype(np.float32)
    g = rng.integers(-16, 17, (B, d)).astype(np.float32)
    w = rng.integers(0, 5, B).astype(np.float32)                   # about a fifth of the rows weigh 0
    wl = rng.integers(0, 5, B).astype(np.float32)
    return f, g, w, wl


def _check_exact(dev, f, g, w, wl, what):
    from deep_cartograph_b200 import ops
    t = lambda a: None if a is None else torch.from_numpy(a).to(dev)
    s = ops.ticacov_sums(t(f), t(g), t(w), t(wl))
    ref = exact_sums(f, g, w, wl)
    for name in SEGMENTS:
        got = s[name].cpu().numpy()
        want = np.asarray(ref[name], dtype=np.float64)
        assert got.shape == want.shape and np.array_equal(got, want), \
            f"{what}: segment {name} differs at {np.argwhere(got != want)[:4].tolist()}"


WEIGHT_MODES = ("both", "w_only", "wl_only", "none")


def _weights(mode, w, wl):
    return {"both": (w, wl), "w_only": (w, None), "wl_only": (None, wl), "none": (None, None)}[mode]


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 2, 127, 128, 129, 255, 256, 1000, 65537])
@pytest.mark.parametrize("d", [1, 2, 3, 7, 8, 15, 16, 17, 31, 32])
def test_sums_bitwise_equal_integer_model(dev, d, B):
    """All seven segments bitwise against int64, for w != wl, w only, wl only and no weights, at tile edges
    (B = 127/128/129, 255/256) and across the one-pass / two-pass thread split (d*d + d + 1 > 256 from d = 16)."""
    f, g, w, wl = _int_data(B, d, seed=B * 33 + d)
    for mode in WEIGHT_MODES:
        _check_exact(dev, f, g, *_weights(mode, w, wl), what=f"B={B} d={d} {mode}")


@pytest.mark.gpu
def test_sums_bitwise_equal_integer_model_large(dev):
    B, d = 2 ** 20 + 3, 10
    f, g, w, wl = _int_data(B, d, seed=5)
    _check_exact(dev, f, g, w, wl, what="B=2^20+3")


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 3, 16, 17, 32])
@pytest.mark.parametrize("B", [129, 256, 300, 1000, ROWS * MAX_CTAS + 1])
def test_sums_marker_rows(dev, d, B):
    """Rows 0, 127, 128 and B-1 carry values 2^0, 2^6, 2^12, 2^18 times a pattern, every other row is zero:
    a dropped, duplicated or misplaced row changes a sum by a distinct power of two."""
    f = np.zeros((B, d), np.float32)
    g = np.zeros((B, d), np.float32)
    pat_f = (1 + np.arange(d) % 7).astype(np.float32)
    pat_g = -(1 + (np.arange(d) + 3) % 5).astype(np.float32)
    for m, r in enumerate(sorted({0, 127, 128, B - 1})):
        f[r] = 2.0 ** (6 * m) * pat_f
        g[r] = 2.0 ** (6 * m) * pat_g
    w = np.full(B, 3, np.float32)
    wl = np.full(B, 2, np.float32)
    for mode in WEIGHT_MODES:
        _check_exact(dev, f, g, *_weights(mode, w, wl), what=f"markers B={B} d={d} {mode}")


# ================================================================================================
# B. sums: real-valued data against float64
# ================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0, 1, 10, 100, 1000])
@pytest.mark.parametrize("B,d", [(4096, 4), (65537, 10), (3000, 17), (300001, 6)])
def test_sums_and_covariances_uncentred(dev, B, d, offset):
    """Gaussian outputs whose mean is ``offset`` standard deviations from zero, w != wl: the raw sums within
    gamma_{R+T+G} sum|w f_i f_j| of a long-double sum, and the centred C0 / C_tau within 1e-5 of the float64
    oracle's largest entry."""
    import oracle
    from deep_cartograph_b200 import ops
    from deep_cartograph_b200.modules.cv_learning.deep_tica import tica_covariances
    rng = np.random.default_rng(B + d + offset)
    z = rng.standard_normal((B + 1, d))
    sig = rng.uniform(0.5, 2.0, d)
    f = ((z[:-1] * sig) + offset * sig * rng.choice([-1, 1], d)).astype(np.float32)
    g = ((0.8 * z[:-1] + 0.6 * z[1:]) * sig + offset * sig * rng.choice([-1, 1], d)).astype(np.float32)
    w = rng.uniform(0.5, 1.5, B).astype(np.float32)
    wl = rng.uniform(0.0, 2.0, B).astype(np.float32)
    tf, tg, tw, twl = (torch.from_numpy(a).to(dev) for a in (f, g, w, wl))
    s = ops.ticacov_sums(tf, tg, tw, twl)
    ref, mag = sums_with_abs(f, g, w, wl)
    tiles = -(-B // ROWS)
    G = min(tiles, MAX_CTAS)
    R, T = min(B, ROWS), -(-tiles // G)
    eps_ld = float(np.finfo(np.longdouble).eps) / 2
    ratio = {}
    for name in SEGMENTS:
        err = np.abs(s[name].cpu().numpy().astype(np.longdouble) - ref[name]).astype(np.float64)
        tol = (_gamma(R + T + G) + _gamma(B, eps_ld)) * mag[name]
        ratio[name] = float(np.max(err / tol))
    C0, Ct = tica_covariances(tf, tg, tw, twl)
    rC0, rCt, _ = oracle.deeptica_cov(f, g, w, wl)
    e0 = np.abs(C0.cpu().numpy() - rC0).max() / np.abs(rC0).max()
    et = np.abs(Ct.cpu().numpy() - rCt).max() / np.abs(rCt).max()
    msg = (f"B={B} d={d} mean/std={offset}: C0 error {e0:.2e}, Ct error {et:.2e} of the largest entry; "
           f"sums at {max(ratio.values()):.2e} of their bound")
    print(msg)
    assert all(r <= 1.0 for r in ratio.values()), f"{msg}: {ratio}"
    assert e0 <= 1e-5 and et <= 1e-5, msg


@pytest.mark.gpu
@pytest.mark.parametrize("B,d", [(65536, 4), (300001, 10), (200000, 32)])
def test_sums_are_bitwise_reproducible(dev, B, d):
    """Real-valued, uncentred outputs: repeated calls give bitwise the same sums (no FP64 atomics), also where
    a CTA takes several tiles (B > 128 * 1024)."""
    from deep_cartograph_b200 import ops
    g0 = torch.Generator(device=dev).manual_seed(B + d)
    f = torch.randn((B, d), generator=g0, device=dev) + 50.0
    g = torch.randn((B, d), generator=g0, device=dev) - 20.0
    w = torch.rand(B, generator=g0, device=dev)
    wl = torch.rand(B, generator=g0, device=dev) + 0.5
    first = ops.ticacov_sums(f, g, w, wl)["flat"].clone()
    for _ in range(5):
        assert torch.equal(ops.ticacov_sums(f, g, w, wl)["flat"], first)


# ================================================================================================
# C. the eigen-loss kernel on chosen sums
# ================================================================================================
def _run_loss(dev, sums, d, reg, n_eig):
    from deep_cartograph_b200 import ops
    r = ops.ticaloss(torch.from_numpy(np.ascontiguousarray(sums, dtype=np.float64)).to(dev), d, reg, n_eig)
    return {k: v.cpu().numpy() for k, v in r.items()}


def _check_loss(got, ref, sums, d, n_eig, gap=None):
    """Everything dcg_ticaloss_f64 returns against the mpmath reference, within the docstring's bounds."""
    kap = ref["kappa"]
    lmax = max(np.abs(ref["ev"]).max(), 1e-300)
    tol_ev = 16 * (d + 1) * U53 * kap * lmax
    used = n_eig if 0 < n_eig < d else d
    if used == d:
        loss, G0, Gt = ref["loss_cf"], ref["G0_cf"], ref["Gt_cf"]
        fac = 1.0
    else:
        loss, G0, Gt = mp_partial(ref, d, n_eig)
        fac = 1.0 + 2.0 * lmax / gap
    assert got["status"] == 0
    assert got["sw"] == sums[0] and got["swl"] == sums[1]
    assert np.array_equal(got["mu"], sums[2:2 + d] / sums[0])            # one IEEE division each
    ev_err = np.abs(got["evals"] - ref["ev"]).max()
    assert ev_err <= tol_ev, f"eigenvalues off by {ev_err:.3e} > {tol_ev:.3e} (kappa {kap:.1e})"
    assert abs(got["loss"] - loss) <= 2 * d * lmax * tol_ev * fac, (got["loss"], loss)
    for name, G, want in (("G0", got["G0"], G0), ("Gt", got["Gt"], Gt)):
        tol = 16 * (d + 1) * d * U53 * kap * fac * np.abs(want).max()
        err = np.abs(G - want).max()
        assert err <= tol, f"{name} off by {err:.3e} > {tol:.3e} (kappa {kap:.1e}, n_eig {n_eig})"
    return ev_err / tol_ev


def _spectrum(d):
    """Distinct, descending, with the largest magnitude negative (so |lam| order is not signed order)."""
    return np.linspace(0.9, -0.97, d) if d > 1 else np.array([-0.6])


@pytest.mark.gpu
@pytest.mark.parametrize("d", list(range(1, 33)))
def test_ticaloss_every_d_every_n_eig(dev, d):
    """d = 1 .. 32, n_eig in {0, 1, d-1, d, d+3, -1}: eigenvalues, loss, gradients, mu, sw, swl."""
    lam = _spectrum(d)
    sums = pencil_sums(d, lam, 1e2, seed=100 + d)
    ref = mp_loss_reference(sums, d, 1e-6)
    gap = float(np.min(-np.diff(lam))) if d > 1 else 1.0
    for n_eig in sorted({0, 1, d - 1, d, d + 3, -1}):
        _check_loss(_run_loss(dev, sums, d, 1e-6, n_eig), ref, sums, d, n_eig, gap)


@pytest.mark.gpu
def test_ticaloss_indefinite_ct_cut_by_signed_order(dev):
    """lam = 0.8, 0.6, 0.3, -0.1, -0.7, -0.99: with n_eig = 2 the loss is -(0.8^2 + 0.6^2) = -1; ranking by
    |lam| would give -(0.99^2 + 0.8^2)."""
    d = 6
    lam = np.array([0.8, 0.6, 0.3, -0.1, -0.7, -0.99])
    sums = pencil_sums(d, lam, 1e3, seed=6)
    ref = mp_loss_reference(sums, d, 1e-6)
    for n_eig in (1, 2, 3, 5):
        got = _run_loss(dev, sums, d, 1e-6, n_eig)
        _check_loss(got, ref, sums, d, n_eig, gap=0.2)
    assert abs(_run_loss(dev, sums, d, 1e-6, 2)["loss"] + 1.0) < 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("d", [4, 8, 32])
def test_ticaloss_repeated_eigenvalues(dev, d):
    """Exactly repeated eigenvalues (n_eig = 0 and d): the closed forms stay defined, the eigenvectors not."""
    lam = np.repeat([0.7, 0.2, -0.4, -0.85], d // 4)
    sums = pencil_sums(d, lam, 1e4, seed=200 + d)
    ref = mp_loss_reference(sums, d, 1e-6)
    for n_eig in (0, d):
        _check_loss(_run_loss(dev, sums, d, 1e-6, n_eig), ref, sums, d, n_eig)


@pytest.mark.gpu
@pytest.mark.parametrize("kappa", [1e2, 1e6, 1e10])
@pytest.mark.parametrize("d", [2, 5, 16, 32])
def test_ticaloss_conditioning(dev, d, kappa):
    """kappa(B) = 1e2, 1e6, 1e10: the tolerance scales with kappa(B); n_eig = 0 and a cut with a clear gap."""
    lam = _spectrum(d)
    sums = pencil_sums(d, lam, kappa, seed=300 + d)
    ref = mp_loss_reference(sums, d, 1e-6)
    gap = float(np.min(-np.diff(lam)))
    for n_eig in (0, 1):
        ratio = _check_loss(_run_loss(dev, sums, d, 1e-6, n_eig), ref, sums, d, n_eig, gap)
        print(f"d={d} kappa={ref['kappa']:.1e} n_eig={n_eig}: eigenvalue error at {ratio:.1e} of the bound")


def _check_flagged(got, d, what):
    assert got["status"] == 1, what
    assert np.isnan(got["loss"]), what
    assert np.isnan(got["evals"]).all(), f"{what}: evals {got['evals']}"
    assert not np.any(got["G0"]) and not np.any(got["Gt"]), what
    assert np.isfinite(got["G0"]).all() and np.isfinite(got["Gt"]).all(), what


@pytest.mark.gpu
def test_ticaloss_negative_reg_is_flagged(dev):
    """C0 with smallest eigenvalue 1e-2 and reg = -5e-2: B indefinite, status 1, NaN loss and evals, zero G."""
    d = 5
    sums = pencil_sums(d, _spectrum(d), 1e2, seed=9, reg=0.0)
    _check_flagged(_run_loss(dev, sums, d, -5e-2, 0), d, "reg < 0")
    _check_loss(_run_loss(dev, sums, d, 0.0, 0), mp_loss_reference(sums, d, 0.0), sums, d, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 5, 32])
def test_ticaloss_non_finite_sums_are_flagged(dev, d):
    """A NaN, +Inf or -Inf in each segment in turn, and sum w = 0, sum wl = 0: status 1, loss and every
    eigenvalue NaN, G0 = Gt = 0.  A good batch afterwards is unaffected."""
    dd = d * d
    good = pencil_sums(d, _spectrum(d), 1e2, seed=11)
    starts = {"sw": 0, "swl": 1, "swf": 2, "sff": 2 + d, "sfg": 2 + d + dd, "slf": 2 + d + 2 * dd,
              "slg": 2 + 2 * d + 2 * dd}
    lens = {"sw": 1, "swl": 1, "swf": d, "sff": dd, "sfg": dd, "slf": d, "slg": d}
    rng = np.random.default_rng(d)
    cases = []
    for name, o in starts.items():
        for k in sorted({0, lens[name] - 1, int(rng.integers(lens[name]))}):
            for v in (math.nan, math.inf, -math.inf):
                cases.append((f"{name}[{k}]={v}", o + k, v))
    cases += [("sw=0", 0, 0.0), ("swl=0", 1, 0.0)]
    for what, pos, v in cases:
        s = good.copy()
        s[pos] = v
        if what == "sw=0":
            s[2:2 + d] = 0.0                                     # all weights zero: sum w f = 0 too (0/0)
        _check_flagged(_run_loss(dev, s, d, 1e-6, 0), d, what)
    _check_loss(_run_loss(dev, good, d, 1e-6, 0), mp_loss_reference(good, d, 1e-6), good, d, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("b", [1, 7, 32])
def test_gen_eig_small_nan_pencil_leaves_the_batch_alone(dev, b):
    """One pencil's H holds a NaN: the other pencils' theta, S and status are bitwise those of the batch
    without it."""
    from deep_cartograph_b200 import ops
    g0 = torch.Generator(device=dev).manual_seed(b)
    nb = 5
    R = torch.randn((nb, b, b + 3), generator=g0, device=dev, dtype=torch.float64)
    G = R @ R.mT + 0.1 * torch.eye(b, device=dev, dtype=torch.float64)
    Q = torch.randn((nb, b, b), generator=g0, device=dev, dtype=torch.float64)
    H = 0.5 * (Q + Q.mT)
    th0, S0, st0 = ops.gen_eig_small(H, G)
    for bad in (0, 2, nb - 1):
        for v in (math.nan, math.inf):
            Hb = H.clone()
            Hb[bad, b // 2, b - 1] = v
            th, S, st = ops.gen_eig_small(Hb, G)
            keep = [k for k in range(nb) if k != bad]
            assert torch.equal(th[keep], th0[keep]) and torch.equal(S[keep], S0[keep]) and torch.equal(st[keep], st0[keep])
            assert not torch.isfinite(th[bad]).all()


# ================================================================================================
# D. backward with distinct weights
# ================================================================================================
def _torch_cov(f, g, w, wl):
    """oracle.deeptica_cov restated in torch (float64, autograd; no ops)."""
    B = f.shape[0]
    w = torch.ones(B, dtype=f.dtype) if w is None else w
    wl = torch.ones(B, dtype=f.dtype) if wl is None else wl
    wn, wln = w / w.sum(), wl / wl.sum()
    mu = (wn[:, None] * f).sum(0)
    ft, gt = f - mu, g - mu
    C0 = (ft * wn[:, None]).T @ ft
    Ct = (ft * wln[:, None]).T @ gt
    return 0.5 * (C0 + C0.T), 0.5 * (Ct + Ct.T)


def _torch_loss(f, g, w, wl, reg, n_eig):
    C0, Ct = _torch_cov(f, g, w, wl)
    d = C0.shape[0]
    L = torch.linalg.cholesky(C0 + reg * torch.eye(d, dtype=C0.dtype))
    Li = torch.linalg.inv(L)
    ev = torch.linalg.eigvalsh(Li @ Ct @ Li.T).flip(0)
    used = ev[:n_eig] if 0 < n_eig < d else ev
    return -(used ** 2).sum(), ev


def _backward_data(B, d, offset, seed):
    rng = np.random.default_rng(seed)
    base = rng.standard_normal((B + 1, d)) @ (np.eye(d) + 0.3 * rng.standard_normal((d, d)))
    rho = np.linspace(0.9, 0.2, d)
    f = base[:-1] + offset
    g = rho * base[:-1] + np.sqrt(1 - rho ** 2) * base[1:] - 0.3 * np.roll(base[:-1], 1, axis=1) + offset
    w = rng.uniform(0.2, 2.0, B)
    wl = rng.uniform(0.0, 3.0, B)
    wl[::7] = 0.0
    return f.astype(np.float32), g.astype(np.float32), w.astype(np.float32), wl.astype(np.float32)


BACKWARD_CASES = [("both", 0.0), ("w_only", 0.0), ("wl_only", 0.0), ("both", 30.0), ("wl_only", 30.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode,offset", BACKWARD_CASES)
@pytest.mark.parametrize("d,n_eig", [(5, 0), (6, 2)])
def test_tica_loss_backward_distinct_weights(dev, mode, offset, d, n_eig):
    """``tica_loss`` (fused kernel + analytic backward): loss, eigenvalues, df and dg against float64 torch
    autograd of the oracle formula, with w != wl, only w, only wl, and outputs 30 spreads off zero."""
    from deep_cartograph_b200.modules.cv_learning.deep_tica import tica_loss
    B = 3000
    f, g, w, wl = _backward_data(B, d, offset, seed=d * 10 + int(offset))
    w, wl = _weights(mode, w, wl)
    t = lambda a: None if a is None else torch.from_numpy(a).to(dev)
    fd, gd = t(f).requires_grad_(True), t(g).requires_grad_(True)
    loss, ev = tica_loss(fd, gd, t(w), t(wl), reg=1e-6, n_eig=n_eig)
    loss.backward()
    t64 = lambda a: None if a is None else torch.from_numpy(a.astype(np.float64))
    f64, g64 = t64(f).requires_grad_(True), t64(g).requires_grad_(True)
    rloss, rev = _torch_loss(f64, g64, t64(w), t64(wl), 1e-6, n_eig)
    rloss.backward()
    assert abs(loss.item() - rloss.item()) <= 1e-9 * abs(rloss.item())
    np.testing.assert_allclose(ev.cpu().numpy(), rev.detach().numpy(), rtol=0, atol=1e-9)
    sc = max(f64.grad.abs().max().item(), g64.grad.abs().max().item())
    np.testing.assert_allclose(fd.grad.cpu().numpy(), f64.grad.numpy(), rtol=0, atol=2e-6 * sc)
    np.testing.assert_allclose(gd.grad.cpu().numpy(), g64.grad.numpy(), rtol=0, atol=2e-6 * sc)


@pytest.mark.gpu
@pytest.mark.parametrize("mode,offset", BACKWARD_CASES)
def test_tica_covariances_backward_distinct_weights(dev, mode, offset):
    """``tica_covariances``: C0, C_tau and the gradient of <R0, C0> + <Rt, C_tau> (R0, Rt not symmetric)
    against float64 torch autograd."""
    from deep_cartograph_b200.modules.cv_learning.deep_tica import tica_covariances
    B, d = 2500, 7
    f, g, w, wl = _backward_data(B, d, offset, seed=77 + int(offset))
    w, wl = _weights(mode, w, wl)
    rng = np.random.default_rng(3)
    R0, Rt = rng.standard_normal((d, d)), rng.standard_normal((d, d))
    t = lambda a: None if a is None else torch.from_numpy(a).to(dev)
    fd, gd = t(f).requires_grad_(True), t(g).requires_grad_(True)
    C0, Ct = tica_covariances(fd, gd, t(w), t(wl))
    ((C0 * t(R0)).sum() + (Ct * t(Rt)).sum()).backward()
    t64 = lambda a: None if a is None else torch.from_numpy(a.astype(np.float64))
    f64, g64 = t64(f).requires_grad_(True), t64(g).requires_grad_(True)
    rC0, rCt = _torch_cov(f64, g64, t64(w), t64(wl))
    ((rC0 * t64(R0)).sum() + (rCt * t64(Rt)).sum()).backward()
    for got, want in ((C0, rC0), (Ct, rCt)):
        want = want.detach().numpy()
        np.testing.assert_allclose(got.detach().cpu().numpy(), want, rtol=0, atol=1e-9 * np.abs(want).max())
    sc = max(f64.grad.abs().max().item(), g64.grad.abs().max().item())
    np.testing.assert_allclose(fd.grad.cpu().numpy(), f64.grad.numpy(), rtol=0, atol=2e-6 * sc)
    np.testing.assert_allclose(gd.grad.cpu().numpy(), g64.grad.numpy(), rtol=0, atol=2e-6 * sc)
