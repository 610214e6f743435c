"""The exact covariance engine (tc_i8x3, csrc/cov_i8.cu) against an exact integer model of its arithmetic.

The engine rounds every value once, to a 23-bit fixed-point integer per column; after that its sums are
integer arithmetic (int8 digit products on the tensor cores) followed by a few FP64 operations.  The model
below restates that arithmetic -- prep, quantiser, digits, the Grams without their d0*d0 term, the H - T
finish, the column sums -- and computes its integer Grams EXACTLY (FP64 GEMMs on 12-bit splits, recombined
in int64).  The device result is then held to the rounding of its FP64 adds instead of a float tolerance:
six to seven orders of magnitude tighter than the float64-checker comparisons in test_gpu_parity.py, which
share the quantiser, the digit scheme and the finish between the two paths they compare.

Model of one call with n rows, lag L, M = n - L pairs (per column j, float32 unless noted):
    c = mean or 0, r = range or 1, amax = max(|xmax - c|, |xmin - c|) (1 if 0 or not finite)
    e = clamp(ilogb(kQMax / (amax * 1.0000002)), -100, 100), and e = min(e, 120 - ilogb(c)) if c != 0
    q = clamp(rint_even(fl32(x - c) * 2^e), +-kQMax),  s = 2^-e / (double) r,  U_t = q_t + q_{t+L}
    S0 = (sum_{t<M} q q^T - sum d0(q) d0(q)^T) s_i s_j                                   (upper triangle)
    St = 1/2 (G - 2 S0_int + H - T) s_i s_j,   G the same Gram of U,  H / T the full q q^T of the rows
         t < L / t >= M                                                                   (both triangles)
    a = (double) sum_{t<M} q * s,  b = (double) sum_{t>=L} q * s                          (bitwise)
"""
import math
import re
from fractions import Fraction

import numpy as np
import pytest
import torch

from conftest import synth_features

KQMAX = 4161536                     # 2^22 - 2^15: |U| <= 2^23 - 2^16, top digit in [-127, 127]
U53 = 2.0 ** -53
KNOBS = ("DCG_I8_FUSED", "DCG_I8_N", "DCG_I8_WINDOW_BYTES", "DCG_I8_ITEM_FRAMES", "DCG_I8_WINDOW_STAGES",
         "DCG_I8_RING", "DCG_I8_RING_BYTES", "DCG_I8_CLUSTERS", "DCG_I8_COOPERATIVE", "DCG_I8_DBG")


# ---- the model ------------------------------------------------------------------------------------
def ilogb(x):
    """ilogbf of finite nonzero float32 values."""
    return np.frexp(np.asarray(x, dtype=np.float32))[1].astype(np.int64) - 1


def prep(mean, rng, xmin, xmax):
    """i8_prep_kernel in float32: shift c, multiplier 2^e (float32), exponent e, scale 2^-e / range (float64)."""
    xmin = np.asarray(xmin, dtype=np.float32)
    xmax = np.asarray(xmax, dtype=np.float32)
    c = np.zeros_like(xmin) if mean is None else np.asarray(mean, dtype=np.float32)
    r = np.ones_like(xmin) if rng is None else np.asarray(rng, dtype=np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        amax = np.maximum(np.abs(xmax - c), np.abs(xmin - c))
        amax = np.where((amax > 0) & np.isfinite(amax), amax, np.float32(1))
        e = ilogb(np.float32(KQMAX) / (amax * np.float32(1.0000002)))
    e = np.clip(e, -100, 100)
    capped = (c != 0) & np.isfinite(c)
    e = np.where(capped, np.minimum(e, 120 - ilogb(np.where(capped, c, np.float32(1)))), e)
    m = np.ldexp(np.ones_like(c), e).astype(np.float32)
    scale = np.ldexp(1.0, -e) / r.astype(np.float64)
    return c, m, e, scale


def quantize(X, c, m):
    """q = clamp(rint_even(fl32(x - c) * 2^e), +-kQMax) as int64, and whether the clamp changed a value."""
    ct = torch.from_numpy(c).to(X.device)
    mt = torch.from_numpy(m).to(X.device)
    y = (X - ct) * mt                                  # float32 subtraction, then an exact power-of-two scaling
    q = torch.round(y).clamp_(-KQMAX, KQMAX).to(torch.int64)
    return q, bool((y.abs() > KQMAX + 0.5).any())


def digits(q):
    """Balanced base-256 digits (d0, d1, d2) of int64 q, each in [-128, 127]: q = d2 2^16 + d1 2^8 + d0."""
    d0 = ((q + 128) & 255) - 128
    r1 = (q - d0) >> 8
    d1 = ((r1 + 128) & 255) - 128
    return d0, d1, (r1 - d1) >> 8


def gram(A, B=None):
    """Exact int64 A^T B of int64 matrices with |entries| < 2^23 and fewer than 2^17 rows.  With A = h 2^12 + l
    (|h| <= 2^11, 0 <= l < 2^12) every partial sum of the four FP64 GEMMs is an integer below 2^53, so any
    summation order is exact, and the recombination stays below 2^63."""
    assert A.shape[0] < 2 ** 17
    def split(T):
        assert T.numel() == 0 or int(T.abs().max()) < 2 ** 23
        return (T >> 12).double(), (T & 4095).double()
    ha, la = split(A)
    hb, lb = (ha, la) if B is None else split(B)
    i64 = lambda t: t.to(torch.int64)                  # noqa: E731
    return (i64(ha.T @ hb) << 24) + ((i64(ha.T @ lb) + i64(la.T @ hb)) << 12) + i64(la.T @ lb)


def gram_no_d0d0(A):
    """What the tensor cores sum: A^T A without the d0 d0 digit product."""
    d0 = digits(A)[0].double()
    return gram(A) - (d0.T @ d0).to(torch.int64)


def abs_gram(A):
    a = A.abs().double()
    return a.T @ a


def tau_factor(M, item_min=128):
    """Relative bound (per unit of Tabs) on the device's rounding of one output entry.
    The digit-product sums of a partial (work item / flush) are bounded by sum |d|-weighted products, and
    |d2| 2^16 + |d1| 2^8 + |d0| <= 3.1 |q| (test_digit_magnitudes_are_at_most_3_1_times_q): 10 Tabs in all.
    A partial is rounded 3 times (digit recombination) and twice more (scaling); every partial is one FP64
    add into the result; the St finish adds 4 roundings and the model 3.  Partials per entry: at most
    one per item (>= item_min frames) and window (>= 4096 frames), plus up to 2 per frame split of the fused
    path (at most one split per cluster: 74 on a 148-SM B200)."""
    K = math.ceil(M / item_min) + math.ceil(M / 4096) + 148
    return 10.0 * (K + 12) * U53


def model_sums(X, lag, mean, rng, xmin, xmax, want_st=True, item_min=128):
    """The engine's outputs, computed exactly from the integers, with Tabs-based tolerances."""
    n = X.shape[0]
    M = n - lag
    tolist = lambda t: None if t is None else t.detach().cpu().numpy()   # noqa: E731
    c, m, _, s_np = prep(tolist(mean), tolist(rng), tolist(xmin), tolist(xmax))
    q, clamped = quantize(X, c, m)
    s = torch.from_numpy(s_np).to(X.device)
    ss = s[:, None] * s[None, :]
    tf = tau_factor(M, item_min)
    Z = q[:M]
    S0_int = gram_no_d0d0(Z)
    assert torch.equal(torch.diagonal(gram(Z)), (Z * Z).sum(0)), "the split GEMM is not exact on this device"
    T0 = abs_gram(Z)
    out = {"S0": S0_int.double() * s[:, None] * s[None, :], "tau0": tf * T0 * ss,
           "a": Z.sum(0).double() * s, "b": q[lag:].sum(0).double() * s, "clamped": clamped, "St": None}
    qmax = Z.abs().max(0).values.double() if M > 0 else torch.zeros_like(s)
    out["delta0"] = torch.where(qmax > 0, 2 * qmax - 1, torch.ones_like(qmax)) * s * s
    if lag > 0 and want_st:
        U = q[:M] + q[lag:]
        St_int = gram_no_d0d0(U) - 2 * S0_int + gram(q[:lag]) - gram(q[M:])
        out["St"] = 0.5 * (St_int.double() * s[:, None] * s[None, :])
        edges = torch.cat([q[:lag], q[M:]])
        out["taut"] = tf * 0.5 * (abs_gram(U) + 2 * T0 + abs_gram(edges)) * ss
        out["umax"] = int(U.abs().max())
    return out


# ---- host-only checks of the model ---------------------------------------------------------------
def _brute_gram(Q, omit_d0d0):
    """Python-int Gram of a small integer matrix (rows = frames), optionally without the d0 d0 term."""
    Q = [[int(v) for v in row] for row in Q.tolist()]
    f = len(Q[0])
    d0 = lambda v: ((v + 128) & 255) - 128           # noqa: E731
    return [[sum(r[i] * r[j] - (d0(r[i]) * d0(r[j]) if omit_d0d0 else 0) for r in Q) for j in range(f)]
            for i in range(f)]


EXTREME_Q = [0, 1, -1, 127, 128, -128, -129, 32895, 32896, -32896, 4095872, -4095872, 4096128, -4096128,
             KQMAX, -KQMAX, 2 * KQMAX, -2 * KQMAX, 2 ** 23 - 1, -(2 ** 23) + 1, 8191744, -8191744]


@pytest.mark.parametrize("kind", ["random_q", "random_u", "extreme"])
def test_split_gemm_gram_is_exact(kind):
    g = torch.Generator().manual_seed(11)
    if kind == "extreme":
        Q = torch.tensor(EXTREME_Q, dtype=torch.int64)[torch.randint(len(EXTREME_Q), (97, 7), generator=g)]
        Q[:, 0] = 4095872                                  # a constant digit-extreme column
        Q[:, 1] = -KQMAX * (1 - 2 * (torch.arange(97) % 2))  # alternating at the clamp limit
    else:
        lim = KQMAX if kind == "random_q" else 2 * KQMAX
        Q = torch.randint(-lim, lim + 1, (131, 6), generator=g, dtype=torch.int64)
    for omit in (False, True):
        got = (gram_no_d0d0(Q) if omit else gram(Q)).tolist()
        assert got == _brute_gram(Q, omit)
    B = torch.randint(-KQMAX, KQMAX + 1, (Q.shape[0], 3), generator=g, dtype=torch.int64)
    cross = [[sum(int(Q[t, i]) * int(B[t, j]) for t in range(Q.shape[0])) for j in range(3)]
             for i in range(Q.shape[1])]
    assert gram(Q, B).tolist() == cross


def test_gram_without_d0d0_is_the_sum_of_the_eight_digit_products():
    """The model's S0_int is what cov_i8_kernel accumulates: A 2^32 + B 2^24 + C 2^16 + D 2^8 over the digit
    products, with d0 d0 the only one left out."""
    g = torch.Generator().manual_seed(3)
    Q = torch.tensor(EXTREME_Q, dtype=torch.int64)[torch.randint(len(EXTREME_Q), (64, 5), generator=g)]
    Q = torch.cat([Q, torch.randint(-2 * KQMAX, 2 * KQMAX + 1, (64, 5), generator=g)])
    d0, d1, d2 = (d.double() for d in digits(Q))
    A = d2.T @ d2
    B = d2.T @ d1 + d1.T @ d2
    C = d2.T @ d0 + d1.T @ d1 + d0.T @ d2
    D = d1.T @ d0 + d0.T @ d1
    ints = [t.to(torch.int64) for t in (A, B, C, D)]
    assert torch.equal((ints[0] << 32) + (ints[1] << 24) + (ints[2] << 16) + (ints[3] << 8), gram_no_d0d0(Q))


def test_digits_reconstruct_q():
    lim = 2 ** 23 - 2 ** 16
    q = torch.arange(-lim, lim + 1, dtype=torch.int32)
    d0, d1, d2 = digits(q)
    assert torch.equal(d2 * 65536 + d1 * 256 + d0, q)
    for d in (d0, d1, d2):
        assert int(d.min()) >= -128 and int(d.max()) <= 127
    assert int(d2.abs().max()) == 127                   # reached at |U| = 2 kQMax
    # the digit-extreme values used on the device
    assert [int(v) for v in (d0[lim + 4095872], d1[lim + 4095872], d2[lim + 4095872])] == [-128, -128, 63]
    assert [int(v) for v in (d0[lim - 4096128], d1[lim - 4096128], d2[lim - 4096128])] == [-128, -128, -62]


def test_digit_magnitudes_are_at_most_3_1_times_q():
    """tau_factor relies on it: the unsigned digit expansion of q is at most 3.1 |q| (3.016 |q| at q = 32640,
    digits -128, -128, 1)."""
    lim = 2 ** 23 - 2 ** 16
    q = torch.arange(-lim, lim + 1, dtype=torch.int32)
    d0, d1, d2 = digits(q)
    P = d2.abs() * 65536 + d1.abs() * 256 + d0.abs()
    assert bool((10 * P <= 31 * q.abs()).all())


def test_lagged_pair_sum_stays_inside_three_digits():
    """|q| <= kQMax after the clamp, so |U| <= 2 kQMax = 2^23 - 2^16: the top digit of U stays in [-127, 127]."""
    x = torch.tensor([[-1e30, 1e30], [1e30, -1e30], [3.0, -3.0], [0.0, 0.0]], dtype=torch.float32)
    c, m, _, _ = prep(None, None, np.array([-1, -1], np.float32), np.array([1, 1], np.float32))
    q, clamped = quantize(x, c, m)
    assert clamped and int(q.abs().max()) == KQMAX
    U = q[:-1] + q[1:]
    assert int(U.abs().max()) <= 2 ** 23 - 2 ** 16 == 2 * KQMAX
    assert int(digits(torch.tensor([2 * KQMAX, -2 * KQMAX]))[2].abs().max()) == 127


def _amax_samples():
    g = np.random.default_rng(5)
    a = np.exp2(g.uniform(-60, 60, 4000)).astype(np.float32)
    edges = []
    for k in range(-30, 31):
        for base in (np.float32(2.0 ** k), np.float32(KQMAX * 2.0 ** k)):
            edges += [base, np.nextafter(base, np.float32(0)), np.nextafter(base, np.float32(np.inf))]
    return np.concatenate([a, np.array(edges, dtype=np.float32)])


def test_exponent_is_the_finest_grid_that_fits():
    """For uncapped columns (c = 0), 2^e is the largest power of two with amax 2^e <= kQMax, up to the one-ulp
    slack i8_prep_kernel allows: amax 2^e <= kQMax < 2 amax 2^e (1 + 2^-21)."""
    amax = _amax_samples()
    _, m, e, scale = prep(None, None, -amax, amax)
    for a, ej, mj, sj in zip(amax.tolist(), e.tolist(), m.tolist(), scale.tolist()):
        lo = Fraction(a) * Fraction(2) ** ej
        assert lo <= KQMAX < 2 * lo * (1 + Fraction(1, 2 ** 21)), (a, ej)
        assert mj == 2.0 ** ej and sj == 2.0 ** -ej


def test_exponent_cap_keeps_the_shift_finite():
    """With a shift c, c 2^e must stay finite in float32 (the fused kernel's single FMA): e <= 120 - ilogb(c)."""
    c = np.array([3e38, 1e30, -1e20, 1.0, 1e-30], dtype=np.float32)
    amax = np.full_like(c, 1e-3)
    _, m, e, _ = prep(c, np.ones_like(c), c - amax, c + amax)
    assert np.all(np.isfinite(c * m))
    assert np.all(e <= 120 - ilogb(c))


def test_quantiser_model_rounds_the_float32_difference():
    """q is rint_even of the float32 difference scaled by 2^e, clamped: checked against float64 arithmetic."""
    g = np.random.default_rng(9)
    X = (g.standard_normal((500, 4)) * [1, 1e3, 1e-4, 7] + [0, 1e5, 1, -3]).astype(np.float32)
    mean = X.astype(np.float64).mean(0).astype(np.float32)
    c, m, e, _ = prep(mean, np.ones(4, np.float32), X.min(0), X.max(0))
    q, clamped = quantize(torch.from_numpy(X), c, m)
    diff = (X - c).astype(np.float64) * np.exp2(e.astype(np.float64))     # float32 difference, exact scaling
    assert not clamped
    assert np.array_equal(q.numpy(), np.clip(np.rint(diff), -KQMAX, KQMAX).astype(np.int64))
    assert int(q.abs().max()) <= KQMAX and int(q.abs().max()) > KQMAX // 2


# ---- device against model -------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from deep_cartograph_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


def standardisation(X):
    """float32 mean and sample standard deviation of the columns (1 where a column is constant)."""
    X64 = X.astype(np.float64)
    sd = X64.std(0, ddof=1) if X.shape[0] > 1 else np.ones(X.shape[1])
    return X64.mean(0).astype(np.float32), np.where(sd > 0, sd, 1.0).astype(np.float32)


def run_engine(X, lag, mean, rng, xmin, xmax, monkeypatch, capfd, block=0, want_st=True, **env):
    """One tc_i8x3 call with the DCG_I8_* knobs in ``env`` (all others unset), DCG_I8_DEBUG on.  Adds the
    fused rounds the engine reported: [(round, rounds, windows)], empty when the two-kernel path ran."""
    from deep_cartograph_b200 import ops
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("DCG_I8_DEBUG", "1")
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    capfd.readouterr()
    out = ops.lagged_covariance(X, lag, mean, rng, block=block, engine="tc_i8x3", want_st=want_st,
                                xmin=xmin, xmax=xmax)
    torch.cuda.synchronize()
    err = capfd.readouterr().err
    out["rounds"] = [tuple(int(v) for v in r)
                     for r in re.findall(r"\[dcg i8 fused\] round (\d+)/(\d+): .* windows (\d+)", err)]
    out["windows"] = err.count("[dcg i8] quantize:")
    return out


def check(out, mdl, block=0, lag=0, want_st=True, what=""):
    f = mdl["S0"].shape[0]
    dev = mdl["S0"].device
    inblock = torch.ones((f, f), dtype=torch.bool, device=dev)
    if block:
        blk = torch.arange(f, device=dev) // block
        inblock = blk[:, None] == blk[None, :]
    assert (int(out["clamped"].item()) != 0) == mdl["clamped"], f"{what}: clamp flag"
    assert torch.equal(out["a"], mdl["a"]), f"{what}: column sums a differ from the model"
    assert torch.equal(out["b"], mdl["b"]), f"{what}: column sums b differ from the model"
    tests = [("S0", inblock.triu(), "tau0")]
    if lag > 0 and want_st:
        tests.append(("St", inblock, "taut"))
    else:
        assert out["St"] is None
    for k, mask, tk in tests:
        err = (out[k] - mdl[k]).abs()
        bad = mask & (err > mdl[tk])
        if bool(bad.any()):
            i, j = (int(v) for v in bad.nonzero()[0])
            pytest.fail(f"{what}: {k}[{i},{j}] = {float(out[k][i, j])!r}, model {float(mdl[k][i, j])!r}, "
                        f"|diff| {float(err[i, j]):.3e} > tau {float(mdl[tk][i, j]):.3e} "
                        f"({int(bad.sum())} entries)")
    # the check must be able to see a one-unit change of the largest |q| in every column
    d = torch.diagonal(mdl["tau0"])
    weak = mdl["delta0"] <= 10 * d
    assert not bool(weak.any()), f"{what}: tolerance too loose to see a +-1 change of q in columns " \
                                 f"{weak.nonzero().flatten()[:8].tolist()}"


def device_inputs(X, dev, ld_pad=0, misalign=False):
    """X on the device, with ``ld_pad`` extra floats per row and, if ``misalign``, a base pointer one float
    off 16-byte alignment."""
    n, f = X.shape
    off = 1 if misalign else 0
    buf = torch.zeros(off + n * (f + ld_pad), dtype=torch.float32, device=dev)
    Xd = buf[off:].view(n, f + ld_pad)[:, :f]
    Xd.copy_(torch.from_numpy(X))
    assert (Xd.data_ptr() % 16 != 0) == misalign
    return Xd


CASES = {
    # name: (n, f, lag, block, ld_pad, standardise, misalign, want_st, fused under DCG_I8_FUSED=2)
    "c1_shape": (164, 54, 1, 0, 0, True, False, True, False),
    "5000x300_lag7": (5000, 300, 7, 0, 0, True, False, True, True),
    "raw_3001x1000_lag3": (3001, 1000, 3, 0, 0, False, False, True, True),
    "lag128": (2500, 640, 128, 0, 0, True, False, True, True),
    "block100_padded": (20011, 1003, 33, 100, 1, True, False, True, True),
    "ragged_block99": (6000, 1000, 4, 99, 0, True, False, True, True),
    "lag0": (9000, 331, 0, 0, 0, True, False, True, True),
    "s0_only_lag5": (4000, 300, 5, 0, 0, True, False, False, True),
    "one_pair": (50, 200, 49, 0, 0, True, False, True, True),
    "f1": (3000, 1, 2, 0, 0, True, False, True, False),
    "f5": (3000, 5, 2, 0, 0, True, False, True, False),
    "misaligned": (4000, 300, 5, 0, 0, True, True, True, True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["0", "2"])
@pytest.mark.parametrize("name", list(CASES))
def test_exact_engine_equals_integer_model(dev, monkeypatch, capfd, name, mode):
    n, f, lag, block, ld_pad, standardise, misalign, want_st, fusable = CASES[name]
    X = synth_features(n, f, seed=n + f)
    Xd = device_inputs(X, dev, ld_pad, misalign)
    mean = rng = None
    if standardise:
        mean, rng = (torch.from_numpy(v).to(dev) for v in standardisation(X))
    xmin, xmax = Xd.amin(0), Xd.amax(0)
    out = run_engine(Xd, lag, mean, rng, xmin, xmax, monkeypatch, capfd, block=block, want_st=want_st,
                     DCG_I8_FUSED=mode)
    assert bool(out["rounds"]) == (mode == "2" and fusable), f"fused rounds {out['rounds']}"
    mdl = model_sums(Xd, lag, mean, rng, xmin, xmax, want_st=want_st)
    assert not mdl["clamped"]
    check(out, mdl, block, lag, want_st, f"{name} fused={mode}")


def edge_columns(n, seed=0):
    """Columns where quantisers go wrong, with their own shift / range (mean 0, range 1 where the column's
    raw values are the point)."""
    g = np.random.default_rng(seed)
    t = np.arange(n)
    cols, raw = [], []
    def add(v, is_raw=False):
        cols.append(np.asarray(v, dtype=np.float32))
        raw.append(is_raw)
    add(np.full(n, 3.7))                                              # constant
    add(1e5 + g.standard_normal(n))                                   # |mean| / std = 1e5
    add(1.0 + 1e-6 * g.standard_normal(n))                            # std = 1e-6
    add(g.standard_cauchy(n))                                         # heavy tails
    add(np.zeros(n))                                                  # all zeros
    add(np.where(t < n // 2, 0.0, 3.0 * g.standard_normal(n)))        # half zeros
    add(np.clip(g.standard_normal(n), -1.5, 1.5))                     # many values exactly at xmin / xmax
    thr = np.float32(KQMAX * 2.0 ** -21)                              # where e steps from 21 to 20
    for a in (np.float32(2.0), np.nextafter(np.float32(2.0), np.float32(0)), np.nextafter(np.float32(2.0), np.float32(4)),
              thr, np.nextafter(thr, np.float32(0)), np.nextafter(thr, np.float32(4)), np.float32(0.25)):
        v = (g.uniform(-0.5, 0.5, n) * a).astype(np.float32)
        v[g.integers(n)] = a if a != np.float32(0.25) else -a         # amax reached once (negative for 0.25)
        add(v, True)
    for qv in (4095872, -4095872, -4096128):                         # digit-extreme constant columns
        add(np.full(n, np.float32(qv * 2.0 ** -20)), True)
    add(np.float32(4095872 * 2.0 ** -20) * np.where(t % 2 == 0, 1, -1), True)      # alternating sign
    add(np.float32(4096128 * 2.0 ** -20) * np.where(t % 3 == 0, -1, 1), True)
    return np.stack(cols, 1), np.array(raw)


def edge_matrix(n, f, seed):
    E, raw = edge_columns(n, seed)
    X = np.ascontiguousarray(np.concatenate([E, synth_features(n, f - E.shape[1], seed=seed)], 1))
    mean, rng = standardisation(X)
    mean[:E.shape[1]][raw] = 0.0
    rng[:E.shape[1]][raw] = 1.0
    return X, mean, rng


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["0", "2"])
def test_exact_engine_edge_columns(dev, monkeypatch, capfd, mode):
    n, f, lag = 5000, 200, 3
    X, mean, rng = edge_matrix(n, f, seed=21)
    Xd = torch.from_numpy(X).to(dev)
    mean, rng = torch.from_numpy(mean).to(dev), torch.from_numpy(rng).to(dev)
    xmin, xmax = Xd.amin(0), Xd.amax(0)
    out = run_engine(Xd, lag, mean, rng, xmin, xmax, monkeypatch, capfd, DCG_I8_FUSED=mode)
    assert bool(out["rounds"]) == (mode == "2")
    mdl = model_sums(Xd, lag, mean, rng, xmin, xmax)
    check(out, mdl, 0, lag, True, f"edge columns fused={mode}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["0", "2"])
def test_exact_engine_long_series_at_the_int32_flush_limit(dev, monkeypatch, capfd, mode):
    """Work items of 32768 frames (the int32 headroom 3 128^2 32768 < 2^31) over digit-extreme columns."""
    n, f, lag = 70000, 256, 10
    X, mean, rng = edge_matrix(n, f, seed=22)
    Xd = torch.from_numpy(X).to(dev)
    mean, rng = torch.from_numpy(mean).to(dev), torch.from_numpy(rng).to(dev)
    xmin, xmax = Xd.amin(0), Xd.amax(0)
    out = run_engine(Xd, lag, mean, rng, xmin, xmax, monkeypatch, capfd, DCG_I8_FUSED=mode,
                     DCG_I8_ITEM_FRAMES=32768)
    assert bool(out["rounds"]) == (mode == "2")
    # items of 32768 frames; the fused path flushes every >= 128 stages of a frame split
    mdl = model_sums(Xd, lag, mean, rng, xmin, xmax, item_min=16384)
    check(out, mdl, 0, lag, True, f"long series fused={mode}")


# ---- geometry sweep: every setting of the knobs gives the same model ------------------------------------
SWEEP_CASES = {
    # name: (n, f, lag, block)
    "standardised": (40000, 384, 10, 0),
    "block200": (12000, 650, 5, 200),     # blocks of 200, 200, 200 and 50 features
}
SWEEP = {
    "split_default": ("0", {}),
    "split_N32": ("0", {"DCG_I8_N": 32}),
    "split_N64": ("0", {"DCG_I8_N": 64}),
    "split_N96": ("0", {"DCG_I8_N": 96}),
    "split_N128": ("0", {"DCG_I8_N": 128}),
    "split_windows4096": ("0", {"DCG_I8_WINDOW_BYTES": 1}),
    "split_items128": ("0", {"DCG_I8_ITEM_FRAMES": 128}),
    "fused_default": ("2", {}),
    "fused_window_stages1": ("2", {"DCG_I8_WINDOW_STAGES": 1}),
    "fused_ring2": ("2", {"DCG_I8_RING": 2}),
    "fused_ring8": ("2", {"DCG_I8_RING": 8}),
    "fused_clusters3": ("2", {"DCG_I8_CLUSTERS": 3}),
}


@pytest.fixture(scope="module")
def sweep_inputs(dev):
    cache = {}

    def get(name):
        if name not in cache:
            n, f, lag, block = SWEEP_CASES[name]
            X = synth_features(n, f, seed=f + lag)
            Xd = torch.from_numpy(X).to(dev)
            mean, rng = (torch.from_numpy(v).to(dev) for v in standardisation(X))
            xmin, xmax = Xd.amin(0), Xd.amax(0)
            cache[name] = (Xd, mean, rng, xmin, xmax, model_sums(Xd, lag, mean, rng, xmin, xmax), {})
        return cache[name]
    return get


@pytest.mark.gpu
@pytest.mark.parametrize("setting", list(SWEEP))
@pytest.mark.parametrize("case", list(SWEEP_CASES))
def test_exact_engine_geometry_sweep(dev, monkeypatch, capfd, sweep_inputs, case, setting):
    n, f, lag, block = SWEEP_CASES[case]
    Xd, mean, rng, xmin, xmax, mdl, seen = sweep_inputs(case)
    mode, env = SWEEP[setting]
    out = run_engine(Xd, lag, mean, rng, xmin, xmax, monkeypatch, capfd, block=block, DCG_I8_FUSED=mode, **env)
    assert bool(out["rounds"]) == (mode == "2")
    if "DCG_I8_WINDOW_BYTES" in env:
        assert out["windows"] == math.ceil((n - lag) / 4096)
    if "DCG_I8_WINDOW_STAGES" in env:
        assert out["rounds"][0][2] > 16, "the window counters must be reused"
    if "DCG_I8_CLUSTERS" in env:
        assert out["rounds"][0][1] > 1, "tiles must outnumber clusters"
    check(out, mdl, block, lag, True, f"{case} {setting}")
    # column sums are integer totals: identical whatever the geometry
    for k in ("a", "b"):
        seen.setdefault(k, out[k].clone())
        assert torch.equal(out[k], seen[k])


# ---- clamping: bounds narrower / wider than the data -------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["0", "2"])
def test_exact_engine_clamps_to_narrow_bounds(dev, monkeypatch, capfd, mode):
    """Bounds of the first half of the frames: values of the second half beyond them are clamped to +-kQMax
    (the flag is set), and the sums are those of the clamped integers."""
    n, f, lag = 6000, 300, 5
    X = synth_features(n, f, seed=31)
    Xd = torch.from_numpy(X).to(dev)
    mean, rng = (torch.from_numpy(v).to(dev) for v in standardisation(X))
    xmin, xmax = Xd[:n // 2].amin(0), Xd[:n // 2].amax(0)
    out = run_engine(Xd, lag, mean, rng, xmin, xmax, monkeypatch, capfd, DCG_I8_FUSED=mode)
    mdl = model_sums(Xd, lag, mean, rng, xmin, xmax)
    assert mdl["clamped"] and int(out["clamped"].item()) > 0
    assert mdl["umax"] == 2 * KQMAX                      # lagged pair sums reach a top digit of 127
    check(out, mdl, 0, lag, True, f"narrow bounds fused={mode}")


@pytest.mark.gpu
@pytest.mark.parametrize("widen", [1, 10])
@pytest.mark.parametrize("mode", ["0", "2"])
def test_exact_engine_bounds_that_contain_the_data(dev, monkeypatch, capfd, mode, widen):
    """Bounds equal to the data's extremes (values exactly at them) or 10x wider (a coarser grid): no flag."""
    n, f, lag = 6000, 300, 5
    X = synth_features(n, f, seed=32)
    Xd = torch.from_numpy(X).to(dev)
    mean, rng = (torch.from_numpy(v).to(dev) for v in standardisation(X))
    xmin, xmax = Xd.amin(0), Xd.amax(0)
    if widen > 1:
        xmin, xmax = mean - widen * (mean - xmin), mean + widen * (xmax - mean)
    out = run_engine(Xd, lag, mean, rng, xmin, xmax, monkeypatch, capfd, DCG_I8_FUSED=mode)
    mdl = model_sums(Xd, lag, mean, rng, xmin, xmax)
    assert int(out["clamped"].item()) == 0 and not mdl["clamped"]
    check(out, mdl, 0, lag, True, f"bounds x{widen} fused={mode}")


# ---- shards ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["0", "2"])
def test_exact_engine_shards_add_up_to_the_whole_series(dev, monkeypatch, capfd, mode):
    """With the global bounds passed to every shard (as the sharded calculator does), frame shards with their
    lag halo quantise every frame as the whole series does, so their sums add up to the whole-series sums:
    what lets a multi-GPU run reproduce a single-GPU one."""
    n, f, lag, cut = 12007, 300, 7, 5003
    X = synth_features(n, f, seed=41)
    Xd = torch.from_numpy(X).to(dev)
    mean, rng = (torch.from_numpy(v).to(dev) for v in standardisation(X))
    xmin, xmax = Xd.amin(0), Xd.amax(0)
    parts = [Xd, Xd[:cut + lag], Xd[cut:]]
    outs = [run_engine(P, lag, mean, rng, xmin, xmax, monkeypatch, capfd, DCG_I8_FUSED=mode) for P in parts]
    mdls = [model_sums(P, lag, mean, rng, xmin, xmax) for P in parts]
    for i, (o, m) in enumerate(zip(outs, mdls)):
        check(o, m, 0, lag, True, f"part {i} fused={mode}")
    whole, s1, s2 = outs
    for k, tk, mask in (("S0", "tau0", torch.ones(f, f, dtype=torch.bool, device=dev).triu()),
                        ("St", "taut", torch.ones(f, f, dtype=torch.bool, device=dev))):
        tol = sum(m[tk] for m in mdls)
        err = (s1[k] + s2[k] - whole[k]).abs()
        assert bool((err[mask] <= tol[mask]).all()), k
    for k in ("a", "b"):
        err = (s1[k] + s2[k] - whole[k]).abs()
        assert bool((err <= 4 * U53 * (s1[k].abs() + s2[k].abs())).all()), k
