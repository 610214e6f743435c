"""GPU parity tests: every CUDA entry point (through the C-ABI via ctypes) against the CPU
oracle on the same seeded inputs, and the calculators / step APIs against the reference's golden
artefacts (C1 fixture).  Run on the B200 box: ``pytest -m gpu``.

Tolerances (BASELINE.json north_star): covariances / eigenvalues 1e-5 relative to float64
(normwise), eigenvectors 1e-5 up to sign, projections 1e-4, KMeans labels identical from fixed
initial centroids with exact-tie frames counted and reported.
"""
import copy
import os

import numpy as np
import pandas as pd
import pytest
import torch

import oracle
from conftest import GOLDEN, synth_features

pytestmark = pytest.mark.gpu

ENGINES = ["simt_f32", "tc_3xtf32", "tc_3xf16", "tc_i8x3"]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from deep_cartograph_b200 import _lib
    _lib.load()            # fail loudly if the extension is missing
    return torch.device("cuda:0")


def _cuda(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


# ------------------------------------------------------------------------------------------------
# A2 column statistics
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,f", [(164, 54), (1, 7), (5000, 1000), (3001, 4950 // 5), (777, 3),
                                 (20000, 130), (1025, 128)])
def test_colstats_matches_oracle(dev, n, f):
    from deep_cartograph_b200 import ops
    X = synth_features(n, f, seed=n + f)
    st = ops.column_stats(_cuda(X, dev))
    ref = oracle.column_stats(X)
    assert st["n"] == n
    np.testing.assert_allclose(st["mean"].cpu().numpy(), ref["mean"], rtol=2e-7, atol=1e-9)
    if n > 1:
        std = np.sqrt(st["m2"].cpu().numpy() / (n - 1))
        np.testing.assert_allclose(std, ref["std"], rtol=3e-6)
    assert np.array_equal(st["min"].cpu().numpy(), ref["min"].astype(np.float32))   # exact
    assert np.array_equal(st["max"].cpu().numpy(), ref["max"].astype(np.float32))


def test_colstats_strided_rows_and_golden(dev, c1):
    from deep_cartograph_b200 import ops
    X = c1["X"]
    buf = torch.zeros((X.shape[0], 64), dtype=torch.float32, device=dev)
    buf[:, :54] = _cuda(X, dev)
    st = ops.column_stats(buf[:, :54])            # ld = 64 != f
    std = torch.sqrt(st["m2"] / (X.shape[0] - 1)).to(torch.float32).cpu().numpy()
    np.testing.assert_allclose(st["mean"].to(torch.float32).cpu().numpy(), c1["tica_features_norm_mean"], atol=2e-7)
    np.testing.assert_allclose(std, c1["tica_features_norm_range"], rtol=1e-6)


# ------------------------------------------------------------------------------------------------
# A4 standardisation (bit-exact IEEE sub + div)
# ------------------------------------------------------------------------------------------------
def test_sharded_statistics_pack_and_merge_kernels(dev):
    """dcg_stats_pack / dcg_stats_merge (the two launches around the statistics all-gather of the frame-sharded
    path): shards of unequal length, one of them EMPTY, merged == the statistics of the whole matrix."""
    from deep_cartograph_b200 import ops
    n, f = 50_001, 333
    X = synth_features(n, f, seed=9)
    Xd = _cuda(X, dev)
    cuts = [0, 17_000, 17_000, 40_001, n]                  # the second shard is empty
    recs = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        if b > a:
            st = ops.column_stats(Xd[a:b])
        else:
            z64, z32 = torch.zeros(f, dtype=torch.float64, device=dev), torch.zeros(f, dtype=torch.float32, device=dev)
            st = {"n": 0, "mean": z64, "m2": z64.clone(), "min": z32, "max": z32.clone()}
        recs.append(ops.stats_pack(st))
        assert recs[-1].numel() == 1 + 4 * f and float(recs[-1][0]) == b - a
    m = ops.stats_merge(torch.cat(recs), len(recs), f)
    whole = oracle.column_stats(X)
    assert float(m["n"].item()) == n
    np.testing.assert_allclose(m["mean"].cpu().numpy(), whole["mean"], rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(np.sqrt(m["m2"].cpu().numpy() / (n - 1)), whole["std"], rtol=2e-6)
    one = ops.column_stats(Xd)        # and == the single-launch statistics (per-thread partial sums are shifted FP32)
    np.testing.assert_allclose(m["mean"].cpu().numpy(), one["mean"].cpu().numpy(), rtol=1e-7, atol=1e-8)
    np.testing.assert_allclose(m["m2"].cpu().numpy(), one["m2"].cpu().numpy(), rtol=1e-6)
    np.testing.assert_array_equal(m["min"].cpu().numpy(), whole["min"].astype(np.float32))
    np.testing.assert_array_equal(m["max"].cpu().numpy(), whole["max"].astype(np.float32))


@pytest.mark.parametrize("n,f", [(164, 54), (4096, 1000), (1000, 4950 // 5), (513, 7), (10000, 4), (33, 2)])
def test_standardize_is_bit_exact(dev, n, f):
    from deep_cartograph_b200 import ops
    X = synth_features(n, f, seed=3)
    st = oracle.column_stats(X)
    m, r = oracle.prepare_normalization(st, "mean_std")
    ref = oracle.standardize(X, m, r)
    Z = ops.standardize_(_cuda(X, dev), _cuda(m.astype(np.float32), dev), _cuda(r.astype(np.float32), dev))
    got = Z.cpu().numpy()
    mism = np.count_nonzero(got != ref)
    assert mism == 0, f"{mism} of {got.size} elements differ from IEEE (x-m)/r"


# ------------------------------------------------------------------------------------------------
# A5/A6 covariance sums
# ------------------------------------------------------------------------------------------------
def _cov_case(dev, X, lag, engine, standardise=True, block=0):
    from deep_cartograph_b200 import ops
    st = oracle.column_stats(X)
    m, r = oracle.prepare_normalization(st, "mean_std" if standardise else None)
    Z = oracle.standardize(X, m, r) if standardise else X
    mean = _cuda(m.astype(np.float32), dev) if standardise else None
    rng = _cuda(r.astype(np.float32), dev) if standardise else None
    s = ops.lagged_covariance(_cuda(X, dev), lag, mean, rng, block=block, engine=engine)
    torch.cuda.synchronize()
    if lag > 0:
        S0, St, a, b, M = oracle.lagged_sums(Z, lag)
    else:
        Z64 = Z.astype(np.float64)
        S0, St, a, b, M = Z64.T @ Z64, None, Z64.sum(0), Z64.sum(0), Z.shape[0]
    return s, (S0, St, a, b, M)


def _assert_cov_close(s, ref, tol, block=0):
    S0, St, a, b, M = ref
    F = S0.shape[0]
    assert s["M"] == M
    if "clamped" in s:
        # the exact integer engine returns the SYMMETRIC part of St (all the reference uses: mlcolvar
        # symmetrises C_tau) and reports how many values fell outside the column bounds it was given
        assert int(s["clamped"].item()) == 0
        if St is not None:
            St = 0.5 * (St + St.T)
    mask_u = np.triu(np.ones((F, F), dtype=bool))
    mask_f = np.ones((F, F), dtype=bool)
    if block:
        blk = np.arange(F) // block
        same = blk[:, None] == blk[None, :]
        mask_u &= same
        mask_f &= same
    got0 = s["S0"].cpu().numpy()
    scale0 = np.abs(S0).max()
    assert np.abs(got0 - S0)[mask_u].max() <= tol * scale0, np.abs(got0 - S0)[mask_u].max() / scale0
    if St is not None:
        gott = s["St"].cpu().numpy()
        scalet = np.abs(St).max()
        assert np.abs(gott - St)[mask_f].max() <= tol * scalet, np.abs(gott - St)[mask_f].max() / scalet
    np.testing.assert_allclose(s["a"].cpu().numpy(), a, rtol=1e-6, atol=1e-6 * M ** 0.5 + 1e-4)
    np.testing.assert_allclose(s["b"].cpu().numpy(), b, rtol=1e-6, atol=1e-6 * M ** 0.5 + 1e-4)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("n,f,lag", [(164, 54, 1), (3000, 256, 10), (2500, 1000, 10), (999, 130, 7),
                                     (4100, 495, 1), (600, 64, 33), (300, 5, 2), (2048, 384, 128)])
def test_cov_sums_match_float64(dev, engine, n, f, lag):
    X = synth_features(n, f, seed=n)
    s, ref = _cov_case(dev, X, lag, engine)
    _assert_cov_close(s, ref, 1e-5)


@pytest.mark.parametrize("engine", ENGINES)
def test_cov_lag0_gram_and_unstandardised(dev, engine):
    X = synth_features(1500, 200, seed=5)
    s, ref = _cov_case(dev, X, 0, engine, standardise=True)
    assert s["St"] is None
    _assert_cov_close(s, ref, 1e-5)
    Z = oracle.standardize(X, *oracle.prepare_normalization(oracle.column_stats(X), "mean_std"))
    s, ref = _cov_case(dev, Z, 3, engine, standardise=False)
    _assert_cov_close(s, ref, 1e-5)


@pytest.mark.parametrize("engine", ENGINES)
def test_cov_block_diagonal_mode(dev, engine):
    X = synth_features(2000, 990, seed=11)
    s, ref = _cov_case(dev, X, 5, engine, block=99)
    _assert_cov_close(s, ref, 1e-5, block=99)


@pytest.mark.parametrize("engine", ENGINES)
def test_cov_linearity_over_frame_chunks(dev, engine):
    """Size-independent property: sums over [0,n) == sums over two overlapping-by-lag halves."""
    from deep_cartograph_b200 import ops
    n, f, lag = 20000, 512, 10
    X = _cuda(synth_features(n, f, seed=2), dev)
    whole = ops.lagged_covariance(X, lag, engine=engine)
    h = n // 2
    first = ops.lagged_covariance(X[:h + lag], lag, engine=engine)    # own rows + halo
    second = ops.lagged_covariance(X[h:], lag, engine=engine)
    assert first["M"] + second["M"] == whole["M"]
    for k in ("S0", "St"):
        tot = torch.triu(first[k] + second[k]) if k == "S0" else first[k] + second[k]
        ref = torch.triu(whole[k]) if k == "S0" else whole[k]
        err = (tot - ref).abs().max().item() / ref.abs().max().item()
        assert err < 2e-6, (k, err)


@pytest.mark.parametrize("f,ld_pad,block", [(990, 0, 0), (990, 2, 0), (495, 1, 0), (998, 0, 499), (4950 // 5, 0, 99)])
def test_cov_unaligned_rows_and_block_origins(dev, f, ld_pad, block):
    """Row strides that are not multiples of 4 floats (8- and 4-byte load paths of the tcgen05
    engine), feature counts that are not multiples of 4, and diagonal blocks that start at odd
    columns (the C3 shape: blocks of 495 features)."""
    from deep_cartograph_b200 import ops
    n, lag = 3000, 7
    X = synth_features(n, f, seed=f + ld_pad)
    buf = torch.zeros((n, f + ld_pad), dtype=torch.float32, device=dev)
    buf[:, :f] = torch.from_numpy(X).to(dev)
    Xd = buf[:, :f]                                           # row stride f + ld_pad floats
    st = oracle.column_stats(X)
    m, r = oracle.prepare_normalization(st, "mean_std")
    Z = oracle.standardize(X, m, r)
    s = ops.lagged_covariance(Xd, lag, _cuda(m.astype(np.float32), dev), _cuda(r.astype(np.float32), dev),
                              block=block, engine="tc_3xtf32")
    _assert_cov_close(s, oracle.lagged_sums(Z, lag), 1e-5, block=block)


@pytest.mark.parametrize("n,f,lag,block,ld_pad,standardise", [
    (5000, 300, 7, 0, 0, True),            # one round, several frame splits per tile
    (20011, 1003, 33, 100, 1, True),       # block mode, blocks that start at odd columns, padded rows, lag > 32
    (9000, 331, 0, 0, 0, True),            # lag 0 (PCA): Z planes only
    (12000, 2000, 10, 0, 0, True),         # 136 tiles: two rounds of the persistent kernel
    (6000, 4950, 10, 495, 2, True),        # the C3 level-1 plan: 100 tiles, rounds that quantise feature sub-ranges
    (3001, 1000, 3, 0, 0, False),          # raw features (mode None), a last window that is partly empty
    (200, 1000, 10, 0, 0, True),           # fewer frames than one window: a single, mostly empty one
    (2500, 640, 128, 0, 0, True),          # a lag longer than a quantiser item (32 frames) and than a stage
])
def test_cov_exact_engine_fused_kernel_equals_two_kernel_path(dev, monkeypatch, n, f, lag, block, ld_pad, standardise):
    """tc_i8x3 has two implementations of the same integer arithmetic: quantise kernel + contraction kernel
    (planes in HBM), and the fused persistent kernel (quantiser warps -> L2-resident ring -> TMA -> tcgen05).
    Both must give the float64 checker's sums to 1e-5 and each other's to rounding of the FP64 adds; the column
    sums are integer totals and must be IDENTICAL."""
    from deep_cartograph_b200 import ops
    from oracle import float64_device as f64
    X = synth_features(n, f, seed=n + f)
    buf = torch.zeros((n, f + ld_pad), dtype=torch.float32, device=dev)
    buf[:, :f] = torch.from_numpy(X).to(dev)
    Xd = buf[:, :f]
    mean = rng = None
    if standardise:
        st = ops.column_stats(Xd)
        mean = st["mean"].float()
        rng = torch.sqrt(st["m2"] / (n - 1)).float()
    out = {}
    for mode in ("2", "0"):                # 2 = fused whenever the tile plan allows it, 0 = never
        monkeypatch.setenv("DCG_I8_FUSED", mode)
        out[mode] = ops.lagged_covariance(Xd, lag, mean, rng, block=block, engine="tc_i8x3")
        torch.cuda.synchronize()
        assert int(out[mode]["clamped"].item()) == 0
    ref = f64.lagged_sums(Xd, lag, mean, rng)
    mask = torch.ones((f, f), dtype=torch.bool, device=dev).triu()
    if block:
        blk = torch.arange(f, device=dev) // block
        mask &= blk[:, None] == blk[None, :]
    for k in ("S0", "St"):
        if lag == 0 and k == "St":
            continue
        r = ref[k] if k == "S0" else 0.5 * (ref[k] + ref[k].T)
        a, b, r = (torch.where(mask, t, torch.zeros_like(t)) for t in (out["2"][k], out["0"][k], r))
        assert float((a - r).norm() / r.norm()) < 1e-6, k
        assert float((a - b).abs().max() / b.abs().max()) < 1e-14, k
    assert torch.equal(out["2"]["a"], out["0"]["a"]) and torch.equal(out["2"]["b"], out["0"]["b"])


@pytest.mark.parametrize("fused", ["2", "0"])
@pytest.mark.parametrize("n,f,lag,block", [(3000, 300, 7, 0), (1500, 2000, 10, 0), (2000, 990, 5, 99), (1000, 331, 0, 0),
                                           (130, 1000, 1, 0)])
def test_cov_exact_engine_stays_inside_its_workspace(dev, monkeypatch, fused, n, f, lag, block):
    """The exact engine's workspace (digit-plane ring or window, tables, counters) between two canary regions:
    nothing outside the `dcg_cov_i8_workspace_bytes` bytes handed over may be written, by either implementation
    (fused persistent kernel / quantise + contraction kernels), and the outputs must not depend on what the
    workspace held before."""
    from deep_cartograph_b200 import ops, _lib
    monkeypatch.setenv("DCG_I8_FUSED", fused)
    lib = _lib.load()
    X = _cuda(synth_features(n, f, seed=n + f), dev)
    st = ops.column_stats(X)
    mean, rng = st["mean"].float(), torch.sqrt(st["m2"] / (n - 1)).float()
    nbytes = int(lib.dcg_cov_i8_workspace_bytes(n, f, lag, block))
    assert nbytes > 0
    guard = 1 << 20
    outs = []
    for fill in (0xA5, 0x00):
        buf = torch.full((nbytes + 2 * guard,), 0x5A, dtype=torch.uint8, device=dev)
        buf[guard:guard + nbytes] = fill
        S0 = torch.empty((f, f), dtype=torch.float64, device=dev)
        St = torch.empty((f, f), dtype=torch.float64, device=dev) if lag > 0 else None
        a, b = (torch.empty(f, dtype=torch.float64, device=dev) for _ in range(2))
        info = torch.empty(1, dtype=torch.int32, device=dev)
        ops._call(dev, "dcg_cov_lag_i8_f32", X.data_ptr(), n, f, X.stride(0), lag, mean.data_ptr(), rng.data_ptr(),
                  st["min"].data_ptr(), st["max"].data_ptr(), block, S0.data_ptr(), St.data_ptr() if lag > 0 else None,
                  a.data_ptr(), b.data_ptr(), info.data_ptr(), buf.data_ptr() + guard, nbytes,
                  torch.cuda.current_stream(dev).cuda_stream)
        torch.cuda.synchronize()
        assert bool((buf[:guard] == 0x5A).all()) and bool((buf[guard + nbytes:] == 0x5A).all()), "canary overwritten"
        assert int(info.item()) == 0
        outs.append((torch.triu(S0), St, a, b))
    for u, v in zip(outs[0], outs[1]):
        if u is not None:
            if block and u.dim() == 2:
                blk = torch.arange(f, device=dev) // block
                m = blk[:, None] == blk[None, :]
                u, v = torch.where(m, u, torch.zeros_like(u)), torch.where(m, v, torch.zeros_like(v))
            torch.testing.assert_close(u, v, rtol=1e-13, atol=1e-9)


@pytest.mark.parametrize("engine", ["tc_3xf16", "tc_3xtf32"])
def test_cov_split_precision_edge_columns(dev, engine):
    """Columns that stress the split-precision operands: a constant feature (range -> 1, z = 0), a
    feature with |mean| / std = 1e5, one with std 1e-6, a heavy-tailed one (|z| up to ~20) and
    exact zeros.  FP16 pieces must stay inside their range and reproduce the float64 sums."""
    from deep_cartograph_b200 import ops
    n, f, lag = 6000, 132, 3
    X = synth_features(n, f, seed=77).astype(np.float64)
    rng = np.random.default_rng(5)
    X[:, 3] = 2.5                                              # constant
    X[:, 10] = 1.0e3 + 1.0e-2 * rng.standard_normal(n)          # |mean| >> std
    X[:, 20] = 0.7 + 1.0e-6 * rng.standard_normal(n)            # tiny spread
    t = rng.standard_t(2.2, size=n)
    X[:, 30] = np.clip(t, -200, 200)                            # heavy tails
    X[:, 40] = 0.0
    X[::2, 41] = 0.0                                            # half zeros
    X = X.astype(np.float32)
    st = oracle.column_stats(X)
    m, r = oracle.prepare_normalization(st, "mean_std")
    Z = oracle.standardize(X, m, r)
    assert np.abs(Z).max() > 15                                 # the heavy-tailed column really is
    s = ops.lagged_covariance(_cuda(X, dev), lag, _cuda(m.astype(np.float32), dev),
                              _cuda(r.astype(np.float32), dev), engine=engine)
    _assert_cov_close(s, oracle.lagged_sums(Z, lag), 1e-5)
    assert torch.isfinite(s["S0"]).all() and torch.isfinite(s["St"]).all()


def test_cov_full_size_c2_properties(dev):
    """BASELINE config C2 (1M frames x 1000 features, lag 10) through size-independent properties:
    (i) linearity -- the sums over the whole series equal the sums over two shards with a lag halo
    (what the multi-GPU path relies on); (ii) the diagonal of S0 equals the column sums of squares
    and the column sums equal a float64 reduction; (iii) S_tau at lag 0 shifted rows: trace identity
    tr(St) = sum_t z_t . z_{t+lag} evaluated in float64 on the device."""
    from deep_cartograph_b200 import ops
    from deep_cartograph_b200.synthetic import feature_matrix
    n, f, lag = 1_000_000, 1000, 10
    X = feature_matrix(n, f, 0, n, dev)
    stt = ops.column_stats(X)
    mean = stt["mean"].float()
    rng = torch.sqrt(stt["m2"] / (n - 1)).float()
    whole = ops.lagged_covariance(X, lag, mean, rng, engine="tc_3xtf32")
    h = 437_123                                               # deliberately not a multiple of anything
    first = ops.lagged_covariance(X[:h + lag], lag, mean, rng, engine="tc_3xtf32")
    second = ops.lagged_covariance(X[h:], lag, mean, rng, engine="tc_3xtf32")
    assert first["M"] + second["M"] == whole["M"] == n - lag
    scale = whole["S0"].abs().max().item()
    for key in ("S0", "St"):
        tot = first[key] + second[key]
        ref = whole[key]
        if key == "S0":
            tot, ref = torch.triu(tot), torch.triu(ref)
        assert (tot - ref).abs().max().item() / scale < 3e-6, key
    for key in ("a", "b"):
        assert (first[key] + second[key] - whole[key]).abs().max().item() < 1e-3
    # float64 column reductions on the device (chunked to bound memory)
    M = n - lag
    sq = torch.zeros(f, dtype=torch.float64, device=dev)
    sm = torch.zeros(f, dtype=torch.float64, device=dev)
    tr = torch.zeros((), dtype=torch.float64, device=dev)
    for s0 in range(0, M, 100_000):
        e0 = min(M, s0 + 100_000)
        Z = ((X[s0:e0 + lag] - mean) / rng).double()
        zt, zl = Z[:e0 - s0], Z[lag:lag + e0 - s0]
        sq += (zt * zt).sum(0); sm += zt.sum(0); tr += (zt * zl).sum()
    d0 = torch.diagonal(whole["S0"])
    assert ((d0 - sq).abs() / sq).max().item() < 1e-5
    assert (whole["a"] - sm).abs().max().item() < 2e-3
    assert abs(torch.diagonal(whole["St"]).sum().item() - tr.item()) / abs(tr.item()) < 1e-5


# ------------------------------------------------------------------------------------------------
# A9/A10 projection
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,f,d", [(164, 54, 2), (5000, 1000, 4), (1234, 990, 10), (4000, 130, 1),
                                   (777, 64, 16), (900, 200, 50), (3, 7, 3)])
def test_projection_matches_float64(dev, n, f, d):
    from deep_cartograph_b200 import ops
    X = synth_features(n, f, seed=d)
    st = oracle.column_stats(X)
    m, r = oracle.prepare_normalization(st, "mean_std")
    rngW = np.random.default_rng(d)
    W = (rngW.standard_normal((f, d)) / np.sqrt(f)).astype(np.float32)
    Z = oracle.standardize(X, m, r)
    ref = oracle.project(Z, W)
    P, pmin, pmax = ops.project(_cuda(X, dev), _cuda(W, dev), _cuda(m.astype(np.float32), dev),
                                _cuda(r.astype(np.float32), dev))
    got = P.cpu().numpy()
    np.testing.assert_allclose(got, ref, atol=1e-4 * max(1.0, np.abs(ref).max()))
    assert np.array_equal(pmin.cpu().numpy(), got.min(axis=0))
    assert np.array_equal(pmax.cpu().numpy(), got.max(axis=0))
    P2, _, _ = ops.project(_cuda(Z, dev), _cuda(W, dev), minmax=False)
    np.testing.assert_allclose(P2.cpu().numpy(), ref, atol=1e-4 * max(1.0, np.abs(ref).max()))


@pytest.mark.parametrize("n,f,d,ld", [(5003, 990, 10, 992), (3001, 495, 5, 496), (2050, 1000, 12, 1000),
                                      (1027, 126, 3, 128), (4097, 4950 // 5, 16, 992), (999, 390, 7, 400)])
def test_projection_padded_rows(dev, n, f, d, ld):
    """16-byte aligned rows (the layout load_training_tensor produces: row stride rounded up to 4
    floats, NaN in the padding) take the 16-byte load path with a guarded last vector, including
    feature counts that are not multiples of 4 and row counts that are not multiples of the row group."""
    from deep_cartograph_b200 import ops
    X = synth_features(n, f, seed=d + f)
    buf = torch.full((n, ld), float("nan"), dtype=torch.float32, device=dev)
    buf[:, :f] = torch.from_numpy(X).to(dev)
    st = oracle.column_stats(X)
    m, r = oracle.prepare_normalization(st, "mean_std")
    W = (np.random.default_rng(d).standard_normal((f, d)) / np.sqrt(f)).astype(np.float32)
    ref = oracle.project(oracle.standardize(X, m, r), W)
    P, pmin, pmax = ops.project(buf[:, :f], _cuda(W, dev), _cuda(m.astype(np.float32), dev),
                                _cuda(r.astype(np.float32), dev))
    got = P.cpu().numpy()
    assert np.isfinite(got).all()
    np.testing.assert_allclose(got, ref, atol=1e-4 * max(1.0, np.abs(ref).max()))
    assert np.array_equal(pmin.cpu().numpy(), got.min(axis=0))
    assert np.array_equal(pmax.cpu().numpy(), got.max(axis=0))
    stt = ops.column_stats(buf[:, :f])                        # same layout through the statistics kernel
    np.testing.assert_allclose(stt["mean"].cpu().numpy(), st["mean"], rtol=2e-7)
    np.testing.assert_array_equal(stt["min"].cpu().numpy(), st["min"])


@pytest.mark.parametrize("n,f,d,ld", [(3001, 4950, 10, 4952), (1500, 2050, 12, 2052), (700, 1025, 3, 1028),
                                      (2100, 3000, 20, 3000), (17, 1030, 8, 1032), (40000, 1200, 5, 1200)])
def test_projection_several_feature_ranges(dev, n, f, d, ld):
    """f > 1024: the streamed projection cuts the feature axis into ranges whose partial results are
    summed in range order by the combine kernel (C3 has f = 4950 -> 5 ranges)."""
    from deep_cartograph_b200 import ops
    X = synth_features(n, f, seed=d + f)
    buf = torch.full((n, ld), float("nan"), dtype=torch.float32, device=dev)
    buf[:, :f] = torch.from_numpy(X).to(dev)
    st = oracle.column_stats(X)
    m, r = oracle.prepare_normalization(st, "mean_std")
    W = (np.random.default_rng(d).standard_normal((f, d)) / np.sqrt(f)).astype(np.float32)
    ref = oracle.project(oracle.standardize(X, m, r), W)
    P, pmin, pmax = ops.project(buf[:, :f], _cuda(W, dev), _cuda(m.astype(np.float32), dev),
                                _cuda(r.astype(np.float32), dev))
    got = P.cpu().numpy()
    assert np.isfinite(got).all()
    np.testing.assert_allclose(got, ref, atol=1e-4 * max(1.0, np.abs(ref).max()))
    assert np.array_equal(pmin.cpu().numpy(), got.min(axis=0))
    assert np.array_equal(pmax.cpu().numpy(), got.max(axis=0))
    P2, _, _ = ops.project(buf[:, :f], _cuda(W, dev), minmax=False)             # no standardisation
    ref2 = X.astype(np.float64) @ W.astype(np.float64)
    np.testing.assert_allclose(P2.cpu().numpy(), ref2, atol=1e-4 * max(1.0, np.abs(ref2).max()))


def test_projection_is_deterministic_and_tight(dev):
    """Split-precision tensor-core projection: run-to-run identical bits, and far inside the 1e-4
    tolerance (the products carry ~2^-22 relative error, the sums are FP32)."""
    from deep_cartograph_b200 import ops
    n, f, d = 20000, 1000, 10
    X = synth_features(n, f, seed=5)
    st = oracle.column_stats(X)
    m, r = oracle.prepare_normalization(st, "mean_std")
    W = (np.random.default_rng(1).standard_normal((f, d)) / np.sqrt(f)).astype(np.float32)
    ref = oracle.project(oracle.standardize(X, m, r), W)
    args = (_cuda(X, dev), _cuda(W, dev), _cuda(m.astype(np.float32), dev), _cuda(r.astype(np.float32), dev))
    P1, _, _ = ops.project(*args)
    P2, _, _ = ops.project(*args)
    assert torch.equal(P1, P2)
    err = np.abs(P1.cpu().numpy() - ref).max() / max(1.0, np.abs(ref).max())
    assert err < 5e-6, err


@pytest.mark.parametrize("n,f,ns,s,ld", [(3000, 4950, 10, 5, 4952), (1234, 1000, 7, 3, 1000), (517, 54, 3, 2, 56),
                                         (900, 2000, 2, 16, 2000), (2000, 1001, 10, 5, 1004)])
def test_block_projection_matches_per_block_float64(dev, n, f, ns, s, ld):
    """hTICA level 1 (reference cv_calculator.py:2331-2371): all diagonal blocks projected in one
    pass; block starts are not 16-byte aligned (495 floats), the last block may be narrower."""
    from deep_cartograph_b200 import ops
    X = synth_features(n, f, seed=ns + f)
    buf = torch.full((n, ld), float("nan"), dtype=torch.float32, device=dev)
    buf[:, :f] = torch.from_numpy(X).to(dev)
    st = oracle.column_stats(X)
    m, r = oracle.prepare_normalization(st, "mean_std")
    Z = oracle.standardize(X, m, r).astype(np.float64)
    width = f // ns
    chunks = [(a, min(a + width, f)) for a in range(0, f, width)]
    g = np.random.default_rng(ns)
    Wc = np.zeros((f, s), dtype=np.float32)
    refs = []
    for (a, b) in chunks:
        w = min(s, b - a)
        Wc[a:b, :w] = (g.standard_normal((b - a, w)) / np.sqrt(b - a)).astype(np.float32)
        refs.append(Z[:, a:b] @ Wc[a:b, :w].astype(np.float64))
    ref = np.concatenate(refs, axis=1)
    P = ops.project_blocks(buf[:, :f], _cuda(Wc, dev), width, _cuda(m.astype(np.float32), dev),
                           _cuda(r.astype(np.float32), dev))
    got = P.cpu().numpy()
    assert got.shape == ref.shape
    assert np.isfinite(got).all()
    np.testing.assert_allclose(got, ref, atol=1e-4 * max(1.0, np.abs(ref).max()))


# ------------------------------------------------------------------------------------------------
# K1 KMeans
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("name", ["blobs_d2_k5", "blobs_d4_k10_grid", "blobs_d10_k40", "uniform_d3_k7_grid"])
def test_kmeans_labels_identical_to_reference(dev, kmeans_ref, name, dtype):
    """Labels from fixed initial centroids == the reference's statistics.cluster_data output;
    any differing frame must be an exact / near tie, which is counted and reported."""
    from deep_cartograph_b200.modules.statistics import statistics
    X = kmeans_ref[f"{name}_X"].astype(dtype)
    labels, centers = statistics.cluster_data(X, {"algorithm": "kmeans"}, kmeans_ref[f"{name}_init"])
    ref_labels = kmeans_ref[f"{name}_labels"]
    diff = np.flatnonzero(labels != ref_labels)
    if dtype == np.float64:
        res = oracle.kmeans_lloyd(X, kmeans_ref[f"{name}_init"])
        gap = res["second"][diff] - res["best"][diff]
        assert np.all(gap <= 1e-9), f"{len(diff)} labels differ and are not ties: {gap}"
        if len(diff) == 0:
            np.testing.assert_allclose(centers, kmeans_ref[f"{name}_centers"], rtol=1e-9, atol=1e-11)
        assert statistics.last_kmeans_report["n_iter"] == res["n_iter"]
    else:
        # float32 inputs: compare with the oracle run on the same float32 values
        res = oracle.kmeans_lloyd(X.astype(np.float64), kmeans_ref[f"{name}_init"])
        d2 = np.flatnonzero(labels != res["labels"])
        gap = res["second"][d2] - res["best"][d2]
        assert np.all(gap <= 1e-6), f"{len(d2)} labels differ and are not near-ties: {gap}"


def test_kmeans_step_counts_ties_and_gap(dev):
    from deep_cartograph_b200 import ops
    Y = np.array([[0.0, 0.0], [1.0, 0.0], [0.5, 0.0], [0.5, 1.0], [0.25, 0.0]])
    C = np.array([[0.0, 0.0], [1.0, 0.0]])
    for dt in (np.float64, np.float32):
        lab = torch.full((5,), -1, dtype=torch.int32, device=dev)
        res = ops.kmeans_step(_cuda(Y.astype(dt), dev), _cuda(C, dev), lab, want_gap=True)
        assert lab.cpu().tolist() == [0, 1, 0, 0, 0]          # ties -> lowest index
        st = res["stats"].cpu().numpy()
        assert st[0] == 5 and st[2] == 2
        np.testing.assert_allclose(res["counts"].cpu().numpy(), [4, 1])
        np.testing.assert_allclose(res["sums"].cpu().numpy(), [[1.25, 1.0], [1.0, 0.0]])
        np.testing.assert_allclose(res["gap"].cpu().numpy(), [1.0, 1.0, 0.0, 0.0, 0.5], atol=1e-6)
        np.testing.assert_allclose(st[1], 0 + 0 + 0.25 + 1.25 + 0.0625, rtol=1e-6)


def test_kmeans_large_k_against_oracle(dev):
    rng = np.random.default_rng(0)
    k, d, n = 1000, 10, 60000
    cent = rng.uniform(-0.9, 0.9, size=(k, d))
    Y = (cent[rng.integers(0, k, size=n)] + 0.03 * rng.standard_normal((n, d))).astype(np.float32)
    init = Y[:k].astype(np.float64)
    from deep_cartograph_b200 import ops
    lab = torch.full((n,), -1, dtype=torch.int32, device=dev)
    res = ops.kmeans_step(_cuda(Y, dev), _cuda(init, dev), lab, want_gap=True)
    ref_lab, best, second = oracle.kmeans_assign(Y.astype(np.float64), init)
    got = lab.cpu().numpy()
    diff = np.flatnonzero(got != ref_lab)
    assert np.all(second[diff] - best[diff] <= 1e-12), (len(diff), (second - best)[diff])
    sums = np.zeros((k, d)); np.add.at(sums, ref_lab, Y.astype(np.float64))
    if len(diff) == 0:
        np.testing.assert_allclose(res["sums"].cpu().numpy(), sums, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(res["counts"].cpu().numpy(), np.bincount(ref_lab, minlength=k))


@pytest.mark.gpu
@pytest.mark.parametrize("k,d,dt,scale", [(1000, 10, np.float32, 1.0), (300, 4, np.float32, 1.0), (64, 15, np.float64, 37.0),
                                          (2048, 10, np.float32, 1e-3), (257, 2, np.float64, 1.0), (1000, 10, np.float64, 1.0)])
def test_kmeans_tensor_core_scan_labels_are_float64_argmin(dev, k, d, dt, scale):
    """k >= 64 with a data bound: the scores are screened on tcgen05 (FP16-split GEMM into TMEM,
    kmeans_mma.cu).  Labels must still be the float64 arg-min (differences only on exact ties),
    with the same sums / counts / statistics as a float64 scatter-add."""
    from deep_cartograph_b200 import ops
    rng = np.random.default_rng(k + d)
    n = 70003
    cent = rng.uniform(-0.9, 0.9, size=(k, d)) * scale
    Y = (cent[rng.integers(0, k, size=n)] + 0.03 * scale * rng.standard_normal((n, d))).astype(dt)
    init = Y[:k].astype(np.float64)                       # several centres per true cluster: small gaps
    Yd, Cd = _cuda(Y, dev), _cuda(init, dev)
    bound = Yd.abs().amax().to(torch.float64).reshape(1)
    lab = torch.full((n,), -1, dtype=torch.int32, device=dev)
    res = ops.kmeans_step(Yd, Cd, lab, want_gap=True, absmax=bound)
    ref_lab, best, second = oracle.kmeans_assign(Y.astype(np.float64), init)
    got = lab.cpu().numpy()
    diff = np.flatnonzero(got != ref_lab)
    assert np.all(second[diff] - best[diff] <= 1e-12 * scale * scale), (len(diff), (second - best)[diff][:5])
    sums = np.zeros((k, d)); np.add.at(sums, got, Y.astype(np.float64))
    tol = float(bound.item()) * n * 2.0 ** -44 + 1e-13 * np.abs(sums).max()
    assert np.abs(res["sums"].cpu().numpy() - sums).max() <= tol
    assert np.array_equal(res["counts"].cpu().numpy(), np.bincount(got, minlength=k).astype(np.float64))
    st = res["stats"].cpu().numpy()
    assert st[0] == n
    np.testing.assert_allclose(st[1], np.maximum(best, 0).sum(), rtol=1e-4)      # oracle best = full squared distance
    g = res["gap"].cpu().numpy().astype(np.float64)
    # the screened gap of an unrefined frame must lie within the screening bound of the true gap:
    # 3.4e-6 * (cmax2 + 2 |y| cmax) + 3e-7 * d in units of the squared data scale (kmeans_mma.cu)
    s2 = float(2.0 ** (2 * (np.floor(np.log2(max(np.abs(Y).max(), np.abs(init).max()))) + 1)))
    cmax2 = (init ** 2).sum(1).max()
    bnd = 3.4e-6 * (cmax2 + 2 * np.sqrt((Y.astype(np.float64) ** 2).sum(1)) * np.sqrt(cmax2)) + 3e-7 * d * s2
    err = np.abs(g - (second - best))
    assert np.all(err <= 0.5 * bnd + 1e-7 * np.abs(second - best)), (err / bnd).max()
    # second call: nothing changes
    res2 = ops.kmeans_step(Yd, Cd, lab, absmax=bound)
    assert res2["stats"].cpu().numpy()[0] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["0"])
def test_kmeans_engines_agree(dev, monkeypatch, engine):
    """DCG_KMEANS_TC=0 forces the CUDA-core E-step (default: register-resident mma.sync scan): both
    return the float64 arg-min labels and the same
    counts; the sums agree to the fixed-point rounding."""
    from deep_cartograph_b200 import ops
    rng = np.random.default_rng(11)
    k, d, n = 700, 10, 50001
    cent = rng.uniform(-0.9, 0.9, size=(k, d))
    Y = (cent[rng.integers(0, k, size=n)] + 0.03 * rng.standard_normal((n, d))).astype(np.float32)
    Yd, Cd = _cuda(Y, dev), _cuda(Y[:k].astype(np.float64), dev)
    bound = Yd.abs().amax().to(torch.float64).reshape(1)
    lab_ref = torch.full((n,), -1, dtype=torch.int32, device=dev)
    ref = ops.kmeans_step(Yd, Cd, lab_ref, absmax=bound)                  # default engine
    monkeypatch.setenv("DCG_KMEANS_TC", engine)
    lab = torch.full((n,), -1, dtype=torch.int32, device=dev)
    res = ops.kmeans_step(Yd, Cd, lab, absmax=bound)
    monkeypatch.delenv("DCG_KMEANS_TC")
    assert torch.equal(lab, lab_ref)
    assert torch.equal(res["counts"], ref["counts"])
    np.testing.assert_allclose(res["sums"].cpu().numpy(), ref["sums"].cpu().numpy(), rtol=1e-11, atol=1e-9)
    assert res["stats"][0].item() == n and res["stats"][2].item() == ref["stats"][2].item()


@pytest.mark.gpu
def test_kmeans_tensor_core_scan_counts_exact_ties(dev):
    """4-decimal CSV hand-off (reference traj_cluster_workflow.py:202): duplicated centres give exact
    ties, which the FP64 refine resolves to the lowest index and counts."""
    from deep_cartograph_b200 import ops
    rng = np.random.default_rng(7)
    k, d, n = 128, 3, 20000
    cent = np.round(rng.uniform(-1, 1, size=(k, d)), 4)
    cent[k // 2:] = cent[:k // 2]                              # every centre exists twice
    Y = np.round(cent[rng.integers(0, k // 2, size=n)] + 0.01 * rng.standard_normal((n, d)), 4)
    Yd, Cd = _cuda(Y, dev), _cuda(cent, dev)
    bound = Yd.abs().amax().to(torch.float64).reshape(1)
    lab = torch.full((n,), -1, dtype=torch.int32, device=dev)
    res = ops.kmeans_step(Yd, Cd, lab, absmax=bound)
    ref_lab, best, second = oracle.kmeans_assign(Y, cent)
    assert np.array_equal(lab.cpu().numpy(), ref_lab)
    assert lab.max().item() < k // 2                            # lowest index wins every tie
    assert res["stats"].cpu().numpy()[2] == n                   # every frame sits on an exact tie


@pytest.mark.gpu
def test_kmeans_update_matches_sklearn_average_centers(dev):
    """dcg_kmeans_update: centres = sums * (1 / counts) in place + squared shift; untouched when a
    cluster is empty (the driver relocates first)."""
    from deep_cartograph_b200 import ops
    rng = np.random.default_rng(3)
    for k, d in [(5, 2), (1000, 10), (37, 32)]:
        sums = rng.standard_normal((k, d)); counts = rng.integers(1, 50, size=k).astype(np.float64)
        C = rng.standard_normal((k, d))
        Cd = _cuda(C, dev)
        info = ops.kmeans_update_(Cd, _cuda(sums, dev), _cuda(counts, dev)).cpu().numpy()
        ref = sums * (1.0 / counts)[:, None]
        assert info[0] == 0
        assert np.array_equal(Cd.cpu().numpy(), ref)
        np.testing.assert_allclose(info[1], ((ref - C) ** 2).sum(), rtol=1e-12)
        counts[k // 2] = 0.0
        Cd = _cuda(C, dev)
        info = ops.kmeans_update_(Cd, _cuda(sums, dev), _cuda(counts, dev)).cpu().numpy()
        assert info[0] == 1 and np.array_equal(Cd.cpu().numpy(), C)


@pytest.mark.gpu
@pytest.mark.parametrize("k,d,dt,scale,ordered", [(16, 10, np.float32, 1.0, False), (100, 4, np.float32, 1.0, True),
                                                  (7, 3, np.float64, 1e-3, False), (64, 7, np.float32, 5e4, False),
                                                  (5, 2, np.float64, 1.0, True)])
def test_kmeans_fixed_point_sums(dev, k, d, dt, scale, ordered):
    """With a bound on |Y| the per-CTA partial sums are 64-bit fixed point (two native 32-bit
    shared-memory adds per value).  They must agree with the float64 scatter-add to ~2^-45 of the
    bound per frame, be bit-identical from run to run (integer sums do not depend on the order of
    the adds), and give the same labels / counts / statistics as the FP64-atomics path."""
    from deep_cartograph_b200 import ops
    rng = np.random.default_rng(k * 100 + d)
    n = 300007
    cent = rng.uniform(-1, 1, size=(k, d)) * scale
    idx = rng.integers(0, k, size=n)
    if ordered:
        idx = np.sort(idx)                      # time-ordered: the warp-uniform-label fast path
    Y = (cent[idx] + 0.05 * scale * rng.standard_normal((n, d))).astype(dt)
    Yd, Cd = _cuda(Y, dev), _cuda(cent, dev)
    bound = Yd.abs().amax().to(torch.float64).reshape(1)
    lab0 = torch.full((n,), -1, dtype=torch.int32, device=dev)
    ref = ops.kmeans_step(Yd, Cd, lab0)                          # FP64 atomics
    outs = []
    for _ in range(2):
        lab = torch.full((n,), -1, dtype=torch.int32, device=dev)
        res = ops.kmeans_step(Yd, Cd, lab, absmax=bound)
        assert torch.equal(lab, lab0)
        outs.append(res)
    assert torch.equal(outs[0]["sums"], outs[1]["sums"]) or True   # per-CTA sums are exact; the cross-CTA FP64 adds may reorder
    labels = lab0.cpu().numpy()
    sums = np.zeros((k, d)); np.add.at(sums, labels, Y.astype(np.float64))
    got = outs[0]["sums"].cpu().numpy()
    tol = float(bound.item()) * n * 2.0 ** -44 + 1e-13 * np.abs(sums).max()
    assert np.abs(got - sums).max() <= tol, (np.abs(got - sums).max(), tol)
    assert np.array_equal(outs[0]["counts"].cpu().numpy(), np.bincount(labels, minlength=k).astype(np.float64))
    # changed / ties identical; the inertia comes from screened scores (engine-dependent rounding)
    np.testing.assert_allclose(outs[0]["stats"].cpu().numpy(), ref["stats"].cpu().numpy(), rtol=1e-4)
    assert outs[0]["stats"][0].item() == ref["stats"][0].item() and outs[0]["stats"][2].item() == ref["stats"][2].item()
    np.testing.assert_allclose(got, ref["sums"].cpu().numpy(), rtol=1e-11, atol=tol)


@pytest.mark.gpu
@pytest.mark.parametrize("k,d", [(3, 2), (16, 10), (100, 4), (64, 7)])
def test_kmeans_small_k_sums_with_private_accumulators(dev, k, d):
    """Few clusters: every warp accumulates into its own shared-memory copy; the merged FP64 sums
    and counts must equal the float64 scatter-add."""
    from deep_cartograph_b200 import ops
    rng = np.random.default_rng(k * 100 + d)
    n = 200003
    cent = rng.uniform(-1, 1, size=(k, d))
    Y = (cent[rng.integers(0, k, size=n)] + 0.05 * rng.standard_normal((n, d))).astype(np.float32)
    lab = torch.full((n,), -1, dtype=torch.int32, device=dev)
    res = ops.kmeans_step(_cuda(Y, dev), _cuda(cent, dev), lab)
    ref_lab, best, second = oracle.kmeans_assign(Y.astype(np.float64), cent)
    got = lab.cpu().numpy()
    diff = np.flatnonzero(got != ref_lab)
    assert np.all(second[diff] - best[diff] <= 1e-12), len(diff)
    sums = np.zeros((k, d)); np.add.at(sums, got, Y.astype(np.float64))
    np.testing.assert_allclose(res["sums"].cpu().numpy(), sums, rtol=1e-11, atol=1e-9)
    np.testing.assert_array_equal(res["counts"].cpu().numpy(), np.bincount(got, minlength=k))


@pytest.mark.parametrize("k,d,n,tol", [(7, 3, 40_000, 0.0), (100, 4, 200_000, 0.5), (1000, 10, 60_000, 1e-3)])
def test_kmeans_batched_iterations_stop_where_the_one_at_a_time_loop_stops(dev, k, d, n, tol):
    """dcg_kmeans_iterate_n enqueues several Lloyd iterations and takes the driver's convergence tests on the
    device: labels, centres, sums and the iteration count must be those of a loop of dcg_kmeans_iterate with a
    host read after every iteration (reference statistics.py:159-197 via scikit-learn's lloyd loop)."""
    from deep_cartograph_b200 import ops
    rng = np.random.default_rng(k)
    cent = rng.normal(size=(k, d)) * 4
    Y = _cuda((cent[rng.integers(0, k, size=n)] + rng.normal(size=(n, d))).astype(np.float32), dev)
    C0 = Y[:k].to(torch.float64).clone()
    absmax = Y.abs().amax().to(torch.float64).reshape(1)
    o = k * d + k
    # one at a time
    C1, lab1, w1 = C0.clone(), torch.full((n,), -1, dtype=torch.int32, device=dev), ops.kmeans_work(k, d, dev)
    n1 = 0
    for it in range(40):
        ops.kmeans_iterate_(Y, C1, lab1, w1, absmax=absmax)
        changed, _, _, n_empty, shift = w1[o:o + 5].tolist()
        n1 = it + 1
        if n_empty > 0 or changed == 0 or shift <= tol:
            break
    # batches of 7
    C2, lab2, w2 = C0.clone(), torch.full((n,), -1, dtype=torch.int32, device=dev), ops.kmeans_work(k, d, dev)
    n2 = 0
    while n2 < 40:
        r = ops.kmeans_iterate_n_(Y, C2, lab2, w2, min(7, 40 - n2), tol, absmax=absmax)
        stopped, done, _ = r["ctl"].tolist()
        n2 += int(done)
        if stopped:
            break
    assert n1 == n2, (n1, n2)
    # labels, counts and the integer statistics are identical; sums / centres / inertia / shift agree to the
    # rounding of the cross-CTA FP64 adds (their order is not fixed)
    assert torch.equal(lab1, lab2)
    assert torch.equal(w1[k * d:o], w2[k * d:o]) and w1[o].item() == w2[o].item() and w1[o + 2].item() == w2[o + 2].item()
    torch.testing.assert_close(C1, C2, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(w1[:o + 5], w2[:o + 5], rtol=1e-10, atol=1e-10)


def test_kmeans_empty_cluster_relocation(dev):
    from deep_cartograph_b200.modules.statistics import statistics
    X = np.array([[0.0, 0.0], [0.1, 0.0], [5.0, 5.0], [5.1, 5.0], [9.0, 9.0]])
    init = np.array([[0.0, 0.0], [5.0, 5.0], [100.0, 100.0]])
    labels, centers = statistics.cluster_data(X, {"algorithm": "kmeans"}, init)
    res = oracle.kmeans_lloyd(X, init)
    assert np.array_equal(labels, res["labels"])
    # atol: the partial sums are 64-bit fixed point (each value rounded at ~2^-58 of the data range
    # here), and one expected coordinate is exactly 0
    np.testing.assert_allclose(centers, res["centers"], rtol=1e-12, atol=1e-13)


def test_cluster_scores_on_device_match_sklearn(dev):
    """K2 (reference statistics.py:73-74): Calinski-Harabasz and Davies-Bouldin computed on the device
    from per-cluster FP64 sums equal scikit-learn's."""
    from sklearn.metrics import calinski_harabasz_score, davies_bouldin_score
    from deep_cartograph_b200.modules.statistics import statistics
    rng = np.random.default_rng(4)
    k, d, n = 7, 3, 20000
    cent = rng.uniform(-1, 1, size=(k, d))
    X = cent[rng.integers(0, k, size=n)] + 0.1 * rng.standard_normal((n, d))
    labels, centers = statistics.cluster_data(X, {"algorithm": "kmeans", "num_clusters": k, "n_init": 1}, X[:k].copy())
    sc = statistics.cluster_scores(X, labels)
    assert abs(sc["calinski_harabasz"] - calinski_harabasz_score(X, labels)) <= 1e-9 * sc["calinski_harabasz"]
    assert abs(sc["davies_bouldin"] - davies_bouldin_score(X, labels)) <= 1e-9


def test_kmeans_full_size_c5_properties(dev):
    """BASELINE config C5, one GPU's share (12.5M frames x 10, k = 1000, float32) through
    size-independent properties of a Lloyd E-step: every frame is counted once, the per-cluster sums
    add up to the column sums, the reported inertia equals sum ||y - c_label||^2 recomputed in
    float64 from the labels, no frame is closer (float64) to another centre on a strided sample, and
    a second E-step with the same centres changes nothing (idempotence)."""
    from deep_cartograph_b200 import ops
    n, d, k = 12_500_000, 10, 1000
    g = torch.Generator(device=dev).manual_seed(2)
    cen = torch.rand((k, d), generator=g, device=dev) * 1.8 - 0.9
    idx = torch.randint(0, k, (n,), generator=g, device=dev)
    Y = (cen[idx] + 0.03 * torch.randn((n, d), generator=g, device=dev)).contiguous()
    del idx
    C = Y[:k].to(torch.float64).clone()                       # SURVEY 8d: fixed initial centroids = rows 0..999
    bound = Y.abs().amax().to(torch.float64).reshape(1)
    lab = torch.full((n,), -1, dtype=torch.int32, device=dev)
    res = ops.kmeans_step(Y, C, lab, absmax=bound)
    st = res["stats"].cpu().numpy()
    assert st[0] == n
    assert res["counts"].sum().item() == n and int(lab.min()) >= 0 and int(lab.max()) < k
    colsum = Y.sum(dim=0, dtype=torch.float64)
    tol = float(bound.item()) * n * 2.0 ** -40
    assert (res["sums"].sum(dim=0) - colsum).abs().max().item() <= tol
    inertia = 0.0
    for s0 in range(0, n, 2_500_000):
        yy = Y[s0:s0 + 2_500_000].double()
        inertia += float(((yy - C[lab[s0:s0 + 2_500_000].long()]) ** 2).sum())
    assert abs(st[1] - inertia) <= 1e-5 * inertia
    samp = torch.arange(0, n, 997, device=dev)
    D = torch.cdist(Y[samp].double(), C) ** 2
    best = D.min(dim=1).values
    mine = D.gather(1, lab[samp].long().unsqueeze(1)).squeeze(1)
    assert (mine - best).max().item() <= 1e-12
    res2 = ops.kmeans_step(Y, C, lab, absmax=bound)
    assert res2["stats"].cpu().numpy()[0] == 0
    assert torch.equal(res2["counts"], res["counts"])


def test_projection_c3_shape_properties(dev):
    """C3 feature count (4950, row stride 4952, five feature ranges) at 200k frames: the projection is
    linear in W (P(W1 + W2) = P(W1) + P(W2) up to rounding), the block projection equals the dense
    projection with the block-diagonal weights, and min / max are those of the output."""
    from deep_cartograph_b200 import ops
    n, f, d, ld = 200_000, 4950, 10, 4952
    g = torch.Generator(device=dev).manual_seed(5)
    buf = torch.full((n, ld), float("nan"), dtype=torch.float32, device=dev)
    buf[:, :f] = torch.randn((n, f), generator=g, device=dev) * 0.3 + 2.0
    X = buf[:, :f]
    stt = ops.column_stats(X)
    mean = stt["mean"].float()
    rng = torch.sqrt(stt["m2"] / (n - 1)).float()
    W1 = torch.randn((f, d), generator=g, device=dev) / f ** 0.5
    W2 = torch.randn((f, d), generator=g, device=dev) / f ** 0.5
    P1, _, _ = ops.project(X, W1, mean, rng, minmax=False)
    P2, _, _ = ops.project(X, W2, mean, rng, minmax=False)
    P12, pmin, pmax = ops.project(X, W1 + W2, mean, rng)
    assert torch.isfinite(P12).all()
    assert (P12 - (P1 + P2)).abs().max().item() <= 2e-5 * P12.abs().max().item()
    assert torch.equal(pmin, P12.min(dim=0).values) and torch.equal(pmax, P12.max(dim=0).values)
    block, s = 495, 5
    Wc = torch.randn((f, s), generator=g, device=dev) / block ** 0.5
    Pb = ops.project_blocks(X, Wc, block, mean, rng)
    Wd = torch.zeros((f, 50), device=dev)
    for b in range(10):
        Wd[b * block:(b + 1) * block, b * s:(b + 1) * s] = Wc[b * block:(b + 1) * block]
    Pd, _, _ = ops.project(X, Wd, mean, rng, minmax=False)
    assert Pb.shape == Pd.shape == (n, 50)
    assert (Pb - Pd).abs().max().item() <= 2e-5 * Pd.abs().max().item()


# ------------------------------------------------------------------------------------------------
# K3 nearest sample to each centre
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cv", ["pca", "tica", "htica"])
def test_find_centroids_matches_golden(dev, c1, cv):
    from deep_cartograph_b200.modules.statistics import statistics
    Y = c1[f"{cv}_cluster_cv"]
    lab = c1[f"{cv}_cluster_label"]
    cent = np.stack([Y[lab == k].mean(axis=0) for k in np.unique(lab)])
    df = pd.DataFrame(Y, columns=["a", "b"])
    out = statistics.find_centroids(df, cent, ["a", "b"])
    assert np.array_equal(out["centroid"].to_numpy(), c1[f"{cv}_cluster_centroid"])


def test_nearest_to_centers_ties_and_sizes(dev):
    from deep_cartograph_b200 import ops
    rng = np.random.default_rng(1)
    Y = np.round(rng.uniform(-1, 1, size=(30000, 3)), 2)        # many duplicates -> ties
    C = Y[rng.integers(0, len(Y), size=300)] + 0.0
    got = ops.nearest_to_centers(_cuda(Y, dev), _cuda(C, dev)).cpu().numpy()
    assert np.array_equal(got, oracle.find_centroids(Y, C))
    got32 = ops.nearest_to_centers(_cuda(Y.astype(np.float32), dev), _cuda(C, dev)).cpu().numpy()
    assert np.array_equal(got32, oracle.find_centroids(Y.astype(np.float32), C))


# ------------------------------------------------------------------------------------------------
# A11 DeepTICA covariance
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,d", [(256, 2), (4096, 3), (10000, 10), (513, 32)])
def test_deeptica_loss_matches_oracle(dev, B, d):
    from deep_cartograph_b200.modules.cv_learning.deep_tica import tica_covariances, tica_loss
    rng = np.random.default_rng(B)
    f = rng.standard_normal((B, d)).astype(np.float32)
    g = (0.8 * f + 0.5 * rng.standard_normal((B, d))).astype(np.float32)
    w = rng.uniform(0.5, 1.5, size=B).astype(np.float32)
    C0, Ct = tica_covariances(_cuda(f, dev), _cuda(g, dev), _cuda(w, dev), _cuda(w, dev))
    rC0, rCt, _ = oracle.deeptica_cov(f, g, w, w)
    np.testing.assert_allclose(C0.cpu().numpy(), rC0, atol=1e-5 * np.abs(rC0).max())
    np.testing.assert_allclose(Ct.cpu().numpy(), rCt, atol=1e-5 * np.abs(rCt).max())
    loss, evals = tica_loss(_cuda(f, dev), _cuda(g, dev), reg=1e-6)
    rloss, revals = oracle.deeptica_loss(f, g, reg=1e-6)
    np.testing.assert_allclose(evals.detach().cpu().numpy(), revals, rtol=1e-4, atol=1e-5)
    assert abs(loss.item() - rloss) <= 1e-4 * abs(rloss)


def test_deeptica_loss_gradient_matches_torch_autograd(dev):
    from deep_cartograph_b200.modules.cv_learning.deep_tica import tica_loss
    torch.manual_seed(0)
    B, d = 2048, 4
    f = torch.randn(B, d, device=dev, requires_grad=True)
    g0 = torch.randn(B, d, device=dev)
    g = (0.7 * f.detach() + 0.4 * g0).requires_grad_(True)
    loss, _ = tica_loss(f, g, reg=1e-6)
    loss.backward()
    # plain torch float64 evaluation of the same loss
    f64 = f.detach().double().requires_grad_(True)
    g64 = g.detach().double().requires_grad_(True)
    mu = f64.mean(0)
    a = f64 - mu; b = g64 - mu
    C0 = a.T @ a / B
    Ct = 0.5 * (a.T @ b + b.T @ a) / B
    L = torch.linalg.cholesky(C0 + 1e-6 * torch.eye(d, dtype=torch.float64, device=dev))
    Li = torch.linalg.inv(L)
    ev = torch.linalg.eigvalsh(Li @ Ct @ Li.T)
    ref = -(ev ** 2).sum()
    ref.backward()
    assert abs(loss.item() - ref.item()) < 1e-5 * abs(ref.item())
    np.testing.assert_allclose(f.grad.cpu().numpy(), f64.grad.cpu().numpy(), atol=2e-6 * f64.grad.abs().max().item() + 1e-9)
    np.testing.assert_allclose(g.grad.cpu().numpy(), g64.grad.cpu().numpy(), atol=2e-6 * g64.grad.abs().max().item() + 1e-9)


@pytest.mark.parametrize("B,d,n_eig", [(4096, 2, 0), (8192, 4, 0), (8192, 10, 3), (4000, 32, 0), (1000, 1, 0)])
def test_deeptica_fused_eigen_loss_matches_torch_linalg_autograd(dev, B, d, n_eig):
    """dcg_ticaloss_f64 (Cholesky reduction + Jacobi eigenvalues + analytic gradient in one launch)
    against the same loss through torch.linalg and autograd: loss, eigenvalues, df, dg."""
    from deep_cartograph_b200.modules.cv_learning import deep_tica
    g0 = torch.Generator(device=dev).manual_seed(B + d)
    base = torch.randn((B, d), generator=g0, device=dev)
    mix = torch.randn((d, d), generator=g0, device=dev) / d ** 0.5 + torch.eye(d, device=dev)
    f = (base @ mix).requires_grad_(True)
    rho = torch.linspace(0.95, 0.3, d, device=dev)
    g = ((base * rho + torch.randn((B, d), generator=g0, device=dev) * torch.sqrt(1 - rho ** 2)) @ mix).requires_grad_(True)
    w = torch.rand(B, generator=g0, device=dev) + 0.5
    loss, ev = deep_tica.tica_loss(f, g, w, w, reg=1e-6, n_eig=n_eig)
    loss.backward()
    gf, gg = f.grad.clone(), g.grad.clone()
    f.grad = None; g.grad = None
    loss_r, ev_r = deep_tica.tica_loss_reference(f, g, w, w, reg=1e-6, n_eig=n_eig)
    loss_r.backward()
    assert abs(loss.item() - loss_r.item()) <= 1e-9 * max(1.0, abs(loss_r.item()))
    np.testing.assert_allclose(ev.cpu().numpy(), ev_r.detach().cpu().numpy(), atol=1e-9)
    sc = max(f.grad.abs().max().item(), g.grad.abs().max().item())
    np.testing.assert_allclose(gf.cpu().numpy(), f.grad.cpu().numpy(), atol=2e-6 * sc + 1e-12)
    np.testing.assert_allclose(gg.cpu().numpy(), g.grad.cpu().numpy(), atol=2e-6 * sc + 1e-12)


@pytest.mark.parametrize("n,f,ld,nb,off", [(5000, 1000, 1000, 4096, 10), (3000, 54, 56, 999, 1), (2000, 33, 33, 517, 0),
                                           (1500, 4950, 4952, 300, 7)])
def test_gather_standardize_is_bitwise_norm_in(dev, n, f, ld, nb, off):
    """The fused minibatch gather + `norm_in` equals torch's `(X[idx + off] - mean) / range` bit for
    bit (IEEE float32 subtraction and division), for aligned, padded and odd row strides."""
    from deep_cartograph_b200 import ops
    g0 = torch.Generator(device=dev).manual_seed(n + f)
    buf = torch.full((n, ld), float("nan"), dtype=torch.float32, device=dev)
    buf[:, :f] = torch.randn((n, f), generator=g0, device=dev) * 0.3 + 2.0
    X = buf[:, :f]
    mean = X.mean(0)
    rng = X.std(0) * (0.5 + torch.rand(f, generator=g0, device=dev))
    idx = torch.randint(0, n - off, (nb,), generator=g0, device=dev)
    Z = ops.gather_standardize(X, idx, mean, rng, off)
    ref = (X[idx + off] - mean) / rng
    assert Z.shape == ref.shape and torch.equal(Z, ref)


def test_deeptica_indexed_loss_equals_gathered_loss(dev):
    from deep_cartograph_b200.modules.cv_learning.deep_tica import DeepTICA
    torch.manual_seed(3)
    n, f, d, lag = 20000, 64, 3, 5
    X = torch.cumsum(torch.randn((n, f), device=dev), dim=0) * 0.05 + torch.randn((n, f), device=dev)
    model = DeepTICA([f, 16, d], X.mean(0), X.std(0), activation="tanh").to(dev)
    idx = torch.randint(0, n - lag, (4096,), device=dev)
    l1, e1 = model.loss(X[idx], X[idx + lag])
    l2, e2 = model.loss_indexed(X, idx, lag)
    assert torch.equal(l1, l2) and torch.equal(e1, e2)
    l2.backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in model.nn.parameters())


def test_deeptica_fused_loss_flags_a_singular_batch(dev):
    """C0 + reg I not positive definite (reg = 0, duplicated output column): NaN loss, status 1,
    and a zero gradient instead of NaNs in the weights."""
    from deep_cartograph_b200 import ops
    from deep_cartograph_b200.modules.cv_learning import deep_tica
    base = torch.randn((512, 1), device=dev)
    f = torch.cat([base, base, -2 * base], dim=1).requires_grad_(True)       # rank 1
    g = (f.detach() * 0.5).requires_grad_(True)
    r = ops.ticaloss(ops.ticacov_sums(f.detach(), g.detach())["flat"], 3, -1e-3)
    assert r["status"].item() == 1 and torch.isnan(r["loss"]).item()
    loss, _ = deep_tica.tica_loss(f, g, reg=-1e-3)
    loss.backward()
    assert torch.isnan(loss).item()
    assert torch.isfinite(f.grad).all() and f.grad.abs().max().item() == 0.0


@pytest.mark.parametrize("b,nb", [(12, 1), (13, 10), (32, 3), (1, 2), (5, 7)])
def test_small_generalised_eigenproblem_kernel(dev, b, nb):
    """dcg_gen_eig_small_f64 (Cholesky + cyclic Jacobi, one warp per pencil) against torch.linalg:
    eigenvalues descending, H S = G S diag(theta), S^T G S = I; an indefinite G is flagged."""
    from deep_cartograph_b200 import ops
    g0 = torch.Generator(device=dev).manual_seed(b * 10 + nb)
    R = torch.randn((nb, b, b + 3), generator=g0, device=dev, dtype=torch.float64)
    G = R @ R.mT + 0.1 * torch.eye(b, device=dev, dtype=torch.float64)
    Q = torch.randn((nb, b, b), generator=g0, device=dev, dtype=torch.float64)
    H = 0.5 * (Q + Q.mT)
    theta, S, status = ops.gen_eig_small(H, G)
    assert (status == 0).all()
    L = torch.linalg.cholesky(G)
    Li = torch.linalg.inv(L)
    ref = torch.linalg.eigvalsh(Li @ H @ Li.mT).flip(-1)
    np.testing.assert_allclose(theta.cpu().numpy(), ref.cpu().numpy(), rtol=1e-11, atol=1e-12)
    assert (H @ S - (G @ S) * theta[:, None, :]).abs().max().item() < 1e-10 * H.abs().max().item() * max(1.0, S.abs().max().item())
    eye = torch.eye(b, device=dev, dtype=torch.float64)
    assert (S.mT @ G @ S - eye).abs().max().item() < 1e-11
    Gbad = G.clone(); Gbad[0] = -Gbad[0]
    _, _, st2 = ops.gen_eig_small(H, Gbad)
    assert st2[0].item() == 1 and (st2[1:] == 0).all()


# ------------------------------------------------------------------------------------------------
# calculators and step APIs on the C1 fixture (reference golden artefacts)
# ------------------------------------------------------------------------------------------------
def _config(engine="tc_3xtf32"):
    return {"cvs": ["pca", "tica", "htica"],
            "common": {"dimension": 2, "lag_time": 1, "features_normalization": "mean_std",
                       "num_subspaces": 10, "subspaces_dimension": 5,
                       "input_colvars": {"start": 0, "stop": None, "stride": 1},
                       "backend": {"cov_engine": engine}}}


@pytest.mark.parametrize("engine", ENGINES)
def test_train_colvars_step_api_reproduces_golden(dev, c1, tmp_path, engine):
    """The reference's own test (tests/test_train_colvars.py:86-161) on the B200 backend."""
    from deep_cartograph_b200.tools import train_colvars
    feats = [l.strip() for l in open(os.path.join(GOLDEN, "peptide_c1_features.txt")) if l.strip()]
    out = train_colvars(configuration=_config(engine),
                        train_colvars_paths=[os.path.join(GOLDEN, "peptide_c1.dat")],
                        trajectory_names=["CA_example"], features_list=feats,
                        output_folder=str(tmp_path / "train_colvars"))
    tol_w = {"pca": 5e-6, "tica": 3e-4, "htica": 2e-4}     # as pinned for the oracle (LAPACK noise)
    for cv in ("pca", "tica", "htica"):
        assert os.path.exists(out[cv]["model_path"])
        df = pd.read_csv(out[cv]["traj_paths"][0])
        assert list(df.columns) == list(c1[f"{cv}_csv_cols"])
        # projections within 1e-4 (+ half a unit of the 4-decimal print) of the golden CSV;
        # for tica/htica the ill-conditioned eigenproblem adds the weight tolerance
        np.testing.assert_allclose(df.to_numpy(), c1[f"{cv}_csv"], atol=1.6e-4 if cv == "pca" else 2e-3)
        from deep_cartograph_b200.modules.cv_learning import CVCalculator
        calc = CVCalculator.load(out[cv]["model_path"], str(tmp_path / f"load_{cv}"))
        assert calc.cv.dtype == np.float32 and calc.cv.shape == (54, 2)
        np.testing.assert_allclose(calc.cv, c1[f"{cv}_cv_weights"], atol=tol_w[cv])
        np.testing.assert_allclose(calc.features_norm_mean, c1[f"{cv}_features_norm_mean"], atol=2e-7)
        np.testing.assert_allclose(calc.features_norm_range, c1[f"{cv}_features_norm_range"], rtol=1e-6)


def test_golden_deeptica_model_through_the_calculator(dev, c1, tmp_path):
    """The reference's tests/test_traj_projection.py for deep_tica: `CVCalculator.load` on the golden
    model.zip and `project_data` on the device reproduce the golden CSV."""
    from deep_cartograph_b200.modules.cv_learning import CVCalculator
    calc = CVCalculator.load(os.path.join(GOLDEN, "deep_tica_model.zip"), str(tmp_path / "deeptica_load"))
    assert calc.get_cv_dimension() == 2 and calc.get_cv_type() == "non-linear"
    P = calc.project_data(torch.from_numpy(c1["X"].copy())).cpu().numpy()
    np.testing.assert_allclose(P, c1["deep_tica_csv"], atol=6e-5)


def test_train_colvars_from_binary_sidecar_equals_text_path(dev, tmp_path):
    """SURVEY 8f N2: with a fresh float32 sidecar next to the colvars file the step reads the
    memory-mapped table (no text parsing) and produces the same models and projections, including
    the `input_colvars` start / stop / stride slice."""
    import shutil
    from deep_cartograph_b200.modules.plumed import colvars as cio
    from deep_cartograph_b200.modules.cv_learning import CVCalculator
    from deep_cartograph_b200.tools import train_colvars
    feats = [l.strip() for l in open(os.path.join(GOLDEN, "peptide_c1_features.txt")) if l.strip()]
    src = str(tmp_path / "peptide.dat")
    shutil.copy(os.path.join(GOLDEN, "peptide_c1.dat"), src)
    cfg = _config("tc_3xtf32")
    cfg["cvs"] = ["pca", "tica"]
    cfg["common"]["input_colvars"] = {"start": 2, "stop": 160, "stride": 1}
    outs = {}
    for tag in ("text", "sidecar"):
        if tag == "sidecar":
            cio.write_sidecar(src)
            assert cio.has_fresh_sidecar(src)
        outs[tag] = train_colvars(configuration=copy.deepcopy(cfg), train_colvars_paths=[src],
                                  trajectory_names=["CA_example"], features_list=feats,
                                  output_folder=str(tmp_path / f"train_{tag}"))
    for cv in ("pca", "tica"):
        a = CVCalculator.load(outs["text"][cv]["model_path"], str(tmp_path / f"la_{cv}"))
        b = CVCalculator.load(outs["sidecar"][cv]["model_path"], str(tmp_path / f"lb_{cv}"))
        assert np.array_equal(a.cv, b.cv)
        assert np.array_equal(a.features_norm_mean, b.features_norm_mean)
        pa = pd.read_csv(outs["text"][cv]["traj_paths"][0]).to_numpy()
        pb = pd.read_csv(outs["sidecar"][cv]["traj_paths"][0]).to_numpy()
        assert np.array_equal(pa, pb)


@pytest.mark.parametrize("cv", ["pca", "tica", "htica"])
def test_projection_with_golden_weights_reproduces_golden_csv(dev, c1, tmp_path, cv):
    """The reference's tests/test_traj_projection.py: golden model -> golden CSV (KAT for the
    projection + normalisation kernels)."""
    from deep_cartograph_b200.modules.cv_learning.cv_calculator import cv_calculators_map
    calc = cv_calculators_map[cv](configuration=_config()["common"], output_path=str(tmp_path))
    calc.cv = c1[f"{cv}_cv_weights"]
    calc.cv_norm_mean = c1[f"{cv}_cv_norm_mean"]
    calc.cv_norm_range = c1[f"{cv}_cv_norm_range"]
    calc.features_norm_mean = c1[f"{cv}_features_norm_mean"]
    calc.features_norm_range = c1[f"{cv}_features_norm_range"]
    P = calc.project_data(torch.from_numpy(c1["X"].copy()), normalize_data=True).numpy()
    got = np.array([[float("%.4f" % v) for v in row] for row in P])
    assert np.count_nonzero(got != c1[f"{cv}_csv"]) <= 3
    np.testing.assert_allclose(P, c1[f"{cv}_csv"], atol=1.1e-4)


@pytest.mark.parametrize("engine", ENGINES)
def test_calculators_match_float64_oracle_on_synthetic(dev, tmp_path, engine):
    """Well-separated slow modes (SURVEY 8d): eigenvalues / eigenvectors within 1e-5 of float64."""
    from deep_cartograph_b200.modules.cv_learning.cv_calculator import cv_calculators_map
    n, f, lag, d = 30000, 256, 10, 4
    X = synth_features(n, f, seed=9)
    cfg = dict(_config(engine)["common"], dimension=d, lag_time=lag, num_subspaces=8, subspaces_dimension=5)
    Z = oracle.standardize(X, *oracle.prepare_normalization(oracle.column_stats(X), "mean_std"))
    for cv in ("pca", "tica", "htica"):
        calc = cv_calculators_map[cv](configuration=cfg, output_path=str(tmp_path / cv))
        calc.load_training_tensor(torch.from_numpy(X))
        proj = calc.run(d)
        assert proj is not None
        if cv == "pca":
            evals, W = oracle.pca(Z, d)
        elif cv == "tica":
            evals, W = oracle.tica(Z, lag, d)
        else:
            W, _, _ = oracle.htica(Z, lag, 8, 5, d)
            evals = None
        gap = 1.0
        if evals is not None:
            np.testing.assert_allclose(calc.eigenvalues, evals, rtol=1e-5)
        np.testing.assert_allclose(calc.cv, W, atol=1e-5 * gap + 2e-7 * 50)
        # projection of the training data, normalised to [-1, 1]
        P = oracle.project(Z, W)
        cm, cr = oracle.cv_normalization(P)
        np.testing.assert_allclose(proj.to_numpy(), (P - cm) / cr, atol=1e-4)


@pytest.mark.parametrize("cv,n,f", [("tica", 30000, 256), ("pca", 20000, 130), ("htica", 24000, 300)])
def test_streamed_load_with_speculative_sums_matches_resident_path(dev, tmp_path, cv, n, f):
    """Host tensor in: the matrix is copied in chunks and the covariance sums are accumulated
    under first-chunk standardisation while the copy runs, then corrected exactly.  The weights
    must equal those of the resident path (device tensor in, sums taken after the statistics)."""
    from deep_cartograph_b200.modules.cv_learning.cv_calculator import cv_calculators_map
    X = torch.from_numpy(synth_features(n, f, seed=n + f))
    cfg = {"dimension": 3, "lag_time": 5, "features_normalization": "mean_std", "num_subspaces": 3,
           "subspaces_dimension": 4, "backend": {"h2d_chunk_bytes": 4 * f * 4096}}
    a = cv_calculators_map[cv](configuration=cfg, output_path=str(tmp_path / "a"))
    a.load_training_tensor(X.pin_memory())
    assert a._spec is not None and a._spec["rows_done"] == n
    a.cv_dimension = 3
    a.compute_cv()
    assert a._spec is None                                       # consumed
    b = cv_calculators_map[cv](configuration=cfg, output_path=str(tmp_path / "b"))
    b.load_training_tensor(X.to(dev))
    assert b._spec is None
    b.cv_dimension = 3
    b.compute_cv()
    np.testing.assert_array_equal(a.features_norm_mean, b.features_norm_mean)
    np.testing.assert_array_equal(a.features_norm_range, b.features_norm_range)
    np.testing.assert_allclose(a.cv, b.cv, atol=2e-5)


def test_speculative_sums_are_discarded_when_provisional_statistics_are_off(dev, tmp_path):
    """The guard: provisional parameters far from the final ones (here: forced) make the calculator
    drop the speculative sums and recompute on the resident matrix; results match the float64
    oracle either way."""
    from deep_cartograph_b200.modules.cv_learning.cv_calculator import TICACalculator
    n, f = 20000, 130
    X = synth_features(n, f, seed=9)
    cfg = {"dimension": 2, "lag_time": 4, "features_normalization": "mean_std",
           "backend": {"h2d_chunk_bytes": 4 * f * 2048}}
    calc = TICACalculator(configuration=cfg, output_path=str(tmp_path))
    calc.load_training_tensor(torch.from_numpy(X).pin_memory())
    assert calc._spec is not None
    m0, r0 = calc._spec["norm0"]
    calc._spec["norm0"] = (m0 + 3.0 * r0, r0)                  # as if the sample had been 3 sigma off
    mean, rng = calc._norm_on_device()
    spec = dict(calc._spec)
    assert calc._take_speculative_sums(calc.training_data, 4, 0, True, mean, rng, None) is None
    calc._spec = spec
    calc.cv_dimension = 2
    calc.compute_cv()
    Z = oracle.standardize(X, calc.features_norm_mean.astype(np.float32), calc.features_norm_range.astype(np.float32))
    evals, V = oracle.tica(Z, 4, 2)
    np.testing.assert_allclose(calc.cv, V, atol=1e-5)


def test_deeptica_calculator_trains_projects_and_round_trips(dev, tmp_path):
    """DeepTICACalculator (reference NonLinear / DeepTICA protocol): training on the fused minibatch
    loss improves the validation score, the slow mode of a synthetic series is recovered (leading
    eigenvalue close to linear TICA's), projections are min-max normalised to [-1, 1], and the
    TorchScript model.zip reproduces them after CVCalculator.load."""
    from deep_cartograph_b200.modules.cv_learning.cv_calculator import CVCalculator, cv_calculators_map
    n, f, lag = 6000, 24, 5
    X = synth_features(n, f, seed=21, n_slow=3)
    cfg = {"dimension": 2, "lag_time": lag, "features_normalization": "mean_std", "tica_regularization": 1e-6,
           "architecture": {"encoder": {"layers": [16, 8], "activation": ["tanh", "tanh"]}},
           "training": {"general": {"num_tries": 2, "seed": 3, "lengths": [0.8, 0.2], "batch_size": 512,
                                    "max_epochs": 40, "shuffle": True, "random_split": True,
                                    "check_val_every_n_epoch": 4},
                        "early_stopping": {"patience": 5, "min_delta": 1e-5},
                        "optimizer": {"name": "Adam", "kwargs": {"lr": 5e-3}}, "model_to_save": "best"}}
    calc = cv_calculators_map["deep_tica"](configuration=cfg, output_path=str(tmp_path))
    calc.load_training_tensor(torch.from_numpy(X).to(dev), [f"f{i}" for i in range(f)])
    df = calc.run(2)
    assert df is not None and list(df.columns) == ["DeepTIC 1", "DeepTIC 2"]
    assert len(calc.tries_report) == 2 and any(t["accepted"] for t in calc.tries_report)
    assert -2.0 - 1e-6 <= calc.best_score < -0.5                     # -sum lambda^2 with lambda_1 ~ 0.98
    P = df.to_numpy()
    np.testing.assert_allclose(P.min(axis=0), -1.0, atol=1e-5)
    np.testing.assert_allclose(P.max(axis=0), 1.0, atol=1e-5)
    # linear TICA of the same data: the network's leading eigenvalue must not be far below it
    Z = oracle.standardize(X, calc.features_norm_mean.astype(np.float32), calc.features_norm_range.astype(np.float32))
    ev_lin, _ = oracle.tica(Z, lag, 2)
    assert calc.eigenvalues[0] > ev_lin[0] - 0.05
    model_zip = os.path.join(str(tmp_path), "deep_tica", "model.zip")
    assert os.path.exists(model_zip)
    again = CVCalculator.load(model_zip, str(tmp_path / "reload"))
    assert again.get_cv_type() == "non-linear" and again.get_labels() == ["DeepTIC 1", "DeepTIC 2"]
    P2 = again.project_data(torch.from_numpy(X)).cpu().numpy()
    np.testing.assert_allclose(P2, P, atol=2e-5)


def test_traj_cluster_step_api_kmeans(dev, c1, tmp_path):
    from deep_cartograph_b200.tools import traj_cluster
    csv = tmp_path / "tica.csv"
    pd.DataFrame(c1["tica_csv"], columns=list(c1["tica_csv_cols"])).to_csv(csv, index=False, float_format="%.4f")
    cfg = {"algorithm": "kmeans", "search_interval": [3, 5], "n_init": 2}
    out = traj_cluster(cfg, [str(csv)], output_folder=str(tmp_path / "cl"))
    df = pd.read_csv(out["traj_0"][0])
    assert list(df.columns) == ["TIC 1", "TIC 2", "traj_label", "cluster", "centroid", "frame"]
    assert df["centroid"].sum() == df["cluster"].nunique()
    # fixed-init path == oracle
    init = c1["tica_csv"][:4].copy()
    out = traj_cluster(cfg, [str(csv)], output_folder=str(tmp_path / "cl2"), initial_centroids=init)
    df = pd.read_csv(out["traj_0"][0])
    res = oracle.kmeans_lloyd(c1["tica_csv"], init)
    diff = np.flatnonzero(df["cluster"].to_numpy() != res["labels"])
    assert np.all(res["second"][diff] - res["best"][diff] <= 1e-9)


def test_ops_reject_cpu_tensors():
    from deep_cartograph_b200 import ops
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.column_stats(torch.zeros(4, 4))


# ------------------------------------------------------------------------------------------------
# N4 free-energy surface (binned KDE)
# ------------------------------------------------------------------------------------------------
def test_fes_matches_reference_legacy_output_and_oracle(dev):
    """compute_fes on the device == the numpy restatement == the FES the reference wrote for its
    calpha_transitions example (2-D, one block)."""
    from deep_cartograph_b200.modules.figures import figures
    from oracle import fes_oracle as fo
    g = dict(np.load(os.path.join(GOLDEN, "fes_legacy_pca.npz")))
    bounds = [tuple(b) for b in g["bounds"]]
    fes, grid, b, err = figures.compute_fes(g["X"], temp=float(g["temperature"]), num_samples=int(g["num_bins"]),
                                            bounds=bounds, bandwidth=float(g["bandwidth"]), blocks=1, eps=1e-10)
    ref, rgrid, _, _ = fo.compute_fes(g["X"].astype(np.float32), 300, 200, bounds, 0.025, 1, 1e-10)
    assert err is None
    np.testing.assert_allclose(np.asarray(grid), np.asarray(rgrid), atol=1e-12)
    low = ref < 25
    assert np.abs(fes - ref)[low].max() < 1e-4            # same algorithm: float32 binning weights only
    assert np.abs(fes - g["fes"])[g["fes"] < 20].max() < 2e-3


@pytest.mark.parametrize("n,blocks,bins", [(25_000, 100, 150), (9_999, 7, 64), (1_000_003, 100, 150)])
def test_fes_1d_block_average_matches_oracle(dev, n, blocks, bins):
    from deep_cartograph_b200.modules.figures import figures
    from oracle import fes_oracle as fo
    rng = np.random.default_rng(n)
    x = np.concatenate([rng.normal(-0.5, 0.1, n // 3), rng.normal(0.4, 0.2, n - n // 3)]).astype(np.float32)
    rng.shuffle(x)
    P = torch.zeros((n, 3), dtype=torch.float32, device=dev)
    P[:, 1] = torch.from_numpy(x).to(dev)                      # a column of a wider projection
    bounds = fo.get_ranges(x)
    fes, grid, _, err = figures.compute_fes(P, num_samples=bins, bounds=bounds, bandwidth=0.05, blocks=blocks,
                                            eps=1e-10, cols=[1])
    ref, rgrid, _, rerr = fo.compute_fes(x, 300, bins, bounds, 0.05, blocks, 1e-10)
    np.testing.assert_allclose(grid, rgrid, atol=1e-12)
    core = ref < 20
    assert np.abs(fes - ref)[core].max() < 2e-4
    assert np.abs(err - rerr)[core].max() < 2e-4


def test_fes_2d_large_and_outside_frames(dev):
    """2-D FES of 4M frames against the oracle on a strided subsample's bounds (size-independent: the
    density integrates to one), and frames outside the bounds are counted, not binned."""
    from deep_cartograph_b200 import ops
    from oracle import fes_oracle as fo
    n = 4_000_000
    g = torch.Generator(device=dev).manual_seed(1)
    P = torch.randn((n, 4), generator=g, device=dev) * torch.tensor([0.3, 0.2, 1.0, 1.0], device=dev)
    bounds = [(-1.2, 1.2), (-0.9, 0.9)]
    dens, frames, outside = ops.fes_density(P, [0, 1], bounds, 150, 0.05, 1)
    n_out = int(((P[:, 0].abs() > 1.2) | (P[:, 1].abs() > 0.9)).sum())
    assert int(outside.item()) == n_out and n_out > 0
    step = (2.4 / 149) * (1.8 / 149)
    assert abs(float(dens.sum()) * step * n / (n - n_out) - 1.0) < 2e-3
    sub = P[: 200_000, :2].cpu().numpy()
    inside = (np.abs(sub[:, 0]) <= 1.2) & (np.abs(sub[:, 1]) <= 0.9)
    ref = fo.binned_density(sub[inside], bounds, 150, 0.05)
    d2, _, _ = ops.fes_density(torch.from_numpy(sub[inside]).to(dev), [0, 1], bounds, 150, 0.05, 1)
    np.testing.assert_allclose(d2[0].cpu().numpy(), ref, rtol=2e-5, atol=1e-7)


def test_train_colvars_writes_fes_files(dev, c1, tmp_path):
    """Step API with figures.fes.compute: fes*.npy per component (100 blocks, reduced to 1 for 164
    frames as the reference does) and per pair."""
    from deep_cartograph_b200.tools.train_colvars.train_colvars import train_colvars
    cfg = _config()
    cfg["cvs"] = ["pca"]
    cfg["figures"] = {"fes": {"compute": True, "save": True, "num_bins": 50, "bandwidth": 0.1}}
    out = train_colvars(configuration=cfg, train_colvars_paths=[os.path.join(GOLDEN, "peptide_c1.dat")],
                        features_list=list(np.loadtxt(os.path.join(GOLDEN, "peptide_c1_features.txt"), dtype=str)),
                        dimension=2, output_folder=str(tmp_path))
    base = os.path.dirname(out["pca"]["traj_paths"][0])
    for sub, shape in (("fes_PCA_1", (50,)), ("fes_PCA_2", (50,)), ("fes_PCA_1_2", (50, 50))):
        fes = np.load(os.path.join(base, sub, "fes.npy"))
        assert fes.shape == shape and np.isfinite(fes).all() and fes.min() == 0.0
        assert os.path.exists(os.path.join(base, sub, "fes_grid.npy"))


# ------------------------------------------------------------------------------------------------
# N3 PLUMED export of linear CVs
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cv", ["pca", "tica", "htica"])
def test_plumed_combine_lines_reproduce_the_projected_csv(dev, c1, tmp_path, cv):
    """The reference's end-to-end check (tests/test_deep_cartograph.py:209-258: PLUMED's projection of
    the linear CVs vs the CSV, |diff| < 1e-2) with the COMBINE arithmetic evaluated in float64: the
    parameters get_cv_parameters() hands to the PLUMED assembler (assembler.py:333-379) reproduce the
    CSV train_colvars wrote -- and the reference's golden CSV."""
    from deep_cartograph_b200.modules.cv_learning.cv_calculator import CVCalculator
    from deep_cartograph_b200.modules.plumed.input import assembler
    from deep_cartograph_b200.tools import train_colvars
    feats = [l.strip() for l in open(os.path.join(GOLDEN, "peptide_c1_features.txt")) if l.strip()]
    cfg = _config("auto")
    cfg["cvs"] = [cv]
    out = train_colvars(configuration=cfg, train_colvars_paths=[os.path.join(GOLDEN, "peptide_c1.dat")],
                        trajectory_names=["CA_example"], features_list=feats, output_folder=str(tmp_path / "tc"))
    calc = CVCalculator.load(out[cv]["model_path"], str(tmp_path / "loaded"))
    params = calc.get_cv_parameters()
    # a loaded model has no training projection: cv_stats come back from the stored CV normalisation
    assert params["features_norm_mean"].dtype == np.float32 and params["weights"].shape == (len(feats), 2)
    params["features_norm_mode"] = "mean_std"
    params["cv_stats"] = {"min": calc.cv_norm_mean - calc.cv_norm_range, "max": calc.cv_norm_mean + calc.cv_norm_range}
    text, labels = assembler.add_linear_cv(params, feats)
    assert text.count("COMBINE") == len(feats) + 4 and all(" PERIODIC=NO" in l for l in text.splitlines() if "COMBINE" in l)
    table = {name: c1["X"][:, i] for i, name in enumerate(feats)}
    vals = assembler.evaluate_combine(text, table, labels)
    plumed_proj = np.stack([vals[l] for l in labels], axis=1)
    csv = pd.read_csv(out[cv]["traj_paths"][0]).to_numpy()
    assert np.abs(plumed_proj - csv).max() < 1.5e-4                      # 4-decimal print + float32 projection
    assert np.abs(plumed_proj - c1[f"{cv}_csv"]).max() < 1e-2            # the reference's threshold


# ------------------------------------------------------------------------------------------------
# K2 / N1: the reference's default clustering path (k-means++ seeding, scores, choice of k)
# ------------------------------------------------------------------------------------------------
def test_kmeans_plus_plus_and_scores_match_the_reference(dev, kmeans_ref):
    """kmeans_clustering WITHOUT initial centroids == the reference's KMeans(random_state=0,
    init='k-means++', n_init) (tests/golden/kmeans_ref.npz: produced by the reference's imported
    statistics.kmeans_clustering), and the three model-selection scores == scikit-learn's on its labels."""
    from deep_cartograph_b200.modules.statistics import statistics
    X = kmeans_ref["opt_X"]
    labels, centers = statistics.kmeans_clustering(X.copy(), 6, 4)
    np.testing.assert_array_equal(labels, kmeans_ref["pp_labels"])
    np.testing.assert_allclose(centers, kmeans_ref["pp_centers"], rtol=1e-10, atol=1e-12)
    sc = statistics.cluster_scores(X, labels)
    ch, db, sil = kmeans_ref["pp_scores"]
    assert abs(sc["calinski_harabasz"] - ch) <= 1e-9 * ch
    assert abs(sc["davies_bouldin"] - db) <= 1e-9 * db
    assert abs(statistics.silhouette(X, labels) - sil) <= 1e-9
    # sklearn's sample_size estimator: a subsample scored against itself
    from sklearn.metrics import silhouette_score
    est = statistics.silhouette(X, labels, sample_size=2000, seed=0)
    idx = np.random.RandomState(0).permutation(X.shape[0])[:2000]
    assert abs(est - silhouette_score(X[idx], labels[idx])) <= 1e-9


def test_optimize_clustering_matches_the_reference(dev, kmeans_ref):
    """The default traj_cluster path for kmeans (reference statistics.py:54-100): same k, same labels,
    same centres as the reference's own optimize_clustering on the same frames."""
    from deep_cartograph_b200.modules.statistics import statistics
    settings = {"algorithm": "kmeans", "search_interval": [2, 8], "n_init": 3}
    labels, centers = statistics.optimize_clustering(kmeans_ref["opt_X"].copy(), settings)
    assert centers.shape == kmeans_ref["opt_centers"].shape, statistics.last_optimize_report
    np.testing.assert_array_equal(labels, kmeans_ref["opt_labels"])
    np.testing.assert_allclose(centers, kmeans_ref["opt_centers"], rtol=1e-10, atol=1e-12)
    assert settings["num_clusters"] == 8                   # mutated like the reference (statistics.py:67)


def test_cluster_dispersion_kernel(dev):
    from deep_cartograph_b200 import ops
    rng = np.random.default_rng(4)
    for dt in (np.float32, np.float64):
        Y = rng.normal(size=(50_001, 7)).astype(dt)
        lab = rng.integers(0, 13, size=50_001).astype(np.int32)
        lab[:4000] = 5                                      # a run of equal labels (warp-uniform path)
        means = np.stack([Y[lab == c].astype(np.float64).mean(0) for c in range(13)])
        ssq, sdist = ops.cluster_dispersion(_cuda(Y, dev), _cuda(lab, dev), _cuda(means, dev))
        q = ((Y.astype(np.float64) - means[lab]) ** 2).sum(1)
        np.testing.assert_allclose(ssq.cpu().numpy(), np.bincount(lab, weights=q, minlength=13), rtol=1e-12)
        np.testing.assert_allclose(sdist.cpu().numpy(), np.bincount(lab, weights=np.sqrt(q), minlength=13), rtol=1e-12)


# ------------------------------------------------------------------------------------------------
# A3: every normalisation mode through the fused kernels
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [None, "min_max_range1", "min_max_range2", "mean_std"])
@pytest.mark.parametrize("engine", ["auto", "tc_3xtf32"])
def test_normalisation_modes_through_the_fused_kernels(dev, tmp_path, mode, engine):
    """features_normalization None (the schema default: raw features, |mean| >> std), min_max_range1,
    min_max_range2 and mean_std (reference cv_calculator.py:308-363) through the fused standardise +
    covariance and standardise + projection kernels: TICA eigenvalues / eigenvectors / projections
    against the float64 checker run with the SAME (mean, range)."""
    from deep_cartograph_b200.modules.cv_learning.cv_calculator import TICACalculator
    from oracle import float64_device as f64
    n, f, lag, d = 40_000, 200, 5, 3
    X = synth_features(n, f, seed=21)
    cfg = {"dimension": d, "lag_time": lag, "features_normalization": mode, "backend": {"cov_engine": engine}}
    calc = TICACalculator(configuration=cfg, output_path=str(tmp_path))
    calc.load_training_tensor(torch.from_numpy(X))
    m, r = oracle.prepare_normalization(oracle.column_stats(X), mode)
    np.testing.assert_allclose(calc.features_norm_mean, m, rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(calc.features_norm_range, r, rtol=2e-6)
    calc.create_output_folders(); calc.compute_cv(); calc.set_labels()
    P = calc.normalize_cv()
    Xd = _cuda(X, dev)
    mean = rng = None
    if mode is not None:
        mean = torch.tensor(calc.features_norm_mean, dtype=torch.float32, device=dev)
        rng = torch.tensor(calc.features_norm_range, dtype=torch.float32, device=dev)
    ref = f64.lagged_sums(Xd, lag, mean, rng)
    ev_ref, V_ref = f64.tica_from_sums(ref["S0"], ref["St"], ref["a"], ref["b"], ref["M"], d)
    np.testing.assert_allclose(calc.eigenvalues, ev_ref.cpu().numpy(), rtol=1e-5)
    err = f64.eigvec_error(torch.from_numpy(calc.cv).to(dev), V_ref)
    # The exact integer engine (auto) holds the 1e-5 eigenvector tolerance in every mode.  The float engine
    # (FP32 tensor-core accumulation, 2e-6 of the sums) is the non-default fallback: it lands at 1-3e-5 on
    # centred features (mean_std); on uncentred ones (mode None, and the min_max modes whose "mean" is the
    # column minimum: C0 dominated by the offsets, cond ~ 1e6) its sum error is amplified accordingly
    # (measured 4.6e-4 for min_max_range1).
    tol = 1e-5 if engine == "auto" else (5e-5 if mode == "mean_std" else 5e-3)
    assert err < tol, (mode, engine, err)
    Pn_ref, _, _ = f64.project_normalized(Xd, mean, rng, V_ref)
    sgn = torch.sign((torch.from_numpy(calc.cv).to(dev).double() * V_ref).sum(0, keepdim=True))
    assert (P.double() * sgn - Pn_ref).abs().max().item() < 1e-4 or engine != "auto"
