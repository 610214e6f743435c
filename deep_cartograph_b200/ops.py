"""Device operators of the CV hot path: thin torch-tensor wrappers over the C-ABI.

Every operator takes CUDA tensors, launches on torch's current stream and returns CUDA
tensors.  CPU tensors raise: the product has no CPU path (the CPU restatement lives in
``oracle/`` and is test infrastructure only).
"""
from __future__ import annotations

import os
from typing import Optional

import torch

from . import _lib
from ._lib import COV_ENGINES, DcgError  # noqa: F401


# Number of libdcg_b200 kernels launched through this module (bench.py reports it).
KERNEL_LAUNCHES = 0


def _count(n: int) -> None:
    global KERNEL_LAUNCHES
    KERNEL_LAUNCHES += n


def _stream(dev) -> int:
    """torch's current stream ON THE DEVICE OF THE TENSORS (not of the current device)."""
    return torch.cuda.current_stream(dev).cuda_stream


def _call(dev, fn: str, *args) -> None:
    """Library call in the device context of the tensors: ``backend.device`` may name a GPU that is
    not torch's current one, and the library keys its attribute caches / arch checks / launches on
    ``cudaGetDevice``."""
    if dev.index is not None and dev.index != torch.cuda.current_device():
        with torch.cuda.device(dev):
            _lib.call(fn, *args)
    else:
        _lib.call(fn, *args)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need_cuda(name: str, t: torch.Tensor, dtype=None) -> None:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: deep_cartograph_b200 has no CPU fallback")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")


def _rows(name: str, t: torch.Tensor):
    """(n, f, ld) of a 2-D tensor whose rows are contiguous."""
    if t.dim() != 2:
        raise ValueError(f"{name} must be 2-D (frames x features)")
    if t.shape[1] > 1 and t.stride(1) != 1:
        raise ValueError(f"{name} rows must be contiguous")
    ld = t.stride(0) if t.shape[0] > 1 else t.shape[1]
    return t.shape[0], t.shape[1], max(ld, t.shape[1])


def _ws(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def default_cov_engine(standardised: bool = True) -> int:
    """Engine used when none is requested: env DCG_COV_ENGINE, else the exact integer tensor-core
    engine (``tc_i8x3``: 23-bit fixed point per column, int32 accumulation -- the only fast engine
    that holds the 1e-5 eigenvector tolerance at the C2 eigenvalue gaps; DESIGN.md 3.1).  The float
    engines stay selectable: ``tc_3xf16`` needs standardised inputs (|z| < 65504), ``tc_3xtf32`` does not."""
    name = os.environ.get("DCG_COV_ENGINE", "auto")
    if name == "auto":
        return COV_ENGINES["tc_i8x3"]
    if name not in COV_ENGINES:
        raise ValueError(f"DCG_COV_ENGINE={name!r}; choose from {sorted(COV_ENGINES)} or 'auto'")
    return COV_ENGINES[name]


def resolve_engine(engine, standardised: bool = True) -> int:
    if engine is None or engine == "auto":
        return default_cov_engine(standardised)
    if isinstance(engine, str):
        return COV_ENGINES[engine]
    return int(engine)


# ---- A2 ---------------------------------------------------------------------------------------
def column_stats(X: torch.Tensor) -> dict:
    """Single-pass per-feature statistics (reference cv_calculator.py:295-297).

    Returns dict(n, mean[f64], m2[f64], min[f32], max[f32]); std(ddof=1) = sqrt(m2/(n-1))."""
    _need_cuda("X", X, torch.float32)
    n, f, ld = _rows("X", X)
    lib = _lib.load()
    dev = X.device
    mean = torch.empty(f, dtype=torch.float64, device=dev)
    m2 = torch.empty(f, dtype=torch.float64, device=dev)
    mn = torch.empty(f, dtype=torch.float32, device=dev)
    mx = torch.empty(f, dtype=torch.float32, device=dev)
    max_rows = 65535 * 1024
    if n <= max_rows:
        ws = _ws(lib.dcg_colstats_workspace_bytes(n, f), dev)
        _call(X.device, "dcg_colstats_f32", X.data_ptr(), n, f, ld, mean.data_ptr(), m2.data_ptr(),
                  mn.data_ptr(), mx.data_ptr(), ws.data_ptr(), ws.numel(), _stream(X.device))
        _count(2)
        return {"n": n, "mean": mean, "m2": m2, "min": mn, "max": mx}
    parts = [column_stats(X[s:s + max_rows]) for s in range(0, n, max_rows)]
    return merge_column_stats(parts)


def merge_column_stats(parts) -> dict:
    """Chan merge of per-shard statistics (FP64); also used across GPUs."""
    n = 0
    mean = m2 = mn = mx = None
    for p in parts:
        if p["n"] == 0:
            continue
        if n == 0:
            n, mean, m2, mn, mx = p["n"], p["mean"].clone(), p["m2"].clone(), p["min"].clone(), p["max"].clone()
            continue
        nb = p["n"]
        nt = n + nb
        dl = p["mean"] - mean
        mean = mean + dl * (nb / nt)
        m2 = m2 + p["m2"] + dl * dl * (n * nb / nt)
        mn = torch.minimum(mn, p["min"])
        mx = torch.maximum(mx, p["max"])
        n = nt
    return {"n": n, "mean": mean, "m2": m2, "min": mn, "max": mx}


# ---- A4 ---------------------------------------------------------------------------------------
def standardize_(X: torch.Tensor, mean: torch.Tensor, rng: torch.Tensor) -> torch.Tensor:
    """In-place IEEE float32 ``(x - mean) / range`` (reference cv_calculator.py:806-837)."""
    _need_cuda("X", X, torch.float32)
    _need_cuda("mean", mean, torch.float32)
    _need_cuda("range", rng, torch.float32)
    n, f, ld = _rows("X", X)
    if mean.numel() != f or rng.numel() != f:
        raise ValueError("mean / range length must equal the number of columns")
    if n == 0:
        return X
    _call(X.device, "dcg_standardize_f32", X.data_ptr(), n, f, ld, mean.contiguous().data_ptr(),
              rng.contiguous().data_ptr(), _stream(X.device))
    _count(1)
    return X


def stats_pack(st: dict) -> torch.Tensor:
    """This rank's column statistics as one FP64 record [n | mean | m2 | min | max] (one launch): the
    contribution to the all-gather of ``FrameShards.merge_stats``."""
    mean, m2, mn, mx = st["mean"], st["m2"], st["min"], st["max"]
    _need_cuda("mean", mean, torch.float64)
    f = mean.numel()
    out = torch.empty(1 + 4 * f, dtype=torch.float64, device=mean.device)
    _call(mean.device, "dcg_stats_pack", float(st["n"]), mean.contiguous().data_ptr(), m2.contiguous().data_ptr(),
          mn.contiguous().data_ptr(), mx.contiguous().data_ptr(), f, out.data_ptr(), _stream(mean.device))
    _count(1)
    return out


def stats_merge(all_packed: torch.Tensor, world: int, f: int) -> dict:
    """Chan merge of ``world`` packed records (one launch, FP64).  Returns dict(mean, m2, min, max, n) with
    ``n`` a 1-element FP64 device tensor (no host read here)."""
    _need_cuda("all_packed", all_packed, torch.float64)
    if all_packed.numel() != world * (1 + 4 * f):
        raise ValueError("all_packed must hold world records of 1 + 4 f doubles")
    dev = all_packed.device
    mean = torch.empty(f, dtype=torch.float64, device=dev)
    m2 = torch.empty(f, dtype=torch.float64, device=dev)
    mn = torch.empty(f, dtype=torch.float32, device=dev)
    mx = torch.empty(f, dtype=torch.float32, device=dev)
    n = torch.empty(1, dtype=torch.float64, device=dev)
    _call(dev, "dcg_stats_merge", all_packed.contiguous().data_ptr(), world, f, mean.data_ptr(), m2.data_ptr(),
          mn.data_ptr(), mx.data_ptr(), n.data_ptr(), _stream(dev))
    _count(1)
    return {"mean": mean, "m2": m2, "min": mn, "max": mx, "n": n}


# ---- A5/A6/A7/A8 ------------------------------------------------------------------------------
def lagged_covariance(X: torch.Tensor, lag: int, mean: Optional[torch.Tensor] = None,
                      rng: Optional[torch.Tensor] = None, block: int = 0, engine=None,
                      want_s0: bool = True, want_st: bool = True,
                      xmin: Optional[torch.Tensor] = None, xmax: Optional[torch.Tensor] = None) -> dict:
    """Raw FP64 sums over the M = n_rows - lag pairs of the (optionally standardised) rows:
    S0 = sum z_t z_t^T (upper triangle valid), St = sum z_t z_{t+lag}^T, a = sum_{t<M} z_t,
    b = sum_{t>=lag} z_t.  Replaces create_timelagged_dataset + TICA.compute's correlation
    sums (reference cv_calculator.py:2244-2261).

    ``xmin`` / ``xmax`` (per-column bounds of X, float32) are used by the exact integer engine
    (``tc_i8x3``); when absent they are taken from X here (one more pass over X).  That engine also
    returns ``clamped`` (int32, device): nonzero if and only if some value of X lay far enough outside
    the bounds to be clamped to the fixed-point range; the number itself is not a count of values."""
    _need_cuda("X", X, torch.float32)
    n, f, ld = _rows("X", X)
    if not (0 <= lag < n):
        raise ValueError(f"lag {lag} out of range for {n} rows")
    if (mean is None) != (rng is None):
        raise ValueError("mean and range must be given together")
    if mean is not None:
        _need_cuda("mean", mean, torch.float32)
        _need_cuda("range", rng, torch.float32)
        mean = mean.contiguous()
        rng = rng.contiguous()
    eng = resolve_engine(engine, standardised=mean is not None)
    lib = _lib.load()
    dev = X.device
    want_st = want_st and lag > 0
    # one flat buffer [S0 | St | a | b | M]: the frame-sharded path all-reduces it in place (no packing copy)
    n0, nt = (f * f if want_s0 else 0), (f * f if want_st else 0)
    flat = torch.empty(n0 + nt + 2 * f + 1, dtype=torch.float64, device=dev)
    S0 = flat[:n0].view(f, f) if want_s0 else None
    St = flat[n0:n0 + nt].view(f, f) if want_st else None
    a = flat[n0 + nt:n0 + nt + f]
    b = flat[n0 + nt + f:n0 + nt + 2 * f]
    flat[-1:].fill_(float(n - lag))
    if eng == _lib.COV_TC_I8X3:
        if xmin is None or xmax is None:
            xmin, xmax = X.amin(dim=0), X.amax(dim=0)
        _need_cuda("xmin", xmin, torch.float32)
        _need_cuda("xmax", xmax, torch.float32)
        info = torch.empty(1, dtype=torch.int32, device=dev)
        ws = _ws(lib.dcg_cov_i8_workspace_bytes(n, f, lag, block), dev)
        _call(X.device, "dcg_cov_lag_i8_f32", X.data_ptr(), n, f, ld, lag, _ptr(mean), _ptr(rng),
              xmin.contiguous().data_ptr(), xmax.contiguous().data_ptr(), block, _ptr(S0), _ptr(St),
              a.data_ptr(), b.data_ptr(), info.data_ptr(), ws.data_ptr(), ws.numel(), _stream(X.device))
        _count(5)                                      # prep + plan + quantise + contraction + column sums (per window)
        return {"S0": S0, "St": St, "a": a, "b": b, "M": n - lag, "clamped": info, "flat": flat}
    ws = _ws(lib.dcg_cov_workspace_bytes(n, f, lag, block, eng), dev)
    _call(X.device, "dcg_cov_lag_f32", X.data_ptr(), n, f, ld, lag, _ptr(mean), _ptr(rng), block,
              _ptr(S0), _ptr(St), a.data_ptr(), b.data_ptr(), eng, ws.data_ptr(), ws.numel(),
              _stream(X.device))
    _count(2 if eng == _lib.COV_SIMT_F32 else 3)      # colsum + engine (+ split reduction)
    return {"S0": S0, "St": St, "a": a, "b": b, "M": n - lag, "flat": flat}


def cov_i8_timing(on: Optional[bool] = None):
    """Switch the exact engine's kernel timing on / off, or (``on`` None) read and reset it:
    returns dict(quantize_ms, contract_ms, launches) summed since the last read."""
    import ctypes
    lib = _lib.load()
    if on is not None:
        _lib.check("dcg_cov_i8_set_timing", lib.dcg_cov_i8_set_timing(1 if on else 0))
        return None
    q, c, n = ctypes.c_float(), ctypes.c_float(), ctypes.c_int()
    _lib.check("dcg_cov_i8_get_timing", lib.dcg_cov_i8_get_timing(ctypes.byref(q), ctypes.byref(c), ctypes.byref(n)))
    return {"quantize_ms": q.value, "contract_ms": c.value, "launches": n.value}


def symmetrize_upper(S: torch.Tensor) -> torch.Tensor:
    """Full symmetric matrix from one whose upper triangle (incl. diagonal) is valid."""
    U = torch.triu(S)
    return U + torch.triu(S, 1).T


# ---- A9/A10 -----------------------------------------------------------------------------------
def project(X: torch.Tensor, W: torch.Tensor, mean: Optional[torch.Tensor] = None,
            rng: Optional[torch.Tensor] = None, minmax: bool = True):
    """``P = ((X - mean)/range) @ W`` in one pass, with per-column min / max of P.
    Replaces LinearCalculator.normalize_cv / project_data (reference cv_calculator.py:918-991).
    Returns (P, pmin, pmax)."""
    _need_cuda("X", X, torch.float32)
    _need_cuda("W", W, torch.float32)
    n, f, ld = _rows("X", X)
    if W.dim() != 2 or W.shape[0] != f:
        raise ValueError(f"W must be ({f}, d)")
    d = W.shape[1]
    if not 1 <= d <= 64:
        raise ValueError("1 <= d <= 64")
    if (mean is None) != (rng is None):
        raise ValueError("mean and range must be given together")
    if mean is not None:
        _need_cuda("mean", mean, torch.float32)
        _need_cuda("range", rng, torch.float32)
        mean = mean.contiguous()
        rng = rng.contiguous()
    lib = _lib.load()
    dev = X.device
    W = W.contiguous()
    P = torch.empty((n, d), dtype=torch.float32, device=dev)
    pmin = torch.empty(d, dtype=torch.float32, device=dev) if minmax else None
    pmax = torch.empty(d, dtype=torch.float32, device=dev) if minmax else None
    if n == 0:
        return P, pmin, pmax
    ws = _ws(lib.dcg_project_workspace_bytes(n, f, d), dev)
    _call(X.device, "dcg_project_f32", X.data_ptr(), n, f, ld, _ptr(mean), _ptr(rng), W.data_ptr(), d,
              P.data_ptr(), _ptr(pmin), _ptr(pmax), ws.data_ptr(), ws.numel(), _stream(X.device))
    passes, nr = (d + 15) // 16, -(-f // 1024)
    if nr > 1 and X.data_ptr() % 16 == 0 and ld % 4 == 0:     # several feature ranges: row batches + combine
        cap = max(16, ((256 << 20) // (nr * 64)) // 16 * 16)
        _count(passes * (1 + 2 * (-(-n // cap))) + (1 if minmax else 0))
    else:
        _count(2 * passes + (1 if minmax else 0))
    return P, pmin, pmax


def project_blocks(X: torch.Tensor, W: torch.Tensor, block: int, mean: Optional[torch.Tensor] = None,
                   rng: Optional[torch.Tensor] = None) -> torch.Tensor:
    """hTICA level 1 (reference cv_calculator.py:2331-2371): every diagonal feature block of width
    ``block`` (torch.split semantics) projected onto its own ``s = W.shape[1]`` columns in ONE pass
    over X.  ``W`` is (f, s): row i holds the weights of feature i inside its block.  Returns
    P (n, sum of min(s, block width)).  Needs 16-byte aligned rows (DcgError -1003 otherwise)."""
    _need_cuda("X", X, torch.float32)
    _need_cuda("W", W, torch.float32)
    n, f, ld = _rows("X", X)
    if W.dim() != 2 or W.shape[0] != f:
        raise ValueError(f"W must be ({f}, s)")
    s = W.shape[1]
    nb = -(-f // block)
    cols = (nb - 1) * s + min(s, f - (nb - 1) * block)
    if (mean is None) != (rng is None):
        raise ValueError("mean and range must be given together")
    if mean is not None:
        _need_cuda("mean", mean, torch.float32)
        _need_cuda("range", rng, torch.float32)
        mean = mean.contiguous()
        rng = rng.contiguous()
    lib = _lib.load()
    dev = X.device
    W = W.contiguous()
    P = torch.empty((n, cols), dtype=torch.float32, device=dev)
    if n == 0:
        return P
    ws = _ws(lib.dcg_project_blocks_workspace_bytes(n, f, block), dev)
    _call(X.device, "dcg_project_blocks_f32", X.data_ptr(), n, f, ld, _ptr(mean), _ptr(rng), W.data_ptr(), block, s,
              P.data_ptr(), cols, ws.data_ptr(), ws.numel(), _stream(X.device))
    _count(2)
    return P


# ---- K1 / K3 ----------------------------------------------------------------------------------
def _dtype_bytes(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return 4
    if t.dtype == torch.float64:
        return 8
    raise TypeError(f"expected float32 or float64, got {t.dtype}")


def _absmax_ptr(absmax: Optional[torch.Tensor], device) -> Optional[int]:
    if absmax is None:
        return None
    if not (isinstance(absmax, torch.Tensor) and absmax.is_cuda and absmax.dtype == torch.float64
            and absmax.numel() == 1 and absmax.device == device):
        raise TypeError("absmax must be a one-element float64 CUDA tensor on the device of Y")
    return absmax.data_ptr()


def kmeans_step(Y: torch.Tensor, centers: torch.Tensor, labels: torch.Tensor,
                update_sums: bool = True, want_gap: bool = False,
                absmax: Optional[torch.Tensor] = None) -> dict:
    """One Lloyd E-step (+ M-step sums).  ``labels`` (int32) holds the previous labels and is
    overwritten.  ``absmax`` (one float64 on the device, optional): a bound on ``|Y|`` that switches
    the partial sums to exact 64-bit fixed point (see dcg.h).
    Returns dict(sums, counts, changed, inertia, ties, gap)."""
    _need_cuda("Y", Y)
    _need_cuda("centers", centers, torch.float64)
    _need_cuda("labels", labels, torch.int32)
    n, d, ld = _rows("Y", Y)
    k = centers.shape[0]
    if centers.dim() != 2 or centers.shape[1] != d:
        raise ValueError("centers must be (k, d)")
    if labels.numel() != n:
        raise ValueError("labels must have one entry per frame")
    dev = Y.device
    centers = centers.contiguous()
    sums = torch.empty((k, d), dtype=torch.float64, device=dev) if update_sums else None
    counts = torch.empty(k, dtype=torch.float64, device=dev) if update_sums else None
    stats = torch.empty(3, dtype=torch.float64, device=dev)
    gap = torch.empty(n, dtype=Y.dtype, device=dev) if want_gap else None
    ws = _ws(256, dev)
    _call(Y.device, "dcg_kmeans_step", Y.data_ptr(), n, d, ld, _dtype_bytes(Y), centers.data_ptr(), k,
              labels.data_ptr(), _ptr(sums), _ptr(counts), stats.data_ptr(), _ptr(gap),
              1 if update_sums else 0, _absmax_ptr(absmax, dev), ws.data_ptr(), ws.numel(), _stream(Y.device))
    _count(1)
    return {"sums": sums, "counts": counts, "stats": stats, "gap": gap}


_KM_WS = {}


def kmeans_step_packed_(Y: torch.Tensor, centers: torch.Tensor, labels: torch.Tensor, work: torch.Tensor,
                        absmax: Optional[torch.Tensor] = None) -> dict:
    """E-step + M-step sums written into ONE buffer ``work = [sums k*d | counts k | stats 3 | ...]``
    (``kmeans_work``): one memset, and a sharded Lloyd iteration can all-reduce ``work[:k*d + k + 3]``
    in place without packing.  Returns views into ``work``."""
    _need_cuda("Y", Y)
    _need_cuda("centers", centers, torch.float64)
    _need_cuda("labels", labels, torch.int32)
    _need_cuda("work", work, torch.float64)
    n, d, ld = _rows("Y", Y)
    k = centers.shape[0]
    if not centers.is_contiguous() or centers.shape[1] != d or work.numel() < k * d + k + 3:
        raise ValueError("centers must be contiguous (k, d) and work at least k*d + k + 3 doubles")
    ws = _KM_WS.get(Y.device)
    if ws is None:
        ws = _KM_WS[Y.device] = _ws(256, Y.device)
    o = k * d
    base = work.data_ptr()
    _call(Y.device, "dcg_kmeans_step", Y.data_ptr(), n, d, ld, _dtype_bytes(Y), centers.data_ptr(), k,
              labels.data_ptr(), base, base + 8 * o, base + 8 * (o + k), None, 1,
              _absmax_ptr(absmax, Y.device), ws.data_ptr(), ws.numel(), _stream(Y.device))
    _count(1)
    return {"sums": work[:o].view(k, d), "counts": work[o:o + k], "stats": work[o + k:o + k + 3],
            "packed": work[:o + k + 3]}


def kmeans_update_(centers: torch.Tensor, sums: torch.Tensor, counts: torch.Tensor,
                   info: Optional[torch.Tensor] = None) -> torch.Tensor:
    """M-step finish on the device: ``info[0]`` = number of empty clusters; when there is none
    ``centers`` (k x d FP64) becomes ``sums * (1 / counts)`` IN PLACE and ``info[1]`` = total squared
    centre shift.  Returns ``info`` (2 x FP64, device); nothing is synchronised."""
    _need_cuda("centers", centers, torch.float64)
    _need_cuda("sums", sums, torch.float64)
    _need_cuda("counts", counts, torch.float64)
    if not (centers.is_contiguous() and sums.is_contiguous() and counts.is_contiguous()):
        raise ValueError("centers, sums and counts must be contiguous")
    k, d = centers.shape
    if info is None:
        info = torch.empty(2, dtype=torch.float64, device=centers.device)
    _call(sums.device, "dcg_kmeans_update", sums.data_ptr(), counts.data_ptr(), k, d, centers.data_ptr(),
              info.data_ptr(), _stream(sums.device))
    _count(1)
    return info


def kmeans_work(k: int, d: int, device) -> torch.Tensor:
    """Work buffer of ``kmeans_iterate_`` / ``kmeans_iterate_n_``:
    [sums k*d | counts k | stats 3 | info 2 | ctl 3] FP64."""
    return torch.empty(k * d + k + 8, dtype=torch.float64, device=device)


def kmeans_iterate_n_(Y: torch.Tensor, centers: torch.Tensor, labels: torch.Tensor, work: torch.Tensor,
                      iters: int, tol: float, absmax: Optional[torch.Tensor] = None) -> dict:
    """Up to ``iters`` Lloyd iterations in ONE library call and without a host round trip: the convergence
    tests (no label changed / centre shift <= ``tol`` / a cluster came out empty) run on the device and the
    launches after the stopping iteration return at once.  Returns views into ``work`` as ``kmeans_iterate_``
    plus ``ctl`` = [stopped, iterations done, tol]."""
    _need_cuda("Y", Y)
    _need_cuda("centers", centers, torch.float64)
    _need_cuda("labels", labels, torch.int32)
    _need_cuda("work", work, torch.float64)
    n, d, ld = _rows("Y", Y)
    k = centers.shape[0]
    if not centers.is_contiguous() or centers.shape[1] != d or work.numel() < k * d + k + 8:
        raise ValueError("centers must be contiguous (k, d) and work at least k*d + k + 8 doubles")
    ws = _KM_WS.get(Y.device)
    if ws is None:
        ws = _KM_WS[Y.device] = _ws(256, Y.device)
    _call(Y.device, "dcg_kmeans_iterate_n", Y.data_ptr(), n, d, ld, _dtype_bytes(Y), centers.data_ptr(), k,
              labels.data_ptr(), work.data_ptr(), _absmax_ptr(absmax, Y.device), int(iters), float(tol),
              ws.data_ptr(), ws.numel(), _stream(Y.device))
    _count(3 * int(iters))
    o = k * d
    return {"sums": work[:o].view(k, d), "counts": work[o:o + k], "stats": work[o + k:o + k + 3],
            "info": work[o + k + 3:o + k + 5], "ctl": work[o + k + 5:o + k + 8]}


def kmeans_iterate_(Y: torch.Tensor, centers: torch.Tensor, labels: torch.Tensor,
                    work: torch.Tensor, absmax: Optional[torch.Tensor] = None) -> dict:
    """One whole Lloyd iteration on one device in ONE library call (memset, E-step + FP64 sums,
    M-step finish): ``centers`` (k x d FP64) and ``labels`` are updated in place.  Returns views
    into ``work``: sums, counts, stats [changed, inertia, ties], info [n_empty, shift]."""
    _need_cuda("Y", Y)
    _need_cuda("centers", centers, torch.float64)
    _need_cuda("labels", labels, torch.int32)
    _need_cuda("work", work, torch.float64)
    n, d, ld = _rows("Y", Y)
    k = centers.shape[0]
    if not centers.is_contiguous() or centers.shape[1] != d or work.numel() < k * d + k + 5:
        raise ValueError("centers must be contiguous (k, d) and work at least k*d + k + 5 doubles")
    ws = _KM_WS.get(Y.device)
    if ws is None:
        ws = _KM_WS[Y.device] = _ws(256, Y.device)
    _call(Y.device, "dcg_kmeans_iterate", Y.data_ptr(), n, d, ld, _dtype_bytes(Y), centers.data_ptr(), k,
              labels.data_ptr(), work.data_ptr(), _absmax_ptr(absmax, Y.device), ws.data_ptr(), ws.numel(),
              _stream(Y.device))
    _count(2)
    o = k * d
    return {"sums": work[:o].view(k, d), "counts": work[o:o + k], "stats": work[o + k:o + k + 3],
            "info": work[o + k + 3:o + k + 5]}


def nearest_to_centers(Y: torch.Tensor, centers: torch.Tensor) -> torch.Tensor:
    """Index of the first arg-min sample per centre (reference statistics.py:370-377)."""
    _need_cuda("Y", Y)
    _need_cuda("centers", centers, torch.float64)
    n, d, ld = _rows("Y", Y)
    k = centers.shape[0]
    lib = _lib.load()
    dev = Y.device
    centers = centers.contiguous()
    out = torch.empty(k, dtype=torch.int64, device=dev)
    ws = _ws(lib.dcg_nearest_workspace_bytes(n, d, k), dev)
    _call(Y.device, "dcg_nearest_to_centers", Y.data_ptr(), n, d, ld, _dtype_bytes(Y), centers.data_ptr(),
              k, out.data_ptr(), ws.data_ptr(), ws.numel(), _stream(Y.device))
    _count(2)
    return out


# ---- A11 --------------------------------------------------------------------------------------
def ticacov_sums(f: torch.Tensor, g: torch.Tensor, w: Optional[torch.Tensor] = None,
                 wl: Optional[torch.Tensor] = None) -> dict:
    """Weighted raw correlation sums of DeepTICA network outputs (B x d, float32).  ``g`` must
    have the shape of ``f``, and ``w`` / ``wl`` (if given) B elements on the same device."""
    # the kernel reads B rows of g and B weights: a shorter tensor would be read past its end
    if f.dim() != 2 or g.shape != f.shape:
        raise ValueError(f"f and g must be (B, d) of one shape, got {tuple(f.shape)} and {tuple(g.shape)}")
    B, d = f.shape
    for name, v in (("w", w), ("wl", wl)):
        if v is not None and (v.dim() != 1 or v.numel() != B or v.device != f.device):
            raise ValueError(f"{name} must be a ({B},) tensor on {f.device}, got {tuple(v.shape)} on {v.device}")
    _need_cuda("f", f, torch.float32)
    _need_cuda("g", g, torch.float32)
    f = f.contiguous()
    g = g.contiguous()
    lib = _lib.load()
    n_out = lib.dcg_ticacov_out_doubles(d)
    if n_out == 0:
        raise ValueError("1 <= d <= 32")
    out = torch.empty(n_out, dtype=torch.float64, device=f.device)
    if w is not None:
        w = w.to(torch.float32).contiguous()
    if wl is not None:
        wl = wl.to(torch.float32).contiguous()
    ws = _ws(lib.dcg_ticacov_workspace_bytes(B, d), f.device)
    _call(f.device, "dcg_ticacov_f32", f.data_ptr(), g.data_ptr(), _ptr(w), _ptr(wl), B, d,
              out.data_ptr(), ws.data_ptr(), ws.numel(), _stream(f.device))
    _count(2)
    o = 2 + d
    return {"flat": out, "sw": out[0], "swl": out[1], "swf": out[2:o],
            "sff": out[o:o + d * d].view(d, d), "sfg": out[o + d * d:o + 2 * d * d].view(d, d),
            "slf": out[o + 2 * d * d:o + 2 * d * d + d], "slg": out[o + 2 * d * d + d:]}


def ticaloss(sums: torch.Tensor, d: int, reg: float, n_eig: int = 0) -> dict:
    """DeepTICA eigen-loss and its gradient from the raw sums of ``ticacov_sums`` in one launch
    (see dcg.h).  Returns dict(loss, status, sw, swl, evals, mu, G0, Gt) of views into one buffer."""
    _need_cuda("sums", sums, torch.float64)
    lib = _lib.load()
    n_out = lib.dcg_ticaloss_out_doubles(d)
    if n_out == 0 or sums.numel() < lib.dcg_ticacov_out_doubles(d) or not sums.is_contiguous():
        raise ValueError("sums must be the contiguous output of ticacov_sums with 1 <= d <= 32")
    res = torch.empty(n_out, dtype=torch.float64, device=sums.device)
    _call(sums.device, "dcg_ticaloss_f64", sums.data_ptr(), d, float(reg), int(n_eig), res.data_ptr(), _stream(sums.device))
    _count(1)
    o = 4
    return {"loss": res[0], "status": res[1], "sw": res[2], "swl": res[3], "evals": res[o:o + d],
            "mu": res[o + d:o + 2 * d], "G0": res[o + 2 * d:o + 2 * d + d * d].view(d, d),
            "Gt": res[o + 2 * d + d * d:].view(d, d)}


def gather_standardize(X: torch.Tensor, idx: torch.Tensor, mean: torch.Tensor, rng: torch.Tensor,
                       offset: int = 0) -> torch.Tensor:
    """``(X[idx + offset] - mean) / range`` (a DeepTICA minibatch through ``norm_in``) in one pass.
    ``idx`` is an int64 CUDA tensor of row indices with ``0 <= idx + offset < X.shape[0]``."""
    _need_cuda("X", X, torch.float32)
    _need_cuda("idx", idx, torch.int64)
    _need_cuda("mean", mean, torch.float32)
    _need_cuda("range", rng, torch.float32)
    n, f, ld = _rows("X", X)
    idx = idx.contiguous()
    nb = idx.numel()
    Z = torch.empty((nb, f), dtype=torch.float32, device=X.device)
    if nb == 0:
        return Z
    _call(X.device, "dcg_gather_standardize_f32", X.data_ptr(), n, f, ld, idx.data_ptr(), nb, int(offset),
              mean.contiguous().data_ptr(), rng.contiguous().data_ptr(), Z.data_ptr(), _stream(X.device))
    _count(1)
    return Z


def gen_eig_small(H: torch.Tensor, G: torch.Tensor):
    """``H s = theta G s`` for a batch of b x b pencils (b <= 32, FP64, G SPD) in one launch:
    returns (theta (nb, b) descending, S (nb, b, b) with G-orthonormal eigenvector columns,
    status (nb,) -- 0 ok, 1 where G was not positive definite).  Nothing is synchronised."""
    _need_cuda("H", H, torch.float64)
    _need_cuda("G", G, torch.float64)
    if H.dim() != 3 or H.shape != G.shape or H.shape[-1] != H.shape[-2] or H.shape[-1] > 32:
        raise ValueError("H and G must be (batch, b, b) with b <= 32")
    nb, b = H.shape[0], H.shape[-1]
    H = H.contiguous()
    G = G.contiguous()
    theta = torch.empty((nb, b), dtype=torch.float64, device=H.device)
    S = torch.empty((nb, b, b), dtype=torch.float64, device=H.device)
    status = torch.empty(nb, dtype=torch.float64, device=H.device)
    _call(H.device, "dcg_gen_eig_small_f64", H.data_ptr(), G.data_ptr(), b, nb, theta.data_ptr(), S.data_ptr(),
              status.data_ptr(), _stream(H.device))
    _count(1)
    return theta, S, status


# ---- N4: free-energy surface (binned KDE) ---------------------------------------------------------
def fes_density(P: torch.Tensor, cols, bounds, num_bins: int, bandwidth: float, blocks: int = 1):
    """Binned Gaussian KDE of the projected frames on an equidistant grid, per block of frames
    (what mlcolvar's ``compute_fes(backend="KDEpy")`` evaluates, reference modules/figures/figures.py:95).

    ``P``: (n, d) float32 CUDA tensor; ``cols``: one or two column indices; ``bounds``: (lo, hi) or
    [(lo, hi), (lo, hi)].  Returns (density (blocks, G) or (blocks, G, G) [iy, ix] FP64, frames per block
    (blocks,) FP64, number of frames outside the bounds)."""
    _need_cuda("P", P, torch.float32)
    n, d, ld = _rows("P", P)
    cols = [int(c) for c in (cols if isinstance(cols, (list, tuple)) else [cols])]
    if len(cols) not in (1, 2) or any(not 0 <= c < d for c in cols):
        raise ValueError("cols must be one or two column indices of P")
    dim = len(cols)
    b = [tuple(map(float, bounds))] if dim == 1 else [tuple(map(float, x)) for x in bounds]
    G = int(num_bins)
    blocks = int(blocks)
    if not 1 <= blocks <= n:
        raise ValueError("1 <= blocks <= number of frames")
    dev = P.device
    shape = (blocks, G) if dim == 1 else (blocks, G, G)
    hist = torch.empty(shape, dtype=torch.float64, device=dev)
    outside = torch.empty(1, dtype=torch.int64, device=dev)
    (lo0, hi0), (lo1, hi1) = b[0], (b[1] if dim == 2 else (0.0, 1.0))
    _call(dev, "dcg_fes_bin_f32", P.data_ptr(), n, ld, cols[0], cols[1] if dim == 2 else -1, lo0, hi0, lo1, hi1,
          G, blocks, hist.data_ptr(), outside.data_ptr(), _stream(dev))
    q, r = divmod(n, blocks)
    frames = torch.tensor([q + 1] * r + [q] * (blocks - r), dtype=torch.float64, device=dev)
    dens = torch.empty_like(hist)
    tmp = torch.empty_like(hist) if dim == 2 else None
    _call(dev, "dcg_fes_smooth_f64", hist.data_ptr(), blocks, G, dim, (hi0 - lo0) / (G - 1),
          (hi1 - lo1) / (G - 1) if dim == 2 else 1.0, float(bandwidth), frames.data_ptr(), dens.data_ptr(),
          _ptr(tmp), _stream(dev))
    _count(2 if dim == 1 else 3)
    return dens, frames, outside


# ---- N1: clustering scores ------------------------------------------------------------------------
def cluster_dispersion(Y: torch.Tensor, labels: torch.Tensor, means: torch.Tensor):
    """Per-cluster ``sum ||y - m_c||^2`` and ``sum ||y - m_c||`` (FP64) in one pass over the frames:
    what Calinski-Harabasz and Davies-Bouldin need besides the counts and the means."""
    _need_cuda("Y", Y)
    _need_cuda("labels", labels, torch.int32)
    _need_cuda("means", means, torch.float64)
    n, d, ld = _rows("Y", Y)
    k = means.shape[0]
    if means.dim() != 2 or means.shape[1] != d or labels.numel() != n:
        raise ValueError("means must be (k, d) and labels must have one entry per frame")
    ssq = torch.empty(k, dtype=torch.float64, device=Y.device)
    sdist = torch.empty(k, dtype=torch.float64, device=Y.device)
    _call(Y.device, "dcg_cluster_dispersion", Y.data_ptr(), n, d, ld, _dtype_bytes(Y), labels.contiguous().data_ptr(),
          means.contiguous().data_ptr(), k, ssq.data_ptr(), sdist.data_ptr(), _stream(Y.device))
    _count(1)
    return ssq, sdist


# ---- N2: agglomerative clustering tree ------------------------------------------------------------------
def linkage(Y: torch.Tensor, method: str = "complete", return_phases: bool = False):
    """Merge tree of the frames ``Y`` (n x d CUDA tensor, float32 or float64) for ``method`` in
    ``single``, ``complete``, ``average``, ``ward``: the (n-1) x 4 FP64 matrix of
    ``scipy.cluster.hierarchy.linkage``, bitwise identical to scikit-learn's ``children_`` /
    ``distances_`` (see dcg.h).  float32 input is widened to float64 (exact, as sklearn does).
    The matrix linkages need 8 n^2 bytes of device memory; the free memory is checked before anything
    is allocated.  ``return_phases``: also return the tree kernel's (row scans, merges) counters."""
    _need_cuda("Y", Y)
    if method not in _lib.LINKAGE_METHODS:
        raise ValueError(f"linkage must be one of {sorted(_lib.LINKAGE_METHODS)}, got {method!r}")
    if Y.dtype not in (torch.float32, torch.float64):
        raise TypeError(f"Y must be float32 or float64, got {Y.dtype}")
    if Y.dim() != 2 or Y.shape[0] < 2 or Y.shape[1] < 1:
        raise ValueError("Y must be (frames x features) with at least 2 frames")
    Y = Y.to(torch.float64).contiguous()
    if not bool(torch.isfinite(Y).all()):
        raise ValueError("Input contains NaN or infinity")
    n, d = Y.shape
    code = _lib.LINKAGE_METHODS[method]
    lib = _lib.load()
    nbytes = int(lib.dcg_linkage_workspace_bytes(n, d, code))
    if nbytes == 0:
        raise ValueError(f"{n} frames are too many for the linkage tree")
    need = nbytes + 32 * (n - 1)
    free, _ = torch.cuda.mem_get_info(Y.device)
    if need > free:
        raise MemoryError(f"{method} linkage of {n} frames needs {need} bytes of device memory "
                          f"({'the 8 N^2-byte distance matrix and ' if code else ''}workspace); {free} bytes are free")
    dev = Y.device
    ws = _ws(nbytes, dev)
    Z = torch.empty((n - 1, 4), dtype=torch.float64, device=dev)
    _call(dev, "dcg_linkage_f64", Y.data_ptr(), n, d, d, code, Z.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev))
    _count(3 if code == 0 else 4)
    phases = ws[:16].view(torch.int64).clone()
    if int(phases[1].item()) != n - 1:
        raise RuntimeError(f"{method} linkage tree of {n} frames stopped after {int(phases[1].item())} merges")
    return (Z, phases) if return_phases else Z


# ---- N3: HDBSCAN core distances and mutual-reachability MST ---------------------------------------------
def _hdbscan_frames(Y: torch.Tensor) -> torch.Tensor:
    """The checks of ``linkage``: a CUDA (frames x features) tensor of at least 2 finite frames, returned
    as contiguous float64 (float32 is widened exactly, as scikit-learn does)."""
    _need_cuda("Y", Y)
    if Y.dtype not in (torch.float32, torch.float64):
        raise TypeError(f"Y must be float32 or float64, got {Y.dtype}")
    if Y.dim() != 2 or Y.shape[0] < 2 or Y.shape[1] < 1:
        raise ValueError("Y must be (frames x features) with at least 2 frames")
    Y = Y.to(torch.float64).contiguous()
    if not bool(torch.isfinite(Y).all()):
        raise ValueError("Input contains NaN or infinity")
    return Y


def _hdbscan_workspace(dev, n: int, d: int, min_samples: int, extra: int, what: str) -> int:
    """Workspace bytes of the HDBSCAN entry points, after checking that they and ``extra`` output bytes fit
    in the free device memory."""
    nbytes = int(_lib.load().dcg_hdbscan_workspace_bytes(n, d, min_samples))
    if nbytes == 0:
        raise ValueError(f"{n} frames are too many for HDBSCAN")
    free, _ = torch.cuda.mem_get_info(dev)
    if nbytes + extra > free:
        raise MemoryError(f"{what} of {n} frames needs {nbytes + extra} bytes of device memory; {free} bytes are free")
    return nbytes


def core_distances(Y: torch.Tensor, min_samples: int) -> torch.Tensor:
    """HDBSCAN core distances of the frames ``Y`` (n x d CUDA tensor, float32 or float64): the FP64
    distance of every frame to its ``min_samples``-th nearest frame, the frame itself counted at distance
    0.  Bitwise ``NearestNeighbors(n_neighbors=min_samples).kneighbors(X)[0][:, -1]`` (see dcg.h);
    1 <= min_samples <= min(n, 64)."""
    Y = _hdbscan_frames(Y)
    n, d = Y.shape
    min_samples = int(min_samples)
    if min_samples > n:
        # the wording of scikit-learn's kneighbors / HDBSCAN.fit check
        raise ValueError(f"Expected n_neighbors <= n_samples_fit, but n_neighbors = {min_samples}, "
                         f"n_samples_fit = {n}, n_samples = {n}")
    if not 1 <= min_samples <= _lib.HDBSCAN_MAX_MIN_SAMPLES:
        raise ValueError(f"min_samples must be in [1, {_lib.HDBSCAN_MAX_MIN_SAMPLES}], got {min_samples}")
    _hdbscan_workspace(Y.device, n, d, min_samples, 8 * n, "core distances")
    dev = Y.device
    core = torch.empty(n, dtype=torch.float64, device=dev)
    _call(dev, "dcg_core_distances_f64", Y.data_ptr(), n, d, d, min_samples, core.data_ptr(), None, 0, _stream(dev))
    _count(1)
    return core


def mreach_mst(Y: torch.Tensor, core: torch.Tensor) -> torch.Tensor:
    """Minimum spanning tree of the HDBSCAN mutual-reachability graph max(core_i, core_j, |y_i - y_j|):
    the (n-1) x 3 FP64 rows (source node, new node, distance) in Prim's visiting order from frame 0,
    bitwise sklearn's ``mst_from_data_matrix`` (sklearn/cluster/_hdbscan/_linkage.pyx; see dcg.h)."""
    Y = _hdbscan_frames(Y)
    n, d = Y.shape
    _need_cuda("core", core, torch.float64)
    if core.shape != (n,):
        raise ValueError(f"core must have shape ({n},), got {tuple(core.shape)}")
    core = core.contiguous()
    if not bool(torch.isfinite(core).all()):
        raise ValueError("core contains NaN or infinity")
    nbytes = _hdbscan_workspace(Y.device, n, d, 1, 24 * (n - 1), "the mutual-reachability MST")
    dev = Y.device
    ws = _ws(nbytes, dev)
    mst = torch.empty((n - 1, 3), dtype=torch.float64, device=dev)
    _call(dev, "dcg_mreach_mst_f64", Y.data_ptr(), n, d, d, core.data_ptr(), mst.data_ptr(), ws.data_ptr(),
          ws.numel(), _stream(dev))
    _count(1)
    steps = int(ws[:16].view(torch.int64)[1].item())
    if steps != n - 1:
        raise RuntimeError(f"mutual-reachability MST of {n} frames stopped after {steps} steps")
    return mst


# ---- N5: nearest clustered frame of supplementary frames -------------------------------------------------
NEAREST_QUERY_BLOCK = 128          # queries of one CTA of the search kernel (kQB, csrc/nearest.cu)


def _nearest_rows(name: str, Y: torch.Tensor) -> torch.Tensor:
    _need_cuda(name, Y)
    if Y.dtype not in (torch.float32, torch.float64):
        raise TypeError(f"{name} must be float32 or float64, got {Y.dtype}")
    if Y.dim() != 2 or Y.shape[1] < 1:
        raise ValueError(f"{name} must be (frames x features) with at least 1 feature")
    Y = Y.to(torch.float64).contiguous()
    if not bool(torch.isfinite(Y).all()):
        raise ValueError(f"{name} contains NaN or infinity")
    return Y


def nearest_frames(X: torch.Tensor, Q: torch.Tensor, return_counters: bool = False):
    """For every query frame of ``Q`` (m x d) its nearest frame of ``X`` (n x d): ``(index int64, dist float64)``.
    CUDA tensors, float32 (widened exactly) or float64, finite, n >= 1.  dist is the FP64 Euclidean distance
    with scikit-learn's KD-tree arithmetic, so it is bitwise ``NearestNeighbors(n_neighbors=1,
    algorithm="kd_tree").fit(X).kneighbors(Q)``'s; among frames at exactly the same distance the lowest index
    is returned (see dcg.h, N5).  ``return_counters``: also return (tiles visited, tiles considered)."""
    X = _nearest_rows("X", X)
    Q = _nearest_rows("Q", Q)
    if X.shape[0] < 1:
        raise ValueError("X must hold at least 1 frame")
    if Q.shape[1] != X.shape[1]:
        raise ValueError(f"X and Q must have the same number of features, got {X.shape[1]} and {Q.shape[1]}")
    if X.device != Q.device:
        raise ValueError(f"X and Q must be on the same device, got {X.device} and {Q.device}")
    n, d = X.shape
    m = Q.shape[0]
    dev = X.device
    if m == 0:
        index, dist = torch.empty(0, dtype=torch.int64, device=dev), torch.empty(0, dtype=torch.float64, device=dev)
        return (index, dist, (0, 0)) if return_counters else (index, dist)
    with torch.cuda.device(dev):
        nbytes = int(_lib.load().dcg_nearest_frames_workspace_bytes(n, m, d))
    if nbytes == 0:
        raise ValueError(f"nearest frames of {m} queries among {n} frames of {d} features: shape out of range")
    free, _ = torch.cuda.mem_get_info(dev)
    if nbytes + 16 * m > free:
        raise MemoryError(f"nearest frames of {m} queries among {n} frames needs {nbytes + 16 * m} bytes of device "
                          f"memory; {free} bytes are free")
    ws = _ws(nbytes, dev)
    index = torch.empty(m, dtype=torch.int64, device=dev)
    dist = torch.empty(m, dtype=torch.float64, device=dev)
    _call(dev, "dcg_nearest_frames_f64", X.data_ptr(), n, d, Q.data_ptr(), m, d, d, index.data_ptr(),
          dist.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev))
    _count(8)                      # box, keys, ordered copies, tile boxes, search; plus two radix sorts
    visited, considered = (int(v) for v in ws[:16].view(torch.int64).tolist())
    blocks = -(-m // NEAREST_QUERY_BLOCK)
    if not (blocks <= visited <= considered and considered % blocks == 0):
        raise ValueError(f"nearest-frame search visited {visited} of {considered} tiles for {blocks} query blocks")
    return (index, dist, (visited, considered)) if return_counters else (index, dist)


# ---- E1: F x F generalised eigenproblem (leading eigenpairs) ---------------------------------------
def tri_inv_blocks_(L: torch.Tensor, out: torch.Tensor, nblk: int, bs: int) -> torch.Tensor:
    """Inverses of the ``nblk`` diagonal blocks (``bs`` x ``bs``, at most 128) of the lower-triangular matrices
    ``L`` (nb, F, F; any strides) into the same blocks of ``out`` (nb, F, F); the rest of ``out`` is left alone."""
    _need_cuda("L", L, torch.float64)
    _need_cuda("out", out, torch.float64)
    if L.dim() != 3 or out.shape != L.shape or nblk * bs > L.shape[-1] or bs > 128:
        raise ValueError("L, out: (nb, F, F) with nblk * bs <= F and bs <= 128")
    _call(L.device, "dcg_tri_inv_blocks_f64", L.data_ptr(), out.data_ptr(), L.shape[0], nblk, bs,
          L.stride(1), L.stride(2), L.stride(0), out.stride(1), out.stride(2), out.stride(0), _stream(L.device))
    _count(1)
    return out
