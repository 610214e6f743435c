"""Small F x F eigen stage, FP64 on one device (torch.linalg -> cuSOLVER).

Takes the raw FP64 sums produced by ``ops.lagged_covariance`` and reproduces the
post-processing of mlcolvar's ``TICA.compute`` / ``cholesky_eigh`` and sklearn's PCA as the
reference calls them (cv_calculator.py:2194-2215, 2249-2267, 2311-2384).  SURVEY appendix A.1/A.2.
"""
from __future__ import annotations

import math
import os
from typing import List, Tuple

import torch


_START_BLOCKS = {}


def _start_block(F: int, b: int, device) -> torch.Tensor:
    """Deterministic F x b starting block (fixed seed, generated once per shape and device)."""
    key = (F, b, str(device))
    if key not in _START_BLOCKS:
        g = torch.Generator(device="cpu").manual_seed(12345)
        _START_BLOCKS[key] = torch.randn((F, b), generator=g, dtype=torch.float64).to(device)
    return _START_BLOCKS[key]


# Counters of the partial eigensolver (tests and bench read them): solves answered by the
# shift-and-invert path, solves that took the dense path, iterations of the last fast solve.
EIG_STATS = {"fast": 0, "dense": 0, "last_iters": 0}

# Below this size the dense path is as fast as the iteration.
_PARTIAL_MIN_F = 192


def _tri_inv_lower(L: torch.Tensor) -> torch.Tensor:
    """Inverse of a batch of lower-triangular matrices (nb, F, F), FP64.

    cuBLAS ``trsm`` with F right-hand sides is a panel-serial algorithm whose time is linear in F at these
    sizes (0.54 ms at F = 1000, 0.064 ms at F = 125, measured: ``tools_dev/tri_time.py``), but it batches for
    free.  So the diagonal is cut into 8 blocks that are inverted as ONE batched call, and the inverse is
    assembled bottom-up from  [[A, 0], [B, C]]^-1 = [[A^-1, 0], [-C^-1 B A^-1, C^-1]]  with batched products
    (three levels): 0.2 ms at F = 1000.  Sizes that are not a multiple of the block count are padded with an
    identity block."""
    nb, F = L.shape[0], L.shape[-1]
    if F < 256:
        eye = torch.eye(F, dtype=L.dtype, device=L.device)
        return torch.linalg.solve_triangular(L, eye.expand(nb, F, F), upper=False)
    nblk = 8 if F >= 512 else 4
    bs = -(-F // nblk)
    Fp = bs * nblk
    if Fp != F:
        Lp = torch.eye(Fp, dtype=L.dtype, device=L.device).repeat(nb, 1, 1)
        Lp[:, :F, :F] = L
    else:
        Lp = L
    # diagonal blocks as one batch
    D = Lp.view(nb, nblk, bs, nblk, bs).diagonal(dim1=1, dim2=3).permute(0, 3, 1, 2)         # (nb, nblk, bs, bs)
    out = torch.zeros_like(Lp)
    if Lp.is_cuda and bs <= 128:
        # one CTA per diagonal block, forward substitution (csrc/eig_dense.cu): cuBLAS' batched trsm loops over
        # the blocks, 56 us each
        from . import ops
        ops.tri_inv_blocks_(Lp, out, nblk, bs)
    else:
        eye = torch.eye(bs, dtype=L.dtype, device=L.device)
        Dinv = torch.linalg.solve_triangular(D.reshape(nb * nblk, bs, bs), eye.expand(nb * nblk, bs, bs), upper=False)
        out.view(nb, nblk, bs, nblk, bs).diagonal(dim1=1, dim2=3).copy_(Dinv.view(nb, nblk, bs, bs).permute(0, 2, 3, 1))
    s, npairs = bs, nblk // 2
    while npairs >= 1:
        # super-blocks of size 2s on the diagonal: their halves are inverted already
        O = out.view(nb, npairs, 2 * s, npairs, 2 * s).diagonal(dim1=1, dim2=3).permute(0, 3, 1, 2)   # views
        S = Lp.view(nb, npairs, 2 * s, npairs, 2 * s).diagonal(dim1=1, dim2=3).permute(0, 3, 1, 2)
        lower = -(O[..., s:, s:] @ (S[..., s:, :s] @ O[..., :s, :s]))
        O[..., s:, :s] = lower
        s, npairs = 2 * s, npairs // 2
    return out[:, :F, :F] if Fp != F else out


def _shift_invert_topk(B: torch.Tensor, Ct: torch.Tensor, out: int, tol: float = 1e-12,
                       max_rounds: int = 10):
    """The `out` largest eigenpairs of Ct v = lambda B v (B SPD) by shift-and-invert subspace
    iteration with Rayleigh-Ritz, FP64.  ``B`` / ``Ct`` are (F, F) or a batch (nb, F, F) of
    independent pencils (hTICA level 1: all blocks in one set of launches).

    K = sigma B - Ct is SPD for sigma > lambda_max (TICA eigenvalues are autocorrelations, <= 1 up
    to estimator noise).  X <- K^-1 B X converges to the eigenvalues closest to sigma at the rate
    (sigma - lambda_out) / (sigma - lambda_{b+1}) per step, whatever the width of the noise bulk.
    K^-1 is applied as two GEMMs with the explicitly inverted Cholesky factor plus one step of
    iterative refinement (cuBLAS triangular solves with a dozen right-hand sides are launch-latency
    bound: 0.9 ms per application at F = 1000, against 20 us per skinny GEMM), so a solve is a
    handful of F x F x b GEMMs instead of the dense route's tridiagonalisation (12 ms at F = 1000).
    Ritz pairs are accepted only when ||Ct x - theta B x|| <= tol ||Ct||_F ||x|| for all `out` of
    them (in every pencil of the batch); returns None otherwise (flat spectrum, shift not found)
    and the caller goes dense."""
    batched = B.dim() == 3
    if not batched:
        B, Ct = B.unsqueeze(0), Ct.unsqueeze(0)
    nb, F = B.shape[0], B.shape[-1]
    b = min(F, out + 8)

    # round 0 (factorisation at sigma = 1.05, 12 steps, Rayleigh-Ritz, residuals) is a fixed sequence of ~150
    # small launches with no host read inside: on the GPU it is replayed as ONE CUDA graph (the stage is
    # host-launch-bound otherwise: 2.4 ms of wall time for ~1.5 ms of GPU time at F = 1000)
    st = _first_round(B, Ct, out, b)
    B, Ct = st["B"], st["Ct"]
    fac, X, theta, sigma, nrm = st["fac"], st["X"], st["theta"], st["sigma"], st["nrm"]
    hostvec = st["host"]
    it = _ROUND0_STEPS
    reshifted = False
    for rnd in range(max_rounds):
        if rnd > 0:
            X, theta, hostvec = _round_on_device(B, Ct, nrm, fac, X, sigma, None, out, 4, False)
            it += 4
        # one host read per round: worst residual + the Ritz values the shift logic needs
        host = hostvec.tolist()
        if host[-1] != 0:
            # sigma = 1.05 was not above the spectrum: checked factorisations with larger shifts, start over
            if rnd > 0:
                return None
            fac = None
            for _ in range(2):
                sigma = sigma * 2.0
                fac = _factor(B, Ct, sigma, check=True)
                if fac is not None:
                    break
            if fac is None:
                return None
            X = _start_block(F, b, B.device).expand(nb, F, b)
            X, theta, hostvec = _round_on_device(B, Ct, nrm, fac, X, sigma, None, out, _ROUND0_STEPS, True)
            host = hostvec.tolist()
            if host[-1] != 0:
                return None
            reshifted = True                   # no second re-shift on this path
        if host[-2] != 0 or host[0] != host[0]:
            return None
        worst = host[0]
        if worst <= tol:
            EIG_STATS["fast"] += nb
            EIG_STATS["last_iters"] = it
            ev, V = theta[:, :out].clone(), X[..., :out].clone()
            return (ev, V) if batched else (ev[0], V[0])
        if not reshifted:
            reshifted = True
            th0, tho, thb, sig = (host[1 + i * nb:1 + (i + 1) * nb] for i in range(4))

            def worst_rate(sg):
                return max((sg[i] - tho[i]) / max(sg[i] - thb[i], 1e-300) for i in range(nb))
            # predicted rate with the current shift; if it is slow, move every shift close to its
            # top Ritz value (which approaches lambda_max from below) and refactorise once
            if worst_rate(sig) > 0.25:
                for mult in (0.05, 0.2, 0.8):
                    s2 = [min(sig[i], th0[i] + mult * max(th0[i] - thb[i], 1e-12) + 1e-9 * max(1.0, abs(th0[i])))
                          for i in range(nb)]
                    s2t = torch.tensor(s2, dtype=B.dtype, device=B.device).reshape(nb, 1, 1)
                    f2 = _factor(B, Ct, s2t, check=True)
                    if f2 is not None:
                        fac, sig, sigma = f2, s2, s2t
                        break
            # flat spectrum below the wanted eigenvalues: more steps than the dense route costs
            rate = worst_rate(sig)
            if rate >= 1.0 or math.log(tol) / math.log(max(rate, 1e-300)) > 4 * max_rounds:
                return None
    return None


def _factor(B, Ct, sig, check=True):
    """sig: (nb, 1, 1).  Returns (K, K^-1, K^-1 B, info) or None if any K is not positive definite.
    ``check=False`` skips the host read of the factorisation status (the caller reads ``info`` later,
    together with the residuals: a failed factor shows there before any result is accepted)."""
    Kmat = sig * B - Ct
    Lk, info = torch.linalg.cholesky_ex(Kmat)
    if check and int(info.abs().max().item()) != 0:
        return None
    Li = _tri_inv_lower(Lk)
    Kinv = Li.mT @ Li                           # two F^3 products (70 us each at F = 1000) buy 1 instead of 6
    return Kmat, Kinv, Kinv @ B, info           # skinny products per cheap step, 4 per accurate one


def _round_on_device(B, Ct, nrm, fac, X, sigma, pending_info, out, n_steps, first):
    """``n_steps`` iterations X <- K^-1 B X, then Rayleigh-Ritz in span(X) and the residuals of the leading
    ``out`` Ritz pairs -- all on the device, no host read.  ``first``: the first _ROUND0_CHEAP steps use the explicitly
    formed K^-1 B (one skinny product; its rounding, eps cond(K), perturbs the operator of these steps only --
    the accurate steps that follow converge to the eigenvectors of the true pencil) and the block is
    re-orthogonalised after steps 4 and 8 (Cholesky QR: the noise directions shrink by (sigma - lambda_max) /
    sigma per step, so 8 plain steps would leave it numerically rank deficient).  Accurate step:
    K^-1 (B X) plus one step of iterative refinement against K itself.  Columns are rescaled every other step.
    Returns (X, theta, hostvec) with hostvec = [worst relative residual | theta_0 | theta_out-1 | theta_b-1 |
    sigma | pencil status | factorisation status]."""
    Kmat, Kinv, KinvB = fac[0], fac[1], fac[2]
    nb, b = X.shape[0], X.shape[-1]
    for i in range(n_steps):
        if first and i < _ROUND0_CHEAP:
            X = KinvB @ X
        else:
            Z = B @ X
            Y = Kinv @ Z
            X = torch.baddbmm(Y, Kinv, torch.baddbmm(Z, Kmat, Y, alpha=-1.0))
        if i & 1:
            X = X / torch.linalg.norm(X, dim=-2, keepdim=True)
        if first and i in (3, 7):
            G = X.mT @ X
            Lg, _ = torch.linalg.cholesky_ex(0.5 * (G + G.mT))
            X = torch.linalg.solve_triangular(Lg.mT, X, upper=True, left=False)      # X <- X Lg^-T
    # Rayleigh-Ritz in span(X):  (X^T Ct X) s = theta (X^T B X) s
    BX = B @ X
    CX = Ct @ X
    Gb = X.mT @ BX
    if X.is_cuda and b <= 32:
        # the b x b pencil in one launch (Cholesky + Jacobi), its status rides on the round's host read
        from . import ops
        theta, S, bad = ops.gen_eig_small(X.mT @ CX, Gb)
    else:
        eye_b = torch.eye(b, dtype=B.dtype, device=B.device)
        Lb, info_b = torch.linalg.cholesky_ex(0.5 * (Gb + Gb.mT))
        Lbi = torch.linalg.solve_triangular(Lb, eye_b.expand(nb, b, b), upper=False)
        Hs = Lbi @ (X.mT @ CX) @ Lbi.mT
        theta, S = torch.linalg.eigh(0.5 * (Hs + Hs.mT))
        theta = theta.flip(-1)
        S = Lbi.mT @ S.flip(-1)
        bad = info_b.abs().to(B.dtype).reshape(nb)
    X = X @ S
    res = torch.linalg.norm(CX @ S[..., :out] - (BX @ S[..., :out]) * theta[:, None, :out], dim=-2)
    rel = res / (nrm * torch.linalg.norm(X[..., :out], dim=-2))
    pend = (pending_info.abs().max().to(B.dtype).reshape(1) if pending_info is not None
            else torch.zeros(1, dtype=B.dtype, device=B.device))
    hostvec = torch.cat([rel.max().reshape(1), theta[:, 0], theta[:, out - 1], theta[:, b - 1],
                         sigma.reshape(-1), bad.max().reshape(1), pend])
    return X, theta, hostvec


def _first_round_eager(B, Ct, out, b):
    nb, F = B.shape[0], B.shape[-1]
    nrm = torch.linalg.matrix_norm(Ct).unsqueeze(-1)         # (nb, 1) Frobenius norms, residual scale
    sigma = torch.full((nb, 1, 1), 1.05, dtype=B.dtype, device=B.device)
    # the first factorisation is used unchecked: its status rides on the round's host read
    fac = _factor(B, Ct, sigma, check=False)
    X0 = _start_block(F, b, B.device).expand(nb, F, b)
    X, theta, hostvec = _round_on_device(B, Ct, nrm, fac, X0, sigma, fac[3], out, _ROUND0_STEPS, True)
    return {"B": B, "Ct": Ct, "fac": fac, "X": X, "theta": theta, "sigma": sigma, "nrm": nrm, "host": hostvec}


_ROUND0_GRAPHS = {}
_ROUND0_GRAPHS_MAX = 8
# Steps before the first Rayleigh-Ritz.  The explicitly formed K^-1 B carries a relative error ~ eps cond(K)
# (1e-8 at C2), i.e. its eigenvectors are ~1e-5 off (gaps 2e-3): 4 cheap steps reach that floor (rate 0.06 per
# step), more are wasted; each accurate step then gains a factor ~0.06, and the 1e-12 acceptance needs 7 of them
# (measured at C2: 8 cheap + 5 accurate end at 1e-11, one round too many).
_ROUND0_CHEAP = 4
_ROUND0_STEPS = 11


def _first_round(B, Ct, out, b):
    """Round 0 of the shift-and-invert iteration; on CUDA a cached CUDA graph per (batch, F, out, device) whose
    inputs are copied into static buffers (``DCG_EIG_GRAPH=0`` or a failed capture: eager).  The returned
    tensors belong to the graph and are valid until its next replay (the caller clones what it returns)."""
    if (not B.is_cuda or os.environ.get("DCG_EIG_GRAPH", "1") == "0" or torch.cuda.is_current_stream_capturing()):
        return _first_round_eager(B, Ct, out, b)
    key = (B.shape[0], B.shape[-1], out, b, B.device.index, B.dtype)
    ent = _ROUND0_GRAPHS.get(key)
    if ent is None:
        while len(_ROUND0_GRAPHS) >= _ROUND0_GRAPHS_MAX:          # each graph keeps ~15 F x F buffers alive
            _ROUND0_GRAPHS.pop(next(iter(_ROUND0_GRAPHS)))
        ent = {"failed": False}
        _ROUND0_GRAPHS[key] = ent
        try:
            Bs, Cs = B.clone().contiguous(), Ct.clone().contiguous()
            side = torch.cuda.Stream(device=B.device)
            side.wait_stream(torch.cuda.current_stream(B.device))
            with torch.cuda.stream(side):
                for _ in range(2):                         # library handles / workspaces before the capture
                    _first_round_eager(Bs, Cs, out, b)
            torch.cuda.current_stream(B.device).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                outs = _first_round_eager(Bs, Cs, out, b)
            ent.update(graph=graph, B=Bs, Ct=Cs, outs=outs)
        except Exception:                                  # capture not possible here: stay eager
            ent["failed"] = True
            torch.cuda.synchronize(B.device)
    if ent["failed"]:
        return _first_round_eager(B, Ct, out, b)
    ent["B"].copy_(B)
    ent["Ct"].copy_(Ct)
    ent["graph"].replay()
    return ent["outs"]


def _cholesky_eigh(C0: torch.Tensor, Ct: torch.Tensor, reg: float, out: int):
    """B = C0 + reg I; L = chol(B); A = L^-1 Ct L^-T; eigh; descending; V = L^-T U;
    unit-L2 columns; sign(row 0) >= 0; first ``out`` (mlcolvar cholesky_eigh + TICA).
    Inputs are (F, F) or a batch (nb, F, F).

    Only the leading ``out`` eigenpairs are needed, so for F >= 192 they come from the
    shift-and-invert iteration above (same generalised eigenvectors: L^-T u solves
    Ct v = lambda B v); the dense route is the fallback and the small-F path."""
    F = C0.shape[-1]
    B = C0 + reg * torch.eye(F, dtype=C0.dtype, device=C0.device)
    out = min(out, F)
    got = None
    if F >= _PARTIAL_MIN_F and 2 * (out + 8) < F:
        # accepted only with residual-checked Ritz pairs of (Ct, B), from Cholesky factorisations
        # of sigma B - Ct and X^T B X; a B that is not positive definite (or not finite) ends up
        # on the dense route below, whose Cholesky of B raises as the reference's does
        got = _shift_invert_topk(B, Ct, out)
    if got is None:
        L, info = torch.linalg.cholesky_ex(B)
        if int(info.abs().max().item()) != 0:
            raise RuntimeError("TICA: C0 + reg*I is not positive definite")
        EIG_STATS["dense"] += 1 if C0.dim() == 2 else C0.shape[0]
        Y = torch.linalg.solve_triangular(L, Ct, upper=False)             # L^-1 Ct
        A = torch.linalg.solve_triangular(L, Y.mT, upper=False).mT        # (L^-1 (L^-1 Ct)^T)^T
        evals, U = torch.linalg.eigh(0.5 * (A + A.mT))
        V = torch.linalg.solve_triangular(L.mT, U.flip(-1)[..., :out], upper=True)    # L^-T U
        got = evals.flip(-1)[..., :out], V
    evals, V = got
    V = V / torch.linalg.norm(V, dim=-2, keepdim=True)
    V = V * torch.sign(V[..., 0:1, :])
    return evals, V


def tica_from_sums(S0, St, a, b, M: int, out: int, reg: float = 1e-6):
    """TICA eigenpairs from raw sums.  ``S0`` must be fully symmetric.  mu = a/M is subtracted
    from BOTH series, covariances are divided by M, C_tau is symmetrised.  Inputs may carry a
    leading batch dimension (independent problems of equal size)."""
    mu = a / M
    nu = b / M
    C0 = S0 / M - mu.unsqueeze(-1) * mu.unsqueeze(-2)
    C0 = 0.5 * (C0 + C0.mT)
    Ct = St / M - mu.unsqueeze(-1) * nu.unsqueeze(-2)
    Ct = 0.5 * (Ct + Ct.mT)
    return _cholesky_eigh(C0, Ct, reg, out)


def restandardize_sums(s: dict, m0: torch.Tensor, r0: torch.Tensor, mean: torch.Tensor,
                       rng: torch.Tensor) -> dict:
    """Raw sums of z' = (x - m0) / r0  ->  raw sums of z = (x - mean) / rng, exactly (FP64):
    z = alpha z' + beta per feature with alpha = r0 / rng, beta = (m0 - mean) / rng, so
        S0 = A S0' A + (A a') beta^T + beta (A a')^T + M beta beta^T
        St = A St' A + (A a') beta^T + beta (A b')^T + M beta beta^T
        a  = A a' + M beta,   b = A b' + M beta                      (A = diag(alpha)).
    Used when the sums were accumulated under provisional standardisation parameters while the
    matrix was still arriving on the device.  ``S0`` must be fully symmetric."""
    al = r0.to(torch.float64) / rng.to(torch.float64)
    be = (m0.to(torch.float64) - mean.to(torch.float64)) / rng.to(torch.float64)
    M = float(s["M"])
    Aa = al * s["a"]
    Ab = al * s["b"]
    out = dict(s)
    bb = M * torch.outer(be, be)
    if s.get("S0") is not None:
        x = torch.outer(Aa, be)
        out["S0"] = al[:, None] * s["S0"] * al[None, :] + x + x.T + bb
    if s.get("St") is not None:
        out["St"] = al[:, None] * s["St"] * al[None, :] + torch.outer(Aa, be) + torch.outer(be, Ab) + bb
    out["a"] = Aa + M * be
    out["b"] = Ab + M * be
    return out


def pca_from_sums(S_all, s_all, N: int, d: int):
    """sklearn covariance-eigh PCA + the reference's sign rule (cv_calculator.py:2204-2215)."""
    mu = s_all / N
    Cm = (S_all - N * torch.outer(mu, mu)) / (N - 1)
    Cm = 0.5 * (Cm + Cm.T)
    evals, V = torch.linalg.eigh(Cm)
    evals = evals.flip(0)[:d]
    W = V.flip(1)[:, :d].clone()
    neg = W[0, :] < 0
    W[:, neg] = -W[:, neg]
    return evals, W


def htica_chunks(F: int, num_subspaces: int) -> List[Tuple[int, int]]:
    """Column chunks exactly as torch.split(x, F // num_subspaces, dim=1) makes them
    (cv_calculator.py:2331-2334)."""
    w = F // num_subspaces
    if w == 0:
        return []
    return [(s, min(s + w, F)) for s in range(0, F, w)]


def htica_level1(S0, St, a, b, M: int, chunks, sub_dim: int, reg: float = 1e-6) -> torch.Tensor:
    """Per-block TICA (level 1); returns the block-diagonal transform T1 (F x S1).  Blocks of equal
    width (all but possibly the last, cv_calculator.py:2331-2334) are solved as ONE batch."""
    F = S0.shape[0]
    blocks = [None] * len(chunks)
    by_width = {}
    for i, (s, e) in enumerate(chunks):
        by_width.setdefault(e - s, []).append(i)
    for width, idxs in by_width.items():
        if len(idxs) == 1:
            s, e = chunks[idxs[0]]
            blocks[idxs[0]] = tica_from_sums(S0[s:e, s:e], St[s:e, s:e], a[s:e], b[s:e], M, sub_dim, reg)[1]
            continue
        sl = [chunks[i] for i in idxs]
        _, Vb = tica_from_sums(torch.stack([S0[s:e, s:e] for s, e in sl]), torch.stack([St[s:e, s:e] for s, e in sl]),
                               torch.stack([a[s:e] for s, e in sl]), torch.stack([b[s:e] for s, e in sl]),
                               M, sub_dim, reg)
        for j, i in enumerate(idxs):
            blocks[i] = Vb[j]
    S1 = sum(v.shape[1] for v in blocks)
    T1 = torch.zeros((F, S1), dtype=S0.dtype, device=S0.device)
    c = 0
    for (s, e), Vb in zip(chunks, blocks):
        T1[s:e, c:c + Vb.shape[1]] = Vb
        c += Vb.shape[1]
    return T1


def htica_from_full_sums(S0, St, a, b, M: int, num_subspaces: int, sub_dim: int, d: int,
                         reg: float = 1e-6):
    """hTICA from the FULL F x F sums (single data pass): level-2 sums are T1^T S T1
    (level-1 projections are uncentred; level 2 re-centres).  Returns (W, T1, V2)."""
    chunks = htica_chunks(S0.shape[0], num_subspaces)
    if not chunks:
        raise ValueError("num_subspaces larger than number of features")
    T1 = htica_level1(S0, St, a, b, M, chunks, sub_dim, reg)
    _, V2 = tica_from_sums(T1.T @ S0 @ T1, T1.T @ St @ T1, T1.T @ a, T1.T @ b, M, d, reg)
    return T1 @ V2, T1, V2
