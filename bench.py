#!/usr/bin/env python
"""Benchmark of the CV hot path (BASELINE.json metric: frames/s for C0/C_tau + projection + KMeans).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload = "C2"): synthetic 1M frames x 1,000 features per GPU, TICA lag 10,
dim 4, KMeans(k=100) with fixed initial centroids and a fixed number of Lloyd iterations in the
4-D CV space.  One "step" = one pass of the whole hot path over the resident matrix:
column statistics -> fused standardise + C0/C_tau -> F x F eigenproblem -> projection (+ CV
min/max, normalisation) -> KMeans.  N > 1: weak scaling, every rank owns a 1M-frame shard of one
N*1M-frame series (lag halo exchanged, partial sums all-reduced every step).

`value`   : frames/s with the matrix resident in HBM (device-timed, max over ranks).
`e2e`     : frames/s through the public calculator API (TICACalculator + kmeans_lloyd) from pinned
            HOST memory, H2D of the matrix and D2H of the results inside the timed region.
`roofline`: the covariance kernel (dominant), timed live with CUDA events on its stream.
`cpu_baseline` / `--impl reference`: the reference's CPU path (oracle/reference_path.py, "port")
            on a bounded sample, all host threads.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# DRAM bytes (read + written) per launch of the dominant kernel, keyed by (engine, frames, features): from the
# committed `ncu --set full` captures under profiles/ (dram__bytes_read.sum + dram__bytes_write.sum).  A shape
# without a capture reports null.
TRAFFIC = {("tc_3xf16", 1_000_000, 1000): 11.88e9, ("tc_3xtf32", 1_000_000, 1000): 9.95e9,
           ("tc_i8x3", 1_000_000, 1000): 5.112e9}

F = 1000
N_PER_GPU = 1_000_000
LAG = 10
DIM = 4
K = 100
KM_ITERS = 10
CPU_SAMPLE_FRAMES = N_PER_GPU          # the reference arm runs the FULL C2 matrix (4 GB: it fits host RAM, BASELINE.md 3.4)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--engine", default=os.environ.get("DCG_COV_ENGINE", "tc_i8x3"),
                    choices=["tc_i8x3", "tc_3xf16", "tc_3xtf32", "tc_1xtf32", "simt_f32"])
    ap.add_argument("--frames", type=int, default=N_PER_GPU, help="frames per GPU (default = C2)")
    ap.add_argument("--features", type=int, default=F)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-legs", action="store_true", help="skip the C3 (hTICA 4950 features) and C5 (KMeans k=1000) legs")
    ap.add_argument("--no-parity", action="store_true", help="skip the float64 parity block")
    ap.add_argument("--c3-frames", type=int, default=0, help="total frames of the C3 leg (default 10M, 1.25M at 1 GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed on rank 0 as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin=None, t_end=None):
        """Summary of the samples that arrived inside [t_begin, t_end] (host clock; the sampler is
        started before the warm-up so that nvidia-smi is already looping when the timed region
        begins -- its start-up alone is longer than a short timed region)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for t, r in self.rows if (t_begin is None or t >= t_begin) and (t_end is None or t <= t_end + 0.02)]
        for r in rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for nm, val in zip(names, parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# reference arm: the reference's CPU path on the host cores
# ----------------------------------------------------------------------------------------------
def host_sample(frames: int, features: int):
    """The first `frames` rows of the synthetic series, generated on the host."""
    import numpy as np
    import torch
    from deep_cartograph_b200.synthetic import feature_matrix
    return feature_matrix(max(frames, 1), features, 0, frames, torch.device("cpu")).numpy()


def time_reference(frames: int, features: int, steps: int, warmup: int):
    from oracle.reference_path import cpu_threads, run_reference_pipeline
    X0 = host_sample(frames, features)
    times = []
    last = None
    for i in range(warmup + steps):
        X = X0.copy()
        t0 = time.perf_counter()
        last = run_reference_pipeline(X, LAG, DIM, K, KM_ITERS)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    mean_s = sum(times) / len(times)
    return {"value": frames / mean_s, "unit": "frames/s", "cores": cpu_threads(), "kind": "port",
            "sample": f"{'the whole C2 matrix: ' if frames >= N_PER_GPU else 'first '}{frames} frames x {features} features "
                      f"of the C2 series, lag {LAG}, d {DIM}, KMeans k={K} x {KM_ITERS} Lloyd iterations from the same fixed "
                      f"centroids (scikit-learn KMeans as reference statistics.py:189-195 calls it, max_iter = {KM_ITERS}, "
                      "tol = 0 so both arms do the same work); stages(s)=" +
                      json.dumps({k: round(v, 4) for k, v in last["timings"].items()})}, mean_s


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1; the reference arm uses every host thread (set before
    # numpy / torch / sklearn are imported)
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    # each step is one pass of the reference's CPU path over the WHOLE C2 matrix (~25 s of host work): at
    # most 4 timed steps and one warm-up so the arm ends within a few minutes whatever --steps / --warmup
    # ask for (the JSON line says what ran)
    steps, warmup = max(1, min(args.steps, 4)), max(0, min(args.warmup, 1))
    cb, mean_s = time_reference(args.frames, args.features, steps, warmup)
    line = {"impl": "reference", "metric": "frames/s, TICA C0/Ctau + projection + KMeans (hot path)",
            "value": cb["value"], "unit": "frames/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": mean_s * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, args.gpus, "cpu"),
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit_json(line)


def workload_config(args, world, engine):
    return {"workload": "C2: synthetic 1M frames x 1,000 features per GPU, TICA lag 10, dim 4, "
                        f"KMeans k={K} x {KM_ITERS} Lloyd iterations (fixed init = first k projected frames)",
            "frames_per_gpu": args.frames, "features": args.features, "lag": LAG, "dim": DIM,
            "kmeans_k": K, "kmeans_iters": KM_ITERS, "cov_engine": engine,
            "parallelism": f"frame-sharded x{world}", "l2": "inputs (4 GB/GPU) larger than L2, no flush needed"}


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
def numa_local_policy(device_index: int):
    """Bind this process's future page allocations (and its CPU affinity, where the cpuset allows) to
    the NUMA node the GPU hangs off, so the pinned staging buffer of each rank is local to its GPU:
    with 8 ranks copying 4 GB each, buffers that all sit on one socket make half of the copies cross
    the inter-socket link.  Best effort (set_mempolicy may be filtered in a container); returns a note
    for the JSON line."""
    try:
        import ctypes
        import torch
        pr = torch.cuda.get_device_properties(device_index)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as fh:
            node = int(fh.read().strip())
        if node < 0:
            return "numa: single node"
        note = f"numa node {node}"
        try:
            with open(f"/sys/devices/system/node/node{node}/cpulist") as fh:
                cpus = set()
                for part in fh.read().strip().split(","):
                    a, _, b = part.partition("-")
                    cpus.update(range(int(a), int(b or a) + 1))
            allowed = os.sched_getaffinity(0) & cpus
            if allowed:
                os.sched_setaffinity(0, allowed)
                note += f", {len(allowed)} local cpus"
        except OSError:
            pass
        libc = ctypes.CDLL(None, use_errno=True)
        mask = (ctypes.c_ulong * 16)()
        mask[node // 64] = 1 << (node % 64)
        MPOL_PREFERRED, SYS_set_mempolicy = 1, 238          # x86_64
        rc = libc.syscall(SYS_set_mempolicy, MPOL_PREFERRED, mask, 16 * 64)
        note += ", mempolicy preferred" if rc == 0 else f", set_mempolicy errno {ctypes.get_errno()}"
        return note
    except Exception as e:  # noqa: BLE001
        return f"numa: unavailable ({type(e).__name__})"


_JSON_FD = None


def _quiet_stdout():
    """stdout carries exactly ONE JSON line: libraries that write to file descriptor 1 from native
    code (NCCL prints its version banner there) are sent to stderr; the JSON line goes to the
    original descriptor."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit_json(line) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


# ----------------------------------------------------------------------------------------------
# parity block and the sharded north_star legs (C3, C5)
# ----------------------------------------------------------------------------------------------
def parity_block(X, lag, d, engine):
    """float64 check of THIS run's kernels on this rank's resident shard (all rows): full S0 / S_tau,
    eigenvalues, eigenvectors (max column L2 distance up to sign) and normalised projections against
    oracle/float64_device.py.  The oracle is the checker here, never the thing timed."""
    import torch
    from deep_cartograph_b200 import linalg, ops
    from oracle import float64_device as f64
    n = X.shape[0]
    st = ops.column_stats(X)
    mean = st["mean"].float()
    rng = torch.sqrt(st["m2"] / (n - 1)).float()
    s = ops.lagged_covariance(X, lag, mean, rng, engine=engine, xmin=st["min"], xmax=st["max"])
    ref = f64.lagged_sums(X, lag, mean, rng)
    err = f64.sums_rel_error(s, ref)
    if engine == "tc_i8x3":
        err["St"] = err["St_sym"]          # the exact engine returns the symmetric part of St (all TICA uses)
    ev, V = linalg.tica_from_sums(ops.symmetrize_upper(s["S0"]), s["St"], s["a"], s["b"], s["M"], d)
    ev_ref, V_ref = f64.tica_from_sums(ref["S0"], ref["St"], ref["a"], ref["b"], ref["M"], d)
    P, pmin, pmax = ops.project(X, V.float(), mean, rng)
    ops.standardize_(P, (pmax + pmin) / 2, (pmax - pmin) / 2)
    Pn_ref, _, _ = f64.project_normalized(X, mean, rng, V_ref)
    sgn = torch.sign((V * V_ref).sum(0, keepdim=True))
    out = {"frames": n, "engine": engine, "cov_rel_err": max(err["S0"], err["St"]),
           "eval_rel_err": float(((ev - ev_ref).abs() / ev_ref.abs()).max()),
           "evec_err": f64.eigvec_error(V, V_ref),
           "proj_err": float((P.double() * sgn - Pn_ref).abs().max()),
           "tolerances": {"cov": 1e-5, "eval": 1e-5, "evec": 1e-5, "proj": 1e-4},
           "checker": "oracle/float64_device.py (torch float64 on the device, dense Cholesky route)"}
    out["ok"] = bool(out["cov_rel_err"] <= 1e-5 and out["eval_rel_err"] <= 1e-5 and out["evec_err"] <= 1e-5
                     and out["proj_err"] <= 1e-4)
    return out


def _log(msg):
    if int(os.environ.get("RANK", "0")) == 0:
        sys.stderr.write("[bench %7.1f s] %s\n" % (time.perf_counter() - _T0, msg))
        sys.stderr.flush()


_T0 = time.perf_counter()


def _max_over_ranks(ms, dev, shards):
    import torch
    import torch.distributed as dist
    t = torch.tensor(ms, dtype=torch.float64, device=dev)
    if shards is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


def run_c3_leg(args, dev, rank, world, shards, peaks, workdir):
    """north_star target configuration C3: 10M frames x 4950 features, hTICA (10 subspaces of 495 ->
    5 each -> d = 10, lag 10) + projection + KMeans(k = 1000, 5 Lloyd iterations), frames sharded over
    the GPUs (strong scaling: the TOTAL is fixed).  At 1 GPU the matrix (198 GB) does not fit: the leg
    then runs one GPU's share of the 8-GPU run (1.25M frames, 24.75 GB) and says so."""
    import torch
    from deep_cartograph_b200 import linalg, ops
    from deep_cartograph_b200.modules.cv_learning.cv_calculator import HTICACalculator
    from deep_cartograph_b200.modules.statistics import statistics
    from deep_cartograph_b200.synthetic import feature_matrix
    f, lag, d, k, iters = 4950, LAG, 10, 1000, 5
    total = args.c3_frames or (10_000_000 if world > 1 else 1_250_000)
    s0, s1 = (rank * total) // world, ((rank + 1) * total) // world
    n = s1 - s0
    ld = (f + 3) // 4 * 4
    buf = torch.empty((n + lag, ld), dtype=torch.float32, device=dev)
    for c0 in range(0, n, 1 << 16):                          # bounded temporaries
        c1 = min(n, c0 + (1 << 16))
        feature_matrix(total, f, s0 + c0, s0 + c1, dev, n_slow=14, out=buf[c0:c1, :f])
    X = buf[:n, :f]
    torch.cuda.synchronize()
    _log(f"C3 leg: shard of {n} x {f} generated")
    cfg = {"dimension": d, "lag_time": lag, "features_normalization": "mean_std", "num_subspaces": 10,
           "subspaces_dimension": 5, "backend": {"cov_engine": args.engine}}
    outdir = os.path.join(workdir, "c3")

    def ev():
        e = torch.cuda.Event(enable_timing=True); e.record(); return e

    def one():
        t = [ev()]
        calc = HTICACalculator(configuration=cfg, output_path=outdir)
        calc.load_training_tensor(X, shards=shards)                  # statistics (+ all-gather merge)
        t.append(ev())
        calc.create_output_folders()
        calc.compute_cv()                                            # level-1 block sums + eigen, block projection, level 2
        t.append(ev())
        calc.set_labels()
        Pn = calc.normalize_cv()                                     # projection + CV min/max (+ all-reduce)
        t.append(ev())
        init = Pn[:k].to(torch.float64).clone()
        if shards is not None:
            shards.broadcast_(init, 0)
        res = statistics.kmeans_lloyd(Pn, init, max_iter=iters, tol=0.0, shards=shards)
        t.append(ev())
        torch.cuda.synchronize()
        assert calc.cv is not None and res["n_iter"] == iters
        return [t[i].elapsed_time(t[i + 1]) for i in range(len(t) - 1)], calc

    one()                                                            # warm-up
    _log("C3 leg: warm-up step done")
    if shards is not None:
        torch.distributed.barrier()
    runs = []
    for _ in range(2):
        ms, calc = one()
        runs.append(_max_over_ranks(ms, dev, shards))
    ms = [min(r[i] for r in runs) for i in range(4)]
    tot = sum(ms)
    W = torch.as_tensor(calc.cv)
    hbm = peaks["hbm_gbs"]
    out = {"workload": f"C3: {total} frames x {f} features (row stride {ld}), hTICA 10 x 495 -> 50 -> {d}, lag {lag}, "
                       f"projection, KMeans k={k} x {iters} Lloyd iterations; frames sharded x{world}",
           "frames_total": total, "frames_per_gpu": n, "n_gpus": world, "scaling": "strong",
           "ms": {"stats": ms[0], "htica_sums_eigen": ms[1], "projection": ms[2], "kmeans": ms[3], "total": tot},
           "frames_per_s": total / (tot * 1e-3),
           "frac_hbm": {"stats": 4.0 * ld * n / (ms[0] * 1e-3) / 1e9 / hbm,
                        "projection": (4.0 * ld + 4.0 * d) * n / (ms[2] * 1e-3) / 1e9 / hbm},
           "weights_finite": bool(torch.isfinite(W).all()), "eig_stats": dict(linalg.EIG_STATS)}
    if world == 1 and total < 10_000_000:
        out["note"] = ("one GPU cannot hold C3 (198 GB): this is ONE GPU's share of the 8-GPU run, resident; the "
                       "8-GPU line's speed-up over it is (its frames_per_s) / (this frames_per_s)")
    del buf, X
    torch.cuda.empty_cache()
    return out


def run_c5_leg(args, dev, rank, world, shards, peaks):
    """C5: KMeans k = 1000 in a 10-D CV space, 12.5M float32 frames per GPU (100M at 8 GPUs, weak
    scaling), fixed initial centroids = the first 1000 frames, 5 sharded Lloyd iterations through
    statistics.kmeans_lloyd (one packed FP64 all-reduce per iteration)."""
    import torch
    from deep_cartograph_b200.modules.statistics import statistics
    from deep_cartograph_b200.synthetic import cluster_points
    n, d, k, iters = 12_500_000, 10, 1000, 5
    Y = cluster_points(n, d, k, dev, seed=2, dtype=torch.float32, start=rank * n)
    init = Y[:k].to(torch.float64).clone()
    if shards is not None:
        shards.broadcast_(init, 0)

    def one():
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        res = statistics.kmeans_lloyd(Y, init, max_iter=iters, tol=0.0, shards=shards)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), res

    one()
    if shards is not None:
        torch.distributed.barrier()
    runs = [one() for _ in range(3)]
    ms = min(_max_over_ranks([r[0]], dev, shards)[0] for r in runs)
    res = runs[-1][1]
    per_iter = ms / (iters + 1)                              # + the final E-step of the driver
    fp32_peak = 148 * 128 * 2 * (peaks.get("sm_max_mhz") or 1965.0) * 1e6 / 1e12
    out = {"workload": f"C5: KMeans k={k}, d={d}, {n} float32 frames per GPU x{world} (weak scaling), fixed init, "
                       f"{iters} Lloyd iterations + final E-step, setup (centring, variance) included",
           "frames_total": n * world, "n_gpus": world, "ms_total": ms, "ms_per_iteration": per_iter,
           "frame_iterations_per_s": n * world * (iters + 1) / (ms * 1e-3),
           "bound": "fp32 / tensor score GEMM + arg-min scan (k/2 = 500 FLOP/B, far above the HBM ridge)",
           "tflops_useful": 2.0 * k * d * n * (iters + 1) / (ms * 1e-3) / 1e12, "fp32_peak_nominal": fp32_peak,
           "ties": res["ties"], "n_iter": res["n_iter"]}
    out["frac_fp32"] = out["tflops_useful"] / fp32_peak
    del Y
    torch.cuda.empty_cache()
    return out


DUMP_ROWS = 1 << 21        # per-frame outputs of more frames are dumped as a fixed sample of this many rows
PER_FRAME = ("cv", "kmeans_labels")


def dump_outputs(path, outputs):
    """Write the outputs of one step as DIR/<name>.npy, in float64 where the step computes float64 and
    float32 otherwise (labels are exact in float32), for output-by-output comparisons of two builds on
    the same seeded inputs.  Beyond DUMP_ROWS frames the per-frame arrays keep the rows of one seeded
    sample, whose frame indices go to frame_index.npy; everything stays under 64 MB.  Two runs of one
    build agree to rounding, not bit for bit (the eigen stage is not bitwise reproducible; at C2 on a
    B200 the eigenvectors differ by ~3e-11, the float32 CVs by an ulp), so compare with a tolerance."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    n = outputs["cv"].shape[0]
    rows = None
    if n > DUMP_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
        np.save(os.path.join(path, "frame_index.npy"), rows.astype(np.float64))
    for name, t in outputs.items():
        a = t.detach().cpu().numpy()
        if rows is not None and name in PER_FRAME:
            a = a[rows]
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))


def main():
    args = parse_args()
    _quiet_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from deep_cartograph_b200 import linalg, ops
    from deep_cartograph_b200.modules.cv_learning.cv_calculator import TICACalculator
    from deep_cartograph_b200.modules.statistics import statistics
    from deep_cartograph_b200.parallel import FrameShards
    from deep_cartograph_b200.synthetic import feature_matrix

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    shards = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        shards = FrameShards()
    n, f = args.frames, args.features
    engine = args.engine
    peaks = measured_peaks()
    # the calculators of the e2e step and the C3 leg write their model files here, outside the tree
    workdir = tempfile.TemporaryDirectory(prefix="dcg_bench_")

    # ---- data: this rank's shard of one world*n-frame series, with room for the lag halo
    buf = torch.empty((n + LAG, f), dtype=torch.float32, device=dev)
    buf[:n] = feature_matrix(world * n, f, rank * n, (rank + 1) * n, dev)
    X = buf[:n]
    torch.cuda.synchronize()

    _log("C2 shard generated")
    cov_ev = []
    pass_ev = {k: [] for k in ("stats", "covariance", "eigen", "projection", "kmeans")}

    class _Timed:
        """CUDA-event bracket around one pass (on torch's current stream, where the kernels launch)."""
        def __init__(self, name, on):
            self.name, self.on = name, on
        def __enter__(self):
            if self.on:
                self.e0 = torch.cuda.Event(enable_timing=True); self.e1 = torch.cuda.Event(enable_timing=True)
                self.e0.record()
        def __exit__(self, *a):
            if self.on:
                self.e1.record()
                pass_ev[self.name].append((self.e0, self.e1))

    # |P| <= 1 after the CV min-max normalisation (+ rounding): bound for the fixed-point KMeans sums
    p_bound = torch.full((1,), 1.0 + 1e-3, dtype=torch.float64, device=dev)

    def step(record=False):
      with _Timed("stats", record):
        st = ops.column_stats(X)
        if shards is not None:
            st = shards.merge_stats(st, n_total=n * world)          # equal shards: no host read
        ntot = st["n"]
        mean = st["mean"].to(torch.float32)
        rng = torch.sqrt(st["m2"] / (ntot - 1)).to(torch.float32)
        rng = torch.where(rng.abs() < 1e-8, torch.ones_like(rng), rng)
      with _Timed("covariance", record):
        Xh = shards.with_halo(X, LAG) if shards is not None else X
        if record:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        s = ops.lagged_covariance(Xh, LAG, mean, rng, engine=engine, xmin=st["min"], xmax=st["max"])
        s.pop("clamped", None)
        if record:
            e1.record()
            cov_ev.append((e0, e1))
        if shards is not None:
            s = shards.allreduce_sums(s, m_total=n * world - LAG)
      with _Timed("eigen", record):
        evals, V = linalg.tica_from_sums(ops.symmetrize_upper(s["S0"]), s["St"], s["a"], s["b"], s["M"], DIM)
        W = V.to(torch.float32)
      with _Timed("projection", record):
        P, pmin, pmax = ops.project(X, W, mean, rng)
        if shards is not None:
            pmin, pmax = shards.allreduce_minmax(pmin, pmax)
        ops.standardize_(P, (pmax + pmin) / 2, (pmax - pmin) / 2)
      with _Timed("kmeans", record):
        # KMeans: fixed init = first K projected frames of rank 0, fixed number of Lloyd iterations
        C = P[:K].to(torch.float64).clone()
        if shards is not None:
            shards.broadcast_(C, 0)
        labels = torch.full((n,), -1, dtype=torch.int32, device=dev)
        work = ops.kmeans_work(K, DIM, dev)
        for _ in range(KM_ITERS):
            if shards is None:
                ops.kmeans_iterate_(P, C, labels, work, absmax=p_bound)   # one library call per Lloyd iteration
                continue
            r = ops.kmeans_step_packed_(P, C, labels, work, absmax=p_bound)      # [sums | counts | stats] in place
            shards.allreduce_sum_(r["packed"])
            ops.kmeans_update_(C, r["sums"], r["counts"], info=work[K * DIM + K + 3:K * DIM + K + 5])
      return {"eigenvalues": evals, "eigenvectors": V, "feature_mean": mean, "feature_scale": rng,
              "cv_min": pmin, "cv_max": pmax, "cv": P, "kmeans_centers": C, "kmeans_labels": labels}

    def sync_all():
        torch.cuda.synchronize()
        if shards is not None:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                    # before the warm-up: nvidia-smi needs ~0.2 s to start looping
    for _ in range(max(args.warmup, 3)):
        step()
    sync_all()
    launches0 = ops.KERNEL_LAUNCHES
    if engine == "tc_i8x3":
        ops.cov_i8_timing(True)            # CUDA events around the quantise and contraction kernels, on their stream
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    host_t0 = time.perf_counter()
    t0.record()
    for _ in range(args.steps):
        outputs = step(record=True)
    t1.record()
    sync_all()
    host_t1 = time.perf_counter()
    clocks = sampler.stop(host_t0, host_t1) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs)
    launches = ops.KERNEL_LAUNCHES - launches0
    i8t = None
    if engine == "tc_i8x3":
        i8t = ops.cov_i8_timing()
        ops.cov_i8_timing(False)
    ms = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device=dev)
    cov_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in cov_ev) / len(cov_ev)], dtype=torch.float64, device=dev)
    if shards is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(cov_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(ms.item()) / args.steps
    value = world * n / (ms_per_step * 1e-3)

    # ---- roofline of the dominant kernel (covariance contraction)
    M = n - LAG if world == 1 else n            # pairs per rank (last rank has n - lag)
    alg_flops = 3.0 * f * f * M                  # SURVEY 8d: 2F^2 (C_tau) + F^2 (upper C0) per pair
    cov_s = float(cov_ms.item()) * 1e-3          # the whole dcg_cov_lag* call (all its kernels)
    if engine == "tc_i8x3":
        # dominant kernel = cov_i8_kernel (tcgen05 kind::i8), timed alone with CUDA events on its stream.
        # peak: the MEASURED dense bf16 figure of MEASURED_PEAKS.json (the contract's tensor denominator;
        # sustained: the kernel is timed inside a long step).  kind::i8 issues at twice the kind::f16 rate
        # (measured: 64 clocks per 256 x 128 x 32 MMA pair-instruction), so the int8 peak derived from the
        # same measurement is 2x; both fractions are reported.
        k_ms = i8t["contract_ms"] / max(1, i8t["launches"])
        q_ms = i8t["quantize_ms"] / max(1, i8t["launches"])
        from deep_cartograph_b200 import _lib as _l
        nb = -(-f // 128)                       # 128-feature blocks; tiles pair two blocks that share a column block
        n_up = sum(((c + 1) - (0 if c & 1 else 1)) // 2 for c in range(nb)) + len(range(0, nb, 4))
        issued_ops = 2.0 * (2 * n_up) * 256 * 128 * 8 * M          # 2 Grams, 8 digit products, MAC = 2 ops
        achieved = alg_flops / (k_ms * 1e-3) / 1e12
        peak = peaks["bf16_tflops_sustained"]
        fused = q_ms < 0.05                     # the fused kernel quantises inside the contraction launch
        roofline = {"bound": "tensor",
                    "kernel": ("cov_i8_fused_kernel (quantiser warps -> L2-resident digit-plane ring -> TMA -> "
                               "tcgen05.mma.cta_group::2.kind::i8, one persistent launch)" if fused else
                               "cov_i8_kernel (tcgen05.mma.cta_group::2.kind::i8, TMA-staged digit planes)"),
                    "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                    "peak_source": f"{peaks['source']} dense bf16, sustained (MEASURED_PEAKS.json)",
                    "kernel_ms": k_ms, "share_of_step": k_ms / ms_per_step,
                    "algorithmic": "3*F^2 FLOP per frame pair (SURVEY 8d); the exact engine issues 8 int8 digit products "
                                   "on 2 x %d tiles of two 128 x 128 blocks of the upper triangle" % n_up,
                    "issued_int8_tops": issued_ops / (k_ms * 1e-3) / 1e12,
                    "int8_peak_derived_tops": 2.0 * peaks["bf16_tflops"],
                    "frac_issued_of_int8_peak_derived": issued_ops / (k_ms * 1e-3) / 1e12 / (2.0 * peaks["bf16_tflops"]),
                    "call_ms": cov_s * 1e3,
                    "traffic": TRAFFIC.get((engine, n, f)),
                    "traffic_note": "dram bytes read + written per launch of this kernel from the committed ncu --set full "
                                    "capture of this shape (profiles/); algorithmic bytes of the whole covariance pass = "
                                    "4*F*n = %.3g" % (4.0 * f * n)}
        if not fused:
            roofline["quantize_kernel"] = {"ms": q_ms, "alg_bytes": 10.0 * f * n, "gbs": 10.0 * f * n / (q_ms * 1e-3) / 1e9,
                                           "frac_hbm": 10.0 * f * n / (q_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                           "note": "4 bytes read + 6 bytes of digit planes written per value (HBM-bound)"}
    else:
        f16_kind = engine == "tc_3xf16"
        tf32_peak = peaks["bf16_tflops_sustained"] if f16_kind else peaks["bf16_tflops_sustained"] / 2.0
        burst_peak = peaks["bf16_tflops"] if f16_kind else peaks["bf16_tflops"] / 2.0
        achieved = alg_flops / cov_s / 1e12
        issued_mult = {"tc_3xf16": 3.0, "tc_3xtf32": 3.0, "tc_1xtf32": 1.0, "simt_f32": 1.0}[engine]
        roofline = {"bound": "tensor", "kernel": f"cov_lag ({engine})", "achieved": achieved, "peak": tf32_peak,
                    "unit": "TFLOP/s", "frac": achieved / tf32_peak, "traffic": TRAFFIC.get((engine, n, f)),
                    "traffic_note": "bytes/launch (ncu); algorithmic bytes/launch = 4*F*n = %.3g" % (4.0 * f * n),
                    "issued_tflops": achieved * issued_mult, "frac_issued": achieved * issued_mult / tf32_peak,
                    "kernel_ms": cov_s * 1e3, "share_of_step": cov_s * 1e3 / ms_per_step,
                    "peak_source": (f"{peaks['source']} bf16 sustained (kind::f16; kernel timed inside a long step)" if f16_kind else
                                    f"{peaks['source']} bf16 sustained / 2 (TF32 : bf16 = 1 : 2 on tcgen05)"),
                    "peak_burst": burst_peak, "frac_issued_of_burst": achieved * issued_mult / burst_peak,
                    "algorithmic": "3*F^2 FLOP per frame pair; issued = x3 for the split-precision engines"}

    # ---- per-pass device times and the HBM fractions of the memory-bound passes (SURVEY 8d bytes)
    def _avg_ms(name):
        ev = pass_ev[name]
        return sum(a.elapsed_time(b) for a, b in ev) / max(1, len(ev))
    hbm = peaks["hbm_gbs"]
    pm = {k: _avg_ms(k) for k in pass_ev}
    passes = {
        "stats": {"ms": pm["stats"], "alg_bytes": 4.0 * f * n, "bound": "hbm"},
        "covariance": {"ms": pm["covariance"], "bound": "tensor", "note": "kernel alone: roofline.kernel_ms"},
        "eigen": {"ms": pm["eigen"], "bound": "none (F x F FP64 eigenproblem, cuSOLVER)"},
        "projection": {"ms": pm["projection"], "alg_bytes": (4.0 * f + 4.0 * DIM) * n + 8.0 * DIM * n, "bound": "hbm",
                       "note": "4F read + 4d written per frame, + 8d for the in-place CV normalisation"},
        "kmeans": {"ms": pm["kmeans"], "alg_bytes": KM_ITERS * (4.0 * DIM + 4.0) * n, "iters": KM_ITERS},
    }
    for v in passes.values():
        if "alg_bytes" in v:
            v["gbs"] = v["alg_bytes"] / (v["ms"] * 1e-3) / 1e9
            v["frac_hbm"] = v["gbs"] / hbm
    # KMeans (SURVEY 8d): 2*k*d FLOP against 4*d + 4 bytes per frame and iteration; HBM-bound only
    # below the FP32 ridge (nominal FMA peak / measured HBM, ~11 FLOP/B, i.e. k <~ 24), FP32-FMA-bound
    # beyond it.  Report the roof that binds.
    fp32_peak = 148 * 128 * 2 * (peaks.get("sm_max_mhz") or 1965.0) * 1e6 / 1e12      # TFLOP/s, nominal
    km = passes["kmeans"]
    km["alg_flop"] = KM_ITERS * 2.0 * K * DIM * n
    km["tflops_fp32"] = km["alg_flop"] / (km["ms"] * 1e-3) / 1e12
    km["intensity_flop_per_byte"] = km["alg_flop"] / km["alg_bytes"]
    if km["intensity_flop_per_byte"] > fp32_peak * 1e3 / hbm:
        km["bound"] = "fp32 fma (k*d/(2d+2) FLOP/B above the ridge)"
        km["frac_fp32"] = km["tflops_fp32"] / fp32_peak
        km["fp32_peak_nominal"] = fp32_peak
    else:
        km["bound"] = "hbm (k small)"
    km["note"] = ("10 whole Lloyd iterations (memset + E-step + FP64/fixed-point sums + centre update per "
                  "iteration) on n x d projected frames: at this size (16 MB) the pass is launch- and "
                  "latency-bound, see profiles/ for the stand-alone E-step at C5 size")

    # ---- e2e through the public API with host buffers
    e2e = None
    host = None
    if not args.no_e2e:
        numa_note = numa_local_policy(local) if world > 1 else None
        host = torch.empty((n, f), dtype=torch.float32, pin_memory=True)
        host.copy_(X)
        cfg = {"dimension": DIM, "lag_time": LAG, "features_normalization": "mean_std",
               "backend": {"cov_engine": engine}}
        outdir = os.path.join(workdir.name, "e2e")

        def e2e_step():
            calc = TICACalculator(configuration=cfg, output_path=outdir)
            calc.load_training_tensor(host, shards=shards)          # H2D of the whole matrix
            calc.create_output_folders()
            calc.compute_cv()
            calc.set_labels()
            Pn = calc.normalize_cv()
            init = Pn[:K].to(torch.float64).clone()
            if shards is not None:
                shards.broadcast_(init, 0)
            res = statistics.kmeans_lloyd(Pn, init, max_iter=KM_ITERS, tol=0.0, shards=shards)
            lab = res["labels"].cpu()                                # D2H of the result
            cen = res["centers"].cpu()
            return lab, cen

        e2e_step()
        sync_all()
        tt = time.perf_counter()
        e2e_steps = args.steps
        for _ in range(e2e_steps):
            e2e_step()
        sync_all()
        el = torch.tensor([time.perf_counter() - tt], dtype=torch.float64, device=dev)
        if shards is not None:
            dist.all_reduce(el, op=dist.ReduceOp.MAX)
        e2e_s = float(el.item()) / e2e_steps
        e2e = {"value": world * n / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": world * n * f * 4,
               "d2h_bytes_per_step": world * n * 4 + K * DIM * 8, "ms_per_step": e2e_s * 1e3,
               "api": "TICACalculator.load_training_tensor/compute_cv/normalize_cv + statistics.kmeans_lloyd"}
        if numa_note:
            e2e["host_buffer"] = numa_note

    _log("C2 timed region + e2e done")
    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_block(X, LAG, DIM, engine)
        _log("parity block done")
    c3 = c5 = None
    if not args.no_legs:
        del buf, X
        torch.cuda.empty_cache()
        c5 = run_c5_leg(args, dev, rank, world, shards, peaks)
        _log("C5 leg done")
        c3 = run_c3_leg(args, dev, rank, world, shards, peaks, workdir.name)
        _log("C3 leg done")

    if rank == 0:
        cpu_baseline = None
        if world == 1 and not args.no_cpu_baseline:
            host = None
            cpu_baseline, _ = time_reference(n, f, 1, 0)                 # the whole matrix, one pass (~25 s)
        line = {"metric": "frames/s, TICA C0/Ctau + projection + KMeans (hot path)", "value": value,
                "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"tc_i8x3": "f32 inputs; 23-bit fixed point in three int8 digit planes, exact int32 tensor-core accumulation, f64 results",
                          "tc_3xf16": "f32 (f16x3 split-precision tensor contraction, f64 accumulation)",
                          "tc_3xtf32": "f32 (tf32x3 split-precision tensor contraction, f64 accumulation)"}.get(engine, "f32"),
                "data": "synthetic", "config": workload_config(args, world, engine),
                "roofline": roofline, "passes": passes, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": launches,
                "clocks": clocks, "eigenvalues": [float(v) for v in outputs["eigenvalues"].cpu().tolist()],
                "parity": parity, "c3": c3, "c5": c5}
        emit_json(line)
    workdir.cleanup()
    if shards is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
