"""Exact silhouette on the device (csrc/silhouette.cu, ops.silhouette) timed on seeded random-walk CVs.

    python tools_dev/silhouette_time.py [--sizes 100000,1000000] [--dims 2,4,10] [--out r7_silhouette_time.json]

For every N x d: the CVs are the seeded random walk of hier_time.py, labelled by the device KMeans for
k = 3..10 (8 labelings, 52 slots), in two row orders: the walk as it is (labels come in long runs) and the same
rows shuffled (labels change at almost every frame: the worst case of the run accumulation).  In the same call
and alternating, after a warm-up: one pass over the 8 labelings, 8 single-labeling passes, and, where it fits,
the torch.cdist routine statistics.silhouette used before the kernel (kept here as the baseline, not in the
product).  scikit-learn's silhouette_score runs on the host at the --sklearn-sizes for one labeling.  Times are
host clocks around calls that end in a device synchronise.  The GPU name and power limit are read in the same
run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deep_cartograph_b200 import ops  # noqa: E402
from deep_cartograph_b200.modules.statistics import statistics  # noqa: E402

KS = list(range(3, 11))
# FP64 instructions per pair and labeling pass: d subtracts, multiplies and adds, the fast path of __dsqrt_rn
# (MUFU.RSQ64H seed, then DMUL / DFMA refinement and rounding: 8 FP64 instructions in the SASS of silhouette.cu),
# and one add per labeling into its running sum (the label compares are integer work on the shared change mask)
SQRT_FP64_OPS = 8


def fp64_ops_per_pair(d, L):
    return 3 * d + SQRT_FP64_OPS + L


def random_walk(n, d, seed):
    rng = np.random.default_rng(seed)
    return np.ascontiguousarray(np.cumsum(0.05 * rng.standard_normal((n, d)), axis=0))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def cdist_silhouette(Y, lab, chunk=2048):
    """The routine statistics.silhouette used before the kernel: 2048-row blocks of torch.cdist, one labeling."""
    n = Y.shape[0]
    _, inv = torch.unique(lab, return_inverse=True)
    k = int(inv.max()) + 1
    onehot = torch.zeros((n, k), dtype=torch.float64, device=Y.device)
    onehot[torch.arange(n, device=Y.device), inv] = 1.0
    cnt = onehot.sum(dim=0)
    total = torch.zeros((), dtype=torch.float64, device=Y.device)
    for s0 in range(0, n, chunk):
        e0 = min(n, s0 + chunk)
        Dc = torch.cdist(Y[s0:e0], Y) @ onehot
        own = inv[s0:e0]
        rows = torch.arange(e0 - s0, device=Y.device)
        n_own = cnt[own]
        a = Dc[rows, own] / (n_own - 1).clamp(min=1.0)
        Dm = Dc / cnt[None, :]
        Dm[rows, own] = float("inf")
        b = Dm.min(dim=1).values
        sil = (b - a) / torch.maximum(a, b)
        sil = torch.where(n_own > 1, sil, torch.zeros_like(sil))
        total += torch.nan_to_num(sil).sum()
    return float((total / n).item())


def save(res, path):
    """Rewritten after every row, so a run cut short keeps what it measured."""
    os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
    with open(path, "w") as fh:
        json.dump(res, fh, indent=1)


def stats(v):
    v = np.asarray(v, dtype=np.float64)
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="100000,1000000")
    ap.add_argument("--dims", default="2,4,10")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--cdist-max", type=int, default=1000000, help="largest N for the torch.cdist baseline")
    ap.add_argument("--sklearn-sizes", default="20000,50000")
    ap.add_argument("--out", default="r7_silhouette_time.json")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "silhouette_time.py measures on the GPU; there is no CPU path"
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "inputs": "random walk, step 0.05 N(0,1) per CV, seed 3; KMeans labels k = 3..10 "
           "(n_init 1)", "fp64_ops_per_pair": "3 d + %d (sqrt) + L" % SQRT_FP64_OPS, "runs": [], "sklearn": []}
    print(json.dumps(res["gpu"]), flush=True)
    Yw = torch.from_numpy(random_walk(5000, 2, 1)).to(dev)                # warm-up: modules, attributes
    lw = [torch.from_numpy(statistics.kmeans_clustering(Yw.cpu().numpy(), k, 1)[0]).to(dev) for k in KS]
    ops.silhouette(Yw, lw)
    for lab in lw:
        ops.silhouette(Yw, lab)
    cdist_silhouette(Yw, lw[0])
    for n in [int(x) for x in a.sizes.split(",")]:
        for d in [int(x) for x in a.dims.split(",")]:
            X = random_walk(n, d, 3)
            labs = np.stack([statistics.kmeans_clustering(X, k, 1)[0] for k in KS]).astype(np.int64)
            perm = np.random.default_rng(0).permutation(n)
            for order in ("walk", "shuffled"):
                Xo, lo = (X, labs) if order == "walk" else (X[perm], labs[:, perm])
                Y = torch.from_numpy(np.ascontiguousarray(Xo)).to(dev)
                lt = [torch.from_numpy(np.ascontiguousarray(l)).to(dev) for l in lo]
                run_cdist = n <= a.cdist_max
                one, eight, old = [], [], []
                s_one = s_eight = s_old = None
                for r in range(a.repeats):
                    t, s_one = timed(lambda: ops.silhouette(Y, lt))
                    one.append(t)
                    t, s_eight = timed(lambda: torch.cat([ops.silhouette(Y, l) for l in lt]))
                    eight.append(t)
                    if run_cdist and (r == 0 or n <= 200000):
                        t, s_old = timed(lambda: [cdist_silhouette(Y, l) for l in lt])
                        old.append(t)
                pairs = float(n) * n
                row = {"n": n, "d": d, "order": order, "labelings": len(KS), "slots": sum(KS),
                       "one_pass_s": stats(one), "eight_passes_s": stats(eight),
                       "eight_over_one": float(np.median(eight) / np.median(one)),
                       "pairs_per_s_one_pass": pairs / float(np.median(one)),
                       "fp64_ops_per_s_one_pass": pairs * fp64_ops_per_pair(d, len(KS)) / float(np.median(one)),
                       "fp64_ops_per_s_single_passes": pairs * len(KS) * fp64_ops_per_pair(d, 1) / float(np.median(eight)),
                       "one_pass_equals_single_passes_bitwise": bool(torch.equal(s_one, s_eight)),
                       "scores": s_one.tolist()}
                if old:
                    row["cdist_baseline_s"] = stats(old)
                    row["cdist_over_one_pass"] = float(np.median(old) / np.median(one))
                    row["cdist_max_abs_diff"] = float(np.abs(np.asarray(s_old) - s_one.cpu().numpy()).max())
                else:
                    row["cdist_baseline_s"] = "not run at this N"
                res["runs"].append(row)
                print(json.dumps(row), flush=True)
                save(res, a.out)
                del Y, lt
                torch.cuda.empty_cache()
    from sklearn.metrics import silhouette_score
    for n in [int(x) for x in a.sklearn_sizes.split(",") if x]:
        X = random_walk(n, 2, 3)
        lab = statistics.kmeans_clustering(X, 5, 1)[0]
        t0 = time.perf_counter()
        ref = silhouette_score(X, lab)
        t_host = time.perf_counter() - t0
        Y = torch.from_numpy(X).to(dev)
        t_dev, got = timed(lambda: ops.silhouette(Y, torch.from_numpy(lab).to(dev)))
        row = {"n": n, "d": 2, "k": 5, "sklearn_host_s": t_host, "device_one_labeling_s": t_dev,
               "abs_diff_of_means": abs(float(got[0]) - ref)}
        res["sklearn"].append(row)
        print(json.dumps(row), flush=True)
    save(res, a.out)


if __name__ == "__main__":
    main()
