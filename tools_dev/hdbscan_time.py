"""Device HDBSCAN (csrc/linkage.cu core_dist_kernel + prim_kernel) timed on seeded random-walk CVs.

    python tools_dev/hdbscan_time.py [--sizes 20000,50000,100000,200000] [--dims 2,10] [--min-samples 3,16]
                                     [--out hdbscan_time.json]

For every N x d x min_samples: three repeats after a warm-up at a small N.  Each repeat times, with CUDA
events, ops.core_distances and ops.mreach_mst, and in the same run torch.profiler gives the device time of
their kernels (core_dist_kernel, prim_kernel); the host finish (numpy argsort + union-find, then the
selection of tree_to_labels at min_cluster_size 5, eom) is timed with a host clock.  scikit-learn's HDBSCAN
runs on the same host and inputs at 20k, with a check that the labels are equal.  The GPU name and power
limit are read in the same run."""
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

KERNELS = {"core": "core_dist_kernel", "mst": "prim_kernel"}


def random_walk(n, d, seed):
    rng = np.random.default_rng(seed)
    return np.ascontiguousarray(np.cumsum(0.05 * rng.standard_normal((n, d)), axis=0))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def one_run(Y, ms):
    from torch.profiler import profile, ProfilerActivity
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ev[0].record()
        core = ops.core_distances(Y, ms)
        ev[1].record()
        mst = ops.mreach_mst(Y, core)
        ev[2].record()
        torch.cuda.synchronize()
    ker = {}
    for e in prof.events():
        for key, name in KERNELS.items():
            if name in e.name:
                ker[key] = ker.get(key, 0.0) + e.device_time / 1e3       # us -> ms
    mst = mst.cpu().numpy()
    t0 = time.perf_counter()
    tree = statistics.single_linkage_from_mst(mst)
    t1 = time.perf_counter()
    labels = statistics.hdbscan_labels(tree, 5)
    t2 = time.perf_counter()
    return labels, {"core_call": ev[0].elapsed_time(ev[1]), "mst_call": ev[1].elapsed_time(ev[2]),
                    "host_tree": (t1 - t0) * 1e3, "host_labels": (t2 - t1) * 1e3}, ker


def stats(v):
    v = np.asarray(v, dtype=np.float64)
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="20000,50000,100000,200000")
    ap.add_argument("--dims", default="2,10")
    ap.add_argument("--min-samples", default="3,16")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--sklearn-n", type=int, default=20000)
    ap.add_argument("--out", default="hdbscan_time.json")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "hdbscan_time.py measures on the GPU; there is no CPU path"
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "inputs": "random walk, step 0.05 N(0,1) per CV, seed 3",
           "labels": "min_cluster_size 5, eom, epsilon 0", "runs": []}
    print(json.dumps(res["gpu"]), flush=True)
    mss = [int(x) for x in a.min_samples.split(",")]
    for ms in mss:                                               # warm-up: modules, attributes, profiler
        one_run(torch.from_numpy(random_walk(2000, 2, 1)).to(dev), ms)
    for n in [int(x) for x in a.sizes.split(",")]:
        for d in [int(x) for x in a.dims.split(",")]:
            X = random_walk(n, d, 3)
            Y = torch.from_numpy(X).to(dev)
            for ms in mss:
                parts, kers = {}, {}
                for _ in range(a.repeats):
                    labels, t, ker = one_run(Y, ms)
                    for k, v in t.items():
                        parts.setdefault(k, []).append(v)
                    for k, v in ker.items():
                        kers.setdefault(k, []).append(v)
                row = {"n": n, "d": d, "min_samples": ms, "ms": {k: stats(v) for k, v in parts.items()},
                       "kernel_ms": {k: stats(v) for k, v in kers.items()},
                       "n_clusters": int(labels.max()) + 1, "noise": int((labels < 0).sum())}
                row["total_ms"] = sum(row["ms"][k]["median"] for k in parts)
                if n == a.sklearn_n:
                    from sklearn.cluster import HDBSCAN
                    t0 = time.perf_counter()
                    ref = HDBSCAN(min_cluster_size=5, min_samples=ms, copy=True).fit_predict(X)
                    row["sklearn_fit_s"] = time.perf_counter() - t0
                    row["speedup_vs_sklearn"] = row["sklearn_fit_s"] * 1e3 / row["total_ms"]
                    row["labels_equal_sklearn"] = bool(np.array_equal(labels, ref))
                res["runs"].append(row)
                print(json.dumps(row), flush=True)
            del Y
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
