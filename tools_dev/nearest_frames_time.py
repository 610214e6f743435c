"""Nearest clustered frame on the device (csrc/nearest.cu, dcg_nearest_frames_f64) timed against scikit-learn's
KD-tree on the same host.

    python tools_dev/nearest_frames_time.py [--sizes 100000,1000000,10000000] [--queries 1000000]
                                            [--dims 2,4,10] [--out profiles/nearest_frames_time.json]

Inputs: the seeded random-walk CVs of hier_time.py (step 0.05 N(0,1) per CV, seed 3), N + M steps, of which a
seeded random choice of M rows are the queries and the rest the frames; plus uniform noise in [-1, 1]^10 for
both, where the tile pruning cannot work.  For every case: the entry point (Morton keys, radix sorts, ordered
copies, tile boxes, search) timed with CUDA events, median of 3 after a warm-up call, and the fraction of tiles
skipped.  scikit-learn's NearestNeighbors(n_neighbors=1, algorithm="kd_tree") build and query are timed with a
host clock; when the query would take more than --sklearn-budget seconds (projected from the first 10^4
queries) only those are timed, and the JSON says how many queries its time covers.  The distances of the queries
scikit-learn answered are checked bitwise against the device's.  The GPU name and power limit are read in the
same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deep_cartograph_b200 import _lib  # noqa: E402


def random_walk(n, d, seed):
    rng = np.random.default_rng(seed)
    return np.ascontiguousarray(np.cumsum(0.05 * rng.standard_normal((n, d)), axis=0))


def make_case(kind, n, m, d):
    if kind == "uniform":
        rng = np.random.default_rng(5)
        return rng.uniform(-1, 1, (n, d)), rng.uniform(-1, 1, (m, d))
    W = random_walk(n + m, d, 3)
    q = np.zeros(n + m, dtype=bool)
    q[np.random.default_rng(4).choice(n + m, m, replace=False)] = True
    return np.ascontiguousarray(W[~q]), np.ascontiguousarray(W[q])


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def device_times(X, Q, repeats):
    """Median / min / max of the entry point's device time (ms), the tiles visited and considered, and the
    result of the last call."""
    n, d = X.shape
    m = Q.shape[0]
    dev = X.device
    ws = torch.empty(int(_lib.load().dcg_nearest_frames_workspace_bytes(n, m, d)), dtype=torch.uint8, device=dev)
    index = torch.empty(m, dtype=torch.int64, device=dev)
    dist = torch.empty(m, dtype=torch.float64, device=dev)
    st = torch.cuda.current_stream(dev)
    args = (X.data_ptr(), n, d, Q.data_ptr(), m, d, d, index.data_ptr(), dist.data_ptr(), ws.data_ptr(),
            ws.numel(), st.cuda_stream)
    _lib.call("dcg_nearest_frames_f64", *args)                    # warm-up
    times = []
    for _ in range(repeats):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record(st)
        _lib.call("dcg_nearest_frames_f64", *args)
        ev[1].record(st)
        torch.cuda.synchronize()
        times.append(ev[0].elapsed_time(ev[1]))
    visited, considered = ws[:16].view(torch.int64).tolist()
    t = np.asarray(times)
    return ({"median": float(np.median(t)), "min": float(t.min()), "max": float(t.max())}, visited, considered,
            index.cpu().numpy(), dist.cpu().numpy())


def sklearn_times(X, Q, budget):
    from sklearn.neighbors import NearestNeighbors
    t0 = time.perf_counter()
    nn = NearestNeighbors(n_neighbors=1, algorithm="kd_tree").fit(X)
    build = time.perf_counter() - t0
    probe = min(10000, Q.shape[0])
    t0 = time.perf_counter()
    dist, idx = nn.kneighbors(Q[:probe])
    t_probe = time.perf_counter() - t0
    if t_probe * Q.shape[0] / probe <= budget and probe < Q.shape[0]:
        t0 = time.perf_counter()
        dist, idx = nn.kneighbors(Q)
        t_probe = time.perf_counter() - t0
    return {"build_s": build, "query_s": t_probe, "queries": int(dist.shape[0])}, dist[:, 0], idx[:, 0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="100000,1000000,10000000")
    ap.add_argument("--queries", type=int, default=1000000)
    ap.add_argument("--dims", default="2,4,10")
    ap.add_argument("--uniform-dim", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--sklearn-budget", type=float, default=60.0)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                  "profiles", "nearest_frames_time.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "nearest_frames_time.py measures on the GPU; there is no CPU path"
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "queries": a.queries,
           "inputs": {"walk": "random walk, step 0.05 N(0,1) per CV, seed 3; M seeded rows are the queries",
                      "uniform": "uniform [-1, 1]^d, seed 5"},
           "device_ms": "dcg_nearest_frames_f64 (keys, sorts, copies, boxes, search), CUDA events, median of "
                        f"{a.repeats} after a warm-up",
           "sklearn": "NearestNeighbors(n_neighbors=1, algorithm='kd_tree'), one host thread", "runs": []}
    print(json.dumps(res["gpu"]), flush=True)
    cases = [("walk", d) for d in (int(x) for x in a.dims.split(","))] + [("uniform", a.uniform_dim)]
    for n in (int(x) for x in a.sizes.split(",")):
        for kind, d in cases:
            Xh, Qh = make_case(kind, n, a.queries, d)
            X, Q = torch.from_numpy(Xh).to(dev), torch.from_numpy(Qh).to(dev)
            t, visited, considered, index, dist = device_times(X, Q, a.repeats)
            row = {"input": kind, "n": n, "m": a.queries, "d": d, "device_ms": t,
                   "tiles_visited": visited, "tiles_considered": considered,
                   "skipped_fraction": 1.0 - visited / considered}
            sk, kdist, kidx = sklearn_times(Xh, Qh, a.sklearn_budget)
            row["sklearn"] = sk
            q = sk["queries"]
            row["speedup_vs_sklearn_build_plus_query"] = (       # only where scikit-learn answered every query
                (sk["build_s"] + sk["query_s"]) * 1e3 / t["median"] if q == a.queries else None)
            row["dist_bitwise_equal_sklearn"] = bool(np.array_equal(dist[:q], kdist))
            row["index_equal_sklearn"] = int((index[:q] == kidx).sum())
            res["runs"].append(row)
            print(json.dumps(row), flush=True)
            del X, Q
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
