"""HDBSCAN on the device (csrc/linkage.cu core_dist_kernel + prim_kernel with core distances,
ops.core_distances / ops.mreach_mst, statistics.hdbscan_tree / hdbscan_labels / hdbscan_clustering, traj_cluster
with backend.hdbscan_on_device): core distances, MST rows and single-linkage tree must be scikit-learn's bit
for bit, and the labels must be sklearn.cluster.HDBSCAN's label for label."""
import ctypes
import functools
import itertools
import os

import numpy as np
import pandas as pd
import pytest
import torch

SELECTION_GRID = list(itertools.product(("eom", "leaf"), (0.0, 0.05, 0.5), (None, 50), (2, 5, 50)))


def random_walk(n, d, seed):
    """Seeded random-walk CVs, like frames of an MD trajectory projected on d CVs."""
    rng = np.random.default_rng(seed)
    return np.ascontiguousarray(np.cumsum(0.05 * rng.standard_normal((n, d)), axis=0))


@functools.lru_cache(maxsize=1)
def golden_cvs():
    """The 164-frame golden CV sets of the reference's bundled peptide test (the conftest's c1 fixture)."""
    c1 = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "peptide_c1.npz"))
    return {cv: np.ascontiguousarray(c1[f"{cv}_cluster_cv"]) for cv in ("pca", "tica", "htica")}


def make_case(name):
    rng = np.random.default_rng(23)
    if name in ("pca", "tica", "htica"):
        return golden_cvs()[name]
    if name == "blobs_noise":              # four blobs of different density over a uniform background
        cent = rng.uniform(-1, 1, size=(4, 2))
        X = np.concatenate([cent[i] + s * rng.standard_normal((m, 2))
                            for i, (m, s) in enumerate([(150, 0.05), (120, 0.1), (80, 0.03), (60, 0.2)])])
        return np.ascontiguousarray(np.concatenate([X, rng.uniform(-1.5, 1.5, size=(90, 2))]))
    if name == "all_noise":                # 60 uniform frames: no split leaves two parts of 50 frames
        return np.ascontiguousarray(rng.uniform(-1, 1, size=(60, 3)))
    if name == "one_blob":
        return np.ascontiguousarray(0.1 * rng.standard_normal((300, 2)))
    if name == "ties5k":                   # 0.01 grid: exact ties and duplicate frames
        return np.ascontiguousarray(np.round(rng.uniform(-1, 1, size=(5000, 2)), 2))
    if name.startswith("walk"):            # walk20k_d2, walk100k_d2, ...
        n, d = name[4:].split("_d")
        return np.round(random_walk(int(n[:-1]) * 1000, int(d), 3), 4)
    raise KeyError(name)


def sk_tree(X, min_samples):
    from sklearn.cluster import HDBSCAN
    return HDBSCAN(min_cluster_size=5, min_samples=min_samples, copy=True).fit(X)._single_linkage_tree_


def sk_mst(X, core):
    from sklearn.cluster._hdbscan._linkage import mst_from_data_matrix
    from sklearn.metrics import DistanceMetric
    m = mst_from_data_matrix(np.ascontiguousarray(X), np.ascontiguousarray(core), DistanceMetric.get_metric("euclidean"))
    return np.stack([m["current_node"].astype(np.float64), m["next_node"].astype(np.float64), m["distance"]], axis=1)


def sk_core(X, k):
    from sklearn.neighbors import NearestNeighbors
    return NearestNeighbors(n_neighbors=k, algorithm="kd_tree").fit(X).kneighbors(X, k)[0][:, -1]


def sk_labels(tree, method, eps, max_size, mcs):
    from sklearn.cluster._hdbscan._tree import tree_to_labels
    return tree_to_labels(tree, mcs, method, False, eps, max_size)[0]


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["blobs_noise", "pca", "tica", "htica", "all_noise", "one_blob"])
def test_hdbscan_labels_equal_sklearn_tree_to_labels(case):
    """The numpy restatement of tree_to_labels on trees scikit-learn builds, over the whole selection grid."""
    from deep_cartograph_b200.modules.statistics import statistics
    X = make_case(case)
    for ms in (1, 3):
        tree = sk_tree(X, ms)
        for method, eps, max_size, mcs in SELECTION_GRID:
            ref = sk_labels(tree, method, eps, max_size, mcs)
            got = statistics.hdbscan_labels(tree, mcs, method, eps, max_size)
            assert np.array_equal(got, ref), (ms, method, eps, max_size, mcs)


def test_hdbscan_labels_all_noise_and_clusters_are_found():
    """The grid holds both outcomes the workflow must handle: only noise, and several clusters with noise."""
    from deep_cartograph_b200.modules.statistics import statistics
    assert (statistics.hdbscan_labels(sk_tree(make_case("all_noise"), 3), 50) == -1).all()
    lab = statistics.hdbscan_labels(sk_tree(make_case("blobs_noise"), 3), 5)
    assert lab.max() >= 3 and (lab == -1).any()


def test_hdbscan_labels_large_walk_equals_sklearn():
    from deep_cartograph_b200.modules.statistics import statistics
    tree = sk_tree(make_case("walk20k_d2"), 3)
    for method, eps, max_size, mcs in SELECTION_GRID:
        if mcs == 2 and method == "eom" and eps == 0.5:
            continue                                  # sklearn's own epsilon search is quadratic here
        assert np.array_equal(statistics.hdbscan_labels(tree, mcs, method, eps, max_size),
                              sk_labels(tree, method, eps, max_size, mcs)), (method, eps, max_size, mcs)


@pytest.mark.parametrize("case", ["blobs_noise", "pca", "tica", "htica", "ties5k"])
def test_single_linkage_from_mst_equals_make_single_linkage(case):
    """numpy's default argsort of the Prim-order MST, then make_single_linkage's union-find, on MSTs with
    tied distances (the golden sets are 4-decimal text, ties5k a 0.01 grid)."""
    from sklearn.cluster._hdbscan.hdbscan import _process_mst
    from sklearn.cluster._hdbscan._linkage import MST_edge_dtype
    from deep_cartograph_b200.modules.statistics import statistics
    X = make_case(case)
    tied = 0
    for ms in (1, 3, 16):
        mst = sk_mst(X, sk_core(X, ms))
        edges = np.empty(len(mst), dtype=MST_edge_dtype)
        edges["current_node"], edges["next_node"], edges["distance"] = mst[:, 0], mst[:, 1], mst[:, 2]
        ref = _process_mst(edges)
        got = statistics.single_linkage_from_mst(mst)
        tied += len(np.unique(mst[:, 2])) < len(mst)
        for f in ("left_node", "right_node", "value", "cluster_size"):
            assert np.array_equal(got[f], ref[f]), (ms, f)
    assert tied or case == "blobs_noise"


def test_schema_device_hdbscan_is_opt_in():
    from deep_cartograph_b200.yaml_schemas.traj_cluster import TrajClusterSchema
    d = TrajClusterSchema().model_dump()
    assert d["backend"]["hdbscan_on_device"] is False
    assert TrajClusterSchema(backend={"hdbscan_on_device": True}).backend.hdbscan_on_device


def test_hdbscan_without_flag_still_exits():
    from deep_cartograph_b200.modules.statistics import statistics
    with pytest.raises(SystemExit):
        statistics.optimize_clustering(np.zeros((4, 2)), {"algorithm": "hdbscan",
                                                          "backend": {"hierarchical_on_device": True}})


def test_hdbscan_argument_errors_without_gpu():
    from deep_cartograph_b200 import _lib
    lib = _lib.load()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    big = 1 << 30
    assert lib.dcg_core_distances_f64(p, 1, 2, 2, 1, p, None, 0, None) == -1001       # n < 2
    assert lib.dcg_core_distances_f64(p, 10, 0, 2, 1, p, None, 0, None) == -1001      # d < 1
    assert lib.dcg_core_distances_f64(p, 10, 3, 2, 1, p, None, 0, None) == -1001      # ld < d
    assert lib.dcg_core_distances_f64(p, 10, 2, 2, 0, p, None, 0, None) == -1001      # min_samples < 1
    assert lib.dcg_core_distances_f64(p, 10, 2, 2, 11, p, None, 0, None) == -1001     # min_samples > n
    assert lib.dcg_core_distances_f64(p, 100, 2, 2, 65, p, None, 0, None) == -1001    # min_samples > 64
    assert lib.dcg_core_distances_f64(p, 10, 2, 2, 3, None, None, 0, None) == -1000   # no output
    assert lib.dcg_mreach_mst_f64(p, 1, 2, 2, p, p, p, big, None) == -1001
    assert lib.dcg_mreach_mst_f64(p, 10, 3, 2, p, p, p, big, None) == -1001
    assert lib.dcg_mreach_mst_f64(p, 10, 2, 2, None, p, p, big, None) == -1000         # no core
    need = lib.dcg_hdbscan_workspace_bytes(10, 2, 3)
    assert lib.dcg_mreach_mst_f64(p, 10, 2, 2, p, p, p, need - 1, None) == -1002       # short workspace
    assert lib.dcg_mreach_mst_f64(p, 10, 2, 2, p, p, None, need, None) == -1002        # no workspace
    assert lib.dcg_hdbscan_workspace_bytes(1, 2, 1) == 0
    assert lib.dcg_hdbscan_workspace_bytes(10, 2, 65) == 0
    assert lib.dcg_hdbscan_workspace_bytes(10, 0, 3) == 0


def test_hdbscan_workspace_is_linear_in_frames():
    from deep_cartograph_b200 import _lib
    lib = _lib.load()
    for n in (4096, 100000, 1000000, 10000000):
        assert 12 * n <= lib.dcg_hdbscan_workspace_bytes(n, 10, 3) <= 12 * n + 1024
    assert lib.dcg_hdbscan_workspace_bytes(50000, 2, 3) == lib.dcg_hdbscan_workspace_bytes(50000, 16, 64)


def test_hdbscan_memory_check_raises_before_allocating(monkeypatch):
    from deep_cartograph_b200 import ops
    monkeypatch.setattr(ops, "_hdbscan_frames", lambda Y: Y)
    monkeypatch.setattr(ops, "_need_cuda", lambda *a, **k: None)
    monkeypatch.setattr(ops, "_ws", lambda *a, **k: pytest.fail("allocated before the memory check"))
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda *a, **k: (1 << 20, 180 << 30))
    with pytest.raises(MemoryError, match="100000 frames needs"):
        ops.mreach_mst(torch.zeros((100000, 2), dtype=torch.float64), torch.zeros(100000, dtype=torch.float64))
    with pytest.raises(MemoryError, match="100000 frames needs"):
        ops.core_distances(torch.zeros((100000, 2), dtype=torch.float64), 3)


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from deep_cartograph_b200 import _lib
    _lib.load()            # fail loudly if the extension is missing
    return torch.device("cuda:0")


def core_input(n, d, kind):
    rng = np.random.default_rng(n * 31 + d)
    X = rng.standard_normal((n, d)) * rng.uniform(0.1, 10, size=d)
    if kind == "grid":                     # 4-decimal text values, as the CV CSVs hold
        X = np.round(X, 4)
    elif kind == "dup":                    # exact duplicate frames and a coarse grid: tied neighbours
        X = np.round(X, 0)
        X[n // 2:] = X[: n - n // 2]
    return np.ascontiguousarray(X)


CORE_CASES = [(n, d, kind) for n in (2, 3, 17, 100, 1000) for d in (1, 2, 3, 10) for kind in ("real", "grid", "dup")] + \
             [(20000, d, kind) for d in (1, 2, 3, 10) for kind in ("grid", "dup")] + \
             [(100000, 2, "grid"), (100000, 3, "dup")]


@pytest.mark.gpu
@pytest.mark.parametrize("n,d,kind", CORE_CASES)
def test_core_distances_bitwise_equal_kd_tree(dev, n, d, kind):
    from deep_cartograph_b200 import ops
    X = core_input(n, d, kind)
    Y = torch.from_numpy(X).to(dev)
    for k in (1, 2, 3, 5, 16, 64):
        if k > n:
            continue
        got = ops.core_distances(Y, k).cpu().numpy()
        ref = sk_core(X, k)
        assert np.array_equal(got, ref), (k, np.flatnonzero(got != ref)[:10])


MST_CASES = ["blobs_noise", "pca", "tica", "htica", "one_blob", "ties5k", "walk20k_d2", "walk20k_d10"]


@functools.lru_cache(maxsize=None)
def cached_sk_tree(case, ms):
    return sk_tree(make_case(case), ms)


@pytest.mark.gpu
@pytest.mark.parametrize("case", MST_CASES)
def test_mreach_mst_and_tree_bitwise_equal_sklearn(dev, case):
    """MST rows (source, new node, distance) in Prim order equal mst_from_data_matrix's, and the
    single-linkage tree equals HDBSCAN's _single_linkage_tree_."""
    from deep_cartograph_b200 import ops
    from deep_cartograph_b200.modules.statistics import statistics
    X = make_case(case)
    Y = torch.from_numpy(X).to(dev)
    for ms in (1, 3, 16):
        core = ops.core_distances(Y, ms)
        mst = ops.mreach_mst(Y, core).cpu().numpy()
        ref = sk_mst(X, core.cpu().numpy())
        assert np.array_equal(mst, ref), (ms, np.flatnonzero((mst != ref).any(axis=1))[:10])
        tree = statistics.hdbscan_tree(X, ms)
        assert np.array_equal(tree, cached_sk_tree(case, ms).astype(statistics.HIERARCHY_DTYPE)), ms


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["pca", "tica", "htica", "blobs_noise", "ties5k", "walk20k_d2", "all_noise"])
def test_hdbscan_clustering_labels_equal_sklearn(dev, case):
    """hdbscan_clustering equals HDBSCAN(...).fit_predict over the selection grid: a full fit_predict for
    every setting on the small sets, and on the large ones one fit per min_samples (the tree) whose labels
    tree_to_labels gives for every setting, plus one full fit_predict."""
    from sklearn.cluster import HDBSCAN
    from deep_cartograph_b200.modules.statistics import statistics
    X = make_case(case)
    big = len(X) > 1000
    for ms in (None, 3):
        for method, eps, max_size, mcs in SELECTION_GRID:
            settings = {"min_cluster_size": mcs, "min_samples": ms, "cluster_selection_method": method,
                        "cluster_selection_epsilon": eps, "max_cluster_size": max_size}
            if big and (ms is None or (mcs == 2 and method == "eom" and eps == 0.5)):
                continue
            labels, centroids = statistics.hdbscan_clustering(X, settings)
            if big:
                ref = sk_labels(cached_sk_tree(case, ms), method, eps, max_size, mcs)
            else:
                ref = HDBSCAN(min_cluster_size=mcs, min_samples=ms, cluster_selection_epsilon=eps,
                              max_cluster_size=max_size, cluster_selection_method=method, copy=True).fit_predict(X)
            assert np.array_equal(labels, ref), (ms, method, eps, max_size, mcs)
            k = ref.max() + 1
            assert centroids.shape == (k, X.shape[1])
            for c in range(k):
                np.testing.assert_array_equal(centroids[c], X[ref == c].mean(axis=0))
    if big:
        ref = HDBSCAN(min_cluster_size=5, min_samples=3, copy=True).fit_predict(X)
        assert np.array_equal(statistics.hdbscan_clustering(X, {"min_cluster_size": 5, "min_samples": 3})[0], ref)


@pytest.mark.gpu
def test_hdbscan_100k_frames_equals_sklearn(dev):
    from sklearn.cluster import HDBSCAN
    from deep_cartograph_b200.modules.statistics import statistics
    X = make_case("walk100k_d2")
    hd = HDBSCAN(min_cluster_size=50, min_samples=3, copy=True).fit(X)
    tree = statistics.hdbscan_tree(X, 3)
    assert np.array_equal(tree, hd._single_linkage_tree_.astype(statistics.HIERARCHY_DTYPE))
    assert np.array_equal(statistics.hdbscan_labels(tree, 50), hd.labels_)


@pytest.mark.gpu
@pytest.mark.parametrize("cv", ["pca", "tica", "htica"])
def test_traj_cluster_hdbscan_writes_sklearn_labels(dev, c1, cv, tmp_path):
    """traj_cluster with the schema's HDBSCAN settings on the golden CV CSVs: the cluster column is
    scikit-learn's labels (-1 for noise) and the centroid column marks the frame nearest each member mean."""
    from sklearn.cluster import HDBSCAN
    from deep_cartograph_b200.tools import traj_cluster
    cols = list(c1[f"{cv}_csv_cols"])
    csv = tmp_path / f"{cv}.csv"
    pd.DataFrame(c1[f"{cv}_cluster_cv"], columns=cols).to_csv(csv, index=False, float_format="%.4f")
    X = pd.read_csv(csv).to_numpy()
    out = traj_cluster({"algorithm": "hdbscan", "backend": {"hdbscan_on_device": True}}, [str(csv)],
                       output_folder=str(tmp_path / "cl"))
    df = pd.read_csv(out["traj_0"][0])
    assert list(df.columns) == cols + ["traj_label", "cluster", "centroid", "frame"]
    ref = HDBSCAN(min_cluster_size=5, min_samples=3, copy=True).fit_predict(X)         # the schema defaults
    assert np.array_equal(df["cluster"].to_numpy(), ref)
    k = ref.max() + 1
    assert k >= 1 and df["centroid"].sum() == k
    for c in range(k):
        mean = X[ref == c].mean(axis=0)
        nearest = int(np.argmin(((X - mean) ** 2).sum(axis=1)))
        assert df["centroid"].iloc[nearest]


@pytest.mark.gpu
def test_traj_cluster_hdbscan_all_noise_completes(dev, tmp_path):
    from deep_cartograph_b200.tools import traj_cluster
    csv = tmp_path / "noise.csv"
    pd.DataFrame(make_case("all_noise"), columns=["a", "b", "c"]).to_csv(csv, index=False, float_format="%.4f")
    out = traj_cluster({"algorithm": "hdbscan", "min_cluster_size": 50, "backend": {"hdbscan_on_device": True}},
                       [str(csv)], output_folder=str(tmp_path / "cl"))
    df = pd.read_csv(out["traj_0"][0])
    assert (df["cluster"] == -1).all() and not df["centroid"].any() and len(df) == 60


@pytest.mark.gpu
def test_optimize_clustering_runs_hdbscan_once_unscored(dev, monkeypatch):
    from sklearn.cluster import HDBSCAN
    from deep_cartograph_b200.modules.statistics import statistics
    X = make_case("tica")
    monkeypatch.setattr(statistics, "cluster_scores", lambda *a, **k: pytest.fail("HDBSCAN is not scored"))
    settings = {"algorithm": "hdbscan", "min_cluster_size": 5, "min_samples": 3, "search_interval": [3, 10],
                "backend": {"hdbscan_on_device": True}}
    labels, _ = statistics.optimize_clustering(X, settings)
    assert np.array_equal(labels, HDBSCAN(min_cluster_size=5, min_samples=3, copy=True).fit_predict(X))
    assert np.array_equal(statistics.cluster_data(X, settings)[0], labels)


@pytest.mark.gpu
def test_hdbscan_float32_input_is_widened_exactly(dev):
    from deep_cartograph_b200 import ops
    X32 = torch.from_numpy(make_case("blobs_noise").astype(np.float32)).to(dev)
    for k in (1, 3, 16):
        c32, c64 = ops.core_distances(X32, k), ops.core_distances(X32.to(torch.float64), k)
        assert torch.equal(c32, c64)
        assert torch.equal(ops.mreach_mst(X32, c32), ops.mreach_mst(X32.to(torch.float64), c64))


@pytest.mark.gpu
def test_hdbscan_rejects_bad_input(dev):
    from deep_cartograph_b200 import ops
    from deep_cartograph_b200.modules.statistics import statistics
    Y = torch.rand((50, 2), dtype=torch.float64, device=dev)
    with pytest.raises(ValueError, match="n_neighbors <= n_samples_fit"):
        ops.core_distances(Y, 51)
    with pytest.raises(ValueError, match=r"min_samples must be in \[1, 64\]"):
        ops.core_distances(torch.rand((100, 2), dtype=torch.float64, device=dev), 65)
    with pytest.raises(ValueError, match=r"min_samples must be in \[1, 64\]"):
        ops.core_distances(Y, 0)
    with pytest.raises(ValueError, match="at least 2 frames"):
        ops.core_distances(Y[:1], 1)
    with pytest.raises(ValueError, match="at least 2 frames"):
        ops.mreach_mst(Y[:1], torch.zeros(1, dtype=torch.float64, device=dev))
    with pytest.raises(ValueError, match="core must have shape"):
        ops.mreach_mst(Y, torch.zeros(49, dtype=torch.float64, device=dev))
    Yn = Y.clone()
    Yn[7, 1] = float("nan")
    with pytest.raises(ValueError, match="NaN"):
        ops.core_distances(Yn, 3)
    with pytest.raises(ValueError, match="NaN"):
        ops.mreach_mst(Yn, torch.zeros(50, dtype=torch.float64, device=dev))
    with pytest.raises(ValueError, match="min_cluster_size must be at least 2"):
        statistics.hdbscan_clustering(Y.cpu().numpy(), {"min_cluster_size": 1, "min_samples": 3})
