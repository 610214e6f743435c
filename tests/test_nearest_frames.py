"""Nearest clustered frame of supplementary frames on the device (csrc/nearest.cu, ops.nearest_frames,
statistics.assign_closest_cluster, traj_cluster with sup_cv_traj_paths).

The device rule: each query takes the lexicographic minimum of (rdist, frame index), rdist = sum_f (q_f - x_f)^2
in ascending feature order with one rounded subtract, multiply and add per term, and dist = sqrt(rdist).  That is
the arithmetic of scikit-learn's KD-tree, so the distances must be bitwise its distances, and the indices must be
its indices wherever the nearest frame is unique (on exact ties the KD-tree returns whichever tied frame it visits
first; the device returns the lowest index)."""
import ctypes

import numpy as np
import pandas as pd
import pytest
import torch

TILE = 256                 # frames of a tile for d <= 24 (kMaxTile, csrc/nearest.cu)
QUERY_BLOCK = 128          # queries of one CTA


def random_walk(n, d, seed, decimals=None, step=0.05):
    """Seeded random-walk CVs, like frames of an MD trajectory projected on d CVs; ``decimals``: rounded as the
    CV CSV files are."""
    rng = np.random.default_rng(seed)
    X = np.cumsum(step * rng.standard_normal((n, d)), axis=0)
    return np.ascontiguousarray(np.round(X, decimals) if decimals is not None else X)


def nearest_reference(X, Q, chunk=256):
    """numpy restatement of the device rule: (index of the lowest-indexed nearest frame, its rdist, the number of
    frames at exactly that rdist).  numpy's subtract, multiply and add are single correctly rounded operations."""
    m = Q.shape[0]
    index = np.empty(m, dtype=np.int64)
    rdist = np.empty(m, dtype=np.float64)
    ties = np.empty(m, dtype=np.int64)
    for a in range(0, m, chunk):
        q = Q[a:a + chunk]
        s = np.zeros((q.shape[0], X.shape[0]))
        for f in range(X.shape[1]):
            t = q[:, f, None] - X[None, :, f]
            s = s + t * t
        i = np.argmin(s, axis=1)                    # first occurrence: the lowest index among the minima
        best = s[np.arange(q.shape[0]), i]
        index[a:a + chunk], rdist[a:a + chunk] = i, best
        ties[a:a + chunk] = (s == best[:, None]).sum(axis=1)
    return index, rdist, ties


def rdist_of(X, Q, idx):
    s = np.zeros(Q.shape[0])
    for f in range(X.shape[1]):
        t = Q[:, f] - X[idx, f]
        s = s + t * t
    return s


def kd_tree(X, Q):
    from sklearn.neighbors import NearestNeighbors
    dist, idx = NearestNeighbors(n_neighbors=1, algorithm="kd_tree").fit(X).kneighbors(Q)
    return idx[:, 0], dist[:, 0]


def check_against_kd_tree(X, Q, index, dist):
    """Distances bitwise the KD-tree's; indices equal to its indices, or, where they differ, a frame at exactly
    the same rdist (a tie)."""
    kidx, kdist = kd_tree(X, Q)
    assert np.array_equal(dist, kdist), np.flatnonzero(dist != kdist)[:10]
    diff = np.flatnonzero(index != kidx)
    if len(diff):
        assert np.array_equal(rdist_of(X, Q[diff], kidx[diff]), rdist_of(X, Q[diff], index[diff])), diff[:10]
        assert np.all(index[diff] < kidx[diff]), diff[:10]            # the device keeps the lowest tied index
    return len(diff)


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
# 4-decimal random walks (what the CV CSV files hold), 20k frames and 20k queries; at d = 2 with a small step the
# walk revisits the 1e-4 grid densely enough for exact ties, some of which the KD-tree breaks by a higher index
WALKS = [(2, 0.003), (3, 0.01)]


def walk_case(d, step):
    W = random_walk(40000, d, 3, decimals=4, step=step)
    return np.ascontiguousarray(W[0::2]), np.ascontiguousarray(W[1::2])


@pytest.mark.parametrize("d,step", WALKS)
def test_restatement_equals_sklearn_kd_tree(d, step):
    """The numpy restatement gives the KD-tree's distances bit for bit, and its indices wherever the minimum is
    unique; where it is not, the KD-tree's frame is tied and the restatement's is the lowest tied index."""
    X, Q = walk_case(d, step)
    index, rdist, ties = nearest_reference(X, Q, chunk=512)
    kidx, kdist = kd_tree(X, Q)
    assert np.array_equal(np.sqrt(rdist), kdist)
    unique = ties == 1
    assert np.array_equal(index[unique], kidx[unique])
    tied = np.flatnonzero(~unique)
    assert np.array_equal(rdist_of(X, Q[tied], kidx[tied]), rdist[tied])
    assert np.all(index[tied] <= kidx[tied])
    if d == 2:                                                      # the data does exercise the tie rule
        assert len(tied) > 0 and np.any(index[tied] < kidx[tied])


def test_restatement_equals_sklearn_kd_tree_above_15_features():
    """scikit-learn's ``auto`` switches to brute force above 15 features; the device keeps the KD-tree's
    arithmetic for every d, so the comparison is with ``algorithm="kd_tree"``."""
    rng = np.random.default_rng(4)
    X, Q = rng.uniform(-1, 1, (3000, 16)), rng.uniform(-1, 1, (500, 16))
    index, rdist, ties = nearest_reference(X, Q)
    kidx, kdist = kd_tree(X, Q)
    assert np.array_equal(np.sqrt(rdist), kdist)
    assert np.all(ties == 1) and np.array_equal(index, kidx)


def test_nearest_frames_argument_errors_without_gpu():
    from deep_cartograph_b200 import _lib
    lib = _lib.load()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    big = 1 << 30
    f = lib.dcg_nearest_frames_f64
    assert f(p, 0, 2, p, 5, 2, 2, p, p, p, big, None) == -1001            # n < 1
    assert f(p, 10, 2, p, -1, 2, 2, p, p, p, big, None) == -1001          # m < 0
    assert f(p, 10, 2, p, 5, 2, 0, p, p, p, big, None) == -1001           # d < 1
    assert f(p, 10, 1, p, 5, 2, 2, p, p, p, big, None) == -1001           # ldx < d
    assert f(p, 10, 2, p, 5, 1, 2, p, p, p, big, None) == -1001           # ldq < d
    assert f(p, 10, 9000, p, 5, 9000, 8193, p, p, p, big, None) == -1001  # d above 8192
    assert f(p, 10, 2, p, 0, 2, 2, None, None, None, 0, None) == 0        # m = 0: nothing to do
    assert f(None, 10, 2, p, 5, 2, 2, p, p, p, big, None) == -1000
    assert f(p, 10, 2, p, 5, 2, 2, None, p, p, big, None) == -1000
    assert f(p, 10, 2, p, 5, 2, 2, p, None, p, big, None) == -1000
    assert lib.dcg_nearest_frames_workspace_bytes(0, 5, 2) == 0
    assert lib.dcg_nearest_frames_workspace_bytes(10, -1, 2) == 0
    assert lib.dcg_nearest_frames_workspace_bytes(10, 5, 0) == 0


def test_ops_nearest_frames_validation_without_gpu(monkeypatch):
    from deep_cartograph_b200 import ops
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        ops.nearest_frames(torch.zeros((4, 2)), torch.zeros((3, 2)))
    monkeypatch.setattr(ops, "_need_cuda", lambda *a, **k: None)
    monkeypatch.setattr(ops, "_ws", lambda *a, **k: (_ for _ in ()).throw(AssertionError("allocated")))
    with pytest.raises(TypeError, match="float32 or float64"):
        ops.nearest_frames(torch.zeros((4, 2), dtype=torch.int32), torch.zeros((3, 2)))
    with pytest.raises(ValueError, match="same number of features"):
        ops.nearest_frames(torch.zeros((4, 2)), torch.zeros((3, 3)))
    with pytest.raises(ValueError, match="at least 1 frame"):
        ops.nearest_frames(torch.zeros((0, 2)), torch.zeros((3, 2)))
    with pytest.raises(ValueError, match="NaN or infinity"):
        ops.nearest_frames(torch.zeros((4, 2)), torch.tensor([[0.0, float("nan")]]))
    with pytest.raises(ValueError, match="NaN or infinity"):
        ops.nearest_frames(torch.tensor([[float("inf"), 0.0]]), torch.zeros((3, 2)))
    with pytest.raises(ValueError, match="2-D|at least 1 feature"):
        ops.nearest_frames(torch.zeros(4), torch.zeros((3, 2)))


def _write_cv(path, X, cols):
    pd.DataFrame(X, columns=cols).to_csv(path, index=False, float_format="%.4f")


@pytest.mark.parametrize("case", ["columns", "name_main", "name_sup"])
def test_traj_cluster_supplementary_errors_before_device_work(case, tmp_path, monkeypatch):
    """Mismatched supplementary CV columns and output-name collisions are reported before any clustering or
    device call, and before any trajectory CSV is written."""
    from deep_cartograph_b200 import ops
    from deep_cartograph_b200.modules.statistics import statistics
    from deep_cartograph_b200.tools import traj_cluster

    def no_device(*a, **k):
        raise AssertionError("device work before the supplementary checks")
    for name in ("optimize_clustering", "cluster_data", "assign_closest_cluster", "_to_device"):
        monkeypatch.setattr(statistics, name, no_device)
    monkeypatch.setattr(ops, "nearest_frames", no_device)
    X = random_walk(50, 2, 1, decimals=4)
    _write_cv(tmp_path / "a.csv", X, ["cv1", "cv2"])
    _write_cv(tmp_path / "s.csv", X, ["cv1", "cvX"] if case == "columns" else ["cv1", "cv2"])
    kw = {}
    if case == "name_main":
        kw = {"trajectories": ["/data/run1.xtc"], "sup_trajectories": ["/other/run1.dcd"]}
    elif case == "name_sup":
        kw = {"sup_cv_traj_paths": [str(tmp_path / "s.csv")] * 2, "sup_trajectories": ["/x/r.xtc", "/y/r.xtc"]}
    kw.setdefault("sup_cv_traj_paths", [str(tmp_path / "s.csv")])
    with pytest.raises(ValueError, match="columns" if case == "columns" else "collides"):
        traj_cluster({"algorithm": "kmeans"}, [str(tmp_path / "a.csv")], output_folder=str(tmp_path / "out"), **kw)
    assert not list((tmp_path / "out").rglob("projected_trajectory.csv"))


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from deep_cartograph_b200 import _lib
    _lib.load()            # fail loudly if the extension is missing
    return torch.device("cuda:0")


def device_nearest(dev, X, Q, counters=False):
    from deep_cartograph_b200 import ops
    out = ops.nearest_frames(torch.from_numpy(X).to(dev), torch.from_numpy(Q).to(dev), return_counters=counters)
    res = (out[0].cpu().numpy(), out[1].cpu().numpy())
    return res + (out[2],) if counters else res


def check_exact(dev, X, Q):
    """Device result equal to the restatement (index and dist) and consistent with the KD-tree."""
    index, dist = device_nearest(dev, X, Q)
    assert index.dtype == np.int64 and dist.dtype == np.float64 and index.shape == dist.shape == (Q.shape[0],)
    if Q.shape[0] == 0:
        return index, dist
    ridx, rdist, _ = nearest_reference(X, Q)
    assert np.array_equal(index, ridx), np.flatnonzero(index != ridx)[:10]
    assert np.array_equal(dist, np.sqrt(rdist)), np.flatnonzero(dist != np.sqrt(rdist))[:10]
    check_against_kd_tree(X, Q, index, dist)
    return index, dist


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 2, 3, 4, 10, 16])
@pytest.mark.parametrize("n", [1, 2, TILE - 1, TILE, TILE + 1])
@pytest.mark.parametrize("m", [0, 1, 3 * QUERY_BLOCK + 5])
def test_nearest_frames_shapes(dev, d, n, m):
    rng = np.random.default_rng(1000 * d + n + m)
    X = rng.uniform(-1, 1, (n, d))
    Q = rng.uniform(-1.2, 1.2, (m, d))
    check_exact(dev, X, Q)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 2, 3, 4, 10])
def test_nearest_frames_ties_and_degenerate_data(dev, d):
    rng = np.random.default_rng(d)
    # duplicated frames: every query's nearest frame exists twice or more; the lowest index must win
    base = np.round(rng.uniform(-1, 1, (300, d)), 2)
    X = np.ascontiguousarray(np.concatenate([base, base[::-1], base[:100]]))
    Q = np.ascontiguousarray(np.round(rng.uniform(-1, 1, (700, d)), 2))
    index, _ = check_exact(dev, X, Q)
    # queries equal to frames: distance 0, lowest index of the duplicates
    index, dist = check_exact(dev, X, np.ascontiguousarray(X[::3]))
    assert np.all(dist == 0.0)
    # every frame identical: one box of zero extent, all keys equal, every frame tied
    Xc = np.ones((3 * TILE + 7, d)) * 0.25
    index, dist = check_exact(dev, Xc, Q)
    assert np.all(index == 0)
    index, dist = check_exact(dev, Xc, np.ascontiguousarray(Xc[:5]))
    assert np.all(index == 0) and np.all(dist == 0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("d,step", WALKS)
def test_nearest_frames_4_decimal_walk_ties_take_the_lowest_index(dev, d, step):
    """The 4-decimal random walks of the CPU test: the device answer is the restatement's (the lowest tied
    index on exact ties), and agrees with the KD-tree wherever the nearest frame is unique."""
    X, Q = walk_case(d, step)
    index, dist = device_nearest(dev, X, Q)
    ridx, rdist, ties = nearest_reference(X, Q, chunk=512)
    assert d != 2 or (ties > 1).any()
    assert np.array_equal(index, ridx)
    assert np.array_equal(dist, np.sqrt(rdist))
    check_against_kd_tree(X, Q, index, dist)


@pytest.mark.gpu
def test_nearest_frames_pruning_effective_on_blobs(dev):
    """Well-separated blobs: exact, and most tiles are skipped."""
    rng = np.random.default_rng(8)
    cent = rng.uniform(-10, 10, (40, 3))
    X = cent[rng.integers(0, 40, 200000)] + 0.05 * rng.standard_normal((200000, 3))
    Q = cent[rng.integers(0, 40, 20000)] + 0.05 * rng.standard_normal((20000, 3))
    index, dist, (visited, considered) = device_nearest(dev, X, Q, counters=True)
    kidx, kdist = kd_tree(X, Q)
    assert np.array_equal(dist, kdist) and np.array_equal(index, kidx)
    assert considered == -(-20000 // QUERY_BLOCK) * -(-200000 // TILE)
    assert visited < 0.1 * considered, (visited, considered)


@pytest.mark.gpu
def test_nearest_frames_tile_bound_equal_to_best_is_not_skipped(dev):
    """The skip tests are strict: a tile whose box bound equals the best already held is still scanned.
    1-D frames in two tiles of TILE: tile 0 is [-10, 0] and holds frame 0 at 0.0; tile 1 is [1, 10] and holds
    frame 2 TILE - 1 at 1.0.  The query 0.5 sorts into tile 1, so the search seeds with frame 2 TILE - 1 at
    rdist 0.25.  Tile 0's bound is (0.5 - 0.0)^2 = 0.25, the same value, and tile 0 holds frame 0 at
    rdist 0.25: the lower index must win.  With >= in either skip test, tile 0 or frame 0 would be passed over
    and the answer would be frame 2 TILE - 1."""
    left = np.concatenate([[0.0], np.linspace(-10.0, -0.5, TILE - 1)])
    right = np.concatenate([np.linspace(1.5, 10.0, TILE - 1), [1.0]])
    X = np.ascontiguousarray(np.concatenate([left, right])[:, None])
    Q = np.array([[0.5]])
    index, dist, (visited, considered) = device_nearest(dev, X, Q, counters=True)
    assert index[0] == 0 and dist[0] == 0.5
    assert (visited, considered) == (2, 2)
    ridx, rdist, ties = nearest_reference(X, Q)
    assert ridx[0] == 0 and rdist[0] == 0.25 and ties[0] == 2


@pytest.mark.gpu
def test_nearest_frames_uniform_d10_defeats_pruning_but_stays_exact(dev):
    rng = np.random.default_rng(9)
    X, Q = rng.uniform(-1, 1, (20000, 10)), rng.uniform(-1, 1, (3000, 10))
    index, dist, (visited, considered) = device_nearest(dev, X, Q, counters=True)
    ridx, rdist, _ = nearest_reference(X, Q)
    assert np.array_equal(index, ridx) and np.array_equal(dist, np.sqrt(rdist))
    check_against_kd_tree(X, Q, index, dist)
    assert visited <= considered


@pytest.mark.gpu
def test_nearest_frames_million_frames(dev):
    """N = 1e6 frames, M = 1e5 queries of a 4-decimal walk: every distance bitwise the KD-tree's, every index the
    KD-tree's or an exactly tied lower one, and a seeded sample of queries checked against all frames with the
    restatement."""
    W = random_walk(1100000, 3, 12, decimals=4)
    X, Q = np.ascontiguousarray(W[:1000000]), np.ascontiguousarray(W[1000000:])
    index, dist = device_nearest(dev, X, Q)
    check_against_kd_tree(X, Q, index, dist)
    sample = np.random.default_rng(0).choice(Q.shape[0], 300, replace=False)
    ridx, rdist, _ = nearest_reference(X, Q[sample], chunk=20)
    assert np.array_equal(index[sample], ridx)
    assert np.array_equal(dist[sample], np.sqrt(rdist))


@pytest.mark.gpu
@pytest.mark.parametrize("d", [2, 4, 10])
def test_nearest_frames_order_independent(dev, d):
    """On tie-free data, permuting the frames and the queries permutes the answer exactly."""
    rng = np.random.default_rng(20 + d)
    X, Q = rng.standard_normal((5000, d)), rng.standard_normal((1500, d))
    index, dist = device_nearest(dev, X, Q)
    px, pq = rng.permutation(5000), rng.permutation(1500)
    index2, dist2 = device_nearest(dev, np.ascontiguousarray(X[px]), np.ascontiguousarray(Q[pq]))
    assert np.array_equal(px[index2], index[pq])
    assert np.array_equal(dist2, dist[pq])


@pytest.mark.gpu
def test_nearest_frames_float32_widened_exactly(dev):
    from deep_cartograph_b200 import ops
    rng = np.random.default_rng(5)
    X = torch.from_numpy(rng.standard_normal((3000, 3)).astype(np.float32)).to(dev)
    Q = torch.from_numpy(rng.standard_normal((700, 3)).astype(np.float32)).to(dev)
    i32, d32 = ops.nearest_frames(X, Q)
    i64, d64 = ops.nearest_frames(X.double(), Q.double())
    assert torch.equal(i32, i64) and torch.equal(d32, d64)


@pytest.mark.gpu
def test_nearest_frames_workspace_is_linear_and_checked(dev):
    from deep_cartograph_b200 import _lib
    lib = _lib.load()
    small = lib.dcg_nearest_frames_workspace_bytes(100000, 10000, 4)
    big = lib.dcg_nearest_frames_workspace_bytes(1000000, 100000, 4)
    assert 0 < small and big < 12 * small                # O(n + m), no n x m buffer
    X = torch.zeros((1000, 4), dtype=torch.float64, device=dev)
    out = torch.empty(10, dtype=torch.float64, device=dev)
    idx = torch.empty(10, dtype=torch.int64, device=dev)
    need = lib.dcg_nearest_frames_workspace_bytes(1000, 10, 4)
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    args = (X.data_ptr(), 1000, 4, X.data_ptr(), 10, 4, 4, idx.data_ptr(), out.data_ptr())
    assert lib.dcg_nearest_frames_f64(*args, ws.data_ptr(), need - 1, None) == -1002
    assert lib.dcg_nearest_frames_f64(*args, None, need, None) == -1002
    torch.cuda.synchronize()


def _labels_case():
    rng = np.random.default_rng(31)
    cent = rng.uniform(-1, 1, (6, 3))
    X = cent[rng.integers(0, 6, 3000)] + 0.12 * rng.standard_normal((3000, 3))
    S = cent[rng.integers(0, 6, 800)] + 0.2 * rng.standard_normal((800, 3))
    return np.ascontiguousarray(X), np.ascontiguousarray(S)


@pytest.mark.gpu
@pytest.mark.parametrize("algorithm", ["kmeans", "hierarchical", "hdbscan"])
def test_assign_closest_cluster_equals_sklearn_restatement(dev, algorithm):
    from sklearn.neighbors import NearestNeighbors
    from deep_cartograph_b200.modules.statistics import statistics
    X, S = _labels_case()
    if algorithm == "kmeans":
        labels, _ = statistics.kmeans_clustering(X, 6, 2)
    elif algorithm == "hierarchical":
        labels, _ = statistics.hierarchical_clustering(X, 6, "complete")
    else:
        labels, _ = statistics.hdbscan_clustering(X, {"min_cluster_size": 30, "min_samples": 10})
        assert (labels < 0).any() and labels.max() >= 1                  # noise is present and propagates
    sup = statistics.assign_closest_cluster(X, labels, S)
    idx = NearestNeighbors(n_neighbors=1).fit(X).kneighbors(S)[1][:, 0]
    assert np.array_equal(sup, labels[idx])
    assert sup.dtype == labels.dtype


@pytest.mark.gpu
@pytest.mark.parametrize("cv", ["pca", "tica"])
def test_traj_cluster_supplementary_golden(dev, c1, cv, tmp_path):
    """traj_cluster on a golden CV set with a perturbed copy as the supplementary trajectory: the supplementary
    CSV has the main layout and the labels of the nearest clustered frames, and the main CSV is byte for byte
    the one written without it."""
    from sklearn.neighbors import NearestNeighbors
    from deep_cartograph_b200.tools import traj_cluster
    cols = list(c1[f"{cv}_csv_cols"])
    X = c1[f"{cv}_cluster_cv"]
    csv, sup = tmp_path / f"{cv}.csv", tmp_path / f"{cv}_sup.csv"
    _write_cv(csv, X, cols)
    _write_cv(sup, X + 0.01 * np.random.default_rng(2).standard_normal(X.shape), cols)
    conf = {"backend": {"hierarchical_on_device": True}}
    plain = traj_cluster(dict(conf), [str(csv)], output_folder=str(tmp_path / "plain"))
    out = traj_cluster(dict(conf), [str(csv)], sup_cv_traj_paths=[str(sup)], sup_trajectories=["/md/extra.xtc"],
                       frames_per_sample=5, output_folder=str(tmp_path / "with_sup"))
    out1 = traj_cluster(dict(conf), [str(csv)], frames_per_sample=5, output_folder=str(tmp_path / "plain5"))
    assert set(out) == {"traj_0", "extra"} and set(plain) == {"traj_0"}
    with open(out["traj_0"][0], "rb") as a, open(out1["traj_0"][0], "rb") as b:
        assert a.read() == b.read()
    main = pd.read_csv(out["traj_0"][0])
    assert np.array_equal(pd.read_csv(plain["traj_0"][0])["cluster"].to_numpy(), main["cluster"].to_numpy())
    df = pd.read_csv(out["extra"][0])
    assert list(df.columns) == cols + ["traj_label", "cluster", "centroid", "frame"]
    assert not df["centroid"].any()
    assert np.array_equal(df["frame"].to_numpy(), 5 * np.arange(len(df)))
    assert np.array_equal(df["traj_label"].to_numpy(), np.zeros(len(df)))
    Xm, Xs = main[cols].to_numpy(), df[cols].to_numpy()
    idx = NearestNeighbors(n_neighbors=1, algorithm="kd_tree").fit(Xm).kneighbors(Xs)[1][:, 0]
    ridx, _, ties = nearest_reference(Xm, Xs)
    assert np.array_equal(df["cluster"].to_numpy(), main["cluster"].to_numpy()[ridx])
    unique = ties == 1
    assert np.array_equal(ridx[unique], idx[unique])
