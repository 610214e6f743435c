"""Exact silhouette of several labelings in one device pass (csrc/silhouette.cu, ops.silhouette,
statistics.silhouette / silhouettes, optimize_clustering, traj_cluster's silhouette_max_samples).

The device computes scikit-learn's silhouette_samples / silhouette_score (Euclidean) with pdist's distance
arithmetic: d(i, j) = sqrt(sum_f (x_f - y_f)^2), features ascending, one rounded subtract, multiply and add per
term.  scikit-learn itself uses the |x|^2 + |y|^2 - 2 x.y expansion, which loses accuracy far from the origin, so
the device is compared frame by frame with a numpy restatement (pdist arithmetic, long-double cluster sums), and
with scikit-learn through the mean score only.

Error bound.  A cluster sum of m non-negative distances, added in any order, is within gamma_m = m u / (1 - m u)
of the exact sum of the same (identically rounded) distances, u = 2^-53.  a_i and b_i add one rounded division:
relative error rho = (1 + gamma_M)(1 + u) - 1, M the largest cluster.  s_i = +-(1 - min/max) then moves by at
most 2 rho / (1 - rho), and the rounded subtract and divide of the kernel add 2.1 u; one more u covers the
rounding of the restatement's long-double s_i to float64."""
import ctypes

import numpy as np
import pandas as pd
import pytest
import torch

U = 2.0 ** -53
ROW_BLOCK = 64             # rows of one CTA (kRows, csrc/silhouette.cu)
MAX_SLOTS = 384            # DCG_SILHOUETTE_MAX_SLOTS


def random_walk(n, d, seed, step=0.05):
    rng = np.random.default_rng(seed)
    return np.ascontiguousarray(np.cumsum(step * rng.standard_normal((n, d)), axis=0))


def pdist_rows(X, rows):
    """Distances of the frames ``rows`` to every frame, with pdist's arithmetic (numpy's subtract, multiply and
    add are single correctly rounded operations)."""
    s = np.zeros((len(rows), X.shape[0]))
    for f in range(X.shape[1]):
        t = X[rows, f, None] - X[None, :, f]
        s = s + t * t
    return np.sqrt(s)


def encode(labels):
    _, inv = np.unique(np.asarray(labels), return_inverse=True)
    return inv.reshape(-1)


def cluster_sums(X, labels, chunk=512):
    """(n, k) long-double sums of the pdist distances of every frame to the members of every cluster."""
    inv = encode(labels)
    k = inv.max() + 1
    n = X.shape[0]
    out = np.zeros((n, k), dtype=np.longdouble)
    for a in range(0, n, chunk):
        D = pdist_rows(X, np.arange(a, min(n, a + chunk))).astype(np.longdouble)
        for c in range(k):
            out[a:a + chunk, c] = D[:, inv == c].sum(axis=1)
    return out, inv


def silhouette_from_sums(S, inv):
    """sklearn's _silhouette_reduce + silhouette_samples finish on the cluster sums S (any float dtype):
    a = own / (n_own - 1), b = min over the other clusters of sum / size, s = (b - a) / max(a, b), NaN -> 0."""
    n, k = S.shape
    sizes = np.bincount(inv, minlength=k).astype(S.dtype)
    rows = np.arange(n)
    with np.errstate(divide="ignore", invalid="ignore"):
        a = S[rows, inv] / (sizes[inv] - 1)
        M = S / sizes[None, :]
        M[rows, inv] = np.inf
        b = M.min(axis=1)
        s = (b - a) / np.maximum(a, b)
    return np.nan_to_num(s)


def restatement(X, labels):
    S, inv = cluster_sums(np.asarray(X, dtype=np.float64), labels)
    return silhouette_from_sums(S, inv), np.bincount(inv).max()


def bound(M):
    g = M * U / (1 - M * U)
    rho = (1 + g) * (1 + U) - 1
    return 2 * rho / (1 - rho) + 4 * U


def offset_duplicates():
    """2-decimal frames offset by 50 with 188 duplicated frames: far from the origin, where scikit-learn's
    expansion differs from direct differences, and with a = b = 0 frames when duplicates are split."""
    rng = np.random.default_rng(11)
    X = np.round(rng.uniform(-1, 1, (1500, 3)), 2) + 50.0
    X = np.concatenate([X, X[rng.choice(1500, 188, replace=False)]])
    lab = rng.integers(0, 4, X.shape[0])
    return np.ascontiguousarray(X), lab


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["blobs", "walk_d4", "walk_singletons"])
def test_restatement_equals_sklearn_per_frame(case):
    from sklearn.metrics import silhouette_samples
    rng = np.random.default_rng(3)
    if case == "blobs":
        cent = rng.uniform(-1, 1, (5, 2))
        X = cent[rng.integers(0, 5, 1200)] + 0.1 * rng.standard_normal((1200, 2))
        lab = rng.integers(0, 5, 1200)
    else:
        X = random_walk(1000, 4 if case == "walk_d4" else 2, 5)
        lab = np.repeat(np.arange(10), 100)
        if case == "walk_singletons":
            lab[[0, 500, 999]] = [20, 21, 22]
    s, _ = restatement(X, lab)
    assert np.abs(s.astype(np.float64) - silhouette_samples(X, lab)).max() <= 1e-12


def test_restatement_mean_equals_sklearn_on_offset_duplicates():
    from sklearn.metrics import silhouette_score
    X, lab = offset_duplicates()
    s, _ = restatement(X, lab)
    assert abs(float(s.astype(np.float64).mean()) - silhouette_score(X, lab)) <= 1e-9


def test_silhouette_argument_errors_without_gpu():
    from deep_cartograph_b200 import _lib
    lib = _lib.load()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    big = 1 << 30
    f = lib.dcg_silhouette_f64
    # Y, n, d, ld, labels, L, offsets, sizes, K, scores, samples, ws, ws_bytes, stream
    assert f(p, 2, 2, 2, p, 1, p, p, 2, p, None, p, big, None) == -1001             # n < 3
    assert f(p, 10, 0, 2, p, 1, p, p, 2, p, None, p, big, None) == -1001            # d < 1
    assert f(p, 10, 2, 1, p, 1, p, p, 2, p, None, p, big, None) == -1001            # ld < d
    assert f(p, 10, 2, 2, p, 0, p, p, 2, p, None, p, big, None) == -1001            # L < 1
    assert f(p, 10, 2, 2, p, 33, p, p, 66, p, None, p, big, None) == -1001          # L above 32
    assert f(p, 10, 2, 2, p, 2, p, p, 3, p, None, p, big, None) == -1001            # K < 2 L
    assert f(p, 1000, 2, 2, p, 2, p, p, MAX_SLOTS + 1, p, None, p, big, None) == -1001   # K above the cap
    assert f(p, 10, 2049, 2049, p, 1, p, p, 2, p, None, p, big, None) == -1001      # d above 2048
    assert f(None, 10, 2, 2, p, 1, p, p, 2, p, None, p, big, None) == -1000
    assert f(p, 10, 2, 2, None, 1, p, p, 2, p, None, p, big, None) == -1000
    assert f(p, 10, 2, 2, p, 1, None, p, 2, p, None, p, big, None) == -1000
    assert f(p, 10, 2, 2, p, 1, p, None, 2, p, None, p, big, None) == -1000
    assert f(p, 10, 2, 2, p, 1, p, p, 2, None, None, p, big, None) == -1000
    need = lib.dcg_silhouette_workspace_bytes(10, 1, 2)
    assert need > 0
    assert f(p, 10, 2, 2, p, 1, p, p, 2, p, None, p, need - 1, None) == -1002        # workspace too small
    assert f(p, 10, 2, 2, p, 1, p, p, 2, p, None, None, need, None) == -1002
    assert lib.dcg_silhouette_workspace_bytes(2, 1, 2) == 0
    assert lib.dcg_silhouette_workspace_bytes(10, 1, MAX_SLOTS + 1) == 0
    # O(n (d + L)): ten times the frames, about ten times the workspace
    assert lib.dcg_silhouette_workspace_bytes(10 ** 7, 8, 52) < 11 * lib.dcg_silhouette_workspace_bytes(10 ** 6, 8, 52)


def test_ops_silhouette_validation_without_gpu(monkeypatch):
    from deep_cartograph_b200 import ops
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        ops.silhouette(torch.zeros((4, 2)), torch.tensor([0, 0, 1, 1]))
    monkeypatch.setattr(ops, "_need_cuda", lambda *a, **k: None)
    monkeypatch.setattr(ops, "_ws", lambda *a, **k: (_ for _ in ()).throw(AssertionError("allocated")))
    Y = torch.rand((6, 2), dtype=torch.float64)
    with pytest.raises(ValueError, match="Number of labels is 1"):
        ops.silhouette(Y, torch.zeros(6, dtype=torch.int64))
    with pytest.raises(ValueError, match="Number of labels is 6"):
        ops.silhouette(Y, torch.arange(6))
    with pytest.raises(ValueError, match="Number of labels is 1"):                 # the second labeling
        ops.silhouette(Y, [torch.tensor([0, 0, 1, 1, 2, 2]), torch.full((6,), 7)])
    Yn = Y.clone()
    Yn[3, 1] = float("nan")
    with pytest.raises(ValueError, match="NaN or infinity"):
        ops.silhouette(Yn, torch.tensor([0, 0, 1, 1, 2, 2]))
    with pytest.raises(ValueError, match="one label per frame"):
        ops.silhouette(Y, torch.tensor([0, 0, 1, 1, 2]))
    with pytest.raises(TypeError, match="integers"):
        ops.silhouette(Y, torch.tensor([0.0, 0, 1, 1, 2, 2]))


def test_silhouette_groups_fit_the_slot_cap():
    from deep_cartograph_b200.ops import _silhouette_groups
    ks = list(range(2, 41))
    groups = _silhouette_groups(ks)
    assert [i for g in groups for i in g] == list(range(len(ks)))
    assert all(sum(ks[i] for i in g) <= MAX_SLOTS and len(g) <= 32 for g in groups) and len(groups) > 1
    assert _silhouette_groups(list(range(3, 11))) == [list(range(8))]            # [3, 10]: K = 52, one pass
    assert _silhouette_groups(list(range(2, 16))) == [list(range(14))]           # [2, 15]: K = 119, one pass
    assert _silhouette_groups([2] * 40) == [list(range(32)), list(range(32, 40))]


def test_schema_silhouette_max_samples():
    from deep_cartograph_b200.yaml_schemas.traj_cluster import TrajClusterSchema
    assert TrajClusterSchema().model_dump()["silhouette_max_samples"] == 50000
    assert TrajClusterSchema(silhouette_max_samples=None).silhouette_max_samples is None
    assert TrajClusterSchema(silhouette_max_samples=1000).silhouette_max_samples == 1000


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from deep_cartograph_b200 import _lib
    _lib.load()            # fail loudly if the extension is missing
    return torch.device("cuda:0")


def device_silhouette(dev, X, labelings):
    from deep_cartograph_b200 import ops
    Y = torch.from_numpy(np.ascontiguousarray(X)).to(dev)
    labs = [torch.from_numpy(np.asarray(lab)).to(dev) for lab in labelings]
    scores, samples = ops.silhouette(Y, labs, return_samples=True)
    return scores.cpu().numpy(), samples.cpu().numpy()


def check_per_frame(dev, X, labelings):
    scores, samples = device_silhouette(dev, X, labelings)
    for l, lab in enumerate(labelings):
        s, M = restatement(np.asarray(X, dtype=np.float64), lab)
        err = np.abs(samples[l] - s.astype(np.float64))
        assert err.max() <= bound(M), (l, err.max(), bound(M), np.argmax(err))
        assert abs(scores[l] - float(s.astype(np.float64).mean())) <= bound(M) + 1e-15
    return scores, samples


@pytest.mark.gpu
def test_exact_lattice_is_bitwise_the_formula(dev):
    """Integer frames, d = 1: every distance and every cluster sum is an exact integer, so s_i must be bitwise
    the float64 formula on the exact sums."""
    rng = np.random.default_rng(1)
    X = rng.integers(-60, 60, (700, 1)).astype(np.float64)
    labs = [rng.integers(0, 5, 700), np.repeat(np.arange(7), 100), rng.integers(0, 40, 700)]
    labs[1][[5, 250]] = [7, 8]                                          # singletons
    _, samples = device_silhouette(dev, X, labs)
    D = np.abs(X[:, 0, None].astype(np.int64) - X[None, :, 0].astype(np.int64))
    for l, lab in enumerate(labs):
        inv = encode(lab)
        k = inv.max() + 1
        S = np.stack([D[:, inv == c].sum(axis=1) for c in range(k)], axis=1).astype(np.float64)    # exact
        assert np.array_equal(samples[l], silhouette_from_sums(S, inv)), l


def _labels(rng, n, k):
    lab = rng.integers(0, k, n)
    lab[:k] = np.arange(k)                                            # every cluster present
    return lab


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 2, 3, 4, 10, 16])
@pytest.mark.parametrize("n", [3, ROW_BLOCK - 1, ROW_BLOCK, ROW_BLOCK + 1, 2 * ROW_BLOCK + 3, 1000])
def test_per_frame_against_restatement(dev, d, n):
    rng = np.random.default_rng(100 * d + n)
    X = rng.standard_normal((n, d)) * 3.0
    labs = [_labels(rng, n, 2), _labels(rng, n, min(n - 1, 7)), _labels(rng, n, min(n - 1, MAX_SLOTS))]   # k = n - 1, the cap
    check_per_frame(dev, X, labs)


@pytest.mark.gpu
def test_per_frame_walk_runs_singletons_and_20k_frames(dev):
    X = random_walk(20000, 2, 7)
    runs = np.repeat(np.arange(10), 2000)                               # long label runs (run accumulation)
    lab2 = runs.copy()
    lab2[[0, 7777, 19999]] = [30, 31, 32]                               # singletons inside and at the ends
    check_per_frame(dev, X, [runs, lab2])


@pytest.mark.gpu
def test_duplicates_split_across_clusters_give_zero(dev):
    """Frames with a = b = 0 (identical frames in two clusters, each cluster one point repeated): 0/0 -> 0."""
    X, lab = offset_duplicates()
    dup = np.zeros((40, 2))
    dup[20:] = 1.0
    lab_dup = np.array([0] * 10 + [1] * 10 + [2] * 10 + [3] * 10)      # clusters 0, 1 at (0, 0); 2, 3 at (1, 1)
    check_per_frame(dev, X, [lab])
    _, samples = check_per_frame(dev, dup, [lab_dup])
    assert np.all(samples == 0.0)


@pytest.mark.gpu
def test_noncontiguous_negative_labels_and_float32(dev):
    from deep_cartograph_b200 import ops
    rng = np.random.default_rng(9)
    X = random_walk(3000, 3, 2)
    lab = rng.choice(np.array([-1, 7, 100, 3]), 3000)
    scores, samples = check_per_frame(dev, X, [lab])
    s_enc, smp_enc = device_silhouette(dev, X, [encode(lab)])
    assert np.array_equal(scores, s_enc) and np.array_equal(samples, smp_enc)
    X32 = torch.from_numpy(X.astype(np.float32)).to(dev)
    lab_t = torch.from_numpy(lab).to(dev)
    a, sa = ops.silhouette(X32, lab_t, return_samples=True)
    b, sb = ops.silhouette(X32.double(), lab_t, return_samples=True)
    assert torch.equal(a, b) and torch.equal(sa, sb)


@pytest.mark.gpu
@pytest.mark.parametrize("cv", ["pca", "tica", "htica"])
def test_mean_equals_sklearn_on_golden_cv_sets(dev, c1, cv):
    from sklearn.metrics import silhouette_score
    from deep_cartograph_b200.modules.statistics import statistics
    X = np.ascontiguousarray(c1[f"{cv}_cluster_cv"], dtype=np.float64)
    labs = [statistics.hierarchical_clustering(X, k, "complete")[0] for k in range(3, 11)]
    got = statistics.silhouettes(X, labs)
    for g, lab in zip(got, labs):
        assert abs(g - silhouette_score(X, lab)) <= 1e-9


@pytest.mark.gpu
def test_mean_equals_sklearn_on_kmeans_ref(dev, kmeans_ref):
    from sklearn.metrics import silhouette_score
    from deep_cartograph_b200.modules.statistics import statistics
    X = kmeans_ref["opt_X"]
    labs = [statistics.kmeans_clustering(X.copy(), k, 1)[0] for k in range(2, 9)]
    got = statistics.silhouettes(X, labs)
    for g, lab in zip(got, labs):
        assert abs(g - silhouette_score(X, lab)) <= 1e-9


@pytest.mark.gpu
def test_mean_equals_sklearn_on_50k_blobs(dev):
    from sklearn.metrics import silhouette_score
    from deep_cartograph_b200.modules.statistics import statistics
    rng = np.random.default_rng(12)
    cent = rng.uniform(-1, 1, (6, 2))
    near = rng.integers(0, 6, 50000)
    X = cent[near] + 0.15 * rng.standard_normal((50000, 2))
    labs = [near, near % 3]
    got = statistics.silhouettes(X, labs)
    for g, lab in zip(got, labs):
        assert abs(g - silhouette_score(X, lab)) <= 1e-9


@pytest.mark.gpu
def test_grouping_and_runs_are_bitwise_reproducible(dev):
    """One call over L labelings == L single calls, bit for bit (each labeling tracks its own label runs), two
    runs are equal, and an interval whose slots exceed the kernel's cap (k = 2..40: 819 slots, several passes)
    gives the per-labeling results."""
    from deep_cartograph_b200 import ops
    from deep_cartograph_b200.modules.statistics import statistics
    X = random_walk(3000, 2, 21)
    tree = statistics.linkage_tree(X, "complete")
    labs = [statistics.cut_tree(tree, k) for k in range(2, 41)]
    Y = torch.from_numpy(X).to(dev)
    lt = [torch.from_numpy(lab).to(dev) for lab in labs]
    all_s, all_smp = ops.silhouette(Y, lt, return_samples=True)
    again_s, again_smp = ops.silhouette(Y, lt, return_samples=True)
    assert torch.equal(all_s, again_s) and torch.equal(all_smp, again_smp)
    for l, lab in enumerate(lt):
        one_s, one_smp = ops.silhouette(Y, lab, return_samples=True)
        assert torch.equal(one_s[0], all_s[l]) and torch.equal(one_smp[0], all_smp[l]), l
    eight_s, eight_smp = ops.silhouette(Y, lt[1:9], return_samples=True)          # [3, 10] in one pass
    assert torch.equal(eight_s, all_s[1:9]) and torch.equal(eight_smp, all_smp[1:9])
    s, _ = restatement(X, labs[5])
    assert np.abs(all_smp[5].cpu().numpy() - s.astype(np.float64)).max() <= bound(np.bincount(labs[5]).max())


@pytest.mark.gpu
def test_large_n_against_chunked_torch_restatement(dev):
    """2e5 frames of a walk, shuffled rows (short label runs), against a chunked torch FP64 direct-difference
    restatement on the device; both sides are bounded by gamma_n."""
    from deep_cartograph_b200 import ops
    n = 200000
    rng = np.random.default_rng(4)
    X = random_walk(n, 3, 13)[rng.permutation(n)]
    Y = torch.from_numpy(np.ascontiguousarray(X)).to(dev)
    labs = [torch.from_numpy(((X[:, 0] > np.median(X[:, 0])) * 2 + (X[:, 1] > 0)).astype(np.int64)).to(dev),
            torch.from_numpy(rng.integers(0, 5, n)).to(dev)]
    _, samples = ops.silhouette(Y, labs, return_samples=True)
    for l, lab in enumerate(labs):
        k = int(lab.max()) + 1
        onehot = torch.nn.functional.one_hot(lab, k).to(torch.float64)
        sizes = onehot.sum(0)
        ref = torch.empty(n, dtype=torch.float64, device=dev)
        for a in range(0, n, 2048):
            e = min(n, a + 2048)
            s = torch.zeros((e - a, n), dtype=torch.float64, device=dev)
            for f in range(3):
                t = Y[a:e, f, None] - Y[None, :, f]
                s = s + t * t
            S = torch.sqrt(s) @ onehot
            rows = torch.arange(e - a, device=dev)
            own = lab[a:e]
            A = S[rows, own] / (sizes[own] - 1)
            M = S / sizes[None, :]
            M[rows, own] = float("inf")
            B = M.min(dim=1).values
            ref[a:e] = torch.nan_to_num((B - A) / torch.maximum(A, B))
        err = (samples[l] - ref).abs().max().item()
        assert err <= 2 * bound(n), (l, err)


def _old_cdist_silhouette(X, labels, sample_size=None, seed=0, chunk=2048):
    """The torch.cdist routine statistics.silhouette used before the kernel (kept here as the yardstick for
    the sampled scores of optimize_clustering)."""
    Y = torch.from_numpy(np.asarray(X, dtype=np.float64)).cuda()
    lab = torch.as_tensor(np.asarray(labels), device=Y.device).long()
    n = Y.shape[0]
    if sample_size is not None and sample_size < n:
        idx = torch.from_numpy(np.random.RandomState(seed).permutation(n)[:sample_size]).to(Y.device)
        Y, lab = Y[idx], lab[idx]
        n = sample_size
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


@pytest.fixture(scope="module")
def frames_55k():
    rng = np.random.default_rng(55)
    cent = rng.uniform(-1, 1, (5, 2))
    X = cent[rng.integers(0, 5, 55000)] + 0.2 * rng.standard_normal((55000, 2))
    return np.ascontiguousarray(np.round(X, 4))


@pytest.mark.gpu
def test_optimize_clustering_exact_above_the_old_cap(dev, frames_55k, monkeypatch):
    """silhouette_max_samples None on 55k frames: one silhouette pass for the whole search, and the same k,
    labels and centres as the selection rule applied to scikit-learn's silhouette_score and the CH / DB."""
    from sklearn.metrics import silhouette_score
    from deep_cartograph_b200 import ops
    from deep_cartograph_b200.modules.statistics import statistics
    X = frames_55k
    calls = []
    real = ops.silhouette

    def counted(*a, **k):
        calls.append(1)
        return real(*a, **k)
    monkeypatch.setattr(ops, "silhouette", counted)
    settings = {"algorithm": "kmeans", "search_interval": [3, 5], "n_init": 1, "silhouette_max_samples": None}
    labels, centers = statistics.optimize_clustering(X.copy(), settings)
    assert len(calls) == 1
    rep = statistics.last_optimize_report
    fits = [statistics.kmeans_clustering(X.copy(), k, 1) for k in rep["k"]]
    sil = np.array([silhouette_score(X, lab) for lab, _ in fits])
    assert np.abs(np.array(rep["silhouette"]) - sil).max() <= 1e-9

    def norm(v):
        v = np.asarray(v, dtype=np.float64)
        return (v - v.min()) / (v.max() - v.min())
    best = int(np.argmax((norm(rep["calinski_harabasz"]) - norm(rep["davies_bouldin"]) + norm(sil)) / 3))
    assert rep["best_k"] == rep["k"][best]
    assert np.array_equal(labels, fits[best][0])
    np.testing.assert_allclose(centers, fits[best][1], rtol=1e-10, atol=1e-12)   # Lloyd's FP64 sum order


@pytest.mark.gpu
def test_optimize_clustering_sampled_scores_unchanged(dev, frames_55k):
    """With the default cap the 55k frames are scored on sklearn's 50k subsample, as before the kernel."""
    from deep_cartograph_b200.modules.statistics import statistics
    X = frames_55k
    settings = {"algorithm": "kmeans", "search_interval": [3, 5], "n_init": 1}
    statistics.optimize_clustering(X.copy(), settings)
    rep = statistics.last_optimize_report
    for k, s in zip(rep["k"], rep["silhouette"]):
        lab, _ = statistics.kmeans_clustering(X.copy(), k, 1)
        assert abs(s - _old_cdist_silhouette(X, lab, sample_size=50000)) <= 1e-12, k


@pytest.mark.gpu
@pytest.mark.parametrize("cv", ["pca", "tica", "htica"])
def test_traj_cluster_exact_silhouette_writes_the_default_csvs(dev, c1, cv, tmp_path):
    """Below 50k frames the default already scores every pair: silhouette_max_samples null changes no byte."""
    from deep_cartograph_b200.tools import traj_cluster
    cols = list(c1[f"{cv}_csv_cols"])
    csv = tmp_path / f"{cv}.csv"
    pd.DataFrame(c1[f"{cv}_cluster_cv"], columns=cols).to_csv(csv, index=False, float_format="%.4f")
    for algorithm in ("hierarchical", "kmeans"):
        conf = {"algorithm": algorithm, "backend": {"hierarchical_on_device": True}}
        a = traj_cluster(dict(conf), [str(csv)], output_folder=str(tmp_path / f"{algorithm}_default"))
        b = traj_cluster(dict(conf, silhouette_max_samples=None), [str(csv)],
                         output_folder=str(tmp_path / f"{algorithm}_exact"))
        with open(a["traj_0"][0], "rb") as fa, open(b["traj_0"][0], "rb") as fb:
            assert fa.read() == fb.read()
