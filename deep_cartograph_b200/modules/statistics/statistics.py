"""KMeans clustering in CV space on the B200 kernels.

Host-side mirror of the reference's ``modules/statistics/statistics.py`` for the KMeans path:
``cluster_data`` (:112-157), ``kmeans_clustering`` (:159-197), ``find_centroids`` (:337-379),
``optimize_clustering`` (:17-110, KMeans only, with the one-pass scores).  The Lloyd driver
reproduces scikit-learn's control flow (sklearn/cluster/_kmeans.py, ``algorithm='lloyd'``) so
that labels from fixed initial centroids are identical to the reference's:

  centre X by its column mean (:1486-1493); tol_eff = tol * mean(var(X, axis=0)) (:285-294);
  per iteration E-step (lowest index wins ties) + FP64 sums / counts; empty clusters relocated
  to the farthest points (_k_means_common.pyx:167-211); centres = sums * (1 / counts);
  stop when labels are unchanged ("strict") or sum ||dc||^2 <= tol_eff (:703-740); one more
  E-step when not strict (:742-754); centres returned un-centred.

Agglomerative clustering (reference ``hierarchical_clustering``, :285) runs on the device when
``settings["backend"]["hierarchical_on_device"]`` is true: ``linkage_tree`` builds the same merge tree as
scikit-learn (``ops.linkage``, csrc/linkage.cu), ``cut_tree`` restates sklearn's ``_hc_cut``, and
``optimize_clustering`` builds the tree once and cuts it for every k.

HDBSCAN runs on the device when ``settings["backend"]["hdbscan_on_device"]`` is true: ``hdbscan_tree``
builds sklearn's single-linkage tree from device core distances and a device mutual-reachability MST
(``ops.core_distances``, ``ops.mreach_mst``) in O(N) memory, and ``hdbscan_labels`` restates sklearn's
``tree_to_labels``.  Without its flag, either algorithm is reported as outside the hot path and the step
exits.
"""
from __future__ import annotations

import heapq
import logging
import sys
from typing import Dict, List, Optional, Tuple

import numpy as np
import pandas as pd
import torch

from ... import ops
from ...parallel import FrameShards

logger = logging.getLogger(__name__)

# set by the last kmeans_clustering call: iterations, strict convergence, tie counts ...
last_kmeans_report: Dict = {}


def _device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("deep_cartograph_b200 needs a CUDA device (B200); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _to_device(features) -> torch.Tensor:
    if isinstance(features, torch.Tensor):
        t = features
    else:
        t = torch.from_numpy(np.ascontiguousarray(features))
    if t.dtype not in (torch.float32, torch.float64):
        t = t.to(torch.float64)
    return t.to(_device()).contiguous()


def _kmeanspp_sklearn(Yc: torch.Tensor, k: int, rs: np.random.RandomState) -> torch.Tensor:
    """scikit-learn's greedy k-means++ (sklearn/cluster/_kmeans.py ``_kmeans_plusplus``, reached from
    reference statistics.py:189-195 with ``init='k-means++'``, ``random_state=0``) on the CENTRED frames
    ``Yc`` (KMeans.fit centres X first, _kmeans.py:1486-1493): the random draws come from the SAME numpy
    ``RandomState`` stream (first centre: ``choice(n, p=uniform)``; then ``2 + int(log k)`` uniform
    draws per centre against the cumulative D^2 potential), the O(n k) distance work runs on the device
    in FP64.  The centres equal scikit-learn's unless a draw lands within rounding of a cumulative-sum
    boundary."""
    n, d = Yc.shape
    Yd = Yc.to(torch.float64)
    n_trials = 2 + int(np.log(k))
    centers = torch.empty((k, d), dtype=torch.float64, device=Yc.device)
    if n <= 5_000_000:
        first = int(rs.choice(n, p=np.full(n, 1.0 / n)))
    else:      # the same draw without the n-vector: choice() searches u in cdf_i = (i + 1) / n -> floor(u n)
        first = min(n - 1, int(np.floor(rs.random_sample() * n)))
    centers[0] = Yd[first]
    closest = ((Yd - centers[0]) ** 2).sum(dim=1)
    pot = float(closest.sum().item())
    for c in range(1, k):
        rand_vals = torch.from_numpy(rs.uniform(size=n_trials) * pot).to(Yc.device)
        cand = torch.searchsorted(torch.cumsum(closest, 0), rand_vals).clamp_(max=n - 1)
        dist = torch.stack([((Yd - Yd[i]) ** 2).sum(dim=1) for i in cand])
        dist = torch.minimum(dist, closest[None, :])
        pots = dist.sum(dim=1)
        best = int(torch.argmin(pots).item())
        pot = float(pots[best].item())
        closest = dist[best]
        centers[c] = Yd[cand[best]]
    return centers


# Lloyd iterations enqueued per host read on one device (dcg_kmeans_iterate_n)
_LLOYD_BATCH = 4


def kmeans_lloyd(Y: torch.Tensor, init_centers: torch.Tensor, max_iter: int = 300, tol: float = 1e-4,
                 shards: Optional[FrameShards] = None, want_gap: bool = False) -> Dict:
    """Lloyd iterations on the device; ``Y`` is this rank's (frames x d) shard (float32/64),
    ``init_centers`` (k x d).  Returns dict(labels, centers, n_iter, strict, inertia, ties, gap)."""
    dev = Y.device
    n, d = Y.shape
    k = init_centers.shape[0]
    C = init_centers.to(dev, torch.float64).clone()

    # centre by the (global) column mean; tolerance from the (global) column variances
    st_n = torch.tensor([float(n)], dtype=torch.float64, device=dev)
    s1 = Y.sum(dim=0, dtype=torch.float64)
    if shards is not None:
        packed = shards.allreduce_sum_(torch.cat([st_n, s1]))
        st_n, s1 = packed[:1], packed[1:]
    n_tot = float(st_n.item())
    x_mean = s1 / n_tot
    Yc = (Y - x_mean.to(Y.dtype)).contiguous()
    s2 = (Yc.to(torch.float64) ** 2).sum(dim=0)
    sc = Yc.sum(dim=0, dtype=torch.float64)
    if shards is not None:
        packed = shards.allreduce_sum_(torch.cat([s2, sc]))
        s2, sc = packed[:d], packed[d:]
    var = s2 / n_tot - (sc / n_tot) ** 2
    tol_eff = float(var.mean().item()) * tol
    C = C - x_mean
    # bound on |Yc| of this shard: lets the E-step accumulate its partial sums in exact 64-bit
    # fixed point (native shared-memory integer adds) instead of FP64 compare-and-swap loops
    absmax = Yc.abs().amax().to(torch.float64).reshape(1) if n > 0 else None

    labels = torch.full((n,), -1, dtype=torch.int32, device=dev)
    strict = False
    n_iter = 0
    res = None
    C = C.contiguous()
    work = ops.kmeans_work(k, d, dev)
    it = 0
    while it < max_iter:
        if shards is None:
            # single device: up to _LLOYD_BATCH whole iterations (zero + E-step + FP64 sums + M-step finish each)
            # per library call; the convergence tests run on the device and the launches after the stopping
            # iteration are no-ops, so the state is the one a one-at-a-time loop would have stopped in
            res = ops.kmeans_iterate_n_(Yc, C, labels, work, min(_LLOYD_BATCH, max_iter - it), tol_eff, absmax=absmax)
            sums, counts = res["sums"], res["counts"]
            changed, _, _, n_empty, shift_tot, _, done, _ = work[k * d + k:k * d + k + 8].tolist()   # ONE host read
            it += int(done)
        else:
            # [sums | counts | stats] land in one buffer and are all-reduced in place
            res = ops.kmeans_step_packed_(Yc, C, labels, work, absmax=absmax)
            shards.allreduce_sum_(res["packed"])
            sums, counts = res["sums"], res["counts"]
            # M-step finish on the device (centres updated in place unless a cluster is empty);
            # ONE host read per iteration: [changed, inertia, ties, n_empty, shift]
            ops.kmeans_update_(C, sums, counts, info=work[k * d + k + 3:k * d + k + 5])
            changed, _, _, n_empty, shift_tot = work[k * d + k:k * d + k + 5].tolist()
            it += 1
        if n_empty > 0:
            empty = torch.nonzero(counts == 0).flatten()
            sums, counts = _relocate_empty(Yc, C, labels, sums, counts, empty, shards)
            C_new = C.clone()
            nz = counts > 0
            C_new[nz] = sums[nz] * (1.0 / counts[nz]).unsqueeze(1)
            shift_tot = float(((C_new - C) ** 2).sum().item())
            C = C_new
        n_iter = it
        if changed == 0:
            strict = True
            break
        if shift_tot <= tol_eff:
            break
    # final E-step with the final centres when not strictly converged (labels consistent with C)
    if not strict:
        res = ops.kmeans_step(Yc, C, labels, update_sums=False, want_gap=want_gap)
    elif want_gap:
        res = ops.kmeans_step(Yc, C, labels, update_sums=False, want_gap=True)
    stats = res["stats"]
    if shards is not None:
        stats = shards.allreduce_sum_(stats.clone())
    return {"labels": labels, "centers": C + x_mean, "n_iter": n_iter, "strict": strict,
            "inertia": float(stats[1].item()), "ties": int(stats[2].item()), "gap": res.get("gap"),
            "tol_eff": tol_eff}


def _relocate_empty(Yc, C, labels, sums, counts, empty, shards):
    """sklearn _relocate_empty_clusters_dense (sklearn/cluster/_k_means_common.pyx:167-211, reached from
    reference statistics.py:189-195): the n_empty frames farthest from their centres become the new
    centres of the empty clusters (in index order of the empty clusters), and leave their old ones.
    Labels are left untouched, as in sklearn.  Rare path, torch ops on the device.

    Frame-sharded: ``sums`` / ``counts`` are the already all-reduced (replicated) global ones; every
    rank offers its n_empty farthest frames (distance, old label, coordinates), the candidates are
    all-gathered, and every rank applies the same global top-n_empty -- ties go to the lower rank,
    then the lower local index, i.e. the lower GLOBAL frame index of the contiguous shards."""
    n_empty = int(empty.numel())
    n, d = Yc.shape
    dev = Yc.device
    dist = ((Yc.to(torch.float64) - C[labels.long()]) ** 2).sum(dim=1)
    m = min(n_empty, n)
    top = torch.topk(dist, m, largest=True, sorted=True) if m > 0 else None
    # candidates: [distance | old label | coordinates], best first; stable for equal distances
    cand = torch.full((n_empty, 2 + d), float("-inf"), dtype=torch.float64, device=dev)
    if m > 0:
        far = top.indices
        order = torch.argsort(far)                                  # equal distances: lower index first
        far = far[order][torch.argsort(-dist[far[order]], stable=True)]
        cand[:m, 0] = dist[far]
        cand[:m, 1] = labels[far].to(torch.float64)
        cand[:m, 2:] = Yc[far].to(torch.float64)
    if shards is not None and shards.world > 1:
        allc = torch.empty((shards.world * n_empty, 2 + d), dtype=torch.float64, device=dev)
        torch.distributed.all_gather_into_tensor(allc, cand.contiguous(), group=shards.group)
        # rank-major order + stable sort = ties to the lower global frame index
        pick = torch.argsort(-allc[:, 0], stable=True)[:n_empty]
        cand = allc[pick]
    sums = sums.clone()
    counts = counts.clone()
    rows = cand.tolist()
    for idx in range(n_empty):
        new_id = int(empty[idx].item())
        if rows[idx][0] == float("-inf"):
            break                                                   # fewer frames than empty clusters
        old_id = int(rows[idx][1])
        x = cand[idx, 2:]
        sums[old_id] -= x
        sums[new_id] = x
        counts[new_id] = 1.0
        counts[old_id] -= 1.0
    return sums, counts


def kmeans_clustering(feature_matrix, num_clusters: int, n_init: int,
                      initial_centroids=None) -> Tuple[np.ndarray, np.ndarray]:
    """Reference statistics.py:159-197: ``KMeans(n_clusters, random_state=0, init, n_init).fit_predict``.
    With ``initial_centroids`` the number of clusters comes from their shape and a single run is made (as
    sklearn does for an ndarray init); otherwise ``n_init`` k-means++ seedings drawn from ONE
    ``RandomState(0)`` stream as sklearn draws them, and the run with the lowest inertia wins (a later
    run replaces the best only if its inertia is lower and its clustering differs, _kmeans.py:1516-1530)."""
    global last_kmeans_report
    logger.debug("Clustering frames with kmeans...")
    Y = _to_device(feature_matrix)
    runs = []
    if initial_centroids is not None:
        init = torch.as_tensor(np.asarray(initial_centroids), dtype=torch.float64)
        num_clusters = init.shape[0]
        runs.append(kmeans_lloyd(Y, init))
    else:
        rs = np.random.RandomState(0)
        x_mean = Y.to(torch.float64).mean(dim=0)
        Yc = (Y - x_mean.to(Y.dtype)).contiguous()
        for _ in range(max(1, int(n_init))):
            runs.append(kmeans_lloyd(Y, _kmeanspp_sklearn(Yc, num_clusters, rs) + x_mean))
    logger.debug("Number of clusters: {}".format(num_clusters))
    best = runs[0]
    for r in runs[1:]:
        if r["inertia"] < best["inertia"]:
            best = r
    last_kmeans_report = {"n_iter": best["n_iter"], "strict": best["strict"], "ties": best["ties"],
                          "inertia": best["inertia"], "n_runs": len(runs)}
    if best["ties"]:
        logger.info(f"KMeans: {best['ties']} frames sit on an exact tie between two centres "
                    "(lowest centre index kept, as in scikit-learn)")
    return best["labels"].cpu().numpy(), best["centers"].cpu().numpy()


def cluster_data(features, settings: Dict, initial_centroids=None) -> Tuple[np.ndarray, np.ndarray]:
    """Reference statistics.py:112-157 (defaults filled in the same way)."""
    settings["algorithm"] = settings.get("algorithm", "kmeans")
    settings["num_clusters"] = settings.get("num_clusters", 10)
    settings["n_init"] = settings.get("n_init", 10)
    if settings["algorithm"] == "kmeans":
        return kmeans_clustering(features, settings["num_clusters"], settings["n_init"], initial_centroids)
    if settings["algorithm"] == "hierarchical" and _hierarchical_on_device(settings):
        return hierarchical_clustering(features, settings["num_clusters"], settings.get("linkage", "complete"))
    if settings["algorithm"] == "hdbscan" and _hdbscan_on_device(settings):
        return hdbscan_clustering(features, settings)
    if settings["algorithm"] in ("hdbscan", "hierarchical"):
        _outside_hot_path(settings["algorithm"])
    raise Exception(f"clustering algorithm {settings['algorithm']} not implemented")


def cluster_scores(features, labels, centers=None) -> Dict[str, float]:
    """Calinski-Harabasz and Davies-Bouldin scores (sklearn definitions, used at reference
    statistics.py:73-74): counts and means of the members from FP64 reductions, the per-cluster
    dispersion sums from one pass of ``dcg_cluster_dispersion``."""
    Y = _to_device(features)
    lab = torch.as_tensor(np.asarray(labels), device=Y.device).long()
    n, d = Y.shape
    ids, inv = torch.unique(lab, return_inverse=True)
    k = ids.numel()
    Yd = Y.to(torch.float64)
    cnt = torch.zeros(k, dtype=torch.float64, device=Y.device).index_add_(0, inv, torch.ones(n, dtype=torch.float64, device=Y.device))
    cent = torch.zeros((k, d), dtype=torch.float64, device=Y.device).index_add_(0, inv, Yd) / cnt[:, None]
    ssq, sdist = ops.cluster_dispersion(Y, inv.to(torch.int32), cent)
    intra_disp = float(ssq.sum().item())
    mean = Yd.mean(dim=0)
    extra_disp = float((cnt * ((cent - mean) ** 2).sum(dim=1)).sum().item())
    ch = 1.0 if intra_disp == 0.0 else extra_disp * (n - k) / (intra_disp * (k - 1.0))
    sk = sdist / cnt
    D = torch.cdist(cent, cent)
    if torch.allclose(sk, torch.zeros_like(sk)) or torch.allclose(D, torch.zeros_like(D)):
        db = 0.0
    else:
        D = D.masked_fill(D == 0, float("inf"))
        db = float(((sk[:, None] + sk[None, :]) / D).max(dim=1).values.mean().item())
    return {"calinski_harabasz": float(ch), "davies_bouldin": db}


def silhouettes(features, labelings, sample_size: Optional[int] = None, seed: int = 0) -> List[float]:
    """Mean silhouette coefficient (sklearn ``silhouette_score``, Euclidean; reference statistics.py:75) of
    every labeling of the same frames, exact in FP64 on the device, all labelings in one pass over the frame
    pairs (``ops.silhouette``): for every frame i, a_i = mean distance to the other members of its cluster,
    b_i = the smallest mean distance to the members of another cluster, s_i = (b_i - a_i) / max(a_i, b_i)
    (0 for singleton clusters and for a_i = b_i = 0).  O(N^2 d) work, O(N (d + L)) memory.  ``sample_size``
    evaluates it on a uniform random subsample of that many frames against each other -- sklearn's own
    ``sample_size`` estimator, the same subsample (``RandomState(seed).permutation(n)[:sample_size]``) for
    every labeling."""
    Y = _to_device(features)
    labs = torch.stack([torch.as_tensor(np.asarray(lab), device=Y.device).long() for lab in labelings])
    n = Y.shape[0]
    if sample_size is not None and sample_size < n:
        idx = torch.from_numpy(np.random.RandomState(seed).permutation(n)[:sample_size]).to(Y.device)
        Y, labs = Y[idx], labs[:, idx]
    return ops.silhouette(Y, labs).tolist()


def silhouette(features, labels, sample_size: Optional[int] = None, seed: int = 0) -> float:
    """Mean silhouette coefficient of one labeling (``silhouettes``)."""
    return silhouettes(features, [labels], sample_size, seed)[0]


def optimize_clustering(features, settings: Dict):
    """Reference statistics.py:17-110 for KMeans and, with ``backend.hierarchical_on_device``, agglomerative
    clustering (the tree is built once and cut at every k; cutting one deterministic tree gives what
    refitting per k gives): every k of ``search_interval`` is clustered and scored
    with Calinski-Harabasz, Davies-Bouldin and the mean silhouette; each score is min-max normalised over
    the interval and the best k maximises (CH - DB + silhouette) / 3.  Like the reference it mutates
    ``settings['num_clusters']`` and ignores ``opt_num_clusters``.  Every k is clustered first, then the
    silhouettes of all k are computed together in one pass over the frame pairs (``silhouettes``).  The
    silhouette is exact up to ``settings['silhouette_max_samples']`` frames (default 50000; None: every frame,
    at any N); beyond that it is sklearn's ``sample_size`` estimator on that many frames (seed 0, the same
    subsample for every k) and a warning says so.
    HDBSCAN (with ``backend.hdbscan_on_device``) takes no number of clusters: it runs once, unscored."""
    algorithm = settings.get("algorithm", "kmeans")
    tree = None
    if algorithm == "hdbscan" and _hdbscan_on_device(settings):
        logger.info("HDBSCAN finds the number of clusters itself: the search over search_interval and its "
                    "scores are skipped")
        labels, centroids = hdbscan_clustering(features, settings)
        if len(centroids) == 0:
            logger.warning("No clusters found using the provided settings. Try different settings or a different algorithm")
        return labels, centroids
    if algorithm == "hierarchical" and _hierarchical_on_device(settings):
        tree = linkage_tree(features, settings.get("linkage", "complete"))     # one tree, cut for every k
    elif algorithm != "kmeans":
        _outside_hot_path(algorithm)
    lo, hi = settings.get("search_interval", [2, 15])
    ks = list(range(lo, hi + 1))
    feats = np.asarray(features)
    max_sil = settings.get("silhouette_max_samples", 50000)
    sample = None
    if max_sil is not None and feats.shape[0] > int(max_sil):
        sample = int(max_sil)
        logger.warning(f"Silhouette score estimated on a random subsample of {sample} of {feats.shape[0]} frames "
                       "(scikit-learn's sample_size estimator); the reference evaluates all pairs")
    ch, db, results = [], [], []
    for k in ks:
        settings["num_clusters"] = k
        if tree is None:
            labels, centroids = cluster_data(feats, settings)
        else:
            labels = cut_tree(tree, k)
            centroids = _member_means(feats, labels, k)
        sc = cluster_scores(feats, labels)
        ch.append(sc["calinski_harabasz"])
        db.append(sc["davies_bouldin"])
        results.append((labels, centroids))
    sil = silhouettes(feats, [labels for labels, _ in results], sample_size=sample)
    for k, c, b, s in zip(ks, ch, db, sil):
        logger.debug(f"k = {k}: Calinski-Harabasz score: {round(c, 3)}, Davies-Bouldin score: {round(b, 3)}, "
                     f"average silhouette score: {round(s, 3)}")

    def norm(v):
        v = np.asarray(v, dtype=np.float64)
        return (v - v.min()) / (v.max() - v.min())
    score = (norm(ch) - norm(db) + norm(sil)) / 3
    best = int(np.argmax(score))
    logger.info(f"Best number of clusters: {ks[best]}")
    labels, centroids = results[best]
    if len(centroids) == 0:
        logger.warning("No clusters found using the provided settings. Try different settings or a different algorithm")
    global last_optimize_report
    last_optimize_report = {"k": ks, "calinski_harabasz": ch, "davies_bouldin": db, "silhouette": sil,
                            "score": score.tolist(), "best_k": ks[best]}
    return labels, centroids


last_optimize_report: Dict = {}


LINKAGES = ("ward", "complete", "average", "single")


def _hierarchical_on_device(settings: Dict) -> bool:
    return bool((settings.get("backend") or {}).get("hierarchical_on_device", False))


def linkage_tree(features, linkage: str = "complete") -> np.ndarray:
    """The (n-1) x 4 merge tree of sklearn ``AgglomerativeClustering(linkage=linkage)`` (scipy ``linkage``
    layout: children, distance, size), built on the device (``ops.linkage``) and returned as numpy."""
    if linkage not in LINKAGES:
        raise ValueError(f"linkage must be one of {list(LINKAGES)}, got {linkage!r}")
    return ops.linkage(_to_device(features), linkage).cpu().numpy()


def cut_tree(Z, n_clusters: int) -> np.ndarray:
    """Labels of the ``n_clusters`` clusters of the merge tree ``Z`` (sklearn ``_hc_cut``,
    sklearn/cluster/_agglomerative.py): the heap of negated node ids is split ``n_clusters - 1`` times at
    its largest node, and a leaf's label is the position of its ancestor in the heap array."""
    children = np.asarray(Z)[:, :2].astype(np.intp)
    n = children.shape[0] + 1
    if n_clusters > n:
        raise ValueError("Cannot extract more clusters than samples: "
                         f"{n_clusters} clusters were given for a tree with {n} leaves.")
    nodes = [-(int(max(children[-1])) + 1)]
    for _ in range(n_clusters - 1):
        these = children[-nodes[0] - n]
        heapq.heappush(nodes, -int(these[0]))
        heapq.heappushpop(nodes, -int(these[1]))
    node_label = np.full(2 * n - 1, -1, dtype=np.intp)
    for i, node in enumerate(nodes):
        node_label[-node] = i
    # children ids are below their parent's: one pass from the root down labels every descendant
    for m in range(n - 2, -1, -1):
        lab = node_label[n + m]
        if lab >= 0:
            node_label[children[m]] = lab
    return node_label[:n].copy()


def _member_means(features: np.ndarray, labels: np.ndarray, k: int) -> np.ndarray:
    """FP64 means of the members of clusters 0..k-1 (the reference's centroids, statistics.py:330-335)."""
    X = np.asarray(features, dtype=np.float64)
    return np.stack([X[labels == c].mean(axis=0) for c in range(k)])


def hierarchical_clustering(feature_matrix, num_clusters: int, linkage: str = "complete") -> Tuple[np.ndarray, np.ndarray]:
    """Reference statistics.py:285: ``AgglomerativeClustering(n_clusters, linkage).fit_predict`` and the
    member means as centroids, with the tree built on the device."""
    logger.debug("Clustering frames with hierarchical clustering...")
    feats = np.asarray(feature_matrix)
    labels = cut_tree(linkage_tree(feats, linkage), num_clusters)
    return labels, _member_means(feats, labels, num_clusters)


# ---- HDBSCAN ------------------------------------------------------------------------------------------------
# sklearn.cluster.HDBSCAN (scikit-learn 1.9.0, sklearn/cluster/_hdbscan/) with metric="euclidean" and
# algorithm="auto" on dense finite data: _hdbscan_prims, then tree_to_labels with allow_single_cluster=False.
HIERARCHY_DTYPE = np.dtype([("left_node", np.intp), ("right_node", np.intp), ("value", np.float64),
                            ("cluster_size", np.intp)])      # sklearn's HIERARCHY_dtype (_tree.pyx)


def _hdbscan_on_device(settings: Dict) -> bool:
    return bool((settings.get("backend") or {}).get("hdbscan_on_device", False))


def single_linkage_from_mst(mst) -> np.ndarray:
    """sklearn's ``_process_mst`` (hdbscan.py) on the (n-1) x 3 rows (source, new node, distance) of
    ``ops.mreach_mst`` in Prim order: the rows are reordered by numpy's default ``argsort`` of the
    distances -- not stable, so the tie order is numpy's own and this must stay a numpy argsort on the
    host -- and ``make_single_linkage`` (_linkage.pyx) merges them with sklearn's ``UnionFind``
    (_hierarchical_fast.pyx): merge i creates node n + i, whose children are the roots of the two
    endpoints, left first.  Returns the HIERARCHY_DTYPE tree."""
    mst = np.asarray(mst, dtype=np.float64)
    n = mst.shape[0] + 1
    mst = mst[np.argsort(mst[:, 2])]
    a = mst[:, 0].astype(np.intp).tolist()
    b = mst[:, 1].astype(np.intp).tolist()
    parent = [-1] * (2 * n - 1)
    size = [1] * n + [0] * (n - 1)
    left, right, csize = [0] * (n - 1), [0] * (n - 1), [0] * (n - 1)

    def find(x):
        r = x
        while parent[r] != -1:
            r = parent[r]
        while x != r and parent[x] != r:          # path compression (does not change any root)
            parent[x], x = r, parent[x]
        return r

    for i in range(n - 1):
        ra, rb = find(a[i]), find(b[i])
        left[i], right[i] = ra, rb
        csize[i] = size[ra] + size[rb]
        parent[ra] = parent[rb] = n + i
        size[n + i] = csize[i]
    tree = np.empty(n - 1, dtype=HIERARCHY_DTYPE)
    tree["left_node"], tree["right_node"], tree["value"], tree["cluster_size"] = left, right, mst[:, 2], csize
    return tree


def hdbscan_tree(features, min_samples: int) -> np.ndarray:
    """sklearn ``HDBSCAN(min_samples=min_samples)._single_linkage_tree_`` (``_hdbscan_prims``): core
    distances and the mutual-reachability MST on the device (``ops.core_distances``, ``ops.mreach_mst``),
    then ``single_linkage_from_mst`` on the host.  O(N) memory."""
    Y = _to_device(features)
    return single_linkage_from_mst(ops.mreach_mst(Y, ops.core_distances(Y, min_samples)).cpu().numpy())


def _bfs_hierarchy(left, right, n: int, root: int) -> List[int]:
    """``bfs_from_hierarchy`` (_tree.pyx): the nodes under ``root`` level by level, left before right."""
    out, queue = [], [root]
    while queue:
        out.extend(queue)
        nxt = []
        for x in queue:
            if x >= n:
                nxt.append(left[x - n])
                nxt.append(right[x - n])
        queue = nxt
    return out


def _condense_tree(tree: np.ndarray, min_cluster_size: int):
    """``_condense_tree`` (_tree.pyx): rows (parent, child, lambda, child size) in sklearn's row order, as
    four numpy arrays."""
    left, right = tree["left_node"].tolist(), tree["right_node"].tolist()
    value, size = tree["value"].tolist(), tree["cluster_size"].tolist()
    n = len(left) + 1
    root = 2 * (n - 1)
    next_label = n + 1
    relabel = [0] * (root + 1)
    relabel[root] = n
    ignore = bytearray(root + 1)
    rows = []
    for node in _bfs_hierarchy(left, right, n, root):
        if ignore[node] or node < n:
            continue
        l, r, dist = left[node - n], right[node - n], value[node - n]
        lam = 1.0 / dist if dist > 0.0 else np.inf
        lc = size[l - n] if l >= n else 1
        rc = size[r - n] if r >= n else 1
        if lc >= min_cluster_size and rc >= min_cluster_size:
            relabel[l] = next_label
            next_label += 1
            rows.append((relabel[node], relabel[l], lam, lc))
            relabel[r] = next_label
            next_label += 1
            rows.append((relabel[node], relabel[r], lam, rc))
            continue
        if lc < min_cluster_size and rc < min_cluster_size:
            fall = (l, r)
        elif lc < min_cluster_size:
            relabel[r] = relabel[node]
            fall = (l,)
        else:
            relabel[l] = relabel[node]
            fall = (r,)
        for sub in fall:
            for sub_node in _bfs_hierarchy(left, right, n, sub):
                if sub_node < n:
                    rows.append((relabel[node], sub_node, lam, 1))
                ignore[sub_node] = 1
    parent, child, lam, csize = zip(*rows)
    return (np.array(parent, dtype=np.intp), np.array(child, dtype=np.intp), np.array(lam, dtype=np.float64),
            np.array(csize, dtype=np.intp))


def hdbscan_labels(tree, min_cluster_size: int = 5, cluster_selection_method: str = "eom",
                   cluster_selection_epsilon: float = 0.0, max_cluster_size: Optional[int] = None) -> np.ndarray:
    """sklearn's ``tree_to_labels`` (sklearn/cluster/_hdbscan/_tree.pyx) with ``allow_single_cluster=False``,
    restated in numpy: condense the single-linkage ``tree`` (HIERARCHY_DTYPE) at ``min_cluster_size``,
    compute the stabilities, select clusters by ``eom`` (excess of mass, capped at ``max_cluster_size``) or
    ``leaf``, merge them upwards to ``cluster_selection_epsilon``, and label each frame with its selected
    cluster (numbered in increasing condensed-node order) or -1 for noise.  Every tie-breaking detail is
    sklearn's: the summation order of the stabilities and the iteration order of its Python sets."""
    if int(min_cluster_size) < 2:
        raise ValueError(f"min_cluster_size must be at least 2, got {min_cluster_size}")
    if cluster_selection_method not in ("eom", "leaf"):
        raise ValueError(f"cluster_selection_method must be 'eom' or 'leaf', got {cluster_selection_method!r}")
    tree = np.asarray(tree)
    parent, child, lam, csize = _condense_tree(tree, int(min_cluster_size))
    eps = float(cluster_selection_epsilon)
    # _compute_stability: sum of (lambda - birth(parent)) * size over the rows, in row order
    root = int(parent.min())
    births = np.full(max(int(child.max()), root) + 1, np.nan)
    births[child] = lam
    births[root] = 0.0
    stab_arr = np.zeros(int(parent.max()) - root + 1)
    np.add.at(stab_arr, parent - root, (lam - births[parent]) * csize.astype(np.float64))
    stability = {root + i: v for i, v in enumerate(stab_arr.tolist())}
    # _get_clusters
    node_list = sorted(stability.keys(), reverse=True)[:-1]
    ct = csize > 1                                                       # the cluster tree's rows
    ct_parent, ct_child, ct_lam = parent[ct].tolist(), child[ct].tolist(), lam[ct].tolist()
    children: Dict[int, List[int]] = {}
    row_of: Dict[int, int] = {}
    for i, (p_, c_) in enumerate(zip(ct_parent, ct_child)):
        children.setdefault(p_, []).append(c_)
        row_of[c_] = i
    cluster_sizes = dict(zip(ct_child, csize[ct].tolist()))
    n_samples = int(child[csize == 1].max()) + 1
    if max_cluster_size is None:
        max_cluster_size = n_samples + 1
    is_cluster = {c: True for c in node_list}

    def below(node):                                                     # bfs_from_cluster_tree, node excluded
        out, queue = [], list(children.get(node, ()))
        while queue:
            out.extend(queue)
            queue = [c for q in queue for c in children.get(q, ())]
        return out

    def epsilon_search(leaves):
        selected, processed = [], set()
        for leaf in leaves:
            if 1 / ct_lam[row_of[leaf]] < eps:
                if leaf not in processed:
                    node = leaf                                          # traverse_upwards
                    while True:
                        up = ct_parent[row_of[node]]
                        if up == root or 1 / ct_lam[row_of[up]] > eps:
                            top = node if up == root else up
                            break
                        node = up
                    selected.append(top)
                    processed.update(below(top))
            else:
                selected.append(leaf)
        return set(selected)

    if cluster_selection_method == "eom":
        for node in node_list:
            sub = np.sum([stability[c] for c in children.get(node, ())])
            if sub > stability[node] or cluster_sizes[node] > max_cluster_size:
                is_cluster[node] = False
                stability[node] = sub
            else:
                for sub_node in below(node):
                    is_cluster[sub_node] = False
        if eps != 0.0 and ct_parent:
            eom_clusters = [c for c in is_cluster if is_cluster[c]]
            if len(eom_clusters) == 1 and eom_clusters[0] == min(ct_parent):
                selected = []
            else:
                selected = epsilon_search(set(eom_clusters))
            for c in is_cluster:
                is_cluster[c] = c in selected
    else:
        leaves = []                                                      # get_cluster_tree_leaves: DFS order
        if ct_parent:
            stack = [min(ct_parent)]
            while stack:
                node = stack.pop()
                kids = children.get(node)
                if kids:
                    stack.extend(reversed(kids))
                else:
                    leaves.append(node)
        leaves = set(leaves)
        selected = epsilon_search(leaves) if eps != 0.0 else leaves
        for c in is_cluster:
            is_cluster[c] = c in selected
    clusters = sorted(c for c in is_cluster if is_cluster[c])
    # _do_labelling: a frame's label is that of its nearest selected ancestor; none below the root is noise.
    # Condensed node ids grow from parent to child, so one increasing pass resolves every node.
    label_of = np.full(int(parent.max()) + 1, -1, dtype=np.intp)
    label_of[clusters] = np.arange(len(clusters))
    up_of = np.empty(int(parent.max()) + 1, dtype=np.intp)
    up_of[child[child >= root]] = parent[child >= root]
    for c in range(root + 1, int(parent.max()) + 1):
        if label_of[c] < 0:
            label_of[c] = label_of[up_of[c]]
    pts = child < root
    labels = np.empty(root, dtype=np.intp)
    labels[child[pts]] = label_of[parent[pts]]
    return labels


def hdbscan_clustering(feature_matrix, settings: Dict) -> Tuple[np.ndarray, np.ndarray]:
    """``HDBSCAN(min_cluster_size, min_samples, cluster_selection_epsilon, max_cluster_size,
    cluster_selection_method).fit_predict`` with the schema's values, the tree built on the device, and
    the FP64 member means of clusters 0..K-1 as centroids (noise, -1, excluded).  The centroid rule is the
    one the reference applies to hierarchical clustering (statistics.py:330-335); its own HDBSCAN wrapper is
    assumed to do the same.  ``min_samples`` None means ``min_cluster_size``, as in scikit-learn."""
    logger.debug("Clustering frames with HDBSCAN...")
    feats = np.asarray(feature_matrix)
    mcs = int(settings.get("min_cluster_size", 5))
    ms = settings.get("min_samples")
    tree = hdbscan_tree(feats, mcs if ms is None else int(ms))
    labels = hdbscan_labels(tree, mcs, settings.get("cluster_selection_method", "eom"),
                            settings.get("cluster_selection_epsilon", 0.0), settings.get("max_cluster_size"))
    k = int(labels.max()) + 1
    means = _member_means(feats, labels, k) if k > 0 else np.empty((0, feats.shape[1]))
    return labels, means


def assign_closest_cluster(clustered, labels, sup) -> np.ndarray:
    """Label of the nearest clustered frame of every supplementary frame (reference
    ``traj_cluster_workflow.py:207-238``, ``assign_closest_cluster``).  The reference's semantics are assumed
    to be ``NearestNeighbors(n_neighbors=1).fit(clustered).kneighbors(sup)``, each supplementary frame taking
    the label of the returned frame; the search runs on the device (``ops.nearest_frames``) with the KD-tree's
    distance arithmetic, and among exactly tied nearest frames the lowest-indexed one wins (scikit-learn's
    KD-tree returns whichever tied frame it visits first).  HDBSCAN noise (-1) propagates: a frame whose
    nearest clustered frame is noise is noise."""
    labels = np.asarray(labels)
    X = _to_device(clustered)
    if labels.shape != (X.shape[0],):
        raise ValueError(f"labels must have one entry per clustered frame ({X.shape[0]}), got shape {labels.shape}")
    Q = _to_device(sup)
    index, _ = ops.nearest_frames(X, Q)
    return labels[index.cpu().numpy()]


def _outside_hot_path(algorithm):
    """hierarchical clustering and hdbscan without their ``backend.*_on_device`` flag are not part of the
    B200 hot path (SURVEY.md section 2): say so the way the reference reports fatal configuration
    problems -- log an error and exit -- instead of a traceback."""
    flag = {"hierarchical": "hierarchical_on_device", "hdbscan": "hdbscan_on_device"}.get(algorithm)
    hint = (f"set traj_cluster.backend.{flag}: true, or algorithm: kmeans" if flag
            else "set traj_cluster.algorithm: kmeans")
    logger.error(f"Clustering algorithm '{algorithm}' is outside the B200 hot path; {hint}, "
                 "or use the reference package for it. Exiting...")
    sys.exit(1)


def find_centroids(data: pd.DataFrame, centroids: np.ndarray, clustering_features: List[str]) -> pd.DataFrame:
    """Mark the sample closest to each centroid (reference statistics.py:337-379) in ONE pass
    over the data instead of k."""
    if len(centroids) == 0:
        logger.warning("No centroids found")
        return pd.DataFrame()
    if len(centroids[0]) != len(clustering_features):
        logger.error("  The dimension of the centroids is not the same as the dimension of the used features for clustering.\n")
        sys.exit(1)
    Y = _to_device(data.loc[:, clustering_features].to_numpy())
    C = torch.as_tensor(np.asarray(centroids), dtype=torch.float64, device=Y.device)
    idx = ops.nearest_to_centers(Y, C).cpu().numpy()
    data["centroid"] = False
    data.loc[data.index[idx], "centroid"] = True
    return data
