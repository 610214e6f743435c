#!/usr/bin/env python
"""Generate the committed golden fixtures from the reference's own test artefacts.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

Writes (all small, committed):
  tests/golden/peptide_c1.npz     C1 fixture: the 164x54 float32 feature matrix of the
      reference's bundled peptide test (virtual_dihedrals.dat filtered by
      filtered_virtual_dihedrals.txt) + the golden weights / normalisations from
      tests/data/input/models/{pca,tica,htica}_model.zip + the golden projected CSVs
      from tests/data/reference/train_colvars/ + the golden traj_cluster CSVs.
  tests/golden/peptide_c1.dat / peptide_c1_features.txt
      the same matrix as a PLUMED colvars text file + feature list, for the step-API tests
      (re-serialised with enough digits to round-trip float32 exactly).
  tests/golden/kmeans_ref.npz     labels / centres produced by the REFERENCE's own
      ``deep_cartograph.modules.statistics.cluster_data`` (sklearn underneath) on seeded inputs
      with fixed initial centroids; the inputs themselves are kept as SHA-256 digests
      (tests/conftest.py:kmeans_inputs regenerates them).
"""
import io
import json
import os
import sys
import zipfile

import numpy as np
import pandas as pd

REF = os.environ.get("DCG_REFERENCE", "/root/reference")
DATA = os.path.join(REF, "deep_cartograph", "tests", "data")
HERE = os.path.dirname(os.path.abspath(__file__))


def read_colvars(path):
    with open(path) as f:
        header = f.readline().split()
    assert header[0] == "#!" and header[1] == "FIELDS"
    names = header[2:]
    df = pd.read_csv(path, sep=r"\s+", dtype=np.float32, comment="#", header=None, names=names)
    return df


def main():
    colvars = os.path.join(DATA, "reference", "compute_features", "virtual_dihedrals.dat")
    feats = [l.strip() for l in open(os.path.join(DATA, "reference", "filter_features",
                                                  "filtered_virtual_dihedrals.txt")) if l.strip()]
    df = read_colvars(colvars)
    time = df["time"].to_numpy()
    X = df[feats].to_numpy(dtype=np.float32)
    out = {"X": X, "features": np.array(feats)}
    for cv in ("pca", "tica", "htica"):
        z = zipfile.ZipFile(os.path.join(DATA, "input", "models", f"{cv}_model.zip"))
        for name in ("cv_weights", "cv_norm_mean", "cv_norm_range", "features_norm_mean",
                     "features_norm_range"):
            out[f"{cv}_{name}"] = np.load(io.BytesIO(z.read(f"model/{name}.npy")))
        meta = json.loads(z.read("model/metadata.json"))
        assert meta["cv_name"] == cv and meta["cv_dimension"] == 2
        labels = z.read("model/features_labels.txt").decode().strip().split("\n")
        assert labels == feats, "model feature order differs from filtered list"
        csv = pd.read_csv(os.path.join(DATA, "reference", "train_colvars",
                                       f"{cv}_projected_trajectory.csv"))
        out[f"{cv}_csv"] = csv.to_numpy(dtype=np.float64)
        out[f"{cv}_csv_cols"] = np.array(list(csv.columns))
        cl = pd.read_csv(os.path.join(DATA, "reference", "traj_cluster",
                                      f"{cv}_projected_trajectory.csv"))
        out[f"{cv}_cluster_cv"] = cl.iloc[:, :2].to_numpy(dtype=np.float64)
        out[f"{cv}_cluster_label"] = cl["cluster"].to_numpy(dtype=np.int64)
        out[f"{cv}_cluster_centroid"] = cl["centroid"].to_numpy(dtype=bool)
    # DeepTICA (SURVEY 8c): the reference's golden TorchScript model and the projection CSV it pins
    # (tests/test_traj_projection.py); the model file is copied as a fixture, it loads with plain torch
    import shutil
    shutil.copy(os.path.join(DATA, "input", "models", "deep_tica_model.zip"),
                os.path.join(HERE, "deep_tica_model.zip"))
    csv = pd.read_csv(os.path.join(DATA, "reference", "train_colvars", "deep_tica_projected_trajectory.csv"))
    out["deep_tica_csv"] = csv.to_numpy(dtype=np.float64)
    out["deep_tica_csv_cols"] = np.array(list(csv.columns))
    np.savez_compressed(os.path.join(HERE, "peptide_c1.npz"), **out)

    # colvars text form for the step-API tests (float32 round-trips with 9 significant digits)
    with open(os.path.join(HERE, "peptide_c1.dat"), "w") as f:
        f.write("#! FIELDS time " + " ".join(feats) + "\n")
        for t, row in zip(time, X):
            f.write(" %.6f " % t + " ".join("%.9g" % v for v in row) + "\n")
    with open(os.path.join(HERE, "peptide_c1_features.txt"), "w") as f:
        f.write("\n".join(feats) + "\n")
    chk = read_colvars(os.path.join(HERE, "peptide_c1.dat"))[feats].to_numpy(dtype=np.float32)
    assert np.array_equal(chk, X), "text round trip is not exact"

    # KMeans: outputs of the reference's own statistics.cluster_data (sklearn underneath).  The inputs are
    # not stored: tests/conftest.py regenerates them from their seed and checks them against the digests.
    sys.path.insert(0, REF)
    from deep_cartograph.modules.statistics import cluster_data  # noqa: E402
    import sklearn
    sys.path.insert(0, os.path.dirname(HERE))
    from conftest import KMEANS_CASES, kmeans_inputs, sha256  # noqa: E402
    km = {"sklearn_version": np.array(sklearn.__version__)}
    inputs = kmeans_inputs()
    for name in KMEANS_CASES:
        X, init = inputs[f"{name}_X"], inputs[f"{name}_init"]
        labels, centers = cluster_data(X.copy(), {"algorithm": "kmeans"}, initial_centroids=init.copy())
        km[f"{name}_X_sha256"] = np.array(sha256(X))
        km[f"{name}_labels"] = labels.astype(np.int32)
        km[f"{name}_centers"] = centers
    # ---- the reference's DEFAULT search path: optimize_clustering (k-means++ with random_state=0, three
    # scores per k) and kmeans_clustering without initial centroids, run by the imported reference module
    from deep_cartograph.modules.statistics.statistics import kmeans_clustering, optimize_clustering
    Xo = inputs["opt_X"]
    lab_o, cen_o = optimize_clustering(Xo.copy(), {"algorithm": "kmeans", "search_interval": [2, 8], "n_init": 3})
    km["opt_X_sha256"], km["opt_labels"], km["opt_centers"] = np.array(sha256(Xo)), lab_o.astype(np.int32), cen_o
    lab_p, cen_p = kmeans_clustering(Xo.copy(), 6, 4)
    km["pp_labels"], km["pp_centers"] = lab_p.astype(np.int32), cen_p
    from sklearn.metrics import calinski_harabasz_score, davies_bouldin_score, silhouette_score
    km["pp_scores"] = np.array([calinski_harabasz_score(Xo, lab_p), davies_bouldin_score(Xo, lab_p),
                                silhouette_score(Xo, lab_p)])
    np.savez_compressed(os.path.join(HERE, "kmeans_ref.npz"), **km)

    # ---- FES: the reference's own legacy output (mlcolvar compute_fes through KDEpy; bandwidth 0.025,
    # 200 bins, 300 K: data/calpha_transitions/input/distances_config.yml:93-95) and the projected
    # trajectory it was computed from

    base = os.path.join(REF, "deep_cartograph", "data", "calpha_transitions", "reference", "1rcs_B-3ssx_R-3",
                        "train_colvars", "pca")
    d = pd.read_csv(os.path.join(base, "projected_trajectory.csv"))
    np.savez_compressed(os.path.join(HERE, "fes_legacy_pca.npz"), X=d[["PC 1", "PC 2"]].to_numpy(),
                        fes=np.load(os.path.join(base, "fes", "fes.npy")).astype(np.float32),
                        grid=np.load(os.path.join(base, "fes", "grid.npy")),
                        bounds=np.load(os.path.join(base, "fes", "bounds.npy")),
                        bandwidth=0.025, num_bins=200, temperature=300)
    print("wrote", os.listdir(HERE))


if __name__ == "__main__":
    main()
