"""traj_cluster step API on the B200 backend (KMeans; agglomerative with ``backend.hierarchical_on_device``;
HDBSCAN with ``backend.hdbscan_on_device``).

Same signature, return value and CSV layout as the reference's
``tools/traj_cluster/traj_cluster.py:18-113`` / ``traj_cluster_workflow.py:240-387``.
Structure extraction (PDB / XTC) and plots are outside the hot path (SURVEY.md section 2).  Supplementary
CV trajectories (``sup_cv_traj_paths``) are assigned on the device: each frame takes the cluster of its
nearest clustered frame (``statistics.assign_closest_cluster``) and is written in the main CSV layout.  ``algorithm: kmeans`` is accelerated, and so is
``algorithm: hierarchical`` (any of sklearn's four linkages, same tree and labels as sklearn) when the
configuration sets ``backend: {hierarchical_on_device: true}``, and ``algorithm: hdbscan`` (sklearn's
labels, -1 for noise, in O(N) device memory) when it sets ``backend: {hdbscan_on_device: true}``.
"""
from __future__ import annotations

import logging
import os
import time
from pathlib import Path
from typing import Dict, List, Optional

import numpy as np
import pandas as pd

from ...modules.common import validate_configuration
from ...modules.statistics import statistics
from ...yaml_schemas.traj_cluster import TrajClusterSchema

logger = logging.getLogger(__name__)


class TrajClusterWorkflow:
    def __init__(self, configuration: Dict, cv_traj_paths: List[str],
                 trajectories: Optional[List[str]] = None, topologies: Optional[List[str]] = None,
                 frames_per_sample: int = 1, output_folder: str = "traj_cluster",
                 initial_centroids: Optional[np.ndarray] = None,
                 sup_cv_traj_paths: Optional[List[str]] = None, sup_trajectories: Optional[List[str]] = None,
                 sup_topologies: Optional[List[str]] = None):
        os.makedirs(output_folder, exist_ok=True)
        self.configuration = validate_configuration(configuration, TrajClusterSchema, output_folder)
        self.cv_traj_paths = cv_traj_paths
        self.trajectories = trajectories
        self.topologies = topologies
        self.frames_per_sample = frames_per_sample
        self.output_folder = output_folder
        self.initial_centroids = initial_centroids
        self.sup_cv_traj_paths = sup_cv_traj_paths
        self.sup_trajectories = sup_trajectories
        self.sup_topologies = sup_topologies

    @staticmethod
    def read_cv_traj_data(paths: List[str]) -> pd.DataFrame:
        """CSV hand-off (4-decimal text -> float64), one 'traj_label' per file (reference :196-205)."""
        data = []
        for traj_index, path in enumerate(paths):
            df = pd.read_csv(path)
            df["traj_label"] = traj_index
            data.append(df)
        return pd.concat(data, ignore_index=True)

    def traj_names(self) -> List[str]:
        return [Path(self.trajectories[i]).stem if self.trajectories else f"traj_{i}"
                for i in range(len(self.cv_traj_paths))]

    def sup_traj_names(self) -> List[str]:
        return [Path(self.sup_trajectories[i]).stem if self.sup_trajectories else f"sup_traj_{i}"
                for i in range(len(self.sup_cv_traj_paths or []))]

    def read_sup_cv_traj_data(self, cv_labels: List[str]) -> Optional[pd.DataFrame]:
        """The supplementary CV trajectories, checked before any clustering: their CV columns must be the main
        ones, and their output folders must not collide with the main trajectories' or with each other."""
        if not self.sup_cv_traj_paths:
            return None
        sup_data = self.read_cv_traj_data(self.sup_cv_traj_paths)
        sup_labels = sup_data.columns[:-1].tolist()
        if sup_labels != cv_labels:
            raise ValueError(f"supplementary CV trajectories have columns {sup_labels}; the clustered ones have "
                             f"{cv_labels}")
        names = self.traj_names()
        for name in self.sup_traj_names():
            if name in names:
                raise ValueError(f"supplementary trajectory name {name!r} collides with another output trajectory "
                                 "name")
            names.append(name)
        return sup_data

    def run(self) -> Dict[str, List[str]]:
        if self.configuration["run"] is False:
            logger.info("traj_cluster workflow set to not run. Exiting...")
            return {}
        output_paths: Dict[str, List[str]] = {}
        cv_data = self.read_cv_traj_data(self.cv_traj_paths)
        cv_labels = cv_data.columns[:-1].tolist()
        sup_data = self.read_sup_cv_traj_data(cv_labels)
        X = cv_data[cv_labels].to_numpy()
        if self.initial_centroids is not None:
            # fixed-k, fixed-init KMeans: the drop-in point for large N (SURVEY row K2)
            labels, centroids = statistics.cluster_data(X, self.configuration, self.initial_centroids)
        else:
            labels, centroids = statistics.optimize_clustering(X, self.configuration)
        cv_data["cluster"] = labels                        # -1: HDBSCAN noise
        if len(centroids) == 0:                             # HDBSCAN found only noise: no frame is a centroid
            cv_data["centroid"] = False
        else:
            cv_data = statistics.find_centroids(cv_data, centroids, cv_labels)
        frames = []
        for traj_index in range(len(self.cv_traj_paths)):
            n_samples = int((cv_data["traj_label"] == traj_index).sum())
            frames.extend(np.arange(0, n_samples * self.frames_per_sample, self.frames_per_sample))
        cv_data["frame"] = frames
        for traj_index, traj_name in enumerate(self.traj_names()):
            out = os.path.join(self.output_folder, traj_name)
            os.makedirs(out, exist_ok=True)
            path = os.path.join(out, "projected_trajectory.csv")
            cv_data[cv_data["traj_label"] == traj_index].to_csv(path, index=False)
            output_paths[traj_name] = [path]
        if sup_data is not None:
            output_paths.update(self.write_supplementary(sup_data, X, labels, cv_labels))
        return output_paths

    def write_supplementary(self, sup_data: pd.DataFrame, X: np.ndarray, labels: np.ndarray,
                            cv_labels: List[str]) -> Dict[str, List[str]]:
        """Every supplementary frame takes the cluster of its nearest clustered frame (noise included; reference
        ``traj_cluster_workflow.py:207-238``) and is written in the main CSV layout; no supplementary frame is a
        centroid."""
        sup_data["cluster"] = statistics.assign_closest_cluster(X, labels, sup_data[cv_labels].to_numpy())
        sup_data["centroid"] = False
        frames = []
        for traj_index in range(len(self.sup_cv_traj_paths)):
            n_samples = int((sup_data["traj_label"] == traj_index).sum())
            frames.extend(np.arange(0, n_samples * self.frames_per_sample, self.frames_per_sample))
        sup_data["frame"] = frames
        output_paths: Dict[str, List[str]] = {}
        for traj_index, traj_name in enumerate(self.sup_traj_names()):
            out = os.path.join(self.output_folder, traj_name)
            os.makedirs(out, exist_ok=True)
            path = os.path.join(out, "projected_trajectory.csv")
            sup_data[sup_data["traj_label"] == traj_index].to_csv(path, index=False)
            output_paths[traj_name] = [path]
        return output_paths


def traj_cluster(configuration: Dict, cv_traj_paths: List[str],
                 trajectories: Optional[List[str]] = None, topologies: Optional[List[str]] = None,
                 sup_cv_traj_paths: Optional[List[str]] = None,
                 sup_trajectories: Optional[List[str]] = None,
                 sup_topologies: Optional[List[str]] = None,
                 frames_per_sample: int = 1, output_folder: str = "traj_cluster",
                 initial_centroids: Optional[np.ndarray] = None) -> Dict[str, List[str]]:
    """Cluster CV trajectories; returns ``{traj_name: [csv]}`` as the reference does.
    ``sup_cv_traj_paths``: CV trajectories that are not clustered; each of their frames takes the cluster of
    its nearest clustered frame and is written to ``<stem of sup_trajectories[i], else sup_traj_i>/``.
    ``initial_centroids`` (extension) runs fixed-init KMeans through ``cluster_data``."""
    start = time.time()
    wf = TrajClusterWorkflow(configuration, cv_traj_paths, trajectories, topologies,
                             frames_per_sample, output_folder, initial_centroids,
                             sup_cv_traj_paths, sup_trajectories, sup_topologies)
    out = wf.run()
    logger.info("Elapsed time (Cluster trajectory): %s", time.strftime("%H h %M min %S s", time.gmtime(time.time() - start)))
    return out
