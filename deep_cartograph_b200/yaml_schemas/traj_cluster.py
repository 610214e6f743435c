"""Configuration contract of the traj_cluster step (reference ``yaml_schemas/traj_cluster.py:18-47``).

The reference default algorithm is ``hierarchical``.  This backend accelerates ``kmeans``; when
``backend.hierarchical_on_device`` is true, ``hierarchical`` (the same tree as scikit-learn, built on the
device); and when ``backend.hdbscan_on_device`` is true, ``hdbscan`` (the same labels as scikit-learn's
HDBSCAN, in O(N) device memory).  Otherwise ``hierarchical`` and ``hdbscan`` log an error and exit
(SURVEY.md section 2).  Supplementary trajectories need no setting: when the step is given
``sup_cv_traj_paths``, their frames take the cluster of their nearest clustered frame, on the device.
Backend knobs live in the optional ``backend`` block."""
from typing import Dict, List, Literal, Optional, Union

from pydantic import BaseModel, ConfigDict


class Backend(BaseModel):
    """B200 backend options (not in the reference)."""
    model_config = ConfigDict(extra="allow")
    # algorithm: hierarchical builds its tree on the device (bitwise the tree scikit-learn builds);
    # off by default, so a reference configuration keeps its current behaviour
    hierarchical_on_device: bool = False
    # algorithm: hdbscan builds its single-linkage tree on the device (label for label scikit-learn's
    # HDBSCAN); off by default for the same reason
    hdbscan_on_device: bool = False


class TrajClusterSchema(BaseModel):
    model_config = ConfigDict(extra="allow")
    run: bool = True
    output_structures: Optional[Literal["centroids", "all"]] = "centroids"
    algorithm: Literal["kmeans", "hdbscan", "hierarchical"] = "hierarchical"
    opt_num_clusters: bool = True
    search_interval: List[int] = [3, 10]
    num_clusters: int = 10
    linkage: str = "complete"
    n_init: int = 20
    min_cluster_size: int = 5
    max_cluster_size: Union[int, None] = None
    min_samples: int = 3
    cluster_selection_epsilon: float = 0
    cluster_selection_method: Literal["eom", "leaf"] = "eom"
    figures: Dict = {}
    backend: Backend = Backend()
