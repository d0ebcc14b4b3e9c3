"""Import the REAL reference classes from a checkout of the original vlfm repository.

TEST INFRASTRUCTURE, used only by oracle/make_golden.py to write tests/golden/: the tests
compare against those stored outputs and never import the reference.  The checkout is
named by the VLFM_REFERENCE environment variable.

``vlfm.mapping.value_map`` imports cleanly (cv2 + numpy only).
``vlfm.mapping.obstacle_map`` needs ``frontier_exploration`` (third-party, unpinned
git dependency, pyproject.toml:25, NOT in the tree); we inject the restated functions
from ``oracle/frontier_exploration_oracle.py`` under that module name so the reference's
own obstacle/explore code runs unmodified around them.
"""
from __future__ import annotations

import os
import sys
import types

REFERENCE_ROOT = os.environ.get("VLFM_REFERENCE", "")


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "vlfm", "mapping"))


def _ensure_path() -> None:
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)


def value_map_class():
    _ensure_path()
    from vlfm.mapping.value_map import ValueMap  # type: ignore

    return ValueMap


def obstacle_map_class():
    _ensure_path()
    if "frontier_exploration" not in sys.modules:
        from . import frontier_exploration_oracle as feo

        pkg = types.ModuleType("frontier_exploration")
        fd = types.ModuleType("frontier_exploration.frontier_detection")
        ut = types.ModuleType("frontier_exploration.utils")
        fow = types.ModuleType("frontier_exploration.utils.fog_of_war")
        fd.detect_frontier_waypoints = feo.detect_frontier_waypoints
        fow.reveal_fog_of_war = feo.reveal_fog_of_war
        pkg.frontier_detection = fd
        pkg.utils = ut
        ut.fog_of_war = fow
        sys.modules["frontier_exploration"] = pkg
        sys.modules["frontier_exploration.frontier_detection"] = fd
        sys.modules["frontier_exploration.utils"] = ut
        sys.modules["frontier_exploration.utils.fog_of_war"] = fow
    from vlfm.mapping.obstacle_map import ObstacleMap  # type: ignore

    return ObstacleMap


def base_map_class():
    _ensure_path()
    from vlfm.mapping.base_map import BaseMap  # type: ignore

    return BaseMap


def frontier_map_class(encoder_cls):
    """vlfm.mapping.frontier_map with its HTTP BLIP-2 client replaced by ``encoder_cls`` (a stub ``vlfm.vlm.blip2itm``)."""
    _ensure_path()
    stub = types.ModuleType("vlfm.vlm.blip2itm")
    stub.BLIP2ITMClient = encoder_cls
    sys.modules["vlfm.vlm.blip2itm"] = stub
    sys.modules.pop("vlfm.mapping.frontier_map", None)
    from vlfm.mapping.frontier_map import FrontierMap  # type: ignore

    return FrontierMap


def geometry_utils():
    _ensure_path()
    import vlfm.utils.geometry_utils as g  # type: ignore

    return g


def img_utils():
    _ensure_path()
    import vlfm.utils.img_utils as g  # type: ignore

    return g


def object_map_module():
    """vlfm.mapping.object_point_cloud_map imports ``open3d`` (absent offline).  A stub module is injected whose
    ``PointCloud.cluster_dbscan`` is scikit-learn's DBSCAN (an independent implementation of the same published algorithm with
    the same sequential cluster numbering), so the reference's own code runs unmodified around it."""
    _ensure_path()
    if "open3d" not in sys.modules:
        import numpy as np

        o3d = types.ModuleType("open3d")
        geometry = types.ModuleType("open3d.geometry")
        utility = types.ModuleType("open3d.utility")

        class PointCloud:
            def __init__(self):
                self.points = None

            def cluster_dbscan(self, eps, min_points, print_progress=False):
                from sklearn.cluster import DBSCAN

                pts = np.asarray(self.points, dtype=np.float64)
                if len(pts) == 0:
                    return []
                return DBSCAN(eps=eps, min_samples=min_points, algorithm="brute").fit(pts).labels_.tolist()

        geometry.PointCloud = PointCloud
        utility.Vector3dVector = lambda a: np.asarray(a, dtype=np.float64)
        o3d.geometry, o3d.utility = geometry, utility
        sys.modules["open3d"] = o3d
        sys.modules["open3d.geometry"] = geometry
        sys.modules["open3d.utility"] = utility
    import vlfm.mapping.object_point_cloud_map as m  # type: ignore

    return m
