"""CPU restatement of vlfm/mapping/object_point_cloud_map.py (SURVEY.md section 8 row f4).

TEST INFRASTRUCTURE (see oracle/__init__.py).

Pinning: everything except the DBSCAN call is checked bit-for-bit against what the REAL reference class, run with a stub
``open3d`` module injected, returned on the same scenarios (tests/test_oracle_object_map.py, tests/golden/).  ``open3d`` itself (``open3d``,
unpinned, README.md:45 / docker/Dockerfile) is ABSENT: ``dbscan_labels`` restates the published DBSCAN algorithm with
Open3D's sequential cluster numbering (``PointCloud::ClusterDBSCAN``: radius neighbourhoods incl. the point itself, a point
is core when it has >= min_points neighbours, clusters are grown one after the other from the lowest-index unlabelled core
point, a border point keeps the FIRST cluster that reaches it) and is pinned against scikit-learn's independent
implementation of the same algorithm (``sklearn.cluster.DBSCAN``, same sequential semantics) on random clouds.  PARITY
UNPINNED with respect to the Open3D binary (its radius test is strict ``<`` in nanoflann, ``<=`` here and in scikit-learn:
they differ only for a pair of points at exactly eps).

Randomness: the reference draws from numpy's GLOBAL generator (``np.random.rand`` for the range ids, ``np.random.choice`` for
the 5000-point subsample); so does this restatement and the GPU class, in the same order -- seed ``np.random.seed`` to compare.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np


def erode_mask(mask: np.ndarray, iterations: int) -> np.ndarray:
    """cv2.erode(mask * 255, None, iterations=k) (object_point_cloud_map.py:153-154): 3x3 kernel, k times = one (2k+1)^2
    erosion; cv2's default border value for erosion is +inf, i.e. the image edge does not erode anything."""
    import cv2

    return cv2.erode(mask * 255, None, iterations=iterations)


def erode_mask_numpy(mask: np.ndarray, iterations: int) -> np.ndarray:
    m = (mask != 0)
    k = int(iterations)
    if k <= 0:
        return (mask * 255)
    h, w = m.shape
    p = np.ones((h + 2 * k, w + 2 * k), dtype=bool)          # outside the image counts as set
    p[k:k + h, k:k + w] = m
    out = np.ones((h, w), dtype=bool)
    for dy in range(2 * k + 1):
        for dx in range(2 * k + 1):
            out &= p[dy:dy + h, dx:dx + w]
    return (out * 255).astype(mask.dtype)


def object_cloud(depth: np.ndarray, mask: np.ndarray, min_depth: float, max_depth: float, fx: float, fy: float) -> np.ndarray:
    """valid-depth conversion + get_point_cloud (object_point_cloud_map.py:156-159, geometry_utils.py:216-236), row-major order"""
    valid = depth.copy()
    valid[valid == 0] = 1
    valid = valid * (max_depth - min_depth) + min_depth
    v, u = np.where(mask)
    z = valid[v, u]
    x = (u - valid.shape[1] // 2) * z / fx
    y = (v - valid.shape[0] // 2) * z / fy
    return np.stack((z, -x, -y), axis=-1)


def dbscan_labels(points: np.ndarray, eps: float = 0.2, min_points: int = 100) -> np.ndarray:
    """Open3D ``cluster_dbscan`` labels (-1 noise, clusters 0.. in order of their lowest-index core point)."""
    n = len(points)
    labels = np.full(n, -1, dtype=np.int64)
    if n == 0:
        return labels
    p = np.asarray(points, dtype=np.float64)[:, :3]
    adj = np.zeros((n, n), dtype=bool)
    step = 1024
    for a in range(0, n, step):
        d = p[a:a + step, None, :] - p[None, :, :]
        d2 = d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]
        d2 = d2 + d[..., 2] * d[..., 2]
        adj[a:a + step] = d2 <= eps * eps
    core = adj.sum(1) >= min_points
    # connected components of the core points (edges = adjacency), numbered by their lowest member
    root = np.arange(n)
    cores = np.nonzero(core)[0]
    comp = np.full(n, -1, dtype=np.int64)
    for i in cores:
        if comp[i] >= 0:
            continue
        stack = [i]
        comp[i] = i
        while stack:
            q = stack.pop()
            nb = np.nonzero(adj[q] & core & (comp < 0))[0]
            comp[nb] = i
            stack.extend(nb.tolist())
    roots = np.unique(comp[cores]) if len(cores) else np.array([], dtype=np.int64)
    number = {int(r): k for k, r in enumerate(roots)}             # ascending root = order in which Open3D seeds them
    for i in cores:
        labels[i] = number[int(comp[i])]
    # border points: the first (lowest-numbered) cluster with a core point within eps
    for i in np.nonzero(~core)[0]:
        nb = np.nonzero(adj[i] & core)[0]
        if len(nb):
            labels[i] = min(number[int(comp[j])] for j in nb)
    return labels


def dbscan_filter(points: np.ndarray, eps: float = 0.2, min_points: int = 100) -> np.ndarray:
    """open3d_dbscan_filtering (object_point_cloud_map.py:192-219): points of the largest non-noise cluster, in input order."""
    labels = dbscan_labels(points, eps, min_points)
    uniq, counts = np.unique(labels, return_counts=True)
    keep = uniq != -1
    uniq, counts = uniq[keep], counts[keep]
    if len(uniq) == 0:
        return np.array([])
    best = uniq[np.argmax(counts)]
    return points[np.where(labels == best)[0]]


def random_subarray(points: np.ndarray, size: int) -> np.ndarray:
    if len(points) <= size:
        return points
    return points[np.random.choice(len(points), size, replace=False)]


def too_offset(mask: np.ndarray) -> bool:
    import cv2

    x, y, w, h = cv2.boundingRect(mask)
    third = mask.shape[1] // 3
    if x + w <= third:
        return x <= int(0.05 * mask.shape[1])
    if x >= 2 * third:
        return x + w >= int(0.95 * mask.shape[1])
    return False


def transform_points(tf: np.ndarray, pts: np.ndarray) -> np.ndarray:
    hom = np.hstack((pts, np.ones((pts.shape[0], 1))))
    out = np.dot(tf, hom.T).T
    return out[:, :3] / out[:, 3:]


def within_fov_cone(origin: np.ndarray, angle: float, fov: float, rng: float, points: np.ndarray) -> np.ndarray:
    d = points[:, :3] - origin
    dist = np.linalg.norm(d, axis=1)
    ang = np.arctan2(d[:, 1], d[:, 0])
    diff = np.mod(ang - angle + np.pi, 2 * np.pi) - np.pi
    return points[np.logical_and(dist <= rng, np.abs(diff) <= fov / 2)]


class ObjectPointCloudMapOracle:
    use_dbscan: bool = True

    def __init__(self, erosion_size: float) -> None:
        self._erosion_size = erosion_size
        self.clouds: Dict[str, np.ndarray] = {}
        self.last_target_coord: Optional[np.ndarray] = None

    def reset(self) -> None:
        self.clouds = {}
        self.last_target_coord = None

    def has_object(self, name: str) -> bool:
        return name in self.clouds and len(self.clouds[name]) > 0

    def extract(self, depth, mask, min_depth, max_depth, fx, fy) -> np.ndarray:
        final = erode_mask(mask, self._erosion_size)
        cloud = random_subarray(object_cloud(depth, final, min_depth, max_depth, fx, fy), 5000)
        return dbscan_filter(cloud) if self.use_dbscan else cloud

    def update_map(self, name, depth, mask, tf, min_depth, max_depth, fx, fy) -> None:
        local = self.extract(depth, mask, min_depth, max_depth, fx, fy)
        if len(local) == 0:
            return
        if too_offset(mask):
            within = np.ones_like(local[:, 0]) * np.random.rand()
        else:
            within = ((local[:, 0] <= max_depth * 0.95) * 1.0).astype(np.float32)
            within[within == 0] = np.random.rand()
        glob = np.concatenate((transform_points(tf, local), within[:, None]), axis=1)
        pos = tf[:3, 3]
        closest = self.closest_point(glob, pos)
        if np.linalg.norm(closest[:3] - pos) < 1.0:
            return
        self.clouds[name] = np.concatenate((self.clouds[name], glob), axis=0) if name in self.clouds else glob

    def closest_point(self, cloud: np.ndarray, pos: np.ndarray) -> np.ndarray:
        nd = pos.shape[0]
        if self.use_dbscan:
            return cloud[np.argmin(np.linalg.norm(cloud[:, :nd] - pos, axis=1))]
        ref = np.concatenate((pos, np.array([0.5]))) if nd == 2 else pos
        order = np.argsort(np.linalg.norm(cloud[:, :3] - ref, axis=1))
        top = order[: int(0.25 * len(cloud))]
        try:
            idx = top[int(len(top) / 2)]
        except IndexError:
            idx = 0
        return cloud[idx]

    def get_target_cloud(self, name: str) -> np.ndarray:
        c = self.clouds[name].copy()
        if np.any(c[:, -1] == 1):
            c = c[c[:, -1] == 1]
        return c

    def get_best_object(self, name: str, pos: np.ndarray) -> np.ndarray:
        p2 = self.closest_point(self.get_target_cloud(name), pos)[:2]
        if self.last_target_coord is None:
            self.last_target_coord = p2
        else:
            delta = np.linalg.norm(p2 - self.last_target_coord)
            if delta < 0.1:
                return self.last_target_coord
            if delta < 0.5 and np.linalg.norm(pos - p2) > 2.0:
                return self.last_target_coord
            self.last_target_coord = p2
        return self.last_target_coord

    def update_explored(self, tf: np.ndarray, max_depth: float, cone_fov: float) -> None:
        cam = tf[:3, 3]
        yaw = float(np.arctan2(tf[1, 0], tf[0, 0]))
        for obj in self.clouds:
            inside = within_fov_cone(cam, yaw, cone_fov, max_depth * 0.5, self.clouds[obj])
            for rid in set(inside[..., -1].tolist()):
                if rid == 1:
                    continue
                self.clouds[obj] = self.clouds[obj][self.clouds[obj][..., -1] != rid]
