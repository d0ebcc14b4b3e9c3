"""oracle/object_map_oracle.py: DBSCAN restatement vs scikit-learn's implementation; the whole class vs what the REAL reference
class (vlfm/mapping/object_point_cloud_map.py, imported with a stub open3d) returned on the same scenarios, stored under
tests/golden/."""
import os

import cv2
import numpy as np
import pytest

from oracle import golden
from oracle import object_map_oracle as om
from vlfm_b200.utils.synthetic import focal_from_hfov, make_object_mask, trajectory


def _clustered(rng, n):
    k = int(rng.integers(1, 5))
    parts = []
    for _ in range(k):
        c = rng.uniform(-2, 2, 3)
        parts.append(c + rng.normal(0, rng.uniform(0.03, 0.25), (int(n // k), 3)))
    parts.append(rng.uniform(-3, 3, (n // 10, 3)))
    p = np.concatenate(parts)
    return p[rng.permutation(len(p))]


def test_dbscan_labels_match_sklearn():
    from sklearn.cluster import DBSCAN

    rng = np.random.default_rng(0)
    for t in range(12):
        pts = _clustered(rng, int(rng.integers(300, 2500)))
        mp = [100, 40, 10][t % 3]
        ref = DBSCAN(eps=0.2, min_samples=mp, algorithm="brute").fit(pts).labels_
        got = om.dbscan_labels(pts, 0.2, mp)
        assert np.array_equal(ref, got), (t, (ref != got).sum())
    assert len(om.dbscan_filter(rng.uniform(-50, 50, (500, 3)))) == 0          # only noise


def test_erode_restatement():
    rng = np.random.default_rng(1)
    for k in (0, 1, 2, 3):
        m = make_object_mask(rng, 120, 160)
        m[:, :3] = 1                                                           # touches the image edge: the border does not erode
        assert np.array_equal(cv2.erode(m * 255, None, iterations=k), om.erode_mask_numpy(m, k))


def _scenario(seed, steps=6, h=240, w=320):
    rng = np.random.default_rng(100 + seed)
    fx = focal_from_hfov(w)
    out = []
    for i, f in enumerate(trajectory(seed, steps, h=h, w=w, bound_m=6.0)):
        side = ["any", "left", "any", "right", "any"][i % 5]
        mask = make_object_mask(rng, h, w, side)
        depth = f.depth.copy()
        if i % 3 == 2:
            depth[mask > 0] = np.float32(0.98)                                # a far detection: out-of-range ids
        out.append((depth, mask, f.tf, fx))
    return out


def run_scenarios(make, use_dbscan):
    """has_object / cloud / best object / target cloud of the map `make()` returns, after each update of three seeded scenarios."""
    out = {}
    for seed in range(3):
        m = make()
        m.use_dbscan = use_dbscan
        for i, (depth, mask, tf, fx) in enumerate(_scenario(seed)):
            np.random.seed(7 + seed)
            m.update_map("chair", depth, mask, tf, 0.5, 5.0, fx, fx)
            m.update_explored(tf, 5.0, np.deg2rad(79))
            key = f"s{seed}_{i}_"
            out[key + "has"] = np.array(m.has_object("chair"))
            if m.has_object("chair"):
                out[key + "cloud"] = m.clouds["chair"]
                out[key + "best"] = m.get_best_object("chair", tf[:2, 3] + 0.3)
                out[key + "target"] = m.get_target_cloud("chair")
    return out


@pytest.mark.parametrize("use_dbscan", [True, False])
def test_oracle_class_matches_the_reference_class(golden_dir, use_dbscan):
    """The reference class's results on the same scenarios are stored in tests/golden/ref_object_map.npz (oracle/make_golden.py)."""
    got = run_scenarios(lambda: om.ObjectPointCloudMapOracle(erosion_size=2), use_dbscan)
    golden.check(got, os.path.join(golden_dir, "ref_object_map.npz"), f"dbscan{int(use_dbscan)}_")
