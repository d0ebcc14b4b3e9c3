import os

import numpy as np
import pytest

from oracle import golden
from oracle.obstacle_map_oracle import ObstacleMapOracle
from vlfm_b200.utils.synthetic import focal_from_hfov, trajectory

OBSTACLE_CASES = [(0, (240, 320), 600, 20), (2, (240, 320), 1500, 50)]


def run_obstacle_half(cls, hole):
    """The obstacle / navigable grids of `cls` (an ObstacleMap-shaped class) after four seeded updates per case."""
    out = {}
    for seed, (h, w), size, ppm in OBSTACLE_CASES:
        m = cls(0.61, 0.88, 0.18, area_thresh=1.5, hole_area_thresh=hole, size=size, pixels_per_meter=ppm)
        fx = focal_from_hfov(w)
        frames = trajectory(seed, 4, h=h, w=w, bound_m=5)
        for f in frames:
            m.update_map(f.depth, f.tf, 0.5, 5.0, fx, fx, np.deg2rad(79), explore=False)
        out[f"s{seed}_inputs"] = np.array(golden.digest(*[a for f in frames for a in (f.depth, f.tf)]))
        out[f"s{seed}_map"], out[f"s{seed}_navigable"] = m._map, m._navigable_map
    return out


@pytest.mark.parametrize("hole", [-1, 100000])
def test_obstacle_half_matches_live_reference(golden_dir, hole):
    """The reference class's grids on the same inputs are stored in tests/golden/ref_obstacle_half.npz (oracle/make_golden.py)."""
    golden.check(run_obstacle_half(ObstacleMapOracle, hole), os.path.join(golden_dir, "ref_obstacle_half.npz"), f"hole{hole}_")


def _depth_with_holes(seed, h=60, w=80):
    rng = np.random.default_rng(seed)
    d = rng.uniform(0.05, 1.0, (h, w)).astype(np.float32)
    yy, xx = np.mgrid[0:h, 0:w]
    for _ in range(int(rng.integers(2, 6))):
        cy, cx, r = rng.integers(0, h), rng.integers(0, w), rng.integers(3, 14)
        d[(yy - cy) ** 2 + (xx - cx) ** 2 <= r * r] = 0
        if r > 6:
            d[(yy - cy) ** 2 + (xx - cx) ** 2 <= (r // 2) ** 2] = 0.5
            d[(yy - cy) ** 2 + (xx - cx) ** 2 <= (r // 4) ** 2] = 0
    d[rng.random((h, w)) < 0.02] = 0
    return d


@pytest.mark.parametrize("thresh", [5, 40, 200, 100000])
def test_fill_holes_restatement_matches_cv2(thresh):
    """oracle.fill_holes_numpy (the rules the GPU kernel follows) against the cv2 calls the reference makes
    (vlfm/utils/img_utils.py:361-390)."""
    cv2 = pytest.importorskip("cv2")
    from oracle import contours as ct
    from oracle.obstacle_map_oracle import fill_holes, fill_holes_numpy

    for seed in range(12):
        d = _depth_with_holes(seed * 13 + thresh)
        assert np.array_equal(fill_holes(d, thresh), fill_holes_numpy(d, thresh))
        holes = (d == 0).astype(np.uint8)
        want = sorted(tuple(map(tuple, c.reshape(-1, 2))) for c in cv2.findContours(holes, cv2.RETR_TREE, cv2.CHAIN_APPROX_NONE)[0])
        got = sorted(tuple(map(tuple, c.reshape(-1, 2))) for c in ct.find_all_contours(holes))
        assert got == want
