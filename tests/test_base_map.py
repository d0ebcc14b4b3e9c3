"""BaseMap conversions (vlfm/mapping/base_map.py:35-60): explicit formulae, and what the reference class returned for the same
points (stored under tests/golden/)."""
import os

import numpy as np
import pytest

from oracle import golden
from vlfm_b200.mapping.base_map import BaseMap


def _ref_xy_to_px(points, size, ppm):          # the reference's arithmetic, array form
    origin = np.array([size // 2, size // 2])
    px = np.rint(points[:, ::-1] * ppm) + origin
    px[:, 0] = size - px[:, 0]
    return px.astype(int)


def _ref_px_to_xy(px, size, ppm):
    origin = np.array([size // 2, size // 2])
    q = px.copy()
    q[:, 0] = size - q[:, 0]
    return ((q - origin) / ppm)[:, ::-1]


@pytest.mark.parametrize("size,ppm", [(1000, 20), (2500, 50), (301, 20), (4000, 40)])
def test_conversions_match_reference_arithmetic(size, ppm):
    rng = np.random.default_rng(size + ppm)
    m = BaseMap(size=size, pixels_per_meter=ppm)
    pts = rng.uniform(-size / ppm / 2, size / ppm / 2, (500, 2))
    pts[:8] = np.array([[0.0, 0.0], [0.025, -0.025], [0.075, 0.125], [1.0, -1.0], [-0.5, 0.5], [2.5 / ppm, 0.5 / ppm], [-1.5 / ppm, 3.5 / ppm], [12.3, -7.7]])
    got = m._xy_to_px(pts)
    assert got.dtype.kind == "i" and np.array_equal(got, _ref_xy_to_px(pts, size, ppm))       # incl. the half-to-even ties
    cells_i = rng.integers(0, size, (200, 2))
    cells_f = rng.uniform(0, size, (200, 2))                                                   # frontier midpoints are fractional
    for cells in (cells_i, cells_f):
        assert np.array_equal(m._px_to_xy(cells), _ref_px_to_xy(cells, size, ppm))
    m.update_agent_traj(np.array([1.0, 2.0]), 0.3)
    assert len(m._camera_positions) == 1 and m._last_camera_yaw == 0.3
    m.reset()
    assert m._camera_positions == []


def run_conversions(m):
    """`m` is a BaseMap-shaped object of size 1000."""
    rng = np.random.default_rng(5)
    pts = rng.uniform(-20, 20, (1000, 2))
    cells = rng.uniform(0, 1000, (300, 2))
    return {"xy_to_px": m._xy_to_px(pts), "px_to_xy": m._px_to_xy(cells), "origin": np.asarray(m._episode_pixel_origin),
            "ppm": np.array(m.pixels_per_meter)}


def test_conversions_match_live_reference_class(golden_dir):
    """The reference class's results on the same points are stored in tests/golden/ref_base_map.npz (oracle/make_golden.py)."""
    golden.check(run_conversions(BaseMap(size=1000)), os.path.join(golden_dir, "ref_base_map.npz"))
