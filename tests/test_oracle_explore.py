"""Explore half of the obstacle map: the cv2-based restatement and the cv2-free one agree, and the reference's
own ObstacleMap code (run with the restated frontier_exploration functions injected) agrees with both: its outputs are stored
under tests/golden/."""
import os

import numpy as np

import oracle.explore_oracle as ex
from oracle import golden
from oracle.obstacle_map_oracle import ObstacleMapOracle
from vlfm_b200.utils.synthetic import focal_from_hfov, trajectory


def _run(prims, seed, steps, hw, size, start=(0.0, 0.0), bound=4.0, depth_scale=1.0):
    ex.PRIMS = prims
    try:
        o = ObstacleMapOracle(0.61, 0.88, 0.18, area_thresh=1.5, hole_area_thresh=-1, size=size)
        fx = focal_from_hfov(hw[1])
        out = []
        for f in trajectory(seed, steps, h=hw[0], w=hw[1], bound_m=bound, start_xy=start):
            o.update_map(f.depth * np.float32(depth_scale), f.tf, 0.5, 5.0, fx, fx, np.deg2rad(79))
            out.append((o.explored_area.copy(), np.asarray(o._frontiers_px).copy(), np.asarray(o.frontiers).copy()))
        return out
    finally:
        ex.PRIMS = "cv2"


def test_cv2_and_numpy_backends_agree():
    for seed in range(3):
        a = _run("cv2", seed, 6, (120, 160), 400)
        b = _run("numpy", seed, 6, (120, 160), 400)
        assert a[-1][0].sum() > 100
        for (ea, fa, xa), (eb, fb, xb) in zip(a, b):
            assert np.array_equal(ea, eb) and fa.shape == fb.shape and np.array_equal(fa, fb) and np.array_equal(xa, xb)


def test_backends_agree_at_the_map_border():
    """agent within max_depth of the grid edge (walls close enough that no obstacle cell leaves the grid, which would be the
    reference's IndexError): the 5 m cone and the occlusion rays are clipped by cv2 (clipLine rules)"""
    for seed, start in ((0, (8.2, 8.2)), (1, (-8.2, 8.2)), (2, (8.2, -8.2)), (3, (-8.2, -8.2)), (4, (0.0, 8.3)), (5, (-8.3, 0.5))):
        a = _run("cv2", seed, 6, (120, 160), 400, start=start, bound=0.4, depth_scale=0.15)
        b = _run("numpy", seed, 6, (120, 160), 400, start=start, bound=0.4, depth_scale=0.15)
        assert a[-1][0].sum() > 50
        for (ea, fa, xa), (eb, fb, xb) in zip(a, b):
            assert np.array_equal(ea, eb) and fa.shape == fb.shape and np.array_equal(fa, fb) and np.array_equal(xa, xb)


def run_reference_class_case(cls):
    """explored area and frontiers of `cls` (an ObstacleMap-shaped class) after each of six seeded updates."""
    m = cls(0.61, 0.88, 0.18, area_thresh=1.5, hole_area_thresh=-1, size=400)
    fx = focal_from_hfov(160)
    frames = trajectory(7, 6, h=120, w=160, bound_m=4)
    out = {"inputs": np.array(golden.digest(*[a for f in frames for a in (f.depth, f.tf)]))}
    for i, f in enumerate(frames):
        m.update_map(f.depth, f.tf, 0.5, 5.0, fx, fx, np.deg2rad(79))
        out[f"explored_{i}"] = m.explored_area.copy()
        out[f"frontiers_px_{i}"] = np.asarray(m._frontiers_px).copy()
        out[f"frontiers_{i}"] = np.asarray(m.frontiers).copy()
    return out


def test_reference_class_with_injected_functions(golden_dir):
    """The reference's own ObstacleMap (restated frontier_exploration functions injected) on the same inputs is stored in
    tests/golden/ref_explore.npz (oracle/make_golden.py)."""
    golden.check(run_reference_class_case(ObstacleMapOracle), os.path.join(golden_dir, "ref_explore.npz"))
