"""Generate tests/golden/*.npz by running the REAL reference.

Usage:  VLFM_REFERENCE=<checkout of the original vlfm repository> python oracle/make_golden.py
Inputs are regenerated from vlfm_b200.utils.synthetic with the recorded seeds (an input
checksum is stored so generator drift is detected); outputs are stored sparsely (flat
indices + values of non-zero cells, bit-packed 0/1 grids).  The ref_*.npz case sets are
produced by the tests' own run_* functions (tests/test_*.py), called here with the
reference classes and there with the oracle / product classes.
"""
from __future__ import annotations

import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import golden, ref_import  # noqa: E402
from vlfm_b200.utils.synthetic import focal_from_hfov, trajectory  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
FOV = float(np.deg2rad(79.0))

VALUE_CASES = [
    # name, channels, use_max_conf, fusion, size, seed, steps, (H, W), bound
    ("vm_weighted", 1, False, "default", 480, 11, 6, (480, 640), 5.0),
    ("vm_maxconf_c2", 2, True, "default", 480, 12, 6, (480, 640), 5.0),
    ("vm_edge_clip", 1, False, "default", 260, 13, 5, (240, 320), 6.2),
    ("vm_replace", 1, False, "replace", 400, 14, 4, (120, 160), 3.0),
    ("vm_equal", 1, False, "equal_weighting", 400, 15, 4, (120, 160), 3.0),
]


def digest(frames) -> str:
    h = hashlib.sha256()
    for f in frames:
        h.update(np.ascontiguousarray(f.depth).tobytes())
        h.update(np.ascontiguousarray(f.tf).tobytes())
    return h.hexdigest()


def sparse(a: np.ndarray):
    flat = a.reshape(-1)
    idx = np.flatnonzero(flat)
    return idx.astype(np.int32), flat[idx]


def value_cases() -> None:
    RV = ref_import.value_map_class()
    for name, ch, maxc, fus, size, seed, steps, (h, w), bound in VALUE_CASES:
        RV._confidence_masks.clear()
        ref = RV(ch, size=size, use_max_confidence=maxc, fusion_type=fus)
        frames = trajectory(seed, steps, h=h, w=w, bound_m=bound)
        rng = np.random.default_rng(seed)
        vals = rng.random((steps, ch))
        for f, v in zip(frames, vals):
            ref.update_map(v, f.depth, f.tf, 0.5, 5.0, FOV)
        ci, cv = sparse(ref._map)
        vi, vv = sparse(ref._value_map)
        wps = np.array([[f.xy[0] + 0.4, f.xy[1] - 0.3] for f in frames])
        red = (lambda s: [max(t) for t in s]) if ch > 1 else None
        sw, sv = ref.sort_waypoints(wps, 0.5, reduce_fn=red)
        np.savez_compressed(
            os.path.join(OUT, name + ".npz"),
            channels=ch, use_max_confidence=maxc, fusion=fus, size=size, seed=seed, steps=steps,
            hw=np.array([h, w]), bound=bound, values=vals, input_sha256=digest(frames),
            conf_idx=ci, conf_val=cv, value_idx=vi, value_val=vv.astype(np.float64),
            value_dtype=str(ref._value_map.dtype), waypoints=wps, sorted_wp=sw,
            sorted_val=np.asarray(sv, dtype=np.float64),
        )
        print(name, "conf nz", ci.size, "value nz", vi.size)


def _save(name: str, arrays) -> None:
    path = os.path.join(OUT, name + ".npz")
    golden.save(path, arrays)
    print(name, len(arrays), "arrays", os.path.getsize(path), "bytes")


def live_cases() -> None:
    """The reference side of the tests that compare a restatement with the reference class on the same inputs."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_base_map
    import test_frontier_map
    import test_oracle_explore
    import test_oracle_object_map
    import test_oracle_obstacle
    import test_oracle_value_map

    RV = ref_import.value_map_class()

    def value_map(ch, size, maxc, fus, ppm=None):
        RV._confidence_masks.clear()
        m = RV(ch, size=size, use_max_confidence=maxc, fusion_type=fus)
        if ppm is not None:            # value_map.py:65 fixes 20 px/m; the cone cache (value_map.py:339) is per class
            m.pixels_per_meter = ppm
        return m

    _save("ref_value_map_live", test_oracle_value_map.run_live_cases(value_map))
    _save("ref_value_map_ppm40", test_oracle_value_map.run_ppm40(lambda size: value_map(1, size, False, "default", ppm=40)))
    RV._confidence_masks.clear()

    RO = ref_import.obstacle_map_class()
    out = {}
    for hole in (-1, 100000):
        out.update({f"hole{hole}_{k}": v for k, v in test_oracle_obstacle.run_obstacle_half(RO, hole).items()})
    _save("ref_obstacle_half", out)
    _save("ref_explore", test_oracle_explore.run_reference_class_case(RO))

    RF = ref_import.frontier_map_class(test_frontier_map.ScriptedEncoder)
    out = {}
    for seed in (0, 1, 2):
        fm = RF()
        fm.frontiers = []              # a class attribute in the reference
        out.update({f"s{seed}_{k}": v for k, v in test_frontier_map.run_stream(fm, seed).items()})
    _save("ref_frontier_map", out)

    R = ref_import.object_map_module().ObjectPointCloudMap

    def object_map():
        m = R(erosion_size=2)
        m.reset()
        return m

    out = {}
    for use_dbscan in (True, False):
        out.update({f"dbscan{int(use_dbscan)}_{k}": v for k, v in test_oracle_object_map.run_scenarios(object_map, use_dbscan).items()})
    _save("ref_object_map", out)

    _save("ref_base_map", test_base_map.run_conversions(ref_import.base_map_class()(size=1000)))


if __name__ == "__main__":
    assert ref_import.available(), "set VLFM_REFERENCE to a checkout of the original vlfm repository"
    os.makedirs(OUT, exist_ok=True)
    value_cases()
    live_cases()
