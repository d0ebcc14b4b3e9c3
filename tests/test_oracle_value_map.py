"""Pin oracle/value_map_oracle.py against the committed fixtures generated from the real
reference (oracle/make_golden.py), with the cv2 and the numpy primitive back-ends."""
import glob
import hashlib
import os

import numpy as np
import pytest

from oracle import golden
from oracle.value_map_oracle import ValueMapOracle
from vlfm_b200.utils.synthetic import trajectory

FOV = float(np.deg2rad(79.0))


def _digest(frames):
    h = hashlib.sha256()
    for f in frames:
        h.update(np.ascontiguousarray(f.depth).tobytes())
        h.update(np.ascontiguousarray(f.tf).tobytes())
    return h.hexdigest()


def load_case(path):
    z = np.load(path)
    h, w = (int(v) for v in z["hw"])
    frames = trajectory(int(z["seed"]), int(z["steps"]), h=h, w=w, bound_m=float(z["bound"]))
    assert _digest(frames) == str(z["input_sha256"]), "synthetic generator drifted from the fixtures"
    return z, frames


def dense(idx, val, shape, dtype):
    out = np.zeros(int(np.prod(shape)), dtype=dtype)
    out[idx] = val
    return out.reshape(shape)


@pytest.mark.parametrize("prims", ["cv2", "numpy"])
def test_oracle_matches_golden(golden_dir, prims):
    paths = sorted(glob.glob(os.path.join(golden_dir, "vm_*.npz")))
    assert paths
    for path in paths:
        z, frames = load_case(path)
        size, ch = int(z["size"]), int(z["channels"])
        o = ValueMapOracle(ch, size=size, use_max_confidence=bool(z["use_max_confidence"]), fusion_type=str(z["fusion"]), prims=prims)
        for f, v in zip(frames, z["values"]):
            o.update_map(v, f.depth, f.tf, 0.5, 5.0, FOV)
        conf = dense(z["conf_idx"], z["conf_val"], (size, size), np.float32)
        val = dense(z["value_idx"], z["value_val"], (size, size, ch), np.float64)
        assert np.array_equal(o._map, conf), path
        assert np.array_equal(o._value_map.astype(np.float64), val), path
        red = (lambda s: [max(t) for t in s]) if ch > 1 else None
        sw, sv = o.sort_waypoints(z["waypoints"], 0.5, reduce_fn=red)
        assert np.array_equal(sw, z["sorted_wp"]) and np.allclose(np.asarray(sv, float), z["sorted_val"], rtol=0, atol=0)


LIVE_CASES = [(1, False, "default", 700, 21), (2, True, "default", 500, 22)]


def run_live_cases(make):
    """make(channels, size, use_max_confidence, fusion_type) -> a value map; the grids after five seeded updates per case."""
    out = {}
    for ch, maxc, fus, size, seed in LIVE_CASES:
        m = make(ch, size, maxc, fus)
        rng = np.random.default_rng(seed)
        frames = trajectory(seed, 5, bound_m=size / 40 - 6)
        for f in frames:
            m.update_map(rng.random(ch), f.depth, f.tf, 0.5, 5.0, FOV)
        out[f"s{seed}_inputs"] = np.array(_digest(frames))
        out[f"s{seed}_conf"], out[f"s{seed}_value"] = m._map, m._value_map
    return out


def run_ppm40(make):
    """make(size) -> a value map at 40 pixels per metre (configs[4]/[5] geometry)."""
    m = make(1000)
    rng = np.random.default_rng(9)
    frames = trajectory(62, 2, h=128, w=128, bound_m=6.0)
    for f in frames:
        m.update_map(rng.random(1), f.depth, f.tf, 0.5, 5.0, FOV)
    return {"inputs": np.array(_digest(frames)), "conf": m._map, "value": m._value_map}


def test_oracle_matches_live_reference(golden_dir):
    """The reference class's grids on the same inputs are stored in tests/golden/ref_value_map_live.npz (oracle/make_golden.py)."""
    got = run_live_cases(lambda ch, size, maxc, fus: ValueMapOracle(ch, size=size, use_max_confidence=maxc, fusion_type=fus,
                                                                      prims="numpy"))
    golden.check(got, os.path.join(golden_dir, "ref_value_map_live.npz"))


def test_oracle_ppm40_matches_patched_reference(golden_dir):
    """configs[4]/[5] geometry: the reference needs `pixels_per_meter` patched and its cone cache cleared
    (value_map.py:65, :339); the oracle takes ppm as a parameter.  Reference grids: tests/golden/ref_value_map_ppm40.npz."""
    got = run_ppm40(lambda size: ValueMapOracle(1, size=size, use_max_confidence=False, pixels_per_meter=40, prims="numpy"))
    golden.check(got, os.path.join(golden_dir, "ref_value_map_ppm40.npz"))
