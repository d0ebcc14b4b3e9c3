"""FrontierMap (vlfm/mapping/frontier_map.py:10-77): host bookkeeping around one cosine call per update that introduces a
new frontier.  Checked against explicit expectations, and against what the REAL reference class (its HTTP encoder replaced by
the same scripted one) returned for the same update streams, stored under tests/golden/."""
import os

import numpy as np
import pytest

from oracle import golden
from vlfm_b200.mapping.frontier_map import FrontierMap


class ScriptedEncoder:
    def __init__(self):
        self.calls = 0

    def cosine(self, image, text):
        self.calls += 1
        return 0.1 * self.calls + float(image.sum() % 7) * 1e-3


def _stream(seed, steps=30):
    rng = np.random.default_rng(seed)
    pool = [rng.uniform(-5, 5, 2).round(2) for _ in range(12)]
    out = []
    for _ in range(steps):
        k = int(rng.integers(0, 6))
        idx = rng.choice(len(pool), size=k, replace=False)
        out.append(([pool[i].copy() for i in idx], rng.integers(0, 255, (4, 4, 3), dtype=np.uint8)))
    return out


def test_update_sort_reset_semantics():
    enc = ScriptedEncoder()
    fm = FrontierMap(encoder=enc)
    img = np.zeros((2, 2, 3), np.uint8)
    a, b, c = np.array([1.0, 2.0]), np.array([3.0, 4.0]), np.array([5.0, 6.0])
    fm.update([a, b], img, "x")
    assert enc.calls == 1 and [f.cosine for f in fm.frontiers] == [0.1, 0.1]            # one encode for both new frontiers
    fm.update([b.copy(), c], img, "x")                                                  # a vanished, b kept (array_equal), c new
    assert enc.calls == 2 and len(fm.frontiers) == 2
    assert np.array_equal(fm.frontiers[0].xyz, b) and fm.frontiers[0].cosine == 0.1 and fm.frontiers[1].cosine == 0.2
    fm.update([b, c], img, "x")
    assert enc.calls == 2                                                               # nothing new: no encode
    pts, vals = fm.sort_waypoints()
    assert vals == [0.2, 0.1] and np.array_equal(pts, np.array([c, b]))
    fm.reset()
    assert fm.frontiers == []
    fm.update([], img, "x")
    assert enc.calls == 2 and fm.frontiers == []


def run_stream(fm, seed):
    """Frontier lists (in stored order) and sorted waypoints of `fm` (its encoder a ScriptedEncoder) after each update of the
    seeded stream, concatenated over the updates."""
    counts, xyz, cos, sorted_xyz, sorted_cos = [], [], [], [], []
    for locs, img in _stream(seed):
        fm.update(locs, img, "a chair")
        counts.append(len(fm.frontiers))
        xyz += [f.xyz for f in fm.frontiers]
        cos += [f.cosine for f in fm.frontiers]
        if fm.frontiers:
            pts, vals = fm.sort_waypoints()
            sorted_xyz.append(pts)
            sorted_cos += vals
    return {"counts": np.array(counts), "xyz": np.array(xyz).reshape(-1, 2), "cosine": np.array(cos, dtype=np.float64),
            "sorted_xyz": np.concatenate(sorted_xyz).reshape(-1, 2), "sorted_cosine": np.array(sorted_cos, dtype=np.float64),
            "encoder_calls": np.array(fm.encoder.calls)}


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_matches_live_reference(golden_dir, seed):
    """The reference class's lists on the same stream are stored in tests/golden/ref_frontier_map.npz (oracle/make_golden.py)."""
    golden.check(run_stream(FrontierMap(encoder=ScriptedEncoder()), seed), os.path.join(golden_dir, "ref_frontier_map.npz"), f"s{seed}_")
