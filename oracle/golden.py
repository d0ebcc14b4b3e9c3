"""Compact storage of reference outputs under tests/golden/ (one compressed .npz per case set).

TEST INFRASTRUCTURE.  A case set is a dict of named arrays.  Small arrays are stored as they are (0/1 grids bit-packed,
mostly-zero grids as flat indices + values); an array whose stored form would exceed INLINE_BYTES compressed is stored as its
shape and the sha256 of its values in float64.  ``check`` compares a freshly computed case set with a stored one exactly, with
``np.array_equal`` semantics either way (values compared, dtype ignored, -0.0 == 0.0).
"""
from __future__ import annotations

import hashlib
import zlib
from typing import Dict

import numpy as np

INLINE_BYTES = 8192


def digest(*arrays) -> str:
    """sha256 over the bytes of the inputs a case set was generated from (detects drift of the synthetic generators)."""
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def value_digest(a: np.ndarray) -> str:
    a = np.asarray(a)
    assert a.dtype.kind in "biuf", a.dtype
    canon = np.ascontiguousarray(a, dtype=np.float64) + 0.0            # + 0.0 turns -0.0 into 0.0
    assert not np.isnan(canon).any()                                    # NaN never compares equal
    return digest(np.array(a.shape, dtype=np.int64), canon)


def _encode(name: str, a: np.ndarray) -> Dict[str, np.ndarray]:
    if a.dtype.kind in "biu" and a.size > 64 and not np.any((a != 0) & (a != 1)):
        return {name + "~bits": np.packbits(a.reshape(-1).astype(bool)), name + "~shape": np.array(a.shape, dtype=np.int64),
                name + "~dtype": np.array(a.dtype.str)}
    if a.dtype.kind == "f" and a.size > 4096 and np.count_nonzero(a) < a.size // 4:
        flat = a.reshape(-1)
        idx = np.flatnonzero(flat)
        return {name + "~idx": idx.astype(np.int32), name + "~val": flat[idx], name + "~shape": np.array(a.shape, dtype=np.int64)}
    return {name: a}


def save(path: str, arrays: Dict[str, np.ndarray]) -> None:
    out = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        enc = _encode(name, a)
        if a.dtype.kind in "biuf" and len(zlib.compress(b"".join(v.tobytes() for v in enc.values()))) > INLINE_BYTES:
            enc = {name + "~sha256": np.array(value_digest(a)), name + "~shape": np.array(a.shape, dtype=np.int64)}
        out.update(enc)
    np.savez_compressed(path, **out)


def load(path: str) -> Dict[str, object]:
    """name -> array, or name -> (shape, sha256) for an array stored as its digest."""
    z = np.load(path)
    got = {}
    for key in z.files:
        name, _, kind = key.partition("~")
        shape = tuple(int(s) for s in z[name + "~shape"]) if kind else None
        if kind == "bits":
            got[name] = np.unpackbits(z[key], count=int(np.prod(shape))).astype(str(z[name + "~dtype"])).reshape(shape)
        elif kind == "val":
            a = np.zeros(int(np.prod(shape)), dtype=z[key].dtype)
            a[z[name + "~idx"]] = z[key]
            got[name] = a.reshape(shape)
        elif kind == "sha256":
            got[name] = (shape, str(z[key]))
        elif not kind:
            got[name] = z[key]
    return got


def check(got: Dict[str, np.ndarray], path: str, prefix: str = "") -> None:
    """Assert that `got` holds exactly the arrays stored under `prefix` in `path`, with equal values."""
    want = {k[len(prefix):]: v for k, v in load(path).items() if k.startswith(prefix)}
    assert sorted(got) == sorted(want), (sorted(got), sorted(want))
    for k, a in got.items():
        a = np.asarray(a)
        if isinstance(want[k], tuple):
            shape, sha = want[k]
            assert a.shape == shape, (k, a.shape, shape)
            assert value_digest(a) == sha, f"{k}: values differ from the stored reference output"
        else:
            assert np.array_equal(a, want[k]), k
