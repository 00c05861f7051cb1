"""Stored outputs of the original project's own leaf classes, for the tests that compare the restated oracle with them.

tests/golden/make_golden.py runs those classes (oracle/_ref, compiled from the original sources by oracle/Makefile) and
records what they computed in tests/golden/reference_leaf.npz, so that the comparisons need nothing outside the repository.
Each array is kept as a SHA-256 of its dtype, shape and exact bytes, plus a fixed sample of its elements: equal digests are
the bit-exact comparison, the sample shows what differs when they are not equal."""
import hashlib
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_leaf.npz")
SAMPLE = 64
_STORED = None


def digest(a: np.ndarray) -> str:
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def _sample(a: np.ndarray) -> np.ndarray:
    flat = np.ascontiguousarray(a).reshape(-1)
    return flat[np.unique(np.linspace(0, flat.size - 1, min(flat.size, SAMPLE)).astype(np.int64))]


def record(out: dict, name: str, arrays: dict) -> None:
    """Add what `name` computed to `out` (the contents of the .npz file)."""
    for k, a in arrays.items():
        out[f"{name}/{k}/sha256"] = np.array(digest(a))
        out[f"{name}/{k}/sample"] = _sample(a)


def check(name: str, arrays: dict) -> None:
    """Assert that every array equals, bit for bit, what the original classes computed for `name`."""
    global _STORED
    if _STORED is None:
        _STORED = dict(np.load(PATH))
    for k, a in arrays.items():
        key = f"{name}/{k}"
        got, want = _sample(a), _STORED[key + "/sample"]
        assert got.dtype == want.dtype and got.tobytes() == want.tobytes(), f"{key}: sampled elements differ: {got[:8]} vs {want[:8]}"
        assert digest(a) == str(_STORED[key + "/sha256"]), f"{key}: differs from the original (shape {a.shape})"
