"""oracle/golden.py -- what the reference computed, stored as test fixtures (TEST INFRASTRUCTURE ONLY).

The tests that compare with the reference project ask a ``Golden`` store for the reference's side of each
comparison.  By default the store reads ``tests/golden/<name>.npz`` and the reference is never touched, so the
comparisons run on any machine.  With ``TGN_GOLDEN_RECORD=<dir>`` set, on a machine where the reference runs
(its checkout for the Python side, ``oracle/_ref`` for its CUDA kernels), every comparison computes the
reference's value live, checks against it as before, and the store writes what was compared to
``<dir>/<name>.npz`` when the process exits; copy those files to ``tests/golden/`` to refresh the fixtures.

To keep the fixtures small, an exact value of more than ``FULL_MAX`` elements is stored as its shape and the
SHA-256 of its bytes; an approximate value is stored as a fixed sample of its elements with the maximum
magnitude of the whole array, which the element-wise criterion of the tests scales by.
"""
from __future__ import annotations

import atexit
import hashlib
import os
import zlib
from typing import Callable, Dict

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
RECORD_DIR = os.environ.get("TGN_GOLDEN_RECORD") or None
FULL_MAX = 4096          # exact values up to this many elements are stored whole
SAMPLE = 2048            # elements kept of a larger approximate value


def _np(a) -> np.ndarray:
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    a = np.asarray(a)
    return a if a.flags.c_contiguous else np.ascontiguousarray(a)


def _digest(a: np.ndarray) -> np.ndarray:
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def sample_index(size: int, key: str, n: int = SAMPLE) -> np.ndarray:
    """A fixed, spread-out set of flat indices into an array of ``size`` elements (the same for the same key)."""
    if size <= n:
        return np.arange(size, dtype=np.int64)
    start = zlib.crc32(key.encode()) % size
    return np.unique((start + np.arange(n, dtype=np.int64) * 2654435761) % size)


def pack(key: str, value) -> Dict[str, np.ndarray]:
    """The entries under which an exact value is stored: itself, or its digest and shape when it is large."""
    w = _np(value)
    if w.size <= FULL_MAX:
        return {key: w}
    return {key + ".sha256": _digest(w), key + ".shape": np.asarray(w.shape, np.int64)}


class Sampled:
    """An approximate reference value: ``values`` at the flat ``index`` of an array of ``shape``, and ``absmax`` of it all."""

    def __init__(self, shape, index, values, absmax):
        self.shape, self.index, self.values, self.absmax = tuple(int(s) for s in shape), index, values, float(absmax)

    def pick(self, a) -> np.ndarray:
        a = _np(a)
        assert a.shape == self.shape, (a.shape, self.shape)
        return a.reshape(-1)[self.index]


class Golden:
    def __init__(self, name: str, record: bool = True):
        """``record=False``: a fixture that another script writes (through ``pack``); it is only read."""
        self.name = name
        self.recording = record and RECORD_DIR is not None
        self._rec: Dict[str, np.ndarray] = {}
        self._fix = None
        if self.recording:
            atexit.register(self._write)

    def _load(self):
        if self._fix is None:
            self._fix = np.load(os.path.join(GOLDEN_DIR, self.name + ".npz"))
        return self._fix

    def _write(self):
        if self._rec:
            os.makedirs(RECORD_DIR, exist_ok=True)
            np.savez_compressed(os.path.join(RECORD_DIR, self.name + ".npz"), **self._rec)

    def array(self, key: str, compute: Callable):
        """The reference's value, stored whole (for inputs the reference produces and small results)."""
        if self.recording:
            a = _np(compute())
            self._rec[key] = a
            return a
        return self._load()[key]

    def exact(self, key: str, got, compute: Callable) -> bool:
        """True when ``got`` equals the reference's value bit for bit (dtype and shape included)."""
        g = _np(got)
        if self.recording:
            w = _np(compute())
            self._rec.update(pack(key, w))
            return g.dtype == w.dtype and g.shape == w.shape and g.tobytes() == w.tobytes()
        fix = self._load()
        if key in fix.files:
            w = fix[key]
            return g.dtype == w.dtype and g.shape == w.shape and g.tobytes() == w.tobytes()
        return bool(np.array_equal(_digest(g), fix[key + ".sha256"]))

    def mismatch(self, key: str, got) -> str:
        """How ``got`` departs from a stored exact value (for the assertion message)."""
        if self.recording:
            return "recording"
        fix, g = self._load(), _np(got)
        if key in fix.files:
            w = fix[key]
            return f"{int((g != w).sum())} of {w.size} elements differ" if g.shape == w.shape else f"shape {g.shape} != {w.shape}"
        shape = tuple(fix[key + ".shape"])
        return f"shape {g.shape} != {shape}" if g.shape != shape else f"{g.dtype} values of shape {shape} differ (SHA-256)"

    def sampled(self, key: str, compute: Callable) -> Sampled:
        """An approximate reference value as a fixed sample of its elements (see ``Sampled``)."""
        if self.recording:
            w = _np(compute())
            idx = sample_index(w.size, key)
            self._rec[key + ".shape"] = np.asarray(w.shape, np.int64)
            self._rec[key + ".sample"] = w.reshape(-1)[idx]
            self._rec[key + ".absmax"] = np.asarray(np.abs(w).max() if w.size else 0.0, np.float64)
            return Sampled(w.shape, idx, w.reshape(-1)[idx], self._rec[key + ".absmax"])
        fix = self._load()
        shape = tuple(fix[key + ".shape"])
        return Sampled(shape, sample_index(int(np.prod(shape)), key), fix[key + ".sample"], fix[key + ".absmax"])
