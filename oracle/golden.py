"""Answers of the reference's own code, stored in tests/golden/reference.npz -- TEST INFRASTRUCTURE.

The tests that pin the oracle, the packers and the file readers to the reference ask for the reference's answer through
``value(key, fn)`` or compare with it through ``check(key, got, fn)``.  ``fn`` computes the answer with the reference's code
(oracle/_ref); it only runs while tests/golden/make_golden_reference.py records the fixture, which runs those same tests, so the
stored answers belong to exactly the inputs the tests build.  Everywhere else the stored answer is used and the reference is not
needed.  ``check`` keeps an answer larger than ``INLINE_BYTES`` as the SHA-256 of its dtype, shape and bytes (NaN payloads
made canonical, as the comparisons treat every NaN alike), which keeps the fixture small; ``value`` always stores the array.
"""
from __future__ import annotations

import hashlib
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "reference.npz")
INLINE_BYTES = 1024
_DIGEST = ".sha256"

_record = None
_store = None
SOURCE = None  # the reference's source tree (a neural-speed checkout), while recording


def recording() -> bool:
    return _record is not None


def start_recording(source: str) -> None:
    global _record, SOURCE
    _record, SOURCE = {}, source


def save_recording(path: str = PATH) -> int:
    np.savez_compressed(path, **_record)
    return len(_record)


def _stored():
    global _store
    if _store is None:
        with np.load(PATH) as z:
            _store = {k: z[k] for k in z.files}
    return _store


def digest(a) -> np.ndarray:
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.array(np.nan, a.dtype), a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def _put(key, v):
    if key in _record:
        assert np.array_equal(_record[key], v), f"{key}: recorded twice with different answers"
    _record[key] = v


def value(key: str, fn) -> np.ndarray:
    """The reference's answer fn() for this key (recorded, or read back from the fixture)."""
    if _record is not None:
        v = np.asarray(fn())
        _put(key, v)
        return v
    return _stored()[key]


def check(key: str, got, fn) -> None:
    """Assert that got equals the reference's answer fn() for this key, element for element and in dtype and shape."""
    got = np.asarray(got)
    if _record is not None:
        want = np.asarray(fn())
        assert got.dtype == want.dtype and got.shape == want.shape, (key, got.dtype, want.dtype, got.shape, want.shape)
        np.testing.assert_array_equal(got, want, err_msg=key)
        if want.nbytes <= INLINE_BYTES:
            _put(key, want)
        else:
            assert np.array_equal(digest(got), digest(want)), f"{key}: equal values, different bytes (signed zeros)"
            _put(key + _DIGEST, digest(want))
        return
    z = _stored()
    if key in z:
        want = z[key]
        assert got.dtype == want.dtype and got.shape == want.shape, (key, got.dtype, want.dtype, got.shape, want.shape)
        np.testing.assert_array_equal(got, want, err_msg=key)
    else:
        assert np.array_equal(digest(got), z[key + _DIGEST]), f"{key}: differs from the reference's answer"
