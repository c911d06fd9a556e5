"""Outputs of the reference's own code (compiled from its sources into oracle/_ref by oracle/Makefile) on the inputs the
parity tests generate, stored in tests/golden/reference_golden.npz by tests/golden/make_reference_golden.py.  The tests
compare the oracle with these, so they run without the reference's sources.

Arrays too large to store whole (distance planes, per-iteration keypoint sets) are stored as a SHA-256 digest of their
values: NaN and -0.0 are canonicalised first, so a digest match means exactly what np.array_equal(..., equal_nan=True)
means."""
import hashlib
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_golden.npz")
_cache = {}


def key(*parts):
    return "/".join(str(p) for p in parts)


def digest(a):
    a = np.asarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.nan, a + 0.0).astype(a.dtype)       # one NaN pattern, -0.0 -> +0.0
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return np.frombuffer(h.digest(), np.uint8).copy()


def load(prefix):
    """Every stored array under `prefix/`, keyed by the rest of its name."""
    if "z" not in _cache:
        with np.load(PATH) as z:
            _cache["z"] = {k: z[k] for k in z.files}
    pre = prefix + "/"
    d = {k[len(pre):]: v for k, v in _cache["z"].items() if k.startswith(pre)}
    assert d, f"no reference outputs stored under {prefix!r} in {PATH}"
    return d
