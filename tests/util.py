"""Shared helpers for the parity tests."""
import numpy as np


def bits32(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def bits64(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def assert_bitexact(a, b, what=""):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if a.dtype == np.float32:
        bad = bits32(a) != bits32(b)
    elif a.dtype == np.float64:
        bad = bits64(a) != bits64(b)
    else:
        bad = a != b
    # NaN payloads are not part of the contract
    if a.dtype.kind == "f":
        bad &= ~(np.isnan(a) & np.isnan(b))
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} differ; first at {np.argwhere(bad)[:5].tolist()} " \
                          f"got {a[bad][:5]} want {b[bad][:5]}"


def row_cosine(a, b):
    a = a.astype(np.float64)
    b = b.astype(np.float64)
    return (a * b).sum(1) / np.sqrt((a * a).sum(1) * (b * b).sum(1) + 1e-300)


def rel_l2(a, b):
    a = a.astype(np.float64)
    b = b.astype(np.float64)
    return float(np.sqrt(((a - b) ** 2).sum() / max((b ** 2).sum(), 1e-300)))


def grad_floor(nd):
    """Least max |refinement gradient| that G's stress weights should give.  Its Linear weights are U(+-sqrt(6 / nd)), so the
    gradient scales like 1 / sqrt(nd): measured max 2.2-69 at nd <= 100, 2.3 at nd 300, 0.60 at 1x16x16 nd 4096."""
    return min(1.0, 10.0 / np.sqrt(nd))
