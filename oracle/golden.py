"""TEST INFRASTRUCTURE ONLY: compact forms of recorded reference outputs (tests/golden/reference_cpu.npz,
tools/make_golden_reference.py).

Outputs that must match exactly are kept as SHA-256 digests when storing them whole would make the fixture large;
floating-point tensors compared under a tolerance are kept at a fixed set of flat positions (``sample_index``).
"""
from __future__ import annotations

import hashlib

import numpy as np


def digest(*parts) -> np.ndarray:
    """SHA-256 over the dtype, shape and bytes of each part (arrays, or str taken as ASCII bytes) -> uint8[32]."""
    h = hashlib.sha256()
    for p in parts:
        a = np.frombuffer(p.encode("ascii"), np.uint8) if isinstance(p, str) else np.ascontiguousarray(p)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def sample_index(size: int, k: int) -> np.ndarray:
    """k flat positions spread over [0, size) by a fixed large-prime stride (no RNG, so no numpy-version dependence)."""
    k = min(k, size)
    return (np.arange(k, dtype=np.int64) * 1000003) % size
