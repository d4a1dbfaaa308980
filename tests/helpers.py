"""Shared helpers for the parity tests (oracle is the checker, never the product)."""
import hashlib
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_CASES = ["cells_default", "cells_nodensity", "cells_regs", "clusters", "cells_spatial"]


def load_golden(name):
    """-> (ctor kwargs for a Mapper-like class, golden outputs dict)."""
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    kw = {}
    for k in z.files:
        if k.startswith("in_"):
            kw[k[3:]] = z[k]
        elif k.startswith("hp_"):
            kw[k[3:]] = float(z[k])
    out = {k: z[k] for k in z.files if not (k.startswith("in_") or k.startswith("hp_"))}
    if "d" not in kw:
        kw["d"] = None
    return kw, out


def rel_fro(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def max_rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-12)))


def sha256_f32(a):
    """Digest of an array's float32 bytes (how the golden files pin the reference's initial mapping)."""
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.float32).tobytes()).hexdigest()


def assert_same_print(ours, ref):
    """The reference's print line `name: value, name: value` (mapping_optimizer.py:300-307):
    same names in the same order; values equal to the printed 3 decimals up to one unit in the
    last printed digit or 1e-6 relative (an fp32 sum differs in its 8th digit)."""
    a = [x.split(": ") for x in ours.split(", ")]
    b = [x.split(": ") for x in ref.split(", ")]
    assert [x[0] for x in a] == [x[0] for x in b], (ours, ref)
    for (_, va), (_, vb) in zip(a, b):
        va, vb = float(va), float(vb)
        assert abs(va - vb) <= 0.0011 + 1e-6 * abs(vb), (ours, ref)


def traj_err(a, b):
    """Error of a loss trajectory that crosses zero: |a - b| relative to max(|b|, a quarter of the trajectory's scale)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 0.25 * np.max(np.abs(b)))))
