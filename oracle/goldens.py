"""Recorded outputs of the compiled reference (TEST INFRASTRUCTURE, see oracle/__init__.py).

Tests that compare bit for bit with the reference at sizes too large to store whole keep, per reference call, a
record of its output: the shape, the SHA-256 of the float32 bytes and a fixed sample of values.  A matching digest
means the arrays are bit-identical; the sample only serves to say how far apart they are when they are not.
tests/golden/gen_reference_runs.py writes the records (tests/golden/reference_runs.json) from oracle/_ref.
"""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np

RUNS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "reference_runs.json")
SAMPLE = 8


def record(a) -> dict:
    a = np.ascontiguousarray(a, np.float32)
    flat = a.ravel()
    idx = np.linspace(0, flat.size - 1, SAMPLE).round().astype(np.int64) if flat.size else np.zeros(0, np.int64)
    return {"shape": list(a.shape), "sha256": hashlib.sha256(a.tobytes()).hexdigest(),
            "sample": [float(v) for v in flat[idx]]}


def mismatch(a, rec: dict) -> str:
    """'' when `a` is bit-identical to the recorded reference output, else how it differs."""
    got = record(a)
    if got["shape"] != rec["shape"]:
        return "shape %s, reference %s" % (got["shape"], rec["shape"])
    if got["sha256"] == rec["sha256"]:
        return ""
    g, w = np.float32(got["sample"]), np.float32(rec["sample"])
    return "not bit-identical to the reference (%d of %d sampled floats differ, max |diff| %.3g)" % (
        int((g.view(np.uint32) != w.view(np.uint32)).sum()), len(w), float(np.abs(g.astype(np.float64) - w).max()))


def check(a, rec: dict, what: str) -> None:
    m = mismatch(a, rec)
    assert not m, "%s: %s" % (what, m)


def load(name: str):
    with open(RUNS) as f:
        return json.load(f)[name]
