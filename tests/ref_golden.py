"""Outputs of the REFERENCE'S OWN code (oracle/_ref, compiled from the original project's sources by `make -C oracle ref` where
those sources are present), stored under tests/golden so that every comparison against the reference runs on any machine.

    gold = RefGolden("ref_match")            # tests/golden/ref_match.npz
    rn, rout = gold("key", lambda: rm.search_by_projection(...))

returns the stored value of `key`.  Where oracle/_ref is present the lambda is run as well and must reproduce the stored value
(guards against a stale or hand-edited fixture).  MCS_RECORD_GOLDEN=1 runs the lambdas and rewrites the store instead:

    MCS_RECORD_GOLDEN=1 python -m pytest tests/test_ref_match_cpu.py tests/test_ref_pin_cpu.py tests/test_bow_cpu.py \
        tests/test_ref_match_gpu.py tests/test_ref_pin_gpu.py

Tests that need a GPU compute their reference outputs first and skip after them in that mode.
A value is a scalar, an array, a list or a tuple of those; it comes back as a python scalar, an array, or a tuple of them."""
import os
import pathlib
import zlib

import numpy as np
import pytest

GOLD = pathlib.Path(__file__).resolve().parent / "golden"
REF_SO = pathlib.Path(__file__).resolve().parents[1] / "oracle" / "_ref"
RECORD = os.environ.get("MCS_RECORD_GOLDEN") == "1"
# for tests that have no reference output to record (GPU-only checks, checks that only read a store another module writes)
not_recording = pytest.mark.skipif(RECORD, reason="MCS_RECORD_GOLDEN=1: only the reference outputs are computed")


def crc(a):
    """32-bit CRC of an array's bytes: stands in for outputs too large to store"""
    return zlib.crc32(np.ascontiguousarray(a).tobytes())


def _out(a):
    a = np.asarray(a)
    return a.item() if a.ndim == 0 else a


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.tobytes() == np.ascontiguousarray(b, a.dtype).tobytes()


class RefGolden:
    def __init__(self, name, lib="libmcs_ref.so"):
        self.path = GOLD / f"{name}.npz"
        self.live = RECORD or (REF_SO / lib).exists()
        self.data = {} if RECORD else self._read()
        self.record = {}

    def __call__(self, key, fn):
        if not self.live:
            return self._load(key)
        v = fn()
        parts = list(v) if isinstance(v, tuple) else [v]
        if RECORD:
            if isinstance(v, tuple):
                self.record.update({f"{key}/{i}": np.asarray(p) for i, p in enumerate(parts)})
            else:
                self.record[key] = np.asarray(v)
            return v
        stored = self._load(key)
        stored = list(stored) if isinstance(v, tuple) else [stored]
        assert len(stored) == len(parts) and all(_same(s, p) for s, p in zip(stored, parts)), \
            f"{self.path.name}[{key}]: the reference library no longer reproduces the stored output"
        return v

    def _load(self, key):
        if key in self.data:
            return _out(self.data[key])
        parts = []
        while f"{key}/{len(parts)}" in self.data:
            parts.append(_out(self.data[f"{key}/{len(parts)}"]))
        if not parts:
            raise KeyError(f"{self.path.name} has no entry {key!r} (regenerate with MCS_RECORD_GOLDEN=1)")
        return tuple(parts)

    def _read(self):
        with np.load(self.path) as z:
            data = {k: z[k] for k in z.files if not k.startswith("scalars:")}
            for kind in ("i", "f"):                          # scalars are packed into two arrays: one entry each would dominate the file
                data.update(zip(z[f"scalars:{kind}:keys"].tolist(), z[f"scalars:{kind}:values"]))
        return data

    def save(self):
        if not (RECORD and self.record):
            return
        arrays = {k: v for k, v in self.record.items() if v.ndim}
        scalars = {k: v for k, v in self.record.items() if not v.ndim}
        for kind, dtype in (("i", np.int64), ("f", np.float64)):
            keys = [k for k, v in scalars.items() if (v.dtype.kind == "f") == (kind == "f")]
            arrays[f"scalars:{kind}:keys"] = np.array(keys, dtype=str)
            arrays[f"scalars:{kind}:values"] = np.array([scalars[k] for k in keys], dtype)
        np.savez_compressed(self.path, **arrays)
