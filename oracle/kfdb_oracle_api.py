"""ctypes wrapper of oracle/libkfdb_oracle.so -- TEST INFRASTRUCTURE (see kfdb_oracle.cpp): the oracle's restatement of
cMultiKeyFrameDatabase, with the interface of multicol_slam_b200.api.KeyFrameDatabase.
Only tests/ and __graft_entry__.smoke() import this."""
import ctypes as C
import pathlib
import subprocess

import numpy as np

_HERE = pathlib.Path(__file__).resolve().parent
_lib = None


def lib():
    global _lib
    if _lib is None:
        so = _HERE / "libkfdb_oracle.so"
        if not so.exists():
            subprocess.check_call(["make", "-s", "-C", str(_HERE), "CXX=g++"])
            subprocess.check_call(["make", "-s", "-C", str(_HERE), "-f", "kfdb.mk", "CXX=g++"])
        _lib = C.CDLL(str(so))
        _lib.mcso_kfdb_create.restype = C.c_void_p
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class OracleKeyFrameDatabase:
    """bow = (words, values), covis = int64 [n, 10] (-1 = none); Detect* return int64 arrays of key-frame ids."""

    def __init__(self, n_words, scoring):
        self.h = C.c_void_p(lib().mcso_kfdb_create(int(n_words), int(scoring)))
        self.top = 0

    def __del__(self):
        if getattr(self, "h", None):
            lib().mcso_kfdb_destroy(self.h); self.h = None

    def add(self, kf_id, bow):
        w, v = np.ascontiguousarray(bow[0], np.int32), np.ascontiguousarray(bow[1], np.float64)
        self.top = max(self.top, int(kf_id) + 1)
        lib().mcso_kfdb_add(self.h, C.c_longlong(kf_id), _p(w), _p(v), len(w))

    def erase(self, kf_id):
        lib().mcso_kfdb_erase(self.h, C.c_longlong(kf_id))

    def clear(self):
        lib().mcso_kfdb_clear(self.h)

    def _detect(self, loop, qid, bow, connected, covis, min_score):
        w, v = np.ascontiguousarray(bow[0], np.int32), np.ascontiguousarray(bow[1], np.float64)
        conn = np.ascontiguousarray(connected if connected is not None else [], np.int64)
        cv = np.ascontiguousarray(np.zeros((0, 10), np.int64) if covis is None else covis, np.int64).reshape(-1, 10)
        out = np.zeros(max(self.top, int(cv.max()) + 1 if cv.size else 0, 1), np.int64)
        n = lib().mcso_kfdb_detect(self.h, int(loop), C.c_longlong(qid), _p(w), _p(v), len(w), _p(conn), len(conn), _p(cv),
                                   C.c_longlong(len(cv)), C.c_double(min_score), _p(out), len(out))
        return out[:n].copy()

    def DetectLoopCandidates(self, kf_id, bow, connected, covis, minScore):
        return self._detect(1, kf_id, bow, connected, covis, minScore)

    def DetectRelocalisationCandidates(self, frame_id, bow, covis):
        return self._detect(0, frame_id, bow, None, covis, 0.0)
