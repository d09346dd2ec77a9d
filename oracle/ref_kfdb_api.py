"""ctypes wrapper of oracle/_ref/libkfdb_ref.so: the REFERENCE's own cMultiKeyFrameDatabase (src/cMultiKeyFrameDatabase.cpp)
compiled in place by `make -C oracle -f kfdb.mk ref` against data-only key-frame stand-ins (ref_kfdb/stub_kfdb.h).  TEST INFRASTRUCTURE:
pins the oracle's restatement (kfdb_oracle.cpp) and generates tests/golden/kfdb_ref.npz.  Same interface as
multicol_slam_b200.api.KeyFrameDatabase."""
import ctypes as C
import pathlib

import numpy as np

_HERE = pathlib.Path(__file__).resolve().parent
SO = _HERE / "_ref" / "libkfdb_ref.so"
VOC_TXT = _HERE / "_ref" / "voc_small_9_6.txt"


def available():
    return SO.exists() and VOC_TXT.exists()


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _bow(bow):
    return np.ascontiguousarray(bow[0], np.int32), np.ascontiguousarray(bow[1], np.float64)


def _covis(covis):
    c = np.ascontiguousarray(np.zeros((0, 10), np.int64) if covis is None else covis, np.int64)
    return c.reshape(-1, 10)


def capacity_for(top, covis):
    """every candidate is an added key frame or a covisibility neighbour: at most this many distinct ids"""
    return max(int(top), int(covis.max()) + 1 if covis.size else 0, 1)


class RefKeyFrameDatabase:
    def __init__(self, scoring, weighting, txt=VOC_TXT):
        self.lib = C.CDLL(str(SO))
        self.lib.refkfdb_create.restype = C.c_void_p
        self.h = C.c_void_p(self.lib.refkfdb_create(str(txt).encode(), int(scoring), int(weighting)))
        if not self.h:
            raise RuntimeError("reference vocabulary did not load")
        self.top = 0

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.refkfdb_free(self.h); self.h = None

    def add(self, kf_id, bow):
        w, v = _bow(bow)
        self.top = max(self.top, int(kf_id) + 1)
        self.lib.refkfdb_add(self.h, C.c_longlong(kf_id), _p(w), _p(v), len(w))

    def erase(self, kf_id):
        self.lib.refkfdb_erase(self.h, C.c_longlong(kf_id))

    def clear(self):
        self.lib.refkfdb_clear(self.h)

    def _detect(self, loop, qid, bow, connected, covis, min_score):
        w, v = _bow(bow)
        conn = np.ascontiguousarray(connected if connected is not None else [], np.int64)
        cv = _covis(covis)
        out = np.zeros(capacity_for(self.top, cv), np.int64)
        n = self.lib.refkfdb_detect(self.h, int(loop), C.c_longlong(qid), _p(w), _p(v), len(w), _p(conn), len(conn), _p(cv),
                                    C.c_longlong(len(cv)), C.c_double(min_score), _p(out), len(out))
        assert n <= len(out)
        return out[:n].copy()

    def DetectLoopCandidates(self, kf_id, bow, connected, covis, minScore):
        return self._detect(1, kf_id, bow, connected, covis, minScore)

    def DetectRelocalisationCandidates(self, frame_id, bow, covis):
        return self._detect(0, frame_id, bow, None, covis, 0.0)
