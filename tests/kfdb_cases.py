"""Scripted call sequences for the key-frame database tests (tests/test_kfdb_cpu.py, tests/test_kfdb_gpu.py).

Every database implementation under test -- the reference's own cMultiKeyFrameDatabase (oracle/ref_kfdb_api.py), the oracle's
restatement (kfdb_oracle_api.OracleKeyFrameDatabase) and the product (multicol_slam_b200.api.KeyFrameDatabase) -- has the same
methods, so one script drives all three.  Inputs are regenerated from seeds; only candidate id lists are stored.

The trajectory: key frame i sits at place(i); the first pass visits places 0..49, the second pass revisits places 10..39, so
revisits share a descriptor pool (and most of their words) with the first visit.  covis row i = the ten best covisibility key
frames of i: its temporal neighbours and the key frames at the same place."""
import pathlib
import sys

import numpy as np

N_KF = 80
N_DESC = 700


def place(i):
    return i if i < 50 else i - 40


def descriptors(seed_place, seed_view, n=N_DESC):
    """a view of a place: 75 % of the descriptors drawn from the place's pool with a few flipped bits, the rest fresh"""
    pool = np.random.default_rng(10_000 + seed_place).integers(0, 256, (1500, 32), dtype=np.uint8)
    rng = np.random.default_rng(seed_view)
    k = n * 3 // 4
    d = pool[rng.integers(0, len(pool), k)].copy()
    flips = rng.integers(0, 256, (k, 4))
    for c in range(4):
        d[np.arange(k), flips[:, c] // 8] ^= (1 << (flips[:, c] % 8)).astype(np.uint8)
    return np.concatenate([d, rng.integers(0, 256, (n - k, 32), dtype=np.uint8)])


def covisibility(n=N_KF):
    cv = -np.ones((n, 10), np.int64)
    for i in range(n):
        same = [j for j in range(n) if j != i and place(j) == place(i)]
        near = sorted((j for j in range(max(0, i - 6), min(n, i + 7)) if j != i), key=lambda j: (abs(j - i), j))
        row = (same + [j for j in near if j not in same])[:10]
        cv[i, :len(row)] = row
    return cv


def bows(transform):
    """transform(desc) -> (words, values): key frames 0..N_KF-1 and the query frames ('f<k>' at place k)"""
    out = {i: transform(descriptors(place(i), i)) for i in range(N_KF)}
    for p in (3, 12, 20, 33, 45):
        out[f"f{p}"] = transform(descriptors(p, 5000 + p))
    out["none"] = (np.zeros(0, np.int32), np.zeros(0))
    return out


def trajectory_script():
    """(op, ...) tuples; detections carry a tag under which their result is stored"""
    cv = covisibility()
    conn = lambda i: [int(j) for j in cv[i] if j >= 0 and abs(j - i) <= 3]           # GetConnectedKeyFrames: temporal neighbours
    s = [("add", i, i) for i in range(49)]
    s += [("erase", 200),                                                               # never added: no effect
          ("reloc", "r_f12", 1000, "f12"),
          ("loop", "l_49", 49, 49, conn(49), 0.0),
          ("loop", "l_49_high", 49, 49, [], 1e9)]                                       # everything below minScore
    s += [("add", i, i) for i in range(49, 64)]
    s += [("loop", "l_64", 64, 64, conn(64), 0.01),                                     # revisit of place 24, its neighbours connected
          ("loop", "l_64_unconnected", 65, 64, [], 0.01),
          ("add", 64, 64),
          ("add", 7, 7),                                                                # duplicate add: 7 counts twice
          ("reloc", "r_f3_dup", 1006, "f3"),
          ("erase", 7),                                                                 # the first of the two copies of 7
          ("erase", 20), ("add", 20, 20),                                               # erase + re-add: 20 moves to the end of its lists
          ("reloc", "r_f20", 1001, "f20"),
          ("reloc", "r_f20_again", 1001, "f33"),                                        # repeated query id
          ("reloc", "r_id0", 0, "f3"),                                                  # query id 0: untouched key frames count as visited
          ("loop", "l_id0", 0, 0, [], 0.0),
          ("reloc", "r_f45", 1002, "f45"),
          ("reloc", "r_none", 1003, "none")]                                            # no shared word
    s += [("add", i, i) for i in range(65, N_KF)]
    s += [("loop", "l_79", 79, 79, conn(79), 0.005),
          ("clear",),
          ("reloc", "r_after_clear", 1004, "f12")]                                      # empty lists: nothing shares a word
    s += [("add", i, i) for i in range(0, 30)]
    s += [("reloc", "r_f20_third", 1001, "f20"),                                        # same id as before the clear: stamps persist
          ("reloc", "r_f12_after", 1005, "f12"),
          ("loop", "l_29", 29, 29, conn(29), 0.0)]
    return s, cv


def reference_db(scoring, weighting):
    """the reference's own cMultiKeyFrameDatabase (oracle/_ref/libkfdb_ref.so)"""
    sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1] / "oracle"))
    import ref_kfdb_api
    return ref_kfdb_api.RefKeyFrameDatabase(scoring, weighting)


def run(db, script, cv, bow):
    out = {}
    for op in script:
        if op[0] == "add":
            db.add(op[1], bow[op[2]])
        elif op[0] == "erase":
            db.erase(op[1])
        elif op[0] == "clear":
            db.clear()
        elif op[0] == "reloc":
            out[op[1]] = np.asarray(db.DetectRelocalisationCandidates(op[2], bow[op[3]], cv), np.int64)
        else:
            out[op[1]] = np.asarray(db.DetectLoopCandidates(op[2], bow[op[3]], op[4], cv, op[5]), np.int64)
    return out


# ---- hand-built BowVectors for the cases a trajectory does not produce on purpose ---------------------------------------------
def _hand(words):
    w = np.asarray(sorted(words), np.int32)
    return w, np.full(len(w), 1.0 / len(w))


def stale_score_script(with_first_query):
    """Key frame 1 (words 100..149) has key frame 2 (words 200..249) as its best covisibility neighbour.  Query A (id 5) is key
    frame 2's own vector: it scores 2 high.  Query B (id 6) shares 25 words with 1 and one word with 2: only 1 is scored, but 2 was
    encountered (mnRelocQuery == 6), so 1's covisibility sum reads 2's score of query A and 2 becomes pBestKF.  Without query A
    the stale score is the initial 0.0 and B returns 1."""
    bow = {1: _hand(range(100, 150)), 2: _hand(range(200, 250)), "qa": _hand(range(200, 250)),
           "qb": _hand(list(range(100, 125)) + [200])}
    cv = -np.ones((3, 10), np.int64)
    cv[1, 0] = 2
    s = [("add", 1, 1), ("add", 2, 2)]
    if with_first_query:
        s.append(("reloc", "a", 5, "qa"))
    s.append(("reloc", "b", 6, "qb"))
    return s, cv, bow


def dedup_tie_script():
    """Key frames 1 and 2 have identical vectors and both name key frame 3 as their best neighbour, 3 being scored higher:
    both accumulate the same score (a tie) and both choose 3, which is returned once.  Key frames 4 and 5 are another identical
    pair without neighbours: a tie returned in add order, and in the other order once 4 is erased and added again."""
    a, b = list(range(300, 340)), list(range(400, 440))
    bow = {1: _hand(a), 2: _hand(a), 3: _hand(a[:30]), 4: _hand(b), 5: _hand(b), "q": _hand(a[:30] + b[:5]), "q45": _hand(b)}
    cv = -np.ones((6, 10), np.int64)
    cv[1, 0] = 3
    cv[2, 0] = 3
    s = [("add", i, i) for i in range(1, 6)]
    s += [("reloc", "dedup", 10, "q"), ("loop", "dedup_loop", 11, "q", [], 0.0),
          ("reloc", "tie", 12, "q45"), ("erase", 4), ("add", 4, 4), ("reloc", "tie_readd", 13, "q45")]
    return s, cv, bow


CONFIGS = [(0, 0), (1, 0), (2, 0), (4, 0), (5, 0), (0, 1)]   # (scoring, weighting): the five types with TF_IDF, L1 with TF
