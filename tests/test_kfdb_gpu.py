"""Key-frame database on the GPU (mcs_kfdb_*, multicol_slam_b200.api.KeyFrameDatabase) against the reference's own database
(candidate lists stored in tests/golden/kfdb_ref.npz, see test_kfdb_cpu.py) and the oracle's restatement (oracle/kfdb_oracle.cpp):
identical candidate lists, in order."""
import ctypes as C
import pathlib

import numpy as np
import pytest

import kfdb_cases as kc
import kfdb_oracle_api as ko
from ref_golden import RefGolden, not_recording

ROOT = pathlib.Path(__file__).resolve().parents[1]
pytestmark = [pytest.mark.gpu, not_recording]


@pytest.fixture(scope="module")
def voc():
    return np.load(ROOT / "tests" / "golden" / "voc_small_9_6.npz")


def test_sequences_match_reference_and_oracle(api, oa, voc):
    gold = RefGolden("kfdb_ref", lib="libkfdb_ref.so")
    n_words = len(voc["word_node"])
    for sc, wg in kc.CONFIGS:
        pv = api.ORBVocabulary(voc, sc, wg)
        ov = oa.OracleVocabulary(voc, sc, wg)
        cases = [("trajectory", kc.trajectory_script() + (kc.bows(lambda d: ov.transform(d, 4)[:2]),)),
                 ("stale", kc.stale_score_script(True)), ("stale_control", kc.stale_score_script(False)),
                 ("dedup_tie", kc.dedup_tie_script())]
        for name, (script, cv, bow) in cases:
            tags = [op[1] for op in script if op[0] in ("reloc", "loop")]
            got = kc.run(api.KeyFrameDatabase(pv), script, cv, bow)
            want = kc.run(ko.OracleKeyFrameDatabase(n_words, sc), script, cv, bow)
            ref = gold(f"{name}/{sc}/{wg}", lambda: tuple(kc.run(kc.reference_db(sc, wg), script, cv, bow)[t] for t in tags))
            for tag, r in zip(tags, ref):
                r = np.asarray(r, np.int64).reshape(-1)
                assert np.array_equal(got[tag], r), (name, sc, wg, tag, got[tag], r)
                assert np.array_equal(want[tag], r), (name, sc, wg, tag)


def scale_map(pv, n_kf, seed=0):
    """n_kf key frames of ~6000 descriptors (-> about 2000 words) on a trajectory that revisits its first places; covis from
    trajectory neighbours and revisits"""
    first = int(n_kf * 0.7)
    place = np.array([i if i < first else (i - first) * 2 % first for i in range(n_kf)])
    rng = np.random.default_rng(seed)
    bows = []
    for i in range(n_kf):
        pool = np.random.default_rng(100_000 + int(place[i])).integers(0, 256, (6000, 32), dtype=np.uint8)
        d = pool[rng.integers(0, len(pool), 4500)]
        d = np.concatenate([d, rng.integers(0, 256, (1500, 32), dtype=np.uint8)])
        bows.append(pv.transform(d, 4)[:2])
    cv = -np.ones((n_kf, 10), np.int64)
    for i in range(n_kf):
        same = [int(j) for j in np.nonzero(place == place[i])[0] if j != i]
        near = sorted((j for j in range(max(0, i - 6), min(n_kf, i + 7)) if j != i), key=lambda j: (abs(j - i), j))
        row = (same + [j for j in near if j not in same])[:10]
        cv[i, :len(row)] = row
    return bows, cv


def test_scale_1000_keyframes(api, oa, voc):
    pv = api.ORBVocabulary(voc)
    bows, cv = scale_map(pv, 1000)
    assert 1500 < np.mean([len(b[0]) for b in bows]) < 3000
    db, odb = api.KeyFrameDatabase(pv), ko.OracleKeyFrameDatabase(len(voc["word_node"]), pv.scoring)
    rng = np.random.default_rng(7)
    both = lambda f, *a: (getattr(db, f)(*a), getattr(odb, f)(*a))
    for i in range(900):
        both("add", i, bows[i])
    n_nonempty = 0
    for k in range(50):
        both("add", 900 + 2 * k, bows[900 + 2 * k]); both("add", 901 + 2 * k, bows[901 + 2 * k])
        if k % 5 == 0:
            victim = int(rng.integers(0, 900))
            both("erase", victim)
            if k % 10 == 0:
                both("add", victim, bows[victim])
        q = int(rng.integers(0, 1000))
        conn = [int(j) for j in cv[q] if j >= 0 and abs(j - q) <= 3]
        g, o = both("DetectLoopCandidates", q, bows[q], conn, cv, 0.02)
        assert np.array_equal(g, o), ("loop", k, g, o)
        f = int(rng.integers(0, 1000))
        g, o = both("DetectRelocalisationCandidates", 10_000 + k % 40, bows[f], cv)   # ids repeat: stale state is exercised
        assert np.array_equal(g, o), ("reloc", k, g, o)
        n_nonempty += len(g) > 0
    assert n_nonempty > 25


def test_segment_rebuild(api, oa, voc):
    """every key frame holds the same 60 words: the segments (8 entries to start with) overflow and are rebuilt on the device
    again and again, with erases leaving tombstones in between"""
    pv = api.ORBVocabulary(voc)
    db, odb = api.KeyFrameDatabase(pv), ko.OracleKeyFrameDatabase(len(voc["word_node"]), pv.scoring)
    rng = np.random.default_rng(3)
    base = np.sort(rng.choice(6999, 60, replace=False)).astype(np.int32)
    cv = -np.ones((300, 10), np.int64)
    for i in range(300):
        cv[i, :3] = [(i + 1) % 300, (i + 7) % 300, (i + 11) % 300]
    for i in range(300):
        w = np.sort(np.concatenate([base, rng.choice(np.setdiff1d(np.arange(6999), base), 20, replace=False)])).astype(np.int32)
        v = rng.random(len(w)); v /= v.sum()
        db.add(i, (w, v)); odb.add(i, (w, v))
        if i % 7 == 3:
            db.erase(i - 2); odb.erase(i - 2)
        if i % 50 == 49:
            q = (base, np.full(len(base), 1.0 / len(base)))
            assert np.array_equal(db.DetectRelocalisationCandidates(5000 + i, q, cv), odb.DetectRelocalisationCandidates(5000 + i, q, cv))
            assert np.array_equal(db.DetectLoopCandidates(i, q, [i - 1], cv, 0.0), odb.DetectLoopCandidates(i, q, [i - 1], cv, 0.0))


def _h(db):
    return db._h


def test_capacity_and_errors(api, voc):
    lib = api.lib()
    pv = api.ORBVocabulary(voc)
    db = api.KeyFrameDatabase(pv)
    for i, words in enumerate(([5, 9, 12], [5, 9, 40], [9, 12, 41])):
        db.add(i, (np.array(words, np.int32), np.full(3, 1 / 3)))
    w, v = np.array([5, 9, 12, 40, 41], np.int32), np.full(5, 0.2)
    cv = -np.ones((3, 10), np.int64)
    want = db.DetectRelocalisationCandidates(77, (w, v), cv)
    assert len(want) == 3
    out, n = np.zeros(3, np.int64), C.c_int32(-1)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = lib.mcs_kfdb_detect_relocalisation_candidates(_h(db), C.c_int64(78), p(w), p(v), 5, p(cv), C.c_int64(3), p(out), 2,
                                                       C.byref(n))
    assert rc == api.MCS_ERR_CAPACITY and n.value == 3
    rc = lib.mcs_kfdb_detect_relocalisation_candidates(_h(db), C.c_int64(79), p(w), p(v), 5, p(cv), C.c_int64(3), p(out), 3,
                                                       C.byref(n))
    assert rc == api.MCS_OK and np.array_equal(out[:n.value], want)
    # malformed vectors and ids
    bad = [(np.array([9, 5], np.int32), np.ones(2)), (np.array([5, 5], np.int32), np.ones(2)),
           (np.array([5, 6999], np.int32), np.ones(2)), (np.array([-1, 5], np.int32), np.ones(2))]
    for b in bad:
        assert lib.mcs_kfdb_add(_h(db), C.c_int64(4), p(b[0]), p(b[1]), 2) == api.MCS_ERR_INVALID
        with pytest.raises(api.McsError):
            db.DetectRelocalisationCandidates(80, b, cv)
    ok = (np.array([5], np.int32), np.ones(1))
    assert lib.mcs_kfdb_add(_h(db), C.c_int64(-3), p(ok[0]), p(ok[1]), 1) == api.MCS_ERR_INVALID
    assert lib.mcs_kfdb_erase(_h(db), C.c_int64(-3)) == api.MCS_ERR_INVALID
    assert lib.mcs_kfdb_erase(_h(db), C.c_int64(12345)) == api.MCS_OK                  # never added: nothing happens
    for bad_cv in (np.full((3, 10), -2, np.int64), np.full((1, 10), -7, np.int64)):
        with pytest.raises(api.McsError) as e:
            db.DetectRelocalisationCandidates(81, ok, bad_cv)
        assert e.value.code == api.MCS_ERR_INVALID
    with pytest.raises(api.McsError) as e:
        db.DetectLoopCandidates(-1, ok, [], cv, 0.0)
    assert e.value.code == api.MCS_ERR_INVALID
    with pytest.raises(api.McsError) as e:
        db.DetectLoopCandidates(2, ok, [-4], cv, 0.0)
    assert e.value.code == api.MCS_ERR_INVALID
    # KL: the bit-exact bar cannot be promised for a device log()
    with pytest.raises(api.McsError) as e:
        api.KeyFrameDatabase(api.ORBVocabulary(voc, scoring=3))
    assert e.value.code == api.MCS_ERR_UNSUPPORTED
