"""Key-frame database, CPU side: the oracle's restatement of cMultiKeyFrameDatabase (oracle/kfdb_oracle.cpp) against
the reference's own database compiled in place (oracle/_ref/libkfdb_ref.so), through the candidate lists stored in
tests/golden/kfdb_ref.npz (tests/ref_golden.py; where oracle/_ref is built the reference is run as well and must reproduce them).
The call sequences are in tests/kfdb_cases.py; BowVectors come from the oracle's DBoW2 transform (pinned by test_bow_cpu.py)."""
import pathlib

import numpy as np
import pytest

import kfdb_cases as kc
import kfdb_oracle_api as ko
from ref_golden import RefGolden

ROOT = pathlib.Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def voc():
    return np.load(ROOT / "tests" / "golden" / "voc_small_9_6.npz")


def trajectory_bows(oa, voc, sc, wg):
    ov = oa.OracleVocabulary(voc, sc, wg)
    return kc.bows(lambda d: ov.transform(d, 4)[:2])


def reference_outputs(oa, voc):
    """{(case, scoring, weighting): {tag: ids}} from the stored reference run (rerun where the reference library exists)"""
    gold = RefGolden("kfdb_ref", lib="libkfdb_ref.so")
    out = {}
    for sc, wg in kc.CONFIGS:
        script, cv = kc.trajectory_script()
        tags = [op[1] for op in script if op[0] in ("reloc", "loop")]
        bow = trajectory_bows(oa, voc, sc, wg)
        ref = gold(f"trajectory/{sc}/{wg}", lambda: tuple(kc.run(kc.reference_db(sc, wg), script, cv, bow)[t] for t in tags))
        out[("trajectory", sc, wg)] = dict(zip(tags, ref))
        for name, (script, cv, bow) in (("stale", kc.stale_score_script(True)), ("stale_control", kc.stale_score_script(False)),
                                        ("dedup_tie", kc.dedup_tie_script())):
            tags = [op[1] for op in script if op[0] in ("reloc", "loop")]
            ref = gold(f"{name}/{sc}/{wg}", lambda: tuple(kc.run(kc.reference_db(sc, wg), script, cv, bow)[t] for t in tags))
            out[(name, sc, wg)] = dict(zip(tags, ref))
    gold.save()
    return out


def oracle_outputs(oa, voc, case, sc, wg):
    if case == "trajectory":
        script, cv = kc.trajectory_script()
        bow = trajectory_bows(oa, voc, sc, wg)
    else:
        script, cv, bow = {"stale": lambda: kc.stale_score_script(True), "stale_control": lambda: kc.stale_score_script(False),
                           "dedup_tie": kc.dedup_tie_script}[case]()
    return kc.run(ko.OracleKeyFrameDatabase(len(voc["word_node"]), sc), script, cv, bow)


def test_oracle_matches_reference(oa, voc):
    ref = reference_outputs(oa, voc)
    for (case, sc, wg), want in ref.items():
        got = oracle_outputs(oa, voc, case, sc, wg)
        for tag, ids in want.items():
            assert np.array_equal(got[tag], np.asarray(ids, np.int64).reshape(-1)), (case, sc, wg, tag, got[tag], ids)


def test_cases_cover_the_contract(oa, voc):
    """the scripted cases produce the situations they are written for (on the reference's stored outputs)"""
    ref = reference_outputs(oa, voc)
    ids = lambda case, sc, wg, tag: np.asarray(ref[(case, sc, wg)][tag], np.int64).reshape(-1).tolist()
    for sc, wg in kc.CONFIGS:
        # a stale mRelocScore of an earlier query changes the returned list
        assert ids("stale", sc, wg, "b") == [2] and ids("stale_control", sc, wg, "b") == [1]
        # two candidates with the same best neighbour: returned once; a tie keeps add order, a re-add moves to the end
        assert ids("dedup_tie", sc, wg, "dedup") == [3] and ids("dedup_tie", sc, wg, "dedup_loop") == [3]
        assert ids("dedup_tie", sc, wg, "tie") == [4, 5] and ids("dedup_tie", sc, wg, "tie_readd") == [5, 4]
        t = lambda tag: ids("trajectory", sc, wg, tag)
        assert t("r_none") == [] and t("l_49_high") == [] and t("r_after_clear") == []
        assert t("r_f12") and t("r_f20") and t("r_f45")
        assert not set(t("l_64")) & {61, 62, 63}               # connected key frames are never listed
