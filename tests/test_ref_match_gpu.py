"""GPU parity against the REFERENCE'S OWN matcher (oracle/_ref/libmcs_ref.so = the original project's src/cORBmatcher.cpp, see
tests/test_ref_match_cpu.py): the CUDA path through the C ABI vs reference-run outputs on the same scenes, stored in
tests/golden/ref_match_cpu.npz (scenes shared with the CPU checks) and tests/golden/ref_match_gpu.npz (tests/ref_golden.py)."""
import numpy as np
import pytest

import test_ref_match_cpu as T
from ref_golden import RECORD, RefGolden, not_recording

pytestmark = pytest.mark.gpu
frames = T.frames
rm = T.rm


@pytest.fixture(scope="module")
def gold():
    return RefGolden("ref_match_cpu")            # read here, written by tests/test_ref_match_cpu.py


@pytest.fixture(scope="module")
def gold_gpu():
    g = RefGolden("ref_match_gpu")
    yield g
    g.save()


@pytest.mark.parametrize("masks", [False, True])
def test_core_searches_gpu_vs_reference(api, rm, gold, gold_gpu, frames, cams, masks):
    F1, F2 = frames
    # SearchByBoW(KF1, KF2) on this test's own scene: brute force with the greedy one-use rule
    rng = np.random.default_rng(17)
    n1, n2 = len(F1.keys), len(F2.keys)
    has1, has2 = rng.random(n1) < 0.7, rng.random(n2) < 0.7
    bad = (rng.random(n1 + n2) < 0.05).astype(np.uint8)
    v1, v2 = (has1 & (bad[:n1] == 0)).astype(np.uint8), (has2 & (bad[n1:] == 0)).astype(np.uint8)
    mp1 = np.where(has1, np.arange(n1), -1).astype(np.int32)
    mp2 = np.where(has2, n1 + np.arange(n2), -1).astype(np.int32)
    bn, bout = gold_gpu(f"search_by_bow_kfkf/{masks}", lambda: rm.search_by_bow_kfkf(
        rm.KF(F1, cams, mp=mp1), rm.KF(F2, cams, mp=mp2), rm.MPTable(3, np.zeros((n1 + n2, 32), np.uint8), bad=bad), 0.9, masks))
    if RECORD:
        pytest.skip("reference outputs recorded")
    m = api.cORBmatcher(0.9, False, 32, masks)
    # SearchForInitialization
    prev = np.stack([F1.keys["x"], F1.keys["y"]], axis=1).astype(np.float64)
    gn, g12 = m.SearchForInitialization(F1, F2, prev.copy(), 50)
    rn, r12, _ = gold(f"search_for_initialization/{masks}/50", lambda: T.sfi_reference(rm, F1, F2, cams, prev, 50, masks))
    assert gn == rn and np.array_equal(g12, r12) and gn > 150
    gn, g12 = m.SearchByBoW(F1.desc, F2.desc, F1.dmask, F2.dmask, v1, v2)
    assert gn == bn and np.array_equal(g12, np.where(bout >= 0, bout - n1, -1)) and gn > 50


@pytest.mark.parametrize("masks", [False, True])
@pytest.mark.parametrize("variant", [1, 2])
@not_recording
def test_fuse_gpu_vs_reference(api, oa, rm, gold, frames, cams, masks, variant):
    """same scene as tests/test_ref_match_cpu.py::test_fuse_equals_reference"""
    KF = frames[0]
    sc = T.make_scene(api, oa, cams, KF, 11 + variant)
    rng = np.random.default_rng(5)
    n = len(sc["world"])
    kf_mp = np.full(len(KF.keys), -1, np.int32)
    occupied = rng.choice(len(KF.keys), len(KF.keys) // 3, replace=False)
    kf_mp[occupied] = n + np.arange(len(occupied))
    bad = np.concatenate([sc["bad"], (rng.random(len(occupied)) < 0.1).astype(np.uint8)])
    in_kf = np.concatenate([(rng.random(n) < 0.1), np.ones(len(occupied), bool)])
    pad = lambda a, fill=0.0: np.concatenate([a, np.full((len(occupied),) + a.shape[1:], fill, a.dtype)])
    points = np.arange(n, dtype=np.int32)
    Scw = None
    if variant == 2:
        Scw = api.inv_rigid(sc["M_t"]).copy()
        Scw[:3, :3] *= 1.3
        Scw[:3, 3] *= 1.3
    m = api.cORBmatcher(0.6, False, 32, masks)
    args = (KF, sc["rig"], kf_mp, points, pad(sc["world"]), pad(sc["min_d"], 1.0), pad(sc["max_d"], 2.0), bad, in_kf, pad(sc["desc"]),
            pad(sc["dmask"]))
    gn, gops, _ = m.Fuse(*args, th=2.5, variant=variant, Scw=Scw)
    table = lambda: rm.MPTable(3, pad(sc["desc"]), dmask=pad(sc["dmask"]), bad=bad, world_pos=pad(sc["world"]), min_dist=pad(sc["min_d"], 1.0),
                               max_dist=pad(sc["max_d"], 2.0), obs_kf=np.where(in_kf, 0, -1).astype(np.int32),
                               obs_idx=np.zeros(len(bad), np.int32))
    rn, rops = gold(f"fuse/{variant}/{masks}", lambda: rm.fuse(
        variant, rm.KF(KF, cams, M_c=sc["M_c"], M_t=sc["M_t"], mp=kf_mp, rays=sc["rays"]), table(), points, 2.5, 0.6, masks, Scw=Scw))
    assert gn == rn and np.array_equal(gops, rops) and len(gops) > 100


@not_recording
@pytest.mark.parametrize("masks", [False, True])
def test_scw_rule_gpu_vs_oracle_multicamera(api, oa, frames, cams, masks):
    """MCS_RULE_SCW on a 3-camera key frame: contiguous id used as the per-camera descriptor row, rows beyond the camera's own
    dropped, keypoint 0 never matched, taken keypoints skipped -- kernel + replay vs the oracle restatement of the same rule"""
    KF = frames[0]
    sc = T.make_scene(api, oa, cams, KF, 41)
    n = len(sc["world"])
    points = np.arange(n, dtype=np.int32)
    matched = np.full(len(KF.keys), -1, np.int32)
    matched[::7] = 0
    Scw = api.inv_rigid(sc["M_t"])
    m = api.cORBmatcher(0.6, False, 32, masks)
    args = (KF, sc["rig"], Scw, points, matched, sc["world"], sc["min_d"], sc["max_d"], sc["bad"], sc["desc"], sc["dmask"])
    gn, gm = m.SearchByProjectionKFScw(*args, th=10)
    on, om = m.SearchByProjectionKFScw(*args, th=10, _sw=oa.search_windows)
    assert gn == on and np.array_equal(gm, om)


@pytest.mark.parametrize("masks", [False, True])
def test_sim3_and_between_cameras_gpu(api, oa, rm, gold, gold_gpu, frames, cams, masks):
    """SearchBySim3 and SearchForTriangulationBetweenCameras as whole entry points over the CUDA window search: the between-cameras
    scene is the CPU check's (tests/test_ref_match_cpu.py), the Sim3 scene this test's own; CUDA vs the reference's outputs"""
    KF = frames[0]
    # Sim3
    sc1 = T.make_scene(api, oa, cams, KF, 51, npts=300)
    rng2 = np.random.default_rng(52)
    w2 = sc1["world"] + rng2.normal(0, 0.003, sc1["world"].shape)
    d2 = T.flip_bits(rng2, KF.desc[sc1["src"]], 30)
    world = np.concatenate([sc1["world"], w2]); desc = np.concatenate([sc1["desc"], d2]); dmask = np.concatenate([sc1["dmask"], sc1["dmask"]])
    bad = np.concatenate([sc1["bad"], np.roll(sc1["bad"], 7)])
    min_d = np.concatenate([sc1["min_d"], sc1["min_d"]]) * 0.5; max_d = np.concatenate([sc1["max_d"], sc1["max_d"]]) * 2.0
    mp1 = np.full(len(KF.keys), -1, np.int32); mp1[sc1["src"]] = np.arange(300)
    mp2 = np.full(len(KF.keys), -1, np.int32); mp2[sc1["src"]] = 300 + np.arange(300)
    a = 0.002
    R12 = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1.0]])
    s12, t12 = 1.002, np.array([0.002, -0.001, 0.003])
    pre = np.full(len(KF.keys), -1, np.int32)
    obs_idx = np.concatenate([sc1["src"], sc1["src"]]).astype(np.int32)
    sn, s12_ref = gold_gpu(f"search_by_sim3/{masks}", lambda: rm.search_by_sim3(
        rm.KF(KF, cams, M_c=sc1["M_c"], M_t=sc1["M_t"], mp=mp1), rm.KF(KF, cams, M_c=sc1["M_c"], M_t=sc1["M_t"], mp=mp2),
        rm.MPTable(3, desc, dmask=dmask, bad=bad, world_pos=world, min_dist=min_d, max_dist=max_d,
                   obs_kf=np.concatenate([np.zeros(300, np.int32), np.ones(300, np.int32)]), obs_idx=obs_idx),
        s12, R12, t12, 7.5, pre, 0.6, masks))
    if RECORD:
        pytest.skip("reference outputs recorded")
    m = api.cORBmatcher(0.6, False, 32, masks)
    gn, g12 = m.SearchBySim3(KF, sc1["rig"], mp1, KF, sc1["rig"], mp2, world, min_d, max_d, bad, desc, dmask, s12, R12, t12, 7.5,
                             matches12=pre, obs_idx2=obs_idx)
    assert gn == sn and np.array_equal(g12, s12_ref) and gn > 10
    # between cameras
    M_c = np.tile(np.eye(4), (3, 1, 1))
    for c in range(3):
        a = 0.05 * c
        M_c[c, :3, :3] = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
        M_c[c, :3, 3] = [0.2 * c, 0.0, 0.0]
    rig = api.Rig(cams, M_c, np.eye(4))
    rays, _, _ = api.frame_prepare(KF.keys, KF.key_cam, cams)
    rng = np.random.default_rng(2)
    kf_mp = np.where(rng.random(len(KF.keys)) < 0.3, 0, -1).astype(np.int32)
    gn, gp = m.SearchForTriangulationBetweenCameras(KF, rig, kf_mp, rays, 0, 1)
    rn, rp = gold(f"search_for_triangulation_between/{masks}/0/1", lambda: rm.search_for_triangulation_between(
        rm.KF(KF, cams, M_c=M_c, mp=kf_mp, rays=rays), rm.MPTable(3, np.zeros((1, 32), np.uint8)), 0, 1, 0.6, masks))
    assert gn == rn and np.array_equal(gp, rp) and gn > 50
