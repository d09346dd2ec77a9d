"""CPU: the matcher restatements (oracle/mcs_oracle.cpp) pinned by the REFERENCE'S OWN matcher -- the original project's
src/cORBmatcher.cpp compiled into oracle/_ref/libmcs_ref.so (oracle/ref_mcs/wrap_match.cpp; the three SLAM container classes it
reads are data-only stand-ins, oracle/ref_mcs/stub_slam.h).  Its outputs on these scenes are stored in
tests/golden/ref_match_cpu.npz (tests/ref_golden.py); where the library is built it is run as well and must reproduce them."""
import pathlib
import sys

import numpy as np
import pytest

from ref_golden import RefGolden, crc

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "oracle"))
SIZES = [(754, 480)] * 3


@pytest.fixture(scope="module")
def rm():
    import ref_match_api
    return ref_match_api


@pytest.fixture(scope="module")
def gold():
    g = RefGolden("ref_match_cpu")
    yield g
    g.save()


@pytest.fixture(scope="module")
def api():
    import multicol_slam_b200.api as a            # holders and host-side compositions only; no device call is made in this file
    return a


@pytest.fixture(scope="module")
def frames(oa, cams):
    """two consecutive 3-camera frames of the sliding-texture stream, extracted by the CPU oracle"""
    import multicol_slam_b200.api as api            # plain array holders only; no device call is made in this file
    from multicol_slam_b200 import synth
    ex = oa.OracleExtractor(nfeatures=350, do_dbrief=True, learn_masks=True)
    sf = [float(ex.info.scale_factor[l]) for l in range(8)]
    out = []
    streams = [synth.texture_stream(cams[c], 2, seed=60 + c) for c in range(3)]
    for t in range(2):
        per = [ex.extract(streams[c][t], synth.mirror_mask(cams[c]), cams[c]) for c in range(3)]
        out.append(api.Frame.from_cameras(per, SIZES, sf))
    return out


def flip_bits(rng, desc, kmax):
    d = desc.copy()
    for i in range(len(d)):
        for b in rng.choice(8 * d.shape[1], rng.integers(0, kmax + 1), replace=False):
            d[i, b // 8] ^= 1 << (b % 8)
    return d


def test_thresholds_and_distances(oa, rm, gold):
    for dim, masks, th in ((32, False, (96, 64)), (32, True, (48, 32)), (16, True, (24, 16)), (64, False, (192, 128))):
        assert gold(f"thresholds/{dim}/{masks}", lambda: rm.thresholds(dim, masks)) == th
    rng = np.random.default_rng(0)
    for dim in (16, 32, 64):
        v = [[rng.integers(0, 256, dim).astype(np.uint8) for _ in range(4)] for _ in range(200)]
        rd = gold(f"distance64/{dim}", lambda: np.array([rm.distance64(a, b, dim) for a, b, _, _ in v]))
        rdm = gold(f"distance64_masked/{dim}", lambda: np.array([rm.distance64_masked(a, b, ma, mb, dim) for a, b, ma, mb in v]))
        assert np.array_equal(rd, [oa.distance64(a, b, dim) for a, b, _, _ in v])
        assert np.array_equal(rdm, [oa.distance64_masked(a, b, ma, mb, dim) for a, b, ma, mb in v])


def test_features_in_area_three_ways(oa, rm, gold, frames, cams):
    """the grid lookup is the one piece of logic the stand-in containers restate: reference-shaped stand-in (stub_slam.h) ==
    C++ oracle == plain-Python restatement, for the frame overload (level filters) and the key-frame overload (<=)"""
    import pyref_match as pm
    from multicol_slam_b200.ctypes_defs import WINDOW_QUERY_DTYPE
    F = frames[0]
    grid = pm.Grid(F.keys, F.key_cam, SIZES)
    rng = np.random.default_rng(1)
    queries = []
    for i in range(150):
        cam, lv, kind = int(rng.integers(0, 3)), int(rng.integers(0, 8)), int(rng.integers(0, 3))
        x, y, r = float(rng.uniform(-30, 790)), float(rng.uniform(-30, 510)), float(rng.uniform(1, 60))
        if i % 5 == 0:                                       # exactly on a keypoint, integer radius: the > r vs <= r boundary
            k = int(rng.integers(0, len(F.keys)))
            cam, x, y, r = int(F.key_cam[k]), float(F.keys["x"][k]) + 7.0, float(F.keys["y"][k]), 7.0
        lo, hi = (-1, -1) if kind == 0 else ((lv, lv) if kind == 1 else (max(lv - 1, 0), lv))
        queries.append((cam, x, y, r, lo, hi))

    def ref_lists(keyframe):                                 # the per-query index lists, concatenated, and their offsets
        kf = rm.KF(F, cams)
        lists = [rm.features_in_area(kf, keyframe, cam, x, y, r, *((-1, -1) if keyframe else (lo, hi))) for cam, x, y, r, lo, hi in queries]
        return np.array([i for l in lists for i in l], np.int64), np.cumsum([0] + [len(l) for l in lists])
    fr, fo = gold("features_in_area/frame", lambda: ref_lists(False))
    kr, ko = gold("features_in_area/keyframe", lambda: ref_lists(True))
    for i, (cam, x, y, r, lo, hi) in enumerate(queries):
        ref = [int(v) for v in fr[fo[i]:fo[i + 1]]]
        assert ref == grid.features_in_area(cam, x, y, r, lo, hi)
        q = np.zeros(1, WINDOW_QUERY_DTYPE)
        q["cam"], q["x"], q["y"], q["r"], q["min_level"], q["max_level"] = cam, x, y, r, lo, hi
        oi, _, oc, rc = oa.window_search(F, q, F.desc, F.dmask, max_cand=1024)
        assert rc == 0 and ref == list(oi[0, :oc[0]])
        refk = [int(v) for v in kr[ko[i]:ko[i + 1]]]
        assert refk == grid.features_in_area_kf(cam, x, y, r) if hasattr(grid, "features_in_area_kf") else True


@pytest.mark.parametrize("masks", [False, True])
def test_search_by_projection_equals_reference(oa, rm, gold, frames, cams, masks):
    import multicol_slam_b200.api as api
    F = frames[0]
    rng = np.random.default_rng(3 + masks)
    nmp, nc = 700, 3
    src = rng.integers(0, len(F.keys), nmp)
    desc, dm = flip_bits(rng, F.desc[src], 40), F.dmask[src].copy()
    in_view = np.zeros((nmp, nc), np.uint8); level = np.zeros((nmp, nc), np.int32)
    px = np.zeros((nmp, nc)); py = np.zeros((nmp, nc)); vc = np.zeros((nmp, nc))
    for i in range(nmp):
        c = F.key_cam[src[i]]
        in_view[i, c] = 1
        level[i, c] = min(7, max(0, F.keys[src[i]]["octave"] + rng.integers(-1, 2)))
        px[i, c] = F.keys[src[i]]["x"] + rng.normal(0, 2); py[i, c] = F.keys[src[i]]["y"] + rng.normal(0, 2)
        vc[i, c] = rng.uniform(0.99, 1.0)
        if rng.random() < 0.2:
            c2 = (c + 1) % nc
            in_view[i, c2] = 1; level[i, c2] = rng.integers(0, 8)
            px[i, c2] = rng.uniform(0, 754); py[i, c2] = rng.uniform(0, 480); vc[i, c2] = rng.uniform(0.9, 1.0)
    bad = (rng.random(nmp) < 0.05).astype(np.uint8)
    mps = api.MapPoints(bad, in_view, level, px, py, vc, desc, dm)
    table = lambda: rm.MPTable(nc, desc, dmask=dm, bad=bad, in_view=in_view, level=level, proj_x=px, proj_y=py, view_cos=vc)
    th_high, _ = gold(f"thresholds/32/{masks}", lambda: rm.thresholds(32, masks))
    for th, pre in ((3.0, None), (1.0, np.where(np.arange(len(F.keys)) % 3 == 0, 0, -1))):
        start = np.full(len(F.keys), -1, np.int32) if pre is None else pre.astype(np.int32)
        on, ofmp = oa.search_by_projection(F, mps, th, 0.8, th_high, masks, start.copy())
        rn, rfmp = gold(f"search_by_projection/{masks}/{th}", lambda: rm.search_by_projection(rm.KF(F, cams, mp=start), table(), th, 0.8, masks))
        assert on == rn and np.array_equal(ofmp, rfmp)
        assert on > 100


def sfi_reference(rm, F1, F2, cams, prev, window, masks):
    """SearchForInitialization of the reference: (matches, matches12, CRC of the updated previous positions)"""
    n, m12, prev = rm.search_for_initialization(rm.KF(F1, cams), rm.KF(F2, cams), prev, window, 0.9, masks)
    return n, m12, crc(prev)


@pytest.mark.parametrize("masks", [False, True])
def test_search_for_initialization_equals_reference(oa, rm, gold, frames, cams, masks):
    F1, F2 = frames
    prev = np.stack([F1.keys["x"], F1.keys["y"]], axis=1).astype(np.float64)
    _, th_low = gold(f"thresholds/32/{masks}", lambda: rm.thresholds(32, masks))
    for window in (50, 100):
        on, om12, oprev = oa.search_for_initialization(F1, F2, prev, window, 0.9, th_low, masks)
        rn, rm12, rprev = gold(f"search_for_initialization/{masks}/{window}", lambda: sfi_reference(rm, F1, F2, cams, prev, window, masks))
        assert on == rn and np.array_equal(om12, rm12) and crc(oprev) == rprev
        assert on > 150


@pytest.mark.parametrize("masks", [False, True])
def test_search_by_bow_kfkf_equals_reference(oa, rm, gold, frames, cams, masks):
    """SearchByBoW(KF1, KF2): all-pairs scan incl. the greedy one-use rule; a third of the keypoints carry no map point, some bad"""
    F1, F2 = frames
    rng = np.random.default_rng(7 + masks)
    n1, n2 = len(F1.keys), len(F2.keys)
    has1, has2 = rng.random(n1) < 0.7, rng.random(n2) < 0.7
    mp1 = np.where(has1, np.arange(n1), -1).astype(np.int32)               # map point ids: KF1 keypoint i -> i, KF2 keypoint j -> n1 + j
    mp2 = np.where(has2, n1 + np.arange(n2), -1).astype(np.int32)
    bad = (rng.random(n1 + n2) < 0.05).astype(np.uint8)
    _, th_low = gold(f"thresholds/32/{masks}", lambda: rm.thresholds(32, masks))
    v1 = (has1 & (bad[:n1] == 0)).astype(np.uint8)
    v2 = (has2 & (bad[n1:] == 0)).astype(np.uint8)
    on, om12 = oa.match_bruteforce(F1.desc, F2.desc, th_low, 0.9, F1.dmask if masks else None, F2.dmask if masks else None, v1, v2)
    rn, rout = gold(f"search_by_bow_kfkf/{masks}", lambda: rm.search_by_bow_kfkf(
        rm.KF(F1, cams, mp=mp1), rm.KF(F2, cams, mp=mp2), rm.MPTable(3, np.zeros((n1 + n2, 32), np.uint8), bad=bad), 0.9, masks))
    ref12 = np.where(rout >= 0, rout - n1, -1)
    assert on == rn and np.array_equal(om12, ref12) and on > 50


def test_check_orientation_constant():
    """every call site passes the compile-time constant checkOrientation == false (include/cORBmatcher.h:40): the wrapper does too"""
    txt = (ROOT / "oracle" / "ref_mcs" / "wrap_match.cpp").read_text()
    assert txt.count("checkOrientation") >= 10


# ---- scenes with 3-D map points for the projection-based searches ---------------------------------------------------------------
def make_scene(api, oa, cams, frame, seed, npts=500, pose_noise=0.0):
    """A key frame = `frame` on a 3-camera rig, and map points that really project near its keypoints: each point sits on the
    bearing ray of a keypoint at a random depth; descriptor = that keypoint's with a few flipped bits."""
    rng = np.random.default_rng(seed)
    nc = 3
    M_c = np.tile(np.eye(4), (nc, 1, 1))
    for c in range(nc):                                            # cameras looking 120 degrees apart, 10 cm off the rig centre
        a = 2 * np.pi * c / nc
        M_c[c, :3, :3] = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
        M_c[c, :3, 3] = [0.1 * np.sin(a), 0.0, 0.1 * np.cos(a)]
    M_t = np.eye(4)
    M_t[:3, 3] = [0.3, -0.2, 0.1]
    rig = api.Rig(cams, M_c, M_t)
    rays, _, _ = oa.frame_prepare(frame.keys, frame.key_cam, cams)
    src = rng.choice(len(frame.keys), npts, replace=False)
    depth = rng.uniform(2.0, 6.0, npts)
    world = np.zeros((npts, 3))
    for i, k in enumerate(src):
        pc = np.append(rays[k] * depth[i], 1.0)
        world[i] = api._mm(rig.MtMc[int(frame.key_cam[k])], pc)[:3] + rng.normal(0, pose_noise, 3)
    desc = flip_bits(rng, frame.desc[src], 30)
    dmask = frame.dmask[src].copy()
    bad = (rng.random(npts) < 0.05).astype(np.uint8)
    min_d, max_d = depth * rng.uniform(0.5, 0.9, npts), depth * rng.uniform(1.2, 3.0, npts)
    return dict(rig=rig, M_c=M_c, M_t=M_t, rays=rays, src=src, world=world, desc=desc, dmask=dmask, bad=bad, min_d=min_d, max_d=max_d)


@pytest.mark.parametrize("masks", [False, True])
@pytest.mark.parametrize("variant", [1, 2])
def test_fuse_equals_reference(oa, rm, gold, api, frames, cams, masks, variant):
    """Fuse(pKF, vpMapPoints, th) -- the live overload whose distance is discarded -- and Fuse(pKF, Scw, vpPoints, th): the host
    composition over the oracle's window search reproduces the reference's map mutations in order"""
    KF = frames[0]
    sc = make_scene(api, oa, cams, KF, 11 + variant)
    rng = np.random.default_rng(5)
    n = len(sc["world"])
    kf_mp = np.full(len(KF.keys), -1, np.int32)                    # a third of the key frame's keypoints already carry a (fresh) map point
    occupied = rng.choice(len(KF.keys), len(KF.keys) // 3, replace=False)
    extra_bad = (rng.random(len(occupied)) < 0.1).astype(np.uint8)
    kf_mp[occupied] = n + np.arange(len(occupied))
    bad = np.concatenate([sc["bad"], extra_bad])
    in_kf = np.concatenate([(rng.random(n) < 0.1), np.ones(len(occupied), bool)])
    obs_kf = np.where(in_kf, 0, -1).astype(np.int32)
    tot = n + len(occupied)
    pad = lambda a, fill=0.0: np.concatenate([a, np.full((len(occupied),) + a.shape[1:], fill, a.dtype)])
    table = lambda: rm.MPTable(3, pad(sc["desc"]), dmask=pad(sc["dmask"]), bad=bad, world_pos=pad(sc["world"]), min_dist=pad(sc["min_d"], 1.0),
                               max_dist=pad(sc["max_d"], 2.0), obs_kf=obs_kf, obs_idx=np.zeros(tot, np.int32))
    points = np.arange(n, dtype=np.int32)
    Scw = None
    if variant == 2:
        s = 1.3
        Tcw = api.inv_rigid(sc["M_t"])
        Scw = Tcw.copy()
        Scw[:3, :3] *= s
        Scw[:3, 3] *= s
    kfr = lambda: rm.KF(KF, cams, M_c=sc["M_c"], M_t=sc["M_t"], mp=kf_mp, rays=sc["rays"])
    rn, rops = gold(f"fuse/{variant}/{masks}", lambda: rm.fuse(variant, kfr(), table(), points, 2.5, 0.6, masks, Scw=Scw))
    m = api.cORBmatcher(0.6, False, 32, masks)
    on, oops, _ = m.Fuse(KF, sc["rig"], kf_mp, points, pad(sc["world"]), pad(sc["min_d"], 1.0), pad(sc["max_d"], 2.0), bad, in_kf,
                         pad(sc["desc"]), pad(sc["dmask"]), th=2.5, variant=variant, Scw=Scw, _sw=oa.search_windows)
    assert rn == on and np.array_equal(rops, oops)
    assert len(rops) > 100 and (rops[:, 0] == 1).sum() > 10 and (rops[:, 0] == 0).sum() > 10


def test_fuse_1420_ignores_the_distance(oa, rm, gold, api, frames, cams):
    """the reference's Fuse(pKF, vpMapPoints, th) returns the same mutations whatever the map point descriptors are"""
    KF = frames[0]
    sc = make_scene(api, oa, cams, KF, 21)
    n = len(sc["world"])
    kf_mp = np.full(len(KF.keys), -1, np.int32)
    out = []
    for i, desc in enumerate((sc["desc"], 255 - sc["desc"])):
        table = lambda: rm.MPTable(3, desc, dmask=sc["dmask"], bad=sc["bad"], world_pos=sc["world"], min_dist=sc["min_d"], max_dist=sc["max_d"])
        out.append(gold(f"fuse_1420/{i}", lambda: rm.fuse(1, rm.KF(KF, cams, M_c=sc["M_c"], M_t=sc["M_t"], mp=kf_mp), table(),
                                                          np.arange(n, dtype=np.int32), 2.5, 0.6, False)))
    assert out[0][0] == out[1][0] and np.array_equal(out[0][1], out[1][1]) and len(out[0][1]) > 100


@pytest.mark.parametrize("masks", [False, True])
def test_search_by_projection_scw_equals_reference(oa, rm, gold, api, frames, cams, masks):
    """SearchByProjection(pKF, Scw, vpPoints, vpMatched, th) with its quirks (camera looked up with the list position, contiguous id
    as descriptor row, bestIdx > 0).  The scene keeps every candidate inside the range where the reference's reads are defined:
    all keypoints of the key frame belong to camera 0 (contiguous id == row)."""
    import multicol_slam_b200.api as apimod
    F = frames[0]
    sel = np.flatnonzero(F.key_cam == 0)
    KF = apimod.Frame(F.keys[sel], F.key_cam[sel], F.desc[sel], F.dmask[sel], SIZES, F.scale_factors)
    sc = make_scene(api, oa, cams, KF, 31, npts=len(sel) - 5)
    n = len(sc["world"])
    # vpPoints entry iMP projects near keypoint src[iMP]; put point 3 at keypoint 0 so that the `bestIdx > 0` rule is exercised
    points = np.arange(n, dtype=np.int32)
    rng = np.random.default_rng(8)
    points[rng.random(n) < 0.05] = -1
    matched = np.full(len(KF.keys), -1, np.int32)
    pre = rng.choice(len(KF.keys), 30, replace=False)
    matched[pre] = rng.choice(n, 30, replace=False)
    Tcw = api.inv_rigid(sc["M_t"])
    Scw = Tcw.copy()
    Scw[:3, :3] *= 0.8
    Scw[:3, 3] *= 0.8
    table = lambda: rm.MPTable(3, sc["desc"], dmask=sc["dmask"], bad=sc["bad"], world_pos=sc["world"], min_dist=sc["min_d"], max_dist=sc["max_d"])
    rn, rmatched = gold(f"search_by_projection_scw/{masks}", lambda: rm.search_by_projection_scw(
        rm.KF(KF, cams, M_c=sc["M_c"], M_t=sc["M_t"]), table(), Scw, points, matched, 10, 0.6, masks))
    m = api.cORBmatcher(0.6, False, 32, masks)
    on, omatched = m.SearchByProjectionKFScw(KF, sc["rig"], Scw, points, matched, sc["world"], sc["min_d"], sc["max_d"], sc["bad"],
                                             sc["desc"], sc["dmask"], th=10, _sw=oa.search_windows)
    assert rn == on and np.array_equal(rmatched, omatched) and rn > 50
    assert omatched[0] == matched[0]                               # keypoint 0 is never assigned (:2385)


def test_search_for_triangulation_between_cameras_equals_reference(oa, rm, gold, api, frames, cams):
    """a rig whose cameras overlap: keypoints of camera 0 searched in camera 1 along their bearing rays"""
    KF = frames[0]
    nc = 3
    M_c = np.tile(np.eye(4), (nc, 1, 1))
    for c in range(nc):                                            # nearly parallel cameras, 20 cm apart
        a = 0.05 * c
        M_c[c, :3, :3] = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
        M_c[c, :3, 3] = [0.2 * c, 0.0, 0.0]
    rig = api.Rig(cams, M_c, np.eye(4))
    rays, _, _ = oa.frame_prepare(KF.keys, KF.key_cam, cams)
    rng = np.random.default_rng(2)
    kf_mp = np.where(rng.random(len(KF.keys)) < 0.3, 0, -1).astype(np.int32)
    for masks in (False, True):
        m = api.cORBmatcher(0.6, False, 32, masks)
        for c1, c2 in ((0, 1), (2, 0)):
            rn, rp = gold(f"search_for_triangulation_between/{masks}/{c1}/{c2}", lambda: rm.search_for_triangulation_between(
                rm.KF(KF, cams, M_c=M_c, mp=kf_mp, rays=rays), rm.MPTable(3, np.zeros((1, 32), np.uint8)), c1, c2, 0.6, masks))
            on, op = m.SearchForTriangulationBetweenCameras(KF, rig, kf_mp, rays, c1, c2, _sw=oa.search_windows)
            assert rn == on and np.array_equal(rp, op)
            assert rn > 50


@pytest.mark.parametrize("masks", [False, True])
def test_search_by_sim3_equals_reference(oa, rm, gold, api, frames, cams, masks):
    """two key frames seeing the same map points from poses related by a similarity; a few matches given beforehand"""
    KF1 = KF2 = frames[0]
    sc1 = make_scene(api, oa, cams, KF1, 51, npts=300)
    # key frame 2 is a second view of the same keypoints: its own map points (ids 300..599) sit where key frame 1's do, up to
    # a few millimetres, with their own descriptor variants -- so that the two projections find each other (mutual check)
    rng2 = np.random.default_rng(52)
    sc2 = dict(sc1)
    sc2["world"] = sc1["world"] + rng2.normal(0, 0.003, sc1["world"].shape)
    sc2["desc"] = flip_bits(rng2, KF1.desc[sc1["src"]], 30)
    n = 600
    world = np.concatenate([sc1["world"], sc2["world"]])
    desc = np.concatenate([sc1["desc"], sc2["desc"]]); dmask = np.concatenate([sc1["dmask"], sc2["dmask"]])
    bad = np.concatenate([sc1["bad"], np.roll(sc1["bad"], 7)])
    min_d = np.concatenate([sc1["min_d"], sc2["min_d"]]) * 0.5; max_d = np.concatenate([sc1["max_d"], sc2["max_d"]]) * 2.0
    mp1 = np.full(len(KF1.keys), -1, np.int32); mp1[sc1["src"]] = np.arange(300)
    mp2 = np.full(len(KF2.keys), -1, np.int32); mp2[sc2["src"]] = 300 + np.arange(300)
    rng = np.random.default_rng(6)
    a = 0.002
    R12 = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1.0]])
    s12, t12 = 1.002, np.array([0.002, -0.001, 0.003])
    pre = np.full(len(KF1.keys), -1, np.int32)
    some = rng.choice(sc1["src"], 10, replace=False)
    pre[some] = 300 + rng.choice(300, 10, replace=False)           # already matched to map points of key frame 2
    obs_kf = np.concatenate([np.zeros(300, np.int32), np.ones(300, np.int32)])
    obs_idx = np.concatenate([sc1["src"], sc2["src"]]).astype(np.int32)
    rn, r12 = gold(f"search_by_sim3/{masks}", lambda: rm.search_by_sim3(
        rm.KF(KF1, cams, M_c=sc1["M_c"], M_t=sc1["M_t"], mp=mp1), rm.KF(KF2, cams, M_c=sc2["M_c"], M_t=sc2["M_t"], mp=mp2),
        rm.MPTable(3, desc, dmask=dmask, bad=bad, world_pos=world, min_dist=min_d, max_dist=max_d, obs_kf=obs_kf, obs_idx=obs_idx),
        s12, R12, t12, 7.5, pre, 0.6, masks))
    m = api.cORBmatcher(0.6, False, 32, masks)
    on, o12 = m.SearchBySim3(KF1, sc1["rig"], mp1, KF2, sc2["rig"], mp2, world, min_d, max_d, bad, desc, dmask, s12, R12, t12, 7.5,
                             matches12=pre, obs_idx2=obs_idx, _sw=oa.search_windows)
    assert rn == on and np.array_equal(r12, o12)
    assert rn > 10


@pytest.mark.parametrize("masks", [False, True])
def test_projection_searches_between_frames_equal_reference(oa, rm, gold, api, frames, cams, masks):
    """SearchByProjection(F1, F2, window) (:476) and SearchByProjection(CurrentFrame, LastFrame, th) (:1990) as whole entry points:
    F1 / LastFrame carry map points that really lie on their bearing rays; F2 / CurrentFrame is the next frame of the stream
    under a slightly different rig pose"""
    F1, F2 = frames
    sc = make_scene(api, oa, cams, F1, 61, npts=600)
    n = 600
    mp1 = np.full(len(F1.keys), -1, np.int32); mp1[sc["src"]] = np.arange(n)
    mp1[sc["src"][5]] = mp1[sc["src"][4]]                              # the same map point twice in F1: only its first keypoint counts
    rng = np.random.default_rng(9)
    M_t2 = sc["M_t"].copy()
    M_t2[:3, 3] += [0.004, -0.003, 0.002]
    rig2 = api.Rig(cams, sc["M_c"], M_t2)
    mp2 = np.full(len(F2.keys), -1, np.int32)
    mp2[rng.choice(len(F2.keys), 80, replace=False)] = rng.choice(n, 80, replace=False)      # some already found in F2
    outlier = (rng.random(len(F1.keys)) < 0.1).astype(np.uint8)
    table = lambda: rm.MPTable(3, sc["desc"], dmask=sc["dmask"], bad=sc["bad"], world_pos=sc["world"], min_dist=sc["min_d"], max_dist=sc["max_d"])
    k1 = lambda: rm.KF(F1, cams, M_c=sc["M_c"], M_t=sc["M_t"], mp=mp1, outlier=outlier)
    k2 = lambda: rm.KF(F2, cams, M_c=sc["M_c"], M_t=M_t2, mp=mp2)
    m = api.cORBmatcher(0.8, False, 32, masks)
    rn, rout = gold(f"search_by_projection_frames/{masks}", lambda: rm.search_by_projection_frames(k1(), k2(), table(), 40, 0.8, masks))
    on, oout = m.SearchByProjectionFramesRig(F1, mp1, F2, rig2, mp2, sc["world"], sc["bad"], 40, _sw=oa.search_windows)
    assert rn == on and np.array_equal(rout, oout) and rn > 50
    rn, rout = gold(f"search_by_projection_last/{masks}", lambda: rm.search_by_projection_last(k2(), k1(), table(), 50.0, 0.8, masks))
    on, oout = m.SearchByProjectionLastRig(F2, rig2, mp2, F1, mp1, outlier, sc["world"], sc["bad"], 50.0, _sw=oa.search_windows)
    assert rn == on and np.array_equal(rout, oout) and rn > 100


@pytest.mark.parametrize("masks", [False, True])
def test_window_search_triangulation_and_bow_frame_equal_reference(oa, rm, gold, api, frames, cams, masks):
    """WindowSearch (:326), SearchForTriangulationRaw (:968, incl. ComputeE / CheckDistEpipolarLine of the reference) and
    SearchByBoW(KF, F) (:179) against the reference's own matcher"""
    F1, F2 = frames
    rng = np.random.default_rng(12 + masks)
    n1, n2 = len(F1.keys), len(F2.keys)
    m = api.cORBmatcher(0.8, False, 32, masks)
    # WindowSearch: F1 keypoints with a (non-bad) map point look into a 60 px window of F2, levels >= 1
    has1 = rng.random(n1) < 0.6
    bad = (rng.random(n1) < 0.05).astype(np.uint8)
    mp1 = np.where(has1, np.arange(n1), -1).astype(np.int32)
    rn, rout = gold(f"window_search/{masks}", lambda: rm.window_search(
        rm.KF(F1, cams, mp=mp1), rm.KF(F2, cams), rm.MPTable(3, np.zeros((n1, 32), np.uint8), bad=bad), 60, 1, 2**31 - 1, 0.8, masks))
    on, o21 = m.WindowSearch(F1, F2, 60, has1 & (bad == 0), 1, _sw=oa.search_windows)
    assert rn == on and np.array_equal(rout, o21) and rn > 50               # map point id == F1 keypoint index here
    # SearchForTriangulationRaw: keypoints WITHOUT map points, same camera only, epipolar check with E from the two rig poses
    sc = make_scene(api, oa, cams, F1, 71, npts=10)
    M_t2 = sc["M_t"].copy()
    M_t2[:3, 3] += [0.05, 0.01, -0.02]
    rays1, _, _ = oa.frame_prepare(F1.keys, F1.key_cam, cams)
    rays2, _, _ = oa.frame_prepare(F2.keys, F2.key_cam, cams)
    free1, free2 = rng.random(n1) < 0.5, rng.random(n2) < 0.5
    rn, rpairs = gold(f"search_for_triangulation_raw/{masks}", lambda: rm.search_for_triangulation_raw(
        rm.KF(F1, cams, M_c=sc["M_c"], M_t=sc["M_t"], mp=np.where(free1, -1, 0).astype(np.int32), rays=rays1),
        rm.KF(F2, cams, M_c=sc["M_c"], M_t=M_t2, mp=np.where(free2, -1, 0).astype(np.int32), rays=rays2),
        rm.MPTable(3, np.zeros((1, 32), np.uint8)), 0.6, masks))
    r1, r2 = api.Rig(cams, sc["M_c"], sc["M_t"]), api.Rig(cams, sc["M_c"], M_t2)
    import ref_mcs_api as ra
    # ComputeE(Get_MtMc_inv(i), Get_MtMc(j))  (ref :989-1000)
    E = gold(f"compute_E/{masks}", lambda: np.array([[ra.compute_E(r1.MtMc_inv[i], r2.MtMc[j]) for j in range(3)] for i in range(3)]))
    th_low = gold(f"thresholds/32/{masks}", lambda: rm.thresholds(32, masks))[1]
    on, om12 = oa.search_for_triangulation(F1.desc, F1.dmask if masks else None, F1.key_cam, free1, rays1, F2.desc, F2.dmask if masks else None,
                                           F2.key_cam, free2, rays2, E, th_low)
    opairs = np.array([(i, om12[i]) for i in range(n1) if om12[i] >= 0], np.int32).reshape(-1, 2)
    assert rn == on and np.array_equal(rpairs, opairs)
    # SearchByBoW(KF, F): feature vectors from the oracle vocabulary (pinned to the reference's DBoW2 elsewhere)
    voc = oa.OracleVocabulary(np.load(ROOT / "tests" / "golden" / "voc_small_9_6.npz"))
    fv1, fv2 = voc.transform(F1.desc, 4)[2:], voc.transform(F2.desc, 4)[2:]
    rn, rout = gold(f"search_by_bow_kff/{masks}", lambda: rm.search_by_bow_kff(
        rm.KF(F1, cams, mp=mp1, featvec=fv1), rm.KF(F2, cams, featvec=fv2), rm.MPTable(3, np.zeros((n1, 32), np.uint8), bad=bad), 0.7, masks))
    on, oout = oa.search_by_bow(F1.desc, F1.dmask if masks else None, (has1 & (bad == 0)).astype(np.uint8), fv1, F2.desc,
                                F2.dmask if masks else None, fv2, th_low, 0.7)
    assert rn == on and np.array_equal(rout, oout) and rn > 30
