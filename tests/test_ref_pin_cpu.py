"""CPU: the extractor restatement (oracle/mcs_oracle.cpp) pinned by outputs of the REFERENCE'S OWN code.

1. against the committed fixtures tests/golden/ref_extract_*.npz, written by tests/golden/make_ref_extract_golden.py from
   oracle/_ref/libmcs_ref.so (= the original project's src/mdBRIEFextractorOct.cpp, cam_model_omni.cpp, misc.cpp compiled in place);
2. against that library's outputs on more seeds and parameter corners, DistributeOctTree alone on adversarial tie-heavy corner
   lists, the camera model and the epipolar test of misc.cpp, stored in tests/golden/ref_pin_cpu.npz (tests/ref_golden.py; where
   the library is built it is run as well and must reproduce them);
3. the stand-in OpenCV primitives underneath the reference build against the real cv2 (only where cv2 is importable).
"""
import glob
import json
import pathlib

import numpy as np
import pytest

from ref_golden import RefGolden, crc

GOLD = pathlib.Path(__file__).resolve().parent / "golden"
FIXTURES = sorted(glob.glob(str(GOLD / "ref_extract_*.npz")))


def _ra():
    import ref_mcs_api as ra
    return ra


@pytest.fixture(scope="module")
def gold():
    g = RefGolden("ref_pin_cpu")
    yield g
    g.save()


def rows_and_crc(a):
    return len(a), crc(a)


def ref_extract_digest(kw, img, mask, cam):
    """the reference extractor's output as (n, crc of keypoints, crc of descriptors, crc of masks)"""
    k, d, m = _ra().RefExtractor(**kw).extract(img, mask, cam)
    return len(k), crc(k), crc(d), crc(m)


def load_case(path):
    from multicol_slam_b200 import synth
    g = np.load(path)
    cam = json.loads(bytes(g["cam_json"]).decode())
    kw = json.loads(bytes(g["params_json"]).decode())
    img = synth.frame(cam, int(g["seed"]))
    assert crc(img) == int(g["image_crc"]), "synthetic image generator changed"
    return g, cam, kw, img, synth.mirror_mask(cam)


def check_against_fixture(g, k, d, m):
    assert len(k) == int(g["n"])
    assert crc(k) == int(g["kps_crc"]) and crc(d) == int(g["desc_crc"]) and crc(m) == int(g["dmask_crc"])
    if "kps" in g.files:
        assert k.tobytes() == g["kps"].tobytes() and np.array_equal(d, g["desc"]) and np.array_equal(m, g["dmask"])


def test_fixture_set_is_complete():
    names = {pathlib.Path(p).stem for p in FIXTURES}
    assert len(names) >= 19 and {"ref_extract_shipped_orb400_cam0", "ref_extract_cfg2_mdbrief2000_cam0",
                                 "ref_extract_cfg4_1920x1080_mdbrief4000"} <= names


@pytest.mark.parametrize("path", FIXTURES, ids=lambda p: pathlib.Path(p).stem[12:])
def test_oracle_equals_reference_fixture(oa, path):
    g, cam, kw, img, mask = load_case(path)
    e = oa.OracleExtractor(**kw)
    k, d, m = e.extract(img, mask, cam)
    check_against_fixture(g, k, d, m)
    for l in range(kw.get("nlevels", 8)):
        # the reference leaves a level blurred iff it produced keypoints (src/mdBRIEFextractorOct.cpp:1293-1301)
        lvl = e.debug_read(l, 1) if int(g["per_level"][l]) else e.debug_read(l, 0)
        assert crc(lvl) == int(g["level_after_crc"][l]), f"pyramid level {l}"
        assert crc(e.debug_read(l, 2)) == int(g["mask_level_crc"][l]), f"mask level {l}"


@pytest.mark.parametrize("path", FIXTURES[::4], ids=lambda p: pathlib.Path(p).stem[12:])
def test_reference_library_reproduces_fixture(path):
    """the fixtures really are what oracle/_ref returns (guards against a stale or hand-edited fixture)"""
    ra = _ra()
    if not ra.available():
        pytest.skip("oracle/_ref/libmcs_ref.so is built only where the original project's sources are present")
    g, cam, kw, img, mask = load_case(path)
    check_against_fixture(g, *ra.RefExtractor(**kw).extract(img, mask, cam))


@pytest.mark.parametrize("seed", range(6))
def test_oracle_equals_reference_live(oa, gold, cams, seed):
    from multicol_slam_b200 import synth
    rng = np.random.default_rng(1000 + seed)
    cam = dict(cams[seed % 3])
    if seed == 4:
        cam = synth.scaled_cam(cam, 640, 400)
    kw = dict(nfeatures=int(rng.integers(150, 2500)), fast_threshold=int(rng.choice([5, 12, 20, 30])),
              nlevels=int(rng.integers(3, 9)), scale_factor=float(rng.choice([1.1, 1.2, 1.3, 1.5])),
              desc_size=int(rng.choice([16, 32, 64])))
    if kw["scale_factor"] == 1.5:
        # a level narrower than 2*22 px makes the reference itself throw (nCols == 0 -> NaN cell size -> vector::resize of a
        # negative count in DistributeOctTree, src/mdBRIEFextractorOct.cpp:886-889, 643-650): keep every level above that
        kw["nlevels"] = min(kw["nlevels"], 5)
    kw.update([dict(), dict(do_dbrief=True), dict(do_dbrief=True, learn_masks=True)][seed % 3])
    img = synth.frame(cam, 500 + seed)
    if seed == 5:                                         # low-texture image: levels with fewer corners than their quota
        img = (img // 64 * 64).astype(np.uint8)
    mask = synth.mirror_mask(cam)
    rn, rk, rd, rm = gold(f"extract/{seed}", lambda: ref_extract_digest(kw, img, mask, cam))
    ok, od, om = oa.OracleExtractor(**kw).extract(img, mask, cam)
    assert len(ok) == rn and crc(ok) == rk
    assert crc(od) == rd and crc(om) == rm


def test_constructor_tables_equal_reference(oa, gold):
    import ctypes as C
    for nf, sf, L in [(400, 1.2, 8), (1000, 1.2, 8), (2000, 1.2, 8), (4000, 1.2, 8), (777, 1.37, 6), (50, 2.0, 3)]:
        q, s, i, um = gold(f"tables/{nf}/{sf}/{L}", lambda: _ra().RefExtractor(nfeatures=nf, scale_factor=sf, nlevels=L).tables())
        e = oa.OracleExtractor(nfeatures=nf, scale_factor=sf, nlevels=L)
        assert list(e.info.features_per_level[:L]) == q.tolist()
        assert np.array_equal(np.array(e.info.scale_factor[:L]), s) and np.array_equal(np.array(e.info.inv_scale_factor[:L]), i)
        oum = (C.c_int * 17)()
        oa.lib().mcso_extractor_umax(e.h, oum)
        assert list(oum) == um.tolist()


@pytest.mark.parametrize("seed", range(8))
def test_octree_equals_reference_with_ties(oa, gold, seed):
    """DistributeOctTree alone (ref :631-861) on corner lists built to provoke equal node sizes (the pointer tie-break, :782)
    and equal responses (first maximum wins, :848-855)."""
    rng = np.random.default_rng(seed)
    W, H = [(710, 436), (584, 356), (166, 90), (1236, 676)][seed % 4]
    n = int(rng.integers(50, 6000))
    if seed % 2:                                          # lattice points: many nodes with identical counts
        xs = (rng.integers(0, W // 8, n) * 8 + rng.integers(0, 2, n)).astype(np.float32)
        ys = (rng.integers(0, H // 8, n) * 8 + rng.integers(0, 2, n)).astype(np.float32)
    else:
        xs, ys = rng.integers(0, W, n).astype(np.float32), rng.integers(0, H, n).astype(np.float32)
    xyr = np.stack([xs, ys, rng.integers(20, 40 if seed % 2 else 255, n).astype(np.float32)], 1)
    xyr = xyr[np.lexsort((xyr[:, 0], xyr[:, 1]))]
    N = int(rng.integers(10, 1500))
    n, r = gold(f"octree/{seed}", lambda: rows_and_crc(_ra().RefExtractor(nfeatures=1000).octree(xyr, 22, 22 + W, 22, 22 + H, N)))
    o = oa.octree(xyr, 22, 22 + W, 22, 22 + H, N)
    assert len(o) == n and crc(np.asarray(o, np.float32)) == r


def test_camera_model_equals_reference(oa, gold, cams, api):
    """WorldToImg / ImgToWorld / undistortPointsOcam / CreateMirrorMask / isPointInMirrorMask of the reference
    (src/cam_model_omni.cpp) vs the oracle and vs the product's host helpers (same double arithmetic, bit for bit)."""
    ra = _ra()
    import ctypes as C
    from multicol_slam_b200 import synth
    from multicol_slam_b200.ctypes_defs import make_ocam
    rng = np.random.default_rng(3)
    for ci, cam in enumerate(list(cams) + [synth.scaled_cam(cams[1], 1920, 1080)]):
        oc = make_ocam(cam)
        ref_mask = gold(f"cam{ci}/mirror_mask_crc", lambda: crc(ra.mirror_mask(cam)))
        assert ref_mask == crc(synth.mirror_mask(cam)) == crc(api.mirror_mask(cam))
        Xs, pxy = [], []
        for _ in range(200):
            Xs.append(rng.normal(size=3) * [1.0, 1.0, 0.6])
            pxy.append((rng.uniform(0, cam["width"]), rng.uniform(0, cam["height"])))
        ref_uv = gold(f"cam{ci}/world_to_img", lambda: np.array([ra.world_to_img(cam, *X) for X in Xs + [(0.0, 0.0, 1.0)]]))
        ref_xyz = gold(f"cam{ci}/img_to_world", lambda: np.array([ra.img_to_world(cam, px, py) for px, py in pxy]))
        for X, (px, py), ruv, rxyz in zip(Xs, pxy, ref_uv, ref_xyz):
            u, v = C.c_double(), C.c_double()
            oa.lib().mcso_cam_world_to_img(C.byref(oc), C.c_double(X[0]), C.c_double(X[1]), C.c_double(X[2]), C.byref(u), C.byref(v))
            assert tuple(ruv) == (u.value, v.value) == api.world_to_img(cam, *X)
            x, y, z = C.c_double(), C.c_double(), C.c_double()
            oa.lib().mcso_cam_img_to_world(C.byref(oc), C.c_double(px), C.c_double(py), C.byref(x), C.byref(y), C.byref(z))
            assert tuple(rxyz) == (x.value, y.value, z.value) == api.img_to_world(cam, px, py)
        assert tuple(ref_uv[-1]) == api.world_to_img(cam, 0.0, 0.0, 1.0)          # norm == 0 branch (:150-151)
        uv = np.stack([rng.uniform(-5, cam["width"] + 5, 500), rng.uniform(-5, cam["height"] + 5, 500)], 1)
        m = synth.mirror_mask(cam)
        ur, vr = np.rint(uv[:, 0]).astype(int), np.rint(uv[:, 1]).astype(int)
        inside = (ur < cam["width"]) & (ur > 0) & (vr < cam["height"]) & (vr > 0)
        exp = np.zeros(500, np.uint8)
        exp[inside] = m[vr[inside], ur[inside]] > 0
        assert np.array_equal(gold(f"cam{ci}/points_in_mask", lambda: ra.points_in_mask(cam, uv)), exp)


def test_epipolar_check_equals_reference(oa, gold):
    """CheckDistEpipolarLine (src/misc.cpp:53-69) vs the oracle's restatement used by SearchForTriangulation"""
    ra = _ra()
    import ctypes as C
    rng = np.random.default_rng(9)
    lib = oa.lib()
    lib.mcso_check_epipolar.restype = C.c_int
    cases = []
    for i in range(2000):
        r1, r2 = rng.normal(size=3), rng.normal(size=3)
        r1 /= np.linalg.norm(r1)
        r2 /= np.linalg.norm(r2)
        E = rng.normal(size=(3, 3)) if i else np.zeros((3, 3))
        cases.append((r1, r2, E, float(rng.choice([1e-2, 1e-3, 0.1]))))
    ref = gold("check_epipolar", lambda: np.array([ra.check_epipolar(*c) for c in cases]))
    for (r1, r2, E, th), r in zip(cases, ref):
        mine = lib.mcso_check_epipolar(r1.ctypes.data_as(C.c_void_p), r2.ctypes.data_as(C.c_void_p), E.ctypes.data_as(C.c_void_p), C.c_double(th))
        assert bool(mine) == bool(r)


def test_reference_constants(gold):
    assert gold("const/0", lambda: _ra().lib().mcsref_const(0)) == 57.2957763671875                      # RHOf (include/misc.h:41)
    assert gold("const/1", lambda: _ra().lib().mcsref_const(1)) == 180.0 / 3.1415926535897932384626433832795


# ---- the stand-in OpenCV primitives underneath the reference build vs the real cv2 -------------------------------------------
def _cv2():
    return pytest.importorskip("cv2")


def test_stub_resize_and_border_vs_cv2(gold, cams):
    ra, cv2 = _ra(), _cv2()
    from multicol_slam_b200 import synth
    rng = np.random.default_rng(1)
    src = synth.frame(cams[0], 7)
    for (w, h) in [(628, 400), (524, 333), (436, 278), (364, 231), (303, 193), (253, 161), (210, 134)]:
        ref = cv2.resize(src, (w, h), interpolation=cv2.INTER_LINEAR)
        assert crc(ref) == gold(f"resize_chain/{w}x{h}/1", lambda: crc(ra.cv_resize(src, w, h, 1)))
        mk = (rng.integers(0, 2, size=src.shape) * 255).astype(np.uint8)
        assert crc(cv2.resize(mk, (w, h), interpolation=cv2.INTER_NEAREST)) == gold(f"resize_chain/{w}x{h}/0", lambda: crc(ra.cv_resize(mk, w, h, 0)))
        src = ref
    for (sw, sh, dw, dh) in [(101, 77, 84, 64), (1920, 1080, 1600, 900), (1280, 720, 1067, 600), (64, 64, 53, 53), (97, 31, 40, 13)]:
        s = rng.integers(0, 256, size=(sh, sw)).astype(np.uint8)
        assert crc(cv2.resize(s, (dw, dh), interpolation=cv2.INTER_LINEAR)) == gold(f"resize/{sw}x{sh}/1", lambda: crc(ra.cv_resize(s, dw, dh, 1)))
        assert crc(cv2.resize(s, (dw, dh), interpolation=cv2.INTER_NEAREST)) == gold(f"resize/{sw}x{sh}/0", lambda: crc(ra.cv_resize(s, dw, dh, 0)))
    s = rng.integers(0, 256, size=(40, 57)).astype(np.uint8)
    assert crc(cv2.copyMakeBorder(s, 25, 25, 25, 25, cv2.BORDER_REFLECT_101)) == gold("border/1", lambda: crc(ra.cv_make_border(s, 25, True)))
    assert crc(cv2.copyMakeBorder(s, 25, 25, 25, 25, cv2.BORDER_CONSTANT, value=0)) == gold("border/0", lambda: crc(ra.cv_make_border(s, 25, False)))


def test_stub_box_filter_vs_cv2(gold, cams):
    ra, cv2 = _ra(), _cv2()
    from multicol_slam_b200 import synth
    rng = np.random.default_rng(2)
    for i, s in enumerate([synth.frame(cams[1], 3), rng.integers(0, 256, size=(61, 87)).astype(np.uint8)]):
        # in place on the ROI of a REFLECT_101-bordered buffer, the reference's use (:1301)
        b = cv2.copyMakeBorder(s, 25, 25, 25, 25, cv2.BORDER_REFLECT_101)
        mine = gold(f"box5/{i}/roi", lambda: crc(ra.cv_box5_roi(b, 25, 25, s.shape[1], s.shape[0])))
        roi = b[25:-25, 25:-25]
        cv2.boxFilter(roi, -1, (5, 5), roi, (-1, -1), True, cv2.BORDER_REFLECT_101)
        assert crc(b) == mine
        # a ROI whose surroundings are NOT its reflection: the C++ API filters a sub-matrix with the parent's pixels
        # (FilterEngine::apply with wholeSize / ofs).  cv2's Python binding cannot express this -- a numpy view arrives as a
        # stand-alone Mat -- so the expectation is the plain 5x5 sum over the parent, (S + 12) / 25 (SURVEY Appendix A.3)
        big = rng.integers(0, 256, size=(s.shape[0] + 20, s.shape[1] + 20)).astype(np.uint8)
        mine = gold(f"box5/{i}/parent", lambda: crc(ra.cv_box5_roi(big, 3, 7, 40, 30)))
        S = sum(big[7 + dy:37 + dy, 3 + dx:43 + dx].astype(np.int64) for dy in range(-2, 3) for dx in range(-2, 3))
        exp = big.copy()
        exp[7:37, 3:43] = (S + 12) // 25
        assert crc(exp) == mine
        # whole image: border extrapolation
        whole = gold(f"box5/{i}/whole", lambda: crc(ra.cv_box5_roi(s, 0, 0, s.shape[1], s.shape[0])))
        assert crc(cv2.boxFilter(s, -1, (5, 5), None, (-1, -1), True, cv2.BORDER_REFLECT_101)) == whole


def test_stub_fast_and_atan2_vs_cv2(gold, cams):
    ra, cv2 = _ra(), _cv2()
    from multicol_slam_b200 import synth
    rng = np.random.default_rng(4)
    yx = [tuple(np.float32(v) for v in rng.normal(size=2) * rng.choice([1, 1e3, 1e6])) for _ in range(3000)]
    yx += [(0, 0), (0, -5), (1, 1), (3, -4), (-7, 2), (5, 0), (-5, 0)]
    ref = gold("fast_atan2", lambda: crc(np.array([ra.cv_fast_atan2(y, x) for y, x in yx], np.float32)))
    assert ref == crc(np.array([cv2.fastAtan2(float(y), float(x)) for y, x in yx], np.float32))
    img = synth.frame(cams[2], 5)
    mask = synth.mirror_mask(cams[2])
    for th in (5, 20, 40):
        fd = cv2.FastFeatureDetector_create(th, True, cv2.FAST_FEATURE_DETECTOR_TYPE_9_16)
        for _ in range(15):                               # reference-sized cells at random places, with their mask cells
            x0, y0 = int(rng.integers(0, 700)), int(rng.integers(0, 430))
            w, h = int(rng.integers(7, 40)), int(rng.integers(7, 40))
            cell, mcell = img[y0:y0 + h, x0:x0 + w], mask[y0:y0 + h, x0:x0 + w]
            kp = fd.detect(cell, mcell)
            exp = np.array([[k.pt[0], k.pt[1], k.response] for k in kp], np.float32).reshape(-1, 3)
            assert np.array_equal(gold(f"fast/{th}/{x0}/{y0}/{w}/{h}", lambda: ra.cv_fast(cell, mcell, th)), exp)
        kp = fd.detect(img, None)
        exp = np.array([[k.pt[0], k.pt[1], k.response] for k in kp], np.float32).reshape(-1, 3)
        assert crc(exp) == gold(f"fast/{th}/whole", lambda: crc(ra.cv_fast(img, None, th)))
    vs = list(rng.normal(size=500) * 100)
    rounded = gold("cv_round", lambda: np.array([ra.lib().mcsref_cv_round(float(v)) for v in vs]))
    for v, r in zip(vs, rounded):
        assert r == cv2.cvRound(float(v)) if hasattr(cv2, "cvRound") else True
    halves = (0.5, 1.5, 2.5, -0.5, -1.5, 3.5)
    assert np.array_equal(gold("cv_round/halves", lambda: np.array([ra.lib().mcsref_cv_round(v) for v in halves])), np.rint(halves))
