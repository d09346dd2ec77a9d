"""GPU parity against outputs of the REFERENCE'S OWN extractor: the CUDA path (through the C ABI) vs the fixtures
tests/golden/ref_extract_*.npz, which tests/golden/make_ref_extract_golden.py wrote from oracle/_ref/libmcs_ref.so
(the original project's src/mdBRIEFextractorOct.cpp, cam_model_omni.cpp, misc.cpp compiled in place).  Bit-exact: keypoint
bytes (incl. the IC angle float), descriptor and mask bytes, pyramid and mask-pyramid levels.  Covers the configuration the
reference ships (plain ORB, 400 features), its init extractor, BASELINE.json configs 1-4 and parameter corners."""
import glob
import json
import pathlib
import zlib

import numpy as np
import pytest

from ref_golden import RECORD, RefGolden, not_recording

pytestmark = pytest.mark.gpu
GOLD = pathlib.Path(__file__).resolve().parent / "golden"
FIXTURES = sorted(glob.glob(str(GOLD / "ref_extract_*.npz")))
KW = {"nfeatures": "nfeatures", "scale_factor": "scaleFactor", "nlevels": "nlevels", "fast_threshold": "fastThreshold",
      "do_dbrief": "do_dBrief", "learn_masks": "learnMasks", "desc_size": "descSize"}


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes())


@not_recording
@pytest.mark.parametrize("path", FIXTURES, ids=lambda p: pathlib.Path(p).stem[12:])
def test_gpu_equals_reference_fixture(api, path):
    from multicol_slam_b200 import synth
    g = np.load(path)
    cam = json.loads(bytes(g["cam_json"]).decode())
    kw = json.loads(bytes(g["params_json"]).decode())
    img = synth.frame(cam, int(g["seed"]))
    assert crc(img) == int(g["image_crc"]), "synthetic image generator changed"
    ex = api.mdBRIEFextractorOct(**{KW[k]: v for k, v in kw.items()})
    k, d, m = ex(img, api.mirror_mask(cam), cam)
    assert len(k) == int(g["n"])
    assert [int((k["octave"] == l).sum()) for l in range(ex.GetLevels())] == g["per_level"].tolist()
    if "kps" in g.files:
        for f in ("x", "y", "size", "response", "octave", "class_id"):
            assert np.array_equal(k[f], g["kps"][f]), f"keypoint field {f}"
        assert np.array_equal(k["angle"].view(np.uint32), g["kps"]["angle"].view(np.uint32)), "IC angle bits"
        assert np.array_equal(d, g["desc"]) and np.array_equal(m, g["dmask"])
    assert crc(k) == int(g["kps_crc"]), "keypoints"
    assert crc(d) == int(g["desc_crc"]), "descriptors"
    assert crc(m) == int(g["dmask_crc"]), "descriptor masks"
    for l in range(ex.GetLevels()):
        lvl = ex.debug_read(l, 1) if int(g["per_level"][l]) else ex.debug_read(l, 0)     # blurred iff the level has keypoints
        assert crc(lvl) == int(g["level_after_crc"][l]), f"pyramid level {l}"
        assert crc(ex.debug_read(l, 2)) == int(g["mask_level_crc"][l]), f"mask level {l}"


def test_gpu_equals_reference_live(api, cams):
    """the reference extractor on three more seeds and modes (tests/golden/ref_pin_gpu.npz, tests/ref_golden.py) next to the CUDA path"""
    import ref_mcs_api as ra
    from multicol_slam_b200 import synth
    gold = RefGolden("ref_pin_gpu")
    cases = []
    for seed, (mode, nf) in enumerate([(dict(), 400), (dict(do_dbrief=True), 900), (dict(do_dbrief=True, learn_masks=True), 2000)]):
        cam = cams[seed]
        img, mask = synth.frame(cam, 900 + seed), synth.mirror_mask(cam)
        ref = gold(f"extract/{seed}", lambda: tuple(crc(a) for a in ra.RefExtractor(nfeatures=nf, **mode).extract(img, mask, cam)))
        cases.append((mode, nf, cam, img, mask, ref))
    gold.save()
    if RECORD:
        pytest.skip("reference outputs recorded")
    for mode, nf, cam, img, mask, ref in cases:
        k, d, m = api.mdBRIEFextractorOct(nfeatures=nf, do_dBrief=mode.get("do_dbrief", False), learnMasks=mode.get("learn_masks", False))(img, mask, cam)
        assert (crc(k), crc(d), crc(m)) == ref
