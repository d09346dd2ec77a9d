"""ctypes binding of libmcs_b200.so (include/mcs_b200.h) plus thin Python mirrors of the reference's
operator/matcher interface for this path:

    mdBRIEFextractorOct(...)(image, mask, camModel) -> keypoints, descriptors, descriptorMasks
        (ref include/mdBRIEFextractorOct.h:333-368, src/mdBRIEFextractorOct.cpp:1244-1337)
    cORBmatcher(nnratio, checkOri, featDim, havingMasks).SearchByProjection / SearchForInitialization /
        SearchByBoW(KF1, KF2)   (ref include/cORBmatcher.h:58-158, src/cORBmatcher.cpp:46-166, 579-726, 885-966)
    ORBVocabulary(voc).transform / score and KeyFrameDatabase(voc).add / erase / clear / DetectLoopCandidates /
        DetectRelocalisationCandidates   (ref include/cMultiKeyFrameDatabase.h, src/cMultiKeyFrameDatabase.cpp)

There is no CPU fallback: the shared library must be present (build it with `python __graft_entry__.py`)
and every compute call needs an sm_100 device, otherwise it raises.
"""
import ctypes as C
import math
import os
import pathlib

import numpy as np

from .ctypes_defs import (ExtractorInfo, ExtractorParams, FrameView, KEYPOINT_DTYPE, MapPointView, Ocam,
                          WINDOW_QUERY_DTYPE, make_ocam, make_params)

_PKG = pathlib.Path(__file__).resolve().parent
# MCS_B200_LIB: load another build of the same C ABI (kernel-variant experiments under tools/); never a CPU library
_LIB_PATH = pathlib.Path(os.environ.get("MCS_B200_LIB", _PKG / "libmcs_b200.so"))
_lib = None

MCS_OK, MCS_ERR_INVALID, MCS_ERR_UNSUPPORTED, MCS_ERR_CUDA, MCS_ERR_CAPACITY, MCS_ERR_NO_DEVICE = 0, -1, -2, -3, -4, -5


class McsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libmcs_b200 error {code}: {msg}")
        self.code = code


def lib():
    """Load libmcs_b200.so; fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            raise ImportError(f"{_LIB_PATH} is missing: the CUDA extension is mandatory (run __graft_entry__.build())")
        _lib = C.CDLL(str(_LIB_PATH))
        _lib.mcs_last_error.restype = C.c_char_p
        _lib.mcs_slot_bytes.restype = C.c_size_t
    return _lib


def _check(rc):
    if rc != 0:
        raise McsError(rc, lib().mcs_last_error().decode())


def _p(a):
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)


def device_count():
    return lib().mcs_device_count()


def as_ocam(cam):
    return cam if isinstance(cam, Ocam) else make_ocam(cam)


def mirror_mask(cam):
    oc = as_ocam(cam)
    out = np.zeros((oc.height, oc.width), np.uint8)
    _check(lib().mcs_cam_mirror_mask(C.byref(oc), _p(out)))
    return out


def distort_table(cam):
    """mcs_cam_distort_table: the per-radius table of the descriptor kernel's tiers 1 and 2 for one camera -> float64 [n, row]"""
    oc = as_ocam(cam)
    n, row = C.c_int32(0), C.c_int32(0)
    _check(lib().mcs_cam_distort_table(C.byref(oc), None, 0, C.byref(n), C.byref(row)))
    out = np.zeros((n.value, row.value), np.float64)
    _check(lib().mcs_cam_distort_table(C.byref(oc), _p(out), n.value, C.byref(n), C.byref(row)))
    return out


def world_to_img(cam, x, y, z):
    oc = as_ocam(cam)
    u, v = C.c_double(), C.c_double()
    lib().mcs_cam_world_to_img(C.byref(oc), C.c_double(x), C.c_double(y), C.c_double(z), C.byref(u), C.byref(v))
    return u.value, v.value


def img_to_world(cam, u, v):
    oc = as_ocam(cam)
    x, y, z = C.c_double(), C.c_double(), C.c_double()
    lib().mcs_cam_img_to_world(C.byref(oc), C.c_double(u), C.c_double(v), C.byref(x), C.byref(y), C.byref(z))
    return x.value, y.value, z.value


class mdBRIEFextractorOct:
    """Same constructor arguments, order and defaults as the reference class."""
    HARRIS_SCORE, FAST_SCORE = 0, 1

    def __init__(self, nfeatures=1000, scaleFactor=1.2, nlevels=8, edgeThreshold=25, firstLevel=0, scoreType=0,
                 patchSize=32, fastThreshold=20, useAgast=False, fastAgastType=2, do_dBrief=False, learnMasks=False,
                 descSize=32):
        self.params = ExtractorParams(nfeatures, scaleFactor, nlevels, edgeThreshold, firstLevel, scoreType, patchSize,
                                      fastThreshold, int(useAgast), fastAgastType, int(do_dBrief), int(learnMasks), descSize)
        self._h = C.c_void_p()
        _check(lib().mcs_extractor_create(C.byref(self.params), C.byref(self._h)))
        self.info = ExtractorInfo()
        _check(lib().mcs_extractor_get_info(self._h, C.byref(self.info)))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().mcs_extractor_destroy(self._h)
            self._h = None

    # reference getters
    def GetLevels(self):
        return self.info.nlevels

    def GetScaleFactor(self):
        return float(np.float32(self.params.scale_factor))

    def GetMasksLearned(self):
        return bool(self.params.learn_masks)

    def GetDescriptorSize(self):
        return self.info.desc_size

    @property
    def capacity(self):
        return self.info.capacity

    def __call__(self, image, mask, camModel):
        """operator(): -> (keypoints structured array [n], descriptors [n,descSize] u8, descriptorMasks [n,descSize] u8).
        An empty image returns None (the reference returns without touching its outputs)."""
        if image is None or image.size == 0:
            return None
        image = np.ascontiguousarray(image, np.uint8)
        mask = np.ascontiguousarray(mask, np.uint8)
        cap, ds = self.info.capacity, self.info.desc_size
        kps = np.zeros(cap, KEYPOINT_DTYPE)
        desc = np.zeros((cap, ds), np.uint8)
        dmask = np.zeros((cap, ds), np.uint8)
        n = C.c_int32(0)
        oc = as_ocam(camModel)
        h, w = image.shape
        _check(lib().mcs_extract(self._h, _p(image), w, h, image.strides[0], _p(mask), mask.strides[0], C.byref(oc),
                                 _p(kps), _p(desc), _p(dmask), cap, C.byref(n)))
        return kps[:n.value].copy(), desc[:n.value].copy(), dmask[:n.value].copy()

    def extract_batch(self, images, masks, cams, cam_of_image):
        """images [B,H,W] u8 host; masks [n_cams,H,W]; cams list; -> (kps [B,cap], desc [B,cap,ds], dmask, counts [B])"""
        images = np.ascontiguousarray(images, np.uint8)
        masks = np.ascontiguousarray(masks, np.uint8)
        coi = np.ascontiguousarray(cam_of_image, np.int32)
        B, H, W = images.shape
        cap, ds = self.info.capacity, self.info.desc_size
        ocs = (Ocam * len(cams))(*[as_ocam(c) for c in cams])
        kps = np.zeros((B, cap), KEYPOINT_DTYPE)
        desc = np.zeros((B, cap, ds), np.uint8)
        dmask = np.zeros((B, cap, ds), np.uint8)
        counts = np.zeros(B, np.int32)
        _check(lib().mcs_extract_batch(self._h, B, _p(images), W, H, W, _p(masks), ocs, len(cams), _p(coi), _p(kps),
                                       _p(desc), _p(dmask), _p(counts), cap))
        return kps, desc, dmask, counts

    def extract_batch_device(self, images_t, masks, cams, cam_of_image, out=None, stream=None, width=None):
        """torch CUDA tensors in/out (plumbing only): images_t [B,H,P] uint8 cuda, P = row pitch >= width (a 16-byte
        aligned pitch lets K1 use 128-bit loads).  Returns dict of cuda tensors {kps [B,cap,7] int32-view,
        desc [B,cap,ds], dmask, counts [B]}; asynchronous on `stream` when given."""
        import torch
        assert images_t.is_cuda and images_t.dtype == torch.uint8 and images_t.is_contiguous()
        B, H, P = images_t.shape
        W = P if width is None else width
        cap, ds = self.info.capacity, self.info.desc_size
        dev = images_t.device
        if out is None:
            out = dict(kps=torch.empty((B, cap, 7), dtype=torch.int32, device=dev),
                       desc=torch.empty((B, cap, ds), dtype=torch.uint8, device=dev),
                       dmask=torch.empty((B, cap, ds), dtype=torch.uint8, device=dev),
                       counts=torch.empty((B,), dtype=torch.int32, device=dev))
        masks = np.ascontiguousarray(masks, np.uint8)
        coi = np.ascontiguousarray(cam_of_image, np.int32)
        ocs = (Ocam * len(cams))(*[as_ocam(c) for c in cams])
        st = C.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream(dev).cuda_stream)
        _check(lib().mcs_extract_batch_device(self._h, B, C.c_void_p(images_t.data_ptr()), W, H, P, _p(masks), ocs, len(cams),
                                              _p(coi), C.c_void_p(out["kps"].data_ptr()), C.c_void_p(out["desc"].data_ptr()),
                                              C.c_void_p(out["dmask"].data_ptr()), C.c_void_p(out["counts"].data_ptr()), cap, st))
        return out

    def packed_views(self, packed_t, n_images):
        """views of a packed feature buffer (mcs_packed_layout) as the four output tensors"""
        import torch
        from . import rig
        cap, ds = self.info.capacity, self.info.desc_size
        offs, total = rig.packed_layout(n_images, cap, ds)
        assert packed_t.numel() >= total
        return dict(counts=packed_t[offs[0]:offs[0] + 4 * n_images].view(torch.int32),
                    kps=packed_t[offs[1]:offs[1] + n_images * cap * 28].view(torch.int32).view(n_images, cap, 7),
                    desc=packed_t[offs[2]:offs[2] + n_images * cap * ds].view(n_images, cap, ds),
                    dmask=packed_t[offs[3]:offs[3] + n_images * cap * ds].view(n_images, cap, ds))

    def extract_batch_packed_device(self, images_t, masks, cams, cam_of_image, packed_t, stream=None, width=None):
        """mcs_extract_batch_packed_device: K3 writes counts | keypoints | descriptors | masks straight into packed_t (uint8
        cuda tensor of rig.packed_layout(B, capacity, descSize)[1] bytes) -- the buffer mcs_allgather_features exchanges."""
        import torch
        B, H, P = images_t.shape
        W = P if width is None else width
        masks = np.ascontiguousarray(masks, np.uint8)
        coi = np.ascontiguousarray(cam_of_image, np.int32)
        ocs = (Ocam * len(cams))(*[as_ocam(c) for c in cams])
        st = C.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream(images_t.device).cuda_stream)
        _check(lib().mcs_extract_batch_packed_device(self._h, B, C.c_void_p(images_t.data_ptr()), W, H, P, _p(masks), ocs, len(cams),
                                                     _p(coi), C.c_void_p(packed_t.data_ptr()), self.info.capacity, st))
        return self.packed_views(packed_t, B)

    def extract_match_stream(self, images, masks, cams, K=2, out=None, packed_t=None, greedy=None):
        """images [F,C,H,W] u8 host (frame-major).  Extract every image and brute-force match each (frame,cam)
        against (frame-1,cam).  Returns dict(kps [F*C,cap], desc, dmask, counts, match_idx [F*C,cap,K], match_dist).
        `out` may hold preallocated (e.g. pinned) numpy arrays with the same keys."""
        images = np.ascontiguousarray(images, np.uint8)
        masks = np.ascontiguousarray(masks, np.uint8)
        F, Cn, H, W = images.shape
        cap, ds, B = self.info.capacity, self.info.desc_size, F * Cn
        ocs = (Ocam * len(cams))(*[as_ocam(c) for c in cams])
        if out is None:
            out = dict(kps=np.zeros((B, cap), KEYPOINT_DTYPE), desc=np.zeros((B, cap, ds), np.uint8),
                       dmask=np.zeros((B, cap, ds), np.uint8), counts=np.zeros(B, np.int32),
                       match_idx=np.zeros((B, cap, K), np.int32), match_dist=np.zeros((B, cap, K), np.int32))
        if packed_t is not None or greedy is not None:
            # packed_t: features also stay in the caller's packed exchange buffer on the GPU; greedy = (th_low, nnratio): the greedy
            # acceptance of SearchByBoW(KF1, KF2) on the device -> out["matches12"] [B,cap], out["nmatches"] [B], out["redo"] [B]
            th, ratio = greedy if greedy is not None else (0, 0.0)
            if greedy is not None:
                for k, shp in (("matches12", (B, cap)), ("nmatches", (B,)), ("redo", (B,))):
                    if k not in out:
                        out[k] = np.zeros(shp, np.int32)
            _check(lib().mcs_extract_match_stream_packed(self._h, F, Cn, _p(images), W, H, W, _p(masks), ocs, _p(out["kps"]),
                                                         _p(out["desc"]), _p(out["dmask"]), _p(out["counts"]), cap, K,
                                                         _p(out["match_idx"]), _p(out["match_dist"]),
                                                         C.c_void_p(packed_t.data_ptr()) if packed_t is not None else None, int(th),
                                                         C.c_double(ratio), _p(out.get("matches12")) if greedy is not None else None,
                                                         _p(out.get("nmatches")) if greedy is not None else None,
                                                         _p(out.get("redo")) if greedy is not None else None))
            return out
        _check(lib().mcs_extract_match_stream(self._h, F, Cn, _p(images), W, H, W, _p(masks), ocs, _p(out["kps"]),
                                              _p(out["desc"]), _p(out["dmask"]), _p(out["counts"]), cap, K,
                                              _p(out["match_idx"]), _p(out["match_dist"])))
        return out

    def set_profiling(self, enable=True):
        _check(lib().mcs_extractor_set_profiling(self._h, int(enable)))

    def tier_stats(self, enable=True):
        """K3 diagnostics: (tier 1, tier 1 repaired, tier 2, tier 3) pattern counts since counting was switched on; enable/disable counting"""
        out = np.zeros(4, np.int64)
        _check(lib().mcs_extractor_tier_stats(self._h, int(enable), _p(out)))
        return out

    def check_status(self, stream=None):
        """mcs_extractor_check_status: overflow report of the last asynchronous extract call (raises MCS_ERR_CAPACITY); synchronises the stream"""
        st = C.c_void_p(stream.cuda_stream) if stream is not None else None
        _check(lib().mcs_extractor_check_status(self._h, st))

    def graph_replays(self):
        """calls served by replaying the cached CUDA graph of the per-frame sequence (mcs_extractor_graph_replays)"""
        n = C.c_int64(0)
        _check(lib().mcs_extractor_graph_replays(self._h, C.byref(n)))
        return n.value

    def get_timings(self):
        """(K1 pyramid+blur+FAST all levels, K2 octree, K3 describe) of the last extract call, milliseconds."""
        ms = (C.c_float * 3)()
        _check(lib().mcs_extractor_get_timings(self._h, ms))
        return tuple(ms)

    def debug_read(self, level, what, image_index=0):
        w, h = C.c_int32(0), C.c_int32(0)
        buf = np.zeros(1 << 24, np.uint8)
        _check(lib().mcs_extractor_debug_read(self._h, image_index, level, what, _p(buf), C.c_size_t(buf.nbytes), C.byref(w), C.byref(h)))
        if what == 3:
            return buf[:w.value * 12].view(np.int32).reshape(-1, 3).copy()
        return buf[:w.value * h.value].reshape(h.value, w.value).copy()


# ---- matcher --------------------------------------------------------------------------------------
def DescriptorDistance64(a, b, dim=32):
    a = np.ascontiguousarray(a, np.uint8)
    b = np.ascontiguousarray(b, np.uint8)
    return lib().mcs_descriptor_distance64(_p(a), _p(b), dim)


def DescriptorDistance64Masked(a, b, ma, mb, dim=32):
    a, b, ma, mb = (np.ascontiguousarray(v, np.uint8) for v in (a, b, ma, mb))
    return lib().mcs_descriptor_distance64_masked(_p(a), _p(b), _p(ma), _p(mb), dim)


def hamming_topk(q, d, K=2, qmask=None, dmask=None, db_skip=None):
    q = np.ascontiguousarray(q, np.uint8)
    d = np.ascontiguousarray(d, np.uint8)
    qmask = None if qmask is None else np.ascontiguousarray(qmask, np.uint8)
    dmask = None if dmask is None else np.ascontiguousarray(dmask, np.uint8)
    db_skip = None if db_skip is None else np.ascontiguousarray(db_skip, np.uint8)
    nq, dim = q.shape
    idx = np.zeros((nq, K), np.int32)
    dist = np.zeros((nq, K), np.int32)
    _check(lib().mcs_hamming_topk(_p(q), _p(qmask), nq, _p(d), _p(dmask), d.shape[0], _p(db_skip), dim, K, _p(idx), _p(dist)))
    return idx, dist


def hamming_topk_device(q_t, d_t, K=2, qmask_t=None, dmask_t=None, skip_t=None, out=None, stream=None):
    """torch CUDA uint8 tensors [nq,dim] / [nd,dim] -> (idx [nq,K] int32, dist [nq,K] int32) cuda tensors."""
    import torch
    nq, dim = q_t.shape
    dev = q_t.device
    if out is None:
        out = (torch.empty((nq, K), dtype=torch.int32, device=dev), torch.empty((nq, K), dtype=torch.int32, device=dev))
    ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    st = C.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream(dev).cuda_stream)
    _check(lib().mcs_hamming_topk_device(ptr(q_t), ptr(qmask_t), nq, ptr(d_t), ptr(dmask_t), d_t.shape[0], ptr(skip_t), dim, K,
                                         ptr(out[0]), ptr(out[1]), st))
    return out


def match_stream_device(desc_t, dmask_t, counts_t, n_frames, n_cams, K=2, out=None, stream=None):
    """torch CUDA tensors: desc [F*C,cap,dim] u8, dmask same or None, counts [F*C] i32 -> (idx, dist) [F*C,cap,K] i32."""
    import torch
    B, cap, dim = desc_t.shape
    dev = desc_t.device
    if out is None:
        out = (torch.empty((B, cap, K), dtype=torch.int32, device=dev), torch.empty((B, cap, K), dtype=torch.int32, device=dev))
    ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    st = C.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream(dev).cuda_stream)
    _check(lib().mcs_match_stream_device(ptr(desc_t), ptr(dmask_t), ptr(counts_t), n_frames, n_cams, cap, dim, K, ptr(out[0]),
                                         ptr(out[1]), st))
    return out


def match_stream_replay_device(idx_t, dist_t, counts_t, desc_t, dmask_t, n_frames, n_cams, th_low, nnratio, out=None, stream=None):
    """mcs_match_stream_replay_device: greedy SearchByBoW acceptance over the K-best lists, on the device.
    -> (matches12 [F*C,cap] i32, nmatches [F*C] i32, redo [F*C] i32) cuda tensors"""
    import torch
    B, cap, K = idx_t.shape
    dev = idx_t.device
    if out is None:
        out = (torch.empty((B, cap), dtype=torch.int32, device=dev), torch.empty(B, dtype=torch.int32, device=dev),
               torch.empty(B, dtype=torch.int32, device=dev))
    ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    st = C.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream(dev).cuda_stream)
    _check(lib().mcs_match_stream_replay_device(ptr(idx_t), ptr(dist_t), ptr(counts_t), ptr(desc_t), ptr(dmask_t), n_frames, n_cams, cap,
                                                desc_t.shape[-1], K, int(th_low), C.c_double(nnratio), ptr(out[0]), ptr(out[1]), ptr(out[2]), st))
    return out


def match_bruteforce_batch_device(q_t, qmask_t, valid1, seg_start, d_t, dmask_t, valid2, th_low, nnratio, stream=None):
    """mcs_match_bruteforce_batch_device: the query sets q_t[seg_start[s]:seg_start[s+1]] each matched against the database as a separate
    SearchByBoW(KF1, KF2) would, K-best lists of all sets from one launch.  Returns (nmatches [n_seg] numpy, matches12 numpy)."""
    import torch
    nq, dim = q_t.shape
    nd = d_t.shape[0]
    seg = np.ascontiguousarray(seg_start, np.int32)
    assert seg[-1] == nq
    v1 = None if valid1 is None else np.ascontiguousarray(valid1, np.uint8)
    v2 = None if valid2 is None else np.ascontiguousarray(valid2, np.uint8)
    m12 = np.zeros(nq, np.int32)
    nm = np.zeros(len(seg) - 1, np.int32)
    ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    st = C.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream(q_t.device).cuda_stream)
    _check(lib().mcs_match_bruteforce_batch_device(ptr(q_t), ptr(qmask_t), _p(v1), _p(seg), len(seg) - 1, ptr(d_t), ptr(dmask_t), _p(v2), nd, dim,
                                                   int(th_low), C.c_double(nnratio), _p(m12), _p(nm), st))
    return nm, m12


def match_stream_greedy_device(desc_t, dmask_t, counts_t, n_frames, n_cams, th_low, nnratio, out=None, stream=None):
    """mcs_match_stream_greedy_device: every image against the same camera's image one frame earlier with SearchByBoW(KF1, KF2)'s
    acceptance rule, lists + replay in one call.  desc_t/dmask_t [F*C,cap,dim] u8 cuda, counts_t [F*C] i32 cuda.
    -> (matches12 [F*C,cap] i32, nmatches [F*C] i32) cuda tensors"""
    import torch
    B, cap, dim = desc_t.shape
    dev = desc_t.device
    if out is None:
        out = (torch.empty((B, cap), dtype=torch.int32, device=dev), torch.empty(B, dtype=torch.int32, device=dev))
    ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    st = C.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream(dev).cuda_stream)
    _check(lib().mcs_match_stream_greedy_device(ptr(desc_t), ptr(dmask_t), ptr(counts_t), n_frames, n_cams, cap, dim, int(th_low),
                                                C.c_double(nnratio), ptr(out[0]), ptr(out[1]), st))
    return out


def match_bruteforce_device(q_t, qmask_t, valid1, d_t, dmask_t, valid2, th_low, nnratio, stream=None):
    """mcs_match_bruteforce_device: SearchByBoW(KF1, KF2) with descriptors resident on the GPU (torch uint8 [n, dim]);
    valid1 / valid2 host uint8 arrays or None.  Returns (nmatches, matches12 numpy)."""
    import torch
    nq, dim = q_t.shape
    nd = d_t.shape[0]
    v1 = None if valid1 is None else np.ascontiguousarray(valid1, np.uint8)
    v2 = None if valid2 is None else np.ascontiguousarray(valid2, np.uint8)
    m12 = np.zeros(nq, np.int32)
    n = C.c_int32(0)
    ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    st = C.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream(q_t.device).cuda_stream)
    _check(lib().mcs_match_bruteforce_device(ptr(q_t), ptr(qmask_t), _p(v1), nq, ptr(d_t), ptr(dmask_t), _p(v2), nd, dim, int(th_low),
                                             C.c_double(nnratio), _p(m12), C.byref(n), st))
    return n.value, m12


class Frame:
    """Flat stand-in for the fields of cMultiFrame / cMultiKeyFrame the matchers read
    (ref include/cMultiFrame.h:90-175): contiguous keypoints in camera-major order."""

    def __init__(self, keys, key_cam, desc, dmask, cam_sizes, scale_factors):
        self.keys = np.ascontiguousarray(keys, KEYPOINT_DTYPE)
        self.key_cam = np.ascontiguousarray(key_cam, np.int32)
        self.desc = np.ascontiguousarray(desc, np.uint8)
        self.dmask = None if dmask is None else np.ascontiguousarray(dmask, np.uint8)
        self.cam_w = np.ascontiguousarray([s[0] for s in cam_sizes], np.int32)
        self.cam_h = np.ascontiguousarray([s[1] for s in cam_sizes], np.int32)
        self.scale_factors = np.ascontiguousarray(scale_factors, np.float64)

    @staticmethod
    def from_cameras(per_cam, cam_sizes, scale_factors):
        """per_cam: list of (kps, desc, dmask) as returned by the extractor, in camera order (ref :168-184)."""
        keys = np.concatenate([p[0] for p in per_cam])
        key_cam = np.concatenate([np.full(len(p[0]), c, np.int32) for c, p in enumerate(per_cam)])
        desc = np.concatenate([p[1] for p in per_cam])
        dmask = np.concatenate([p[2] for p in per_cam]) if per_cam[0][2] is not None else None
        return Frame(keys, key_cam, desc, dmask, cam_sizes, scale_factors)

    def view(self):
        v = FrameView()
        v.n_cams, v.n_keys = len(self.cam_w), len(self.keys)
        v.keys, v.key_cam, v.desc = _p(self.keys).value, _p(self.key_cam).value, _p(self.desc).value
        v.dmask = _p(self.dmask).value if self.dmask is not None else None
        v.cam_width, v.cam_height = _p(self.cam_w).value, _p(self.cam_h).value
        v.dim, v.n_levels = self.desc.shape[1], len(self.scale_factors)
        v.scale_factors = _p(self.scale_factors).value
        return v


class MapPoints:
    """Parallel arrays of the cMapPoint tracking fields (ref include/cMapPoint.h: mbTrackInView, mnTrackScaleLevel,
    mTrackProjX/Y, mTrackViewCos; GetDescriptorPtr / GetDescriptorMaskPtr)."""

    def __init__(self, bad, in_view, level, proj_x, proj_y, view_cos, desc, dmask=None):
        self.bad = np.ascontiguousarray(bad, np.uint8)
        self.in_view = np.ascontiguousarray(in_view, np.uint8)
        self.level = np.ascontiguousarray(level, np.int32)
        self.proj_x = np.ascontiguousarray(proj_x, np.float64)
        self.proj_y = np.ascontiguousarray(proj_y, np.float64)
        self.view_cos = np.ascontiguousarray(view_cos, np.float64)
        self.desc = np.ascontiguousarray(desc, np.uint8)
        self.dmask = None if dmask is None else np.ascontiguousarray(dmask, np.uint8)

    def view(self):
        v = MapPointView()
        v.n_points = len(self.bad)
        v.bad, v.in_view, v.level = _p(self.bad).value, _p(self.in_view).value, _p(self.level).value
        v.proj_x, v.proj_y, v.view_cos = _p(self.proj_x).value, _p(self.proj_y).value, _p(self.view_cos).value
        v.desc = _p(self.desc).value
        v.dmask = _p(self.dmask).value if self.dmask is not None else None
        return v


def window_search(frame, queries, qdesc, qmask=None, max_cand=64):
    queries = np.ascontiguousarray(queries, WINDOW_QUERY_DTYPE)
    qdesc = np.ascontiguousarray(qdesc, np.uint8)
    qmask = None if qmask is None else np.ascontiguousarray(qmask, np.uint8)
    nq = len(queries)
    idx = np.zeros((nq, max_cand), np.int32)
    dist = np.zeros((nq, max_cand), np.int32)
    cnt = np.zeros(nq, np.int32)
    fv = frame.view()
    rc = lib().mcs_window_search(C.byref(fv), _p(queries), nq, _p(qdesc), _p(qmask), max_cand, _p(idx), _p(dist), _p(cnt))
    if rc not in (MCS_OK, MCS_ERR_CAPACITY):
        _check(rc)
    return idx, dist, cnt, rc


def frame_prepare(keys, key_cam, cams):
    """GPU epilogue of the cMultiFrame constructor (ref src/cMultiFrame.cpp:143-184): bearing rays [n,3] and the 64x48 grid as
    CSR (cell_start [n_cams*64*48+1], cell_items [n_in_grid])."""
    keys = np.ascontiguousarray(keys, KEYPOINT_DTYPE)
    key_cam = np.ascontiguousarray(key_cam, np.int32)
    nc, n = len(cams), len(keys)
    ocs = (Ocam * nc)(*[as_ocam(c) for c in cams])
    rays = np.zeros((n, 3))
    start = np.zeros(nc * 64 * 48 + 1, np.int32)
    items = np.zeros(max(n, 1), np.int32)
    ning = C.c_int32(0)
    _check(lib().mcs_frame_prepare(_p(keys), _p(key_cam), n, ocs, nc, _p(rays), _p(start), _p(items), C.byref(ning)))
    return rays, start, items[:ning.value].copy()


def project_mappoints(mtmc_inv, mtmc, cams, masks, world_pos, normal, min_dist, max_dist, scale_factors):
    """Batched cMultiFrame::isInFrustum (ref src/cMultiFrame.cpp:218-270): mtmc_inv / mtmc [n_cams,4,4], masks [n_cams,H,W],
    world_pos / normal [n,3].  Returns (in_view [n,n_cams] u8, level i32, proj_x, proj_y, view_cos f64) -- the MapPoints fields."""
    mi = np.ascontiguousarray(mtmc_inv, np.float64)
    mm = np.ascontiguousarray(mtmc, np.float64)
    masks = np.ascontiguousarray(masks, np.uint8)
    pos = np.ascontiguousarray(world_pos, np.float64)
    nrm = np.ascontiguousarray(normal, np.float64)
    dmin = np.ascontiguousarray(min_dist, np.float64)
    dmax = np.ascontiguousarray(max_dist, np.float64)
    sf = np.ascontiguousarray(scale_factors, np.float64)
    nc, n = len(cams), len(pos)
    ocs = (Ocam * nc)(*[as_ocam(c) for c in cams])
    in_view = np.zeros((n, nc), np.uint8)
    level = np.zeros((n, nc), np.int32)
    px, py, vc = np.zeros((n, nc)), np.zeros((n, nc)), np.zeros((n, nc))
    _check(lib().mcs_project_mappoints(nc, _p(mi), _p(mm), ocs, _p(masks), n, _p(pos), _p(nrm), _p(dmin), _p(dmax), _p(sf), len(sf),
                                       _p(in_view), _p(level), _p(px), _p(py), _p(vc)))
    return in_view, level, px, py, vc


RULE_RATIO, RULE_BEST, RULE_LEVEL_RATIO, RULE_BEST_FREE, RULE_FIRST_FREE, RULE_SCW = 0, 1, 2, 3, 4, 5


def search_windows(frame, queries, qdesc, qmask, query_tag, rule, nnratio, threshold, assigned):
    """mcs_search_windows: generic projection-window search + greedy acceptance (see include/mcs_b200.h)."""
    queries = np.ascontiguousarray(queries, WINDOW_QUERY_DTYPE)
    qdesc = np.ascontiguousarray(qdesc, np.uint8)
    qmask = None if qmask is None else np.ascontiguousarray(qmask, np.uint8)
    tags = np.ascontiguousarray(query_tag, np.int32)
    assigned = np.ascontiguousarray(assigned, np.int32)
    n = C.c_int32(0)
    fv = frame.view()
    if qmask is None:
        fv.dmask = None
    _check(lib().mcs_search_windows(C.byref(fv), _p(queries), len(queries), _p(qdesc), _p(qmask), _p(tags), rule,
                                    C.c_double(nnratio), threshold, _p(assigned), C.byref(n)))
    return n.value, assigned


def _queries(cam, x, y, r, min_level, max_level, desc_index):
    q = np.zeros(len(cam), WINDOW_QUERY_DTYPE)
    q["cam"], q["x"], q["y"], q["r"] = cam, x, y, r
    q["min_level"], q["max_level"], q["desc_index"] = min_level, max_level, desc_index
    return q


def _mm(A, B):
    """cv::Matx product: s = 0; s += a(i,k) * b(k,j) in index order, plain doubles (no FMA, no BLAS reordering)"""
    A, B = np.asarray(A, np.float64), np.asarray(B, np.float64)
    B2 = B.reshape(B.shape[0], -1)
    out = np.zeros((A.shape[0], B2.shape[1]))
    for i in range(A.shape[0]):
        for j in range(B2.shape[1]):
            acc = 0.0
            for k in range(A.shape[1]):
                acc += float(A[i, k]) * float(B2[k, j])
            out[i, j] = acc
    return out.reshape((A.shape[0],) + B.shape[1:])


def inv_rigid(M):
    """cConverter::invMat (ref src/cConverter.cpp:31-44): [R^T | -R^T t]"""
    M = np.asarray(M, np.float64)
    Rt = M[:3, :3].T.copy()
    t = _mm(-Rt, M[:3, 3])
    out = np.eye(4)
    out[:3, :3], out[:3, 3] = Rt, t
    return out


class Rig:
    """cMultiCamSys_ as the matchers use it (ref include/cam_system_omni.h:53-206): MCS pose M_t, camera offsets M_c[c], interior
    orientations; MtMc = M_t * M_c[c] and its rigid inverse kept like the reference does (flagMcMt)."""

    def __init__(self, cams, M_c=None, M_t=None):
        self.cams = list(cams)
        n = len(self.cams)
        self.M_c = np.ascontiguousarray(np.tile(np.eye(4), (n, 1, 1)) if M_c is None else M_c, np.float64)
        self.masks = [mirror_mask(c) for c in self.cams]
        self.set_pose(np.eye(4) if M_t is None else M_t)

    def set_pose(self, M_t):
        self.M_t = np.ascontiguousarray(M_t, np.float64)
        self.MtMc = np.stack([_mm(self.M_t, self.M_c[c]) for c in range(len(self.cams))])
        self.MtMc_inv = np.stack([inv_rigid(m) for m in self.MtMc])

    def world_to_cam(self, c, p3):
        """WorldToCamHom_fast (ref src/cam_system_omni.cpp:92-133) -> (u, v, camera-frame point)"""
        pc = _mm(self.MtMc_inv[c], np.array([p3[0], p3[1], p3[2], 1.0]))
        u, v = world_to_img(self.cams[c], float(pc[0]), float(pc[1]), float(pc[2]))
        return u, v, pc

    def in_mirror_mask(self, c, u, v):
        """isPointInMirrorMask(u, v, 0) (ref src/cam_model_omni.cpp:163-178)"""
        if not (np.isfinite(u) and np.isfinite(v)):
            return False
        ur, vr = int(np.rint(u)), int(np.rint(v))
        m = self.masks[c]
        if ur >= m.shape[1] or ur <= 0 or vr >= m.shape[0] or vr <= 0:
            return False
        return bool(m[vr, ur] > 0)


def compute_E_rel(Trel):
    """inline ComputeE(const cv::Matx44d& Trel) (ref include/misc.h:232-241): [t/|t|]_x * R"""
    Trel = np.asarray(Trel, np.float64)
    R = Trel[:3, :3]
    t = Trel[:3, 3].copy()
    n = float(np.sqrt(t[0] * t[0] + t[1] * t[1] + t[2] * t[2]))
    t = t / n
    tx = np.array([[0.0, -t[2], t[1]], [t[2], 0.0, -t[0]], [-t[1], t[0], 0.0]])
    return _mm(tx, R)


def check_epipolar(ray1, ray2, E, thresh):
    """CheckDistEpipolarLine (ref src/misc.cpp:53-69), cv::Matx accumulation order"""
    r1, r2, E = (np.asarray(a, np.float64) for a in (ray1, ray2, E))
    nom = float(_mm(_mm(r2.reshape(1, 3), E), r1.reshape(3, 1))[0, 0])
    ex1 = _mm(E, r1.reshape(3, 1)).ravel()
    etx2 = _mm(E.T.copy(), r2.reshape(3, 1)).ravel()
    den = float(ex1[0] * ex1[0] + ex1[1] * ex1[1] + ex1[2] * ex1[2] + etx2[0] * etx2[0] + etx2[1] * etx2[1] + etx2[2] * etx2[2])
    if den == 0.0:
        return False
    return (nom * nom) / den < thresh


def _predict_level(scale_factors, ratio):
    """lower_bound over the scale factors, clamped to the last level (ref src/cORBmatcher.cpp:1313-1317)"""
    return min(int(np.searchsorted(scale_factors, ratio, side="left")), len(scale_factors) - 1)


class cORBmatcher:
    """ref include/cORBmatcher.h:55-178; thresholds as in src/cORBmatcher.cpp:46-64."""

    def __init__(self, nnratio=0.6, checkOri=True, featDim=32, havingMasks=False):
        self.mfNNratio, self.mbCheckOrientation, self.mbFeatDim, self.havingMasks = nnratio, checkOri, featDim, havingMasks
        if havingMasks:
            self.TH_HIGH_, self.TH_LOW_ = int(math.floor(1.5 * featDim)), int(math.floor(featDim))
        else:
            self.TH_HIGH_, self.TH_LOW_ = 3 * featDim, 2 * featDim

    def SearchByProjection(self, F, mapPoints, th, frame_mp=None):
        """SearchByProjection(cMultiFrame&, vector<cMapPoint*>&, th) (ref :67-166).
        frame_mp: F.mvpMapPoints as int32 indices (-1 = none), updated in place.  Returns (nmatches, frame_mp)."""
        if frame_mp is None:
            frame_mp = np.full(len(F.keys), -1, np.int32)
        frame_mp = np.ascontiguousarray(frame_mp, np.int32)
        n = C.c_int32(0)
        fv, mv = F.view(), mapPoints.view()
        _check(lib().mcs_search_by_projection(C.byref(fv), C.byref(mv), C.c_double(th), C.c_double(self.mfNNratio), self.TH_HIGH_,
                                              int(self.havingMasks), _p(frame_mp), C.byref(n)))
        return n.value, frame_mp

    def SearchForInitialization(self, F1, F2, vbPrevMatched, windowSize=10):
        """ref :579-726.  vbPrevMatched [n1,2] float64 updated in place.  Returns (nmatches, vnMatches12)."""
        prev = np.ascontiguousarray(vbPrevMatched, np.float64)
        m12 = np.zeros(len(F1.keys), np.int32)
        n = C.c_int32(0)
        f1, f2 = F1.view(), F2.view()
        _check(lib().mcs_search_for_initialization(C.byref(f1), C.byref(f2), _p(prev), windowSize, C.c_double(self.mfNNratio),
                                                   self.TH_LOW_, int(self.havingMasks), _p(m12), C.byref(n)))
        if prev is not vbPrevMatched:
            vbPrevMatched[...] = prev
        return n.value, m12

    def WindowSearch(self, F1, F2, windowSize, valid1, minScaleLevel=0, maxScaleLevel=2**31 - 1, _sw=None):
        """WindowSearch(F1, F2, windowSize, vpMapPointMatches2, minScaleLevel, maxScaleLevel) (ref :326-474).
        valid1[i1]: F1 keypoint i1 carries a non-bad map point.  Returns (nmatches, vnMatches21: F1 index per F2 keypoint)."""
        lv = F1.keys["octave"]
        sel = np.flatnonzero((np.asarray(valid1) != 0) & ((minScaleLevel <= 0) | (lv >= minScaleLevel)) &
                             ((maxScaleLevel >= 2**31 - 1) | (lv <= maxScaleLevel)))
        q = _queries(F1.key_cam[sel], F1.keys["x"][sel].astype(np.float64), F1.keys["y"][sel].astype(np.float64),
                     float(windowSize), -1, -1, sel)
        return (search_windows if _sw is None else _sw)(F2, q, F1.desc, F1.dmask if self.havingMasks else None, sel, RULE_RATIO,
                                                        self.mfNNratio, self.TH_HIGH_, np.full(len(F2.keys), -1, np.int32))

    def SearchByProjectionFrames(self, F1, F2, windowSize, valid1, uv, in_mask, assigned2=None):
        """SearchByProjection(F1, F2, windowSize, vpMapPointMatches2) (ref :476-573).  valid1[i1]: keypoint i1 of F1 carries a
        map point that is not bad, not already found in F2 and not seen before in F1 (the caller's bookkeeping, :490-499);
        uv[i1, c] = projection of that map point into camera c of F2 (WorldToCamHom_fast), in_mask[i1, c] = isPointInMirrorMask.
        assigned2 = F2.mvpMapPoints as indices (-1 = NULL).  Returns (nmatches, assigned2 with F1 indices for new matches)."""
        n1, nc = len(F1.keys), len(F2.cam_w)
        if assigned2 is None:
            assigned2 = np.full(len(F2.keys), -1, np.int32)
        i1, c = np.nonzero((np.asarray(valid1) != 0)[:, None] & (np.asarray(in_mask) != 0))      # i1 outer, camera inner
        lv = F1.keys["octave"][i1]
        q = _queries(c, np.asarray(uv)[i1, c, 0], np.asarray(uv)[i1, c, 1], float(windowSize), lv, lv, i1)
        return search_windows(F2, q, F1.desc, F1.dmask if self.havingMasks else None, i1, RULE_RATIO, self.mfNNratio,
                              self.TH_HIGH_, assigned2)

    def SearchByProjectionLast(self, CurrentFrame, LastFrame, th, valid_last, uv, in_mask, assigned_cur=None):
        """SearchByProjection(CurrentFrame, LastFrame, th) (ref :1990-2118, motion model).  valid_last[i]: LastFrame keypoint i has a
        non-bad, non-outlier map point; uv[i] = its projection into its own camera of CurrentFrame, in_mask[i] = mirror-mask test.
        Returns (nmatches, CurrentFrame.mvpMapPoints as LastFrame indices)."""
        if assigned_cur is None:
            assigned_cur = np.full(len(CurrentFrame.keys), -1, np.int32)
        sel = np.flatnonzero((np.asarray(valid_last) != 0) & (np.asarray(in_mask) != 0))
        lv = LastFrame.keys["octave"][sel]
        r = th * CurrentFrame.scale_factors[lv]
        q = _queries(LastFrame.key_cam[sel], np.asarray(uv)[sel, 0], np.asarray(uv)[sel, 1], r, lv - 1, lv + 1, sel)
        return search_windows(CurrentFrame, q, LastFrame.desc, LastFrame.dmask if self.havingMasks else None, sel, RULE_BEST,
                              self.mfNNratio, self.TH_HIGH_, assigned_cur)

    def FuseCandidates(self, KF, uv, in_mask, level, th, mp_desc, mp_dmask=None, first_wins=False):
        """Matching core of Fuse(pKF, curKF, vpMapPoints, th) (ref :1265-1418) and Fuse(pKF, Scw, vpPoints, th) (:1570-1719): for map
        point i and camera c (in_mask[i,c]) the best keypoint of KF within th*scale[level] of uv[i,c] on levels {level-1, level},
        accepted when its distance <= TH_LOW_.  first_wins=True is Fuse(pKF, vpMapPoints, th) (:1420-1568) as the reference behaves:
        the distance is discarded there, the first in-level candidate of the window wins (MCS_RULE_FIRST_FREE).
        Returns best [n, n_cams] (keypoint index or -1); replacing / adding observations stays with the caller (host map bookkeeping)."""
        in_mask = np.asarray(in_mask) != 0
        i, c = np.nonzero(in_mask)
        lv = np.asarray(level)[i, c]
        q = _queries(c, np.asarray(uv)[i, c, 0], np.asarray(uv)[i, c, 1], th * KF.scale_factors[lv], lv - 1, lv, i)
        n, res = search_windows(KF, q, mp_desc, mp_dmask if self.havingMasks else None, np.zeros(len(q), np.int32),
                                RULE_FIRST_FREE if first_wins else RULE_BEST_FREE,
                                self.mfNNratio, self.TH_LOW_, np.full(max(len(q), len(KF.keys)), -1, np.int32))
        best = np.full(in_mask.shape, -1, np.int32)
        best[i, c] = res[:len(q)]
        return best

    def SearchByProjectionScw(self, KF, query_cam, uv, level, th, valid, mp_desc, mp_dmask=None, matched=None):
        """Matching part of SearchByProjection(pKF, Scw, vpPoints, vpMatched, th) (ref :2265-2392) as written there.  Entry i of
        vpPoints: valid[i] (not NULL / bad / already found, projected inside the mirror mask, distance in range), query_cam[i] =
        keypoint_to_cam[i] -- the reference looks the camera up with the POINT's list position (:2326) --, uv[i], level[i] the
        predicted level.  matched = vpMatched as map point ids per keypoint (-1 = NULL), updated.  Candidate descriptors are read
        the way the reference does (contiguous id as per-camera row; MCS_RULE_SCW) and keypoint 0 can never be matched (:2385)."""
        if matched is None:
            matched = np.full(len(KF.keys), -1, np.int32)
        sel = np.flatnonzero(np.asarray(valid) != 0)
        lv = np.asarray(level)[sel]
        q = _queries(np.asarray(query_cam)[sel], np.asarray(uv)[sel, 0], np.asarray(uv)[sel, 1], th * KF.scale_factors[lv], lv - 1, lv, sel)
        return search_windows(KF, q, mp_desc, mp_dmask if self.havingMasks else None, sel, RULE_SCW, self.mfNNratio, self.TH_LOW_,
                              matched)

    def _project_for_fuse(self, KF, rig, Ow, world_pos, min_dist, max_dist, idx, float_dist):
        """projection front-end shared by the Fuse overloads and SearchByProjection(KF, Scw): WorldToCamHom_fast ->
        isPointInMirrorMask -> distance range -> predicted level (ref :1288-1318)"""
        nc = len(rig.cams)
        uv = np.zeros((len(idx), nc, 2)); ok = np.zeros((len(idx), nc), np.uint8); lvl = np.zeros((len(idx), nc), np.int32)
        for k, i in enumerate(idx):
            p = world_pos[i]
            for c in range(nc):
                u, v, _ = rig.world_to_cam(c, p)
                if not rig.in_mirror_mask(c, u, v):
                    continue
                po = p - Ow
                d = float(np.sqrt(po[0] * po[0] + po[1] * po[1] + po[2] * po[2]))
                if float_dist:
                    d = float(np.float32(d))                      # `const float dist3D = cv::norm(PO);` (ref :1301, :1472)
                if d < min_dist[i] or d > max_dist[i]:
                    continue
                uv[k, c] = (u, v); ok[k, c] = 1
                lvl[k, c] = _predict_level(KF.scale_factors, d / min_dist[i])
        return uv, ok, lvl

    def Fuse(self, KF, rig, kf_mp, points, world_pos, min_dist, max_dist, bad, in_kf, mp_desc, mp_dmask=None, th=2.5, variant=1,
             Scw=None, cur_rays=None, kf_rays=None, cur_rig=None, _sw=None):
        """The three Fuse overloads of the reference as whole entry points (projection on the host with the reference's double
        arithmetic, window search + distances on the GPU, map bookkeeping replayed in order):
          variant 0  Fuse(pKF, curKF, vpMapPoints, th)  (ref :1265-1418): points[i] is the map point of keypoint i of curKF; a hit
                     on an occupied keypoint needs the epipolar check of the two bearing rays (cur_rays, kf_rays, cur_rig)
          variant 1  Fuse(pKF, vpMapPoints, th)         (ref :1420-1568): distance discarded, first in-level candidate wins
          variant 2  Fuse(pKF, Scw, vpPoints, th)       (ref :1570-1719): the rig pose is replaced by the Sim3's rigid part
        kf_mp [n_keys] map point id per keypoint (-1 none), updated like pKF->AddMapPoint does; points: candidate map point ids
        (-1 = NULL); bad / in_kf (IsInKeyFrame(pKF)) per map point.  Returns (nFused, ops) with ops rows (0, mp, keypoint) =
        AddObservation + AddMapPoint and (1, mp, other) = Replace(other), in the reference's call order."""
        sw = search_windows if _sw is None else _sw
        kf_mp = np.ascontiguousarray(kf_mp, np.int32).copy()
        world_pos = np.asarray(world_pos, np.float64)
        if variant == 2:
            S = np.asarray(Scw, np.float64)
            sR = S[:3, :3]
            inv_s = 1.0 / float(np.sqrt(sR[0, 0] * sR[0, 0] + sR[0, 1] * sR[0, 1] + sR[0, 2] * sR[0, 2]))
            T = np.eye(4)
            T[:3, :3], T[:3, 3] = inv_s * sR, inv_s * S[:3, 3]
            rig = Rig(rig.cams, rig.M_c, inv_rigid(T))            # camSys.Set_M_t(invMat(Rt2Hom(Rcw, tcw)))  (ref :1576-1584)
            already = set(int(m) for m in kf_mp if m >= 0 and not bad[m])
            idx = [int(i) for i in points if not bad[i] and int(i) not in already]
        else:
            idx = [int(i) for i in points if i >= 0 and not bad[i] and not in_kf[i]]
        Ow = rig.M_t[:3, 3].copy()
        uv, ok, lvl = self._project_for_fuse(KF, rig, Ow, world_pos, min_dist, max_dist, idx, float_dist=(variant != 2))
        k, c = np.nonzero(ok)
        lv = lvl[k, c]
        q = _queries(c, uv[k, c, 0], uv[k, c, 1], th * KF.scale_factors[lv], lv - 1, lv, np.asarray(idx, np.int64)[k])
        n, res = sw(KF, q, mp_desc, mp_dmask if self.havingMasks else None, np.zeros(len(q), np.int32),
                    RULE_FIRST_FREE if variant == 1 else RULE_BEST_FREE, self.mfNNratio, self.TH_LOW_,
                    np.full(max(len(q), len(KF.keys)), -1, np.int32))
        best = np.full(ok.shape, -1, np.int32)
        best[k, c] = res[:len(q)]
        ops, fused = [], 0
        pos_of = {}
        if variant == 0:
            pos_of = {int(i): j for j, i in enumerate(points) if i >= 0}     # keypoint of curKF that carries map point i
        for kk, i in enumerate(idx):
            for cam in range(ok.shape[1]):
                b = int(best[kk, cam])
                if b < 0:
                    continue
                other = int(kf_mp[b])
                if other >= 0:
                    good = not bad[other]
                    if variant == 0 and good:
                        T1 = inv_rigid(cur_rig.MtMc[cam]) if cur_rig is not None else np.eye(4)
                        E = compute_E_rel(_mm(T1, rig.MtMc[cam]))
                        good = check_epipolar(cur_rays[pos_of[i]], kf_rays[b], E, 1e-2)
                    if good:
                        ops.append((1, i, other)); fused += 1
                else:
                    ops.append((0, i, b)); kf_mp[b] = i
        return fused, np.asarray(ops, np.int32).reshape(-1, 3), kf_mp

    def SearchByProjectionKFScw(self, KF, rig, Scw, points, matched, world_pos, min_dist, max_dist, bad, mp_desc, mp_dmask=None, th=10,
                                _sw=None):
        """SearchByProjection(pKF, Scw, vpPoints, vpMatched, th) (ref :2265-2392) as a whole entry point, quirks included: the
        camera of entry iMP of vpPoints is keypoint_to_cam[iMP] (:2326), candidate descriptors are read with the contiguous id as
        per-camera row (:2367, :2372) and keypoint 0 is never matched (:2385).  points: map point ids (-1 = NULL), len <= n_keys;
        matched: vpMatched as map point ids per keypoint (-1 = NULL).  Returns (nmatches, vpMatched)."""
        sw = search_windows if _sw is None else _sw
        S = np.asarray(Scw, np.float64)
        sR = S[:3, :3]
        inv_s = 1.0 / float(np.sqrt(sR[0, 0] * sR[0, 0] + sR[0, 1] * sR[0, 1] + sR[0, 2] * sR[0, 2]))
        T = np.eye(4)
        T[:3, :3], T[:3, 3] = inv_s * sR, inv_s * S[:3, 3]
        rig = Rig(rig.cams, rig.M_c, inv_rigid(T))
        Ow = rig.M_t[:3, 3].copy()
        matched = np.ascontiguousarray(matched, np.int32).copy()
        found = set(int(m) for m in matched if m >= 0)
        world_pos = np.asarray(world_pos, np.float64)
        qc, quv, qlv, qi = [], [], [], []
        for iMP, i in enumerate(points):
            i = int(i)
            if i < 0 or bad[i] or i in found:
                continue
            cam = int(KF.key_cam[iMP])
            u, v, _ = rig.world_to_cam(cam, world_pos[i])
            if not rig.in_mirror_mask(cam, u, v):
                continue
            po = world_pos[i] - Ow
            d = float(np.sqrt(po[0] * po[0] + po[1] * po[1] + po[2] * po[2]))
            if d < min_dist[i] or d > max_dist[i]:
                continue
            qc.append(cam); quv.append((u, v)); qlv.append(_predict_level(KF.scale_factors, d / min_dist[i])); qi.append(i)
        if not qi:
            return 0, matched
        lv = np.asarray(qlv)
        quv = np.asarray(quv)
        q = _queries(np.asarray(qc), quv[:, 0], quv[:, 1], float(int(th)) * KF.scale_factors[lv], lv - 1, lv, np.asarray(qi))
        return sw(KF, q, mp_desc, mp_dmask if self.havingMasks else None, np.asarray(qi, np.int32), RULE_SCW, self.mfNNratio,
                  self.TH_LOW_, matched)

    def SearchByProjectionFramesRig(self, F1, mp1, F2, rig2, mp2, world_pos, bad, windowSize, _sw=None):
        """SearchByProjection(F1, F2, windowSize, vpMapPointMatches2) (ref :476-577) as a whole entry point: every map point of F1
        (first occurrence only, not bad, not already in F2) is projected into EVERY camera of F2's rig and searched there on the level
        of its F1 keypoint; ratio test + TH_HIGH_, greedy.  mp1 / mp2: map point id per keypoint (-1 none).
        Returns (nmatches, vpMapPointMatches2 as map point ids)."""
        sw = search_windows if _sw is None else _sw
        out = np.ascontiguousarray(mp2, np.int32).copy()
        already = set(int(x) for x in out)                   # spMapPointsAlreadyFound holds NULL as well: harmless
        world_pos = np.asarray(world_pos, np.float64)
        seen = set()
        qc, quv, qlv, qi, tags = [], [], [], [], []
        for i1 in range(len(F1.keys)):
            p = int(mp1[i1])
            if p < 0 or bad[p] or p in already or p in seen:
                continue
            seen.add(p)
            for c in range(len(rig2.cams)):
                u, v, _ = rig2.world_to_cam(c, world_pos[p])
                if rig2.in_mirror_mask(c, u, v):
                    qc.append(c); quv.append((u, v)); qlv.append(int(F1.keys["octave"][i1])); qi.append(i1); tags.append(p)
        if not qi:
            return 0, out
        quv, lv = np.asarray(quv), np.asarray(qlv)
        q = _queries(np.asarray(qc), quv[:, 0], quv[:, 1], float(int(windowSize)), lv, lv, np.asarray(qi))
        return sw(F2, q, F1.desc, F1.dmask if self.havingMasks else None, np.asarray(tags, np.int32), RULE_RATIO, self.mfNNratio,
                  self.TH_HIGH_, out)

    def SearchByProjectionLastRig(self, CurrentFrame, rig_cur, cur_mp, LastFrame, last_mp, last_outlier, world_pos, bad, th, _sw=None):
        """SearchByProjection(CurrentFrame, LastFrame, th) (ref :1990-2118, motion model) as a whole entry point: the map point of
        every LastFrame keypoint (not bad, not an outlier) is projected into the SAME camera of the current rig pose and searched
        on levels octave-1 .. octave+1 within th*scale[octave]; best distance <= TH_HIGH_, greedy on CurrentFrame.mvpMapPoints.
        Returns (nmatches, CurrentFrame.mvpMapPoints as map point ids)."""
        sw = search_windows if _sw is None else _sw
        out = np.ascontiguousarray(cur_mp, np.int32).copy()
        world_pos = np.asarray(world_pos, np.float64)
        qc, quv, qlv, qi, tags = [], [], [], [], []
        for i in range(len(LastFrame.keys)):
            p = int(last_mp[i])
            if p < 0 or bad[p] or (last_outlier is not None and last_outlier[i]):
                continue
            cam = int(LastFrame.key_cam[i])
            u, v, _ = rig_cur.world_to_cam(cam, world_pos[p])
            if not rig_cur.in_mirror_mask(cam, u, v):
                continue
            qc.append(cam); quv.append((u, v)); qlv.append(int(LastFrame.keys["octave"][i])); qi.append(i); tags.append(p)
        if not qi:
            return 0, out
        quv, lv = np.asarray(quv), np.asarray(qlv)
        q = _queries(np.asarray(qc), quv[:, 0], quv[:, 1], th * CurrentFrame.scale_factors[lv], lv - 1, lv + 1, np.asarray(qi))
        return sw(CurrentFrame, q, LastFrame.desc, LastFrame.dmask if self.havingMasks else None, np.asarray(tags, np.int32), RULE_BEST,
                  self.mfNNratio, self.TH_HIGH_, out)

    def SearchBySim3(self, KF1, rig1, mp1, KF2, rig2, mp2, world_pos, min_dist, max_dist, bad, mp_desc, mp_dmask, s12, R12, t12, th,
                     matches12=None, obs_idx2=None, _sw=None):
        """SearchBySim3(pKF1, pKF2, vpMatches12, s12, R12, t12, th) (ref :1721-1988) as a whole entry point: the map points of each
        key frame are carried into the other one by the similarity, searched in a th*scale[level] window on levels {l-1, l}
        (best distance <= TH_HIGH_), and only mutual agreements are kept.  mp1 / mp2: map point id per keypoint (-1 none);
        matches12 [n1]: already matched map point ids (-1 none) -- their keypoints are excluded, obs_idx2[id] = keypoint of KF2 that
        observes map point id (GetIndexInKeyFrame(pKF2)[0]).  Returns (nFound, vpMatches12 as map point ids)."""
        sw = search_windows if _sw is None else _sw
        n1, n2 = len(KF1.keys), len(KF2.keys)
        m12 = np.full(n1, -1, np.int32) if matches12 is None else np.ascontiguousarray(matches12, np.int32).copy()
        world_pos = np.asarray(world_pos, np.float64)
        R12, t12 = np.asarray(R12, np.float64), np.asarray(t12, np.float64)
        T1, T2 = inv_rigid(rig1.M_t), inv_rigid(rig2.M_t)                       # GetPoseInverse()
        sR12 = s12 * R12
        sR21 = (1.0 / s12) * R12.T.copy()
        t21 = _mm(-sR21, t12)
        done1, done2 = np.zeros(n1, bool), np.zeros(n2, bool)
        for i in range(n1):
            if m12[i] >= 0:
                done1[i] = True
                j = int(obs_idx2[m12[i]]) if obs_idx2 is not None else -1
                if 0 <= j < n2:
                    done2[j] = True

        def one_way(KFa, mpa, Ta, sR, tt, KFb, rigb, skip_a):
            """points of a -> frame b; returns best keypoint of b per keypoint of a (-1 none)"""
            qc, quv, qlv, qi, qd = [], [], [], [], []
            for i in range(len(KFa.keys)):
                p = int(mpa[i])
                if p < 0 or skip_a[i] or bad[p]:
                    continue
                cam = int(KFa.key_cam[i])
                pa = _mm(Ta[:3, :3], world_pos[p]) + Ta[:3, 3]                  # point in the MCS frame of a
                pb = _mm(sR, pa) + tt                                           # ... of b
                p4 = _mm(inv_rigid(rigb.M_c[cam]), np.array([pb[0], pb[1], pb[2], 1.0]))
                if pb[2] < 0.0:
                    continue
                u, v = world_to_img(rigb.cams[cam], float(p4[0]), float(p4[1]), float(p4[2]))
                if not rigb.in_mirror_mask(cam, u, v):
                    continue
                d = float(np.sqrt(p4[0] * p4[0] + p4[1] * p4[1] + p4[2] * p4[2]))
                if d < min_dist[p] or d > max_dist[p]:
                    continue
                qc.append(cam); quv.append((u, v)); qlv.append(_predict_level(KFb.scale_factors, d / min_dist[p])); qi.append(i); qd.append(p)
            best = np.full(len(KFa.keys), -1, np.int32)
            if qi:
                lv, quv2 = np.asarray(qlv), np.asarray(quv)
                q = _queries(np.asarray(qc), quv2[:, 0], quv2[:, 1], th * KFb.scale_factors[lv], lv - 1, lv, np.asarray(qd))
                _, res = sw(KFb, q, mp_desc, mp_dmask if self.havingMasks else None, np.zeros(len(q), np.int32), RULE_BEST_FREE,
                            self.mfNNratio, self.TH_HIGH_, np.full(max(len(q), len(KFb.keys)), -1, np.int32))
                best[np.asarray(qi)] = res[:len(q)]
            return best
        b1 = one_way(KF1, mp1, T1, sR21, t21, KF2, rig2, done1)
        b2 = one_way(KF2, mp2, T2, sR12, t12, KF1, rig1, done2)
        found = 0
        for i1 in range(n1):
            i2 = int(b1[i1])
            if i2 >= 0 and int(b2[i2]) == i1:
                m12[i1] = mp2[i2]
                found += 1
        return found, m12

    def SearchForTriangulationBetweenCameras(self, KF, rig, kf_mp, rays, cam1, cam2, _sw=None):
        """SearchForTriangulationBetweenCameras(pKF1, cam1, cam2, ...) (ref :1158-1263): every keypoint of camera cam1 without a
        map point is carried along its bearing ray into camera cam2 of the same rig (relative orientation of the two cameras),
        searched in a 40 px window (all levels, nothing skipped), and accepted when the best distance is <= 100 and the two rays
        satisfy the epipolar constraint.  Returns (nmatches, pairs [n,2] of contiguous keypoint ids)."""
        sw = search_windows if _sw is None else _sw
        rel = _mm(inv_rigid(rig.M_c[cam1]), rig.M_c[cam2])
        E12 = compute_E_rel(rel)
        Rrel = rel[:3, :3].T.copy()
        trel = _mm(-Rrel, rel[:3, 3])
        qi, quv = [], []
        for i in range(len(KF.keys)):
            if kf_mp[i] >= 0 or int(KF.key_cam[i]) != cam1:
                continue
            rp = _mm(Rrel, rays[i]) + trel
            rp = rp / float(np.sqrt(rp[0] * rp[0] + rp[1] * rp[1] + rp[2] * rp[2]))
            u, v = world_to_img(rig.cams[cam2], float(rp[0]), float(rp[1]), float(rp[2]))
            if not rig.in_mirror_mask(cam2, u, v):
                continue
            qi.append(i); quv.append((u, v))
        pairs = []
        if qi:
            quv = np.asarray(quv)
            q = _queries(np.full(len(qi), cam2), quv[:, 0], quv[:, 1], 40.0, -1, -1, np.asarray(qi))
            _, res = sw(KF, q, KF.desc, KF.dmask if self.havingMasks else None, np.zeros(len(q), np.int32), RULE_BEST_FREE, self.mfNNratio,
                        100, np.full(max(len(q), len(KF.keys)), -1, np.int32))
            for k, i in enumerate(qi):
                b = int(res[k])
                # the reference evaluates the epipolar test with the best candidate even when its distance fails (:1247-1249);
                # RULE_BEST_FREE already applied bestDist <= 100
                if b >= 0 and check_epipolar(rays[i], rays[b], E12, 1e-2):
                    pairs.append((i, b))
        return len(pairs), np.asarray(pairs, np.int32).reshape(-1, 2)

    def SearchForTriangulationRaw(self, desc1, mask1, cam1, free1, rays1, desc2, mask2, cam2, free2, rays2, E, epi_thresh=1e-2):
        """SearchForTriangulationRaw(KF1, KF2, ...) (ref :968-1156): free1/free2 flag keypoints WITHOUT a map point, rays = bearing
        vectors [n,3], E [n_cams,n_cams,3,3] from ComputeE.  Returns (nmatches, vMatches12)."""
        d1, d2 = np.ascontiguousarray(desc1, np.uint8), np.ascontiguousarray(desc2, np.uint8)
        use = self.havingMasks and mask1 is not None and mask2 is not None
        m1 = np.ascontiguousarray(mask1, np.uint8) if use else None
        m2 = np.ascontiguousarray(mask2, np.uint8) if use else None
        c1, c2 = np.ascontiguousarray(cam1, np.int32), np.ascontiguousarray(cam2, np.int32)
        f1, f2 = np.ascontiguousarray(free1, np.uint8), np.ascontiguousarray(free2, np.uint8)
        r1, r2 = np.ascontiguousarray(rays1, np.float64), np.ascontiguousarray(rays2, np.float64)
        Em = np.ascontiguousarray(E, np.float64)
        m12 = np.zeros(len(d1), np.int32)
        n = C.c_int32(0)
        _check(lib().mcs_search_for_triangulation(_p(d1), _p(m1), _p(c1), _p(f1), _p(r1), len(d1), _p(d2), _p(m2), _p(c2), _p(f2), _p(r2),
                                                  len(d2), d1.shape[1], self.TH_LOW_, _p(Em), Em.shape[0], C.c_double(epi_thresh), _p(m12), C.byref(n)))
        return n.value, m12

    def SearchByBoW(self, desc1, desc2, mask1=None, mask2=None, valid1=None, valid2=None):
        """SearchByBoW(cMultiKeyFrame*, cMultiKeyFrame*, vpMatches12) (ref :885-966): all-pairs scan over the
        map-point-bearing keypoints of two keyframes.  Returns (nmatches, matches12 indices into desc2)."""
        d1 = np.ascontiguousarray(desc1, np.uint8)
        d2 = np.ascontiguousarray(desc2, np.uint8)
        use = self.havingMasks and mask1 is not None and mask2 is not None
        m1 = np.ascontiguousarray(mask1, np.uint8) if use else None
        m2 = np.ascontiguousarray(mask2, np.uint8) if use else None
        v1 = None if valid1 is None else np.ascontiguousarray(valid1, np.uint8)
        v2 = None if valid2 is None else np.ascontiguousarray(valid2, np.uint8)
        m12 = np.zeros(len(d1), np.int32)
        n = C.c_int32(0)
        _check(lib().mcs_match_bruteforce(_p(d1), _p(m1), _p(v1), len(d1), _p(d2), _p(m2), _p(v2), len(d2), d1.shape[1],
                                          self.TH_LOW_, C.c_double(self.mfNNratio), _p(m12), C.byref(n)))
        return n.value, m12

    def SearchByBoWFrame(self, desc_kf, featvec_kf, desc_f, featvec_f, mask_kf=None, mask_f=None, valid_kf=None):
        """SearchByBoW(cMultiKeyFrame* pKF, cMultiFrame& F, vpMapPointMatches) (ref src/cORBmatcher.cpp:179-324): matching
        restricted to keypoints that fall into the same vocabulary node.  featvec_* = (nodes, offsets, features) as returned
        by ORBVocabulary.transform.  Returns (nmatches, match_of_f) with match_of_f[i] = key-frame keypoint or -1."""
        d1 = np.ascontiguousarray(desc_kf, np.uint8)
        d2 = np.ascontiguousarray(desc_f, np.uint8)
        use = self.havingMasks and mask_kf is not None and mask_f is not None
        m1 = np.ascontiguousarray(mask_kf, np.uint8) if use else None
        m2 = np.ascontiguousarray(mask_f, np.uint8) if use else None
        v1 = None if valid_kf is None else np.ascontiguousarray(valid_kf, np.uint8)
        a = [np.ascontiguousarray(x, np.int32) for x in featvec_kf]
        b = [np.ascontiguousarray(x, np.int32) for x in featvec_f]
        out = np.zeros(len(d2), np.int32)
        n = C.c_int32(0)
        _check(lib().mcs_search_by_bow(_p(d1), _p(m1), _p(v1), len(d1), _p(a[0]), _p(a[1]), len(a[0]), _p(a[2]), _p(d2), _p(m2), len(d2),
                                       _p(b[0]), _p(b[1]), len(b[0]), _p(b[2]), d1.shape[1], self.TH_LOW_, C.c_double(self.mfNNratio),
                                       _p(out), C.byref(n)))
        return n.value, out


class ORBVocabulary:
    """Mirror of ORBVocabulary = DBoW2::TemplatedVocabulary<FORB::TDescriptor, FORB> (ref include/cORBVocabulary.h:34) for the
    calls the SLAM front end makes: load, transform(features, BowVector, FeatureVector, levelsup), score, size.
    The tree lives on the GPU (mcs_vocabulary_create); `voc` is a mapping with k, L, scoring, weighting, parent, weight,
    desc, word_node and optionally node_order (tools/extract_vocabulary.py writes that layout)."""

    def __init__(self, voc, scoring=None, weighting=None):
        self.k, self.L = int(voc["k"]), int(voc["L"])
        self.scoring = int(voc["scoring"] if scoring is None else scoring)
        self.weighting = int(voc["weighting"] if weighting is None else weighting)
        par = np.ascontiguousarray(voc["parent"], np.int32)
        wt = np.ascontiguousarray(voc["weight"], np.float64)
        ds = np.ascontiguousarray(voc["desc"], np.uint8)
        wn = np.ascontiguousarray(voc["word_node"], np.int32)
        order = voc["node_order"] if "node_order" in voc else None
        order = None if order is None else np.ascontiguousarray(order, np.int32)
        if ds.shape != (len(par), 32) or len(wt) != len(par):
            raise ValueError("vocabulary arrays disagree in size")
        self._n_words = len(wn)
        self._h = C.c_void_p()
        _check(lib().mcs_vocabulary_create(self.k, self.L, self.scoring, self.weighting, len(par), _p(par), _p(wt), _p(ds), _p(order),
                                           len(wn), _p(wn), C.byref(self._h)))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().mcs_vocabulary_destroy(self._h)
            self._h = None

    @staticmethod
    def loadFromTextFile(path, **kw):
        """DBoW2 text layout (ref TemplatedVocabulary.h:1338-1425): 'k L scoring weighting', then one line per node
        'parent isLeaf d0..d31 weight', node ids and word ids in line order."""
        lines = [ln for ln in open(path).read().split("\n") if ln.strip()]
        k, L, sc, wg = (int(t) for t in lines[0].split()[:4])
        n = len(lines)
        parent = np.zeros(n, np.int32); weight = np.zeros(n); desc = np.zeros((n, 32), np.uint8); words = []
        for i, ln in enumerate(lines[1:], start=1):
            t = ln.split()
            parent[i] = int(t[0]); desc[i] = [int(x) for x in t[2:34]]; weight[i] = float(t[34])
            if int(t[1]) > 0:
                words.append(i)
        return ORBVocabulary(dict(k=k, L=L, scoring=sc, weighting=wg, parent=parent, weight=weight, desc=desc,
                                  word_node=np.asarray(words, np.int32)), **kw)

    @staticmethod
    def load(path, **kw):
        """DBoW2 YAML layout as cv::FileStorage writes it (ref TemplatedVocabulary.h:1476-1624)."""
        import re
        txt = open(path).read()
        head = {key: int(re.search(r"\b%s:\s*(\d+)" % key, txt).group(1)) for key in ("k", "L", "scoringType", "weightingType")}
        nodes = re.findall(r"nodeId:(\d+),\s*parentId:(\d+),\s*weight:([-+0-9.eE]+),\s*descriptor:\"([^\"]*)\"", txt)
        words = re.findall(r"wordId:(\d+),\s*nodeId:(\d+)", txt)
        n = len(nodes) + 1
        parent = np.zeros(n, np.int32); weight = np.zeros(n); desc = np.zeros((n, 32), np.uint8); order = np.zeros(n - 1, np.int32)
        for i, (nid, pid, w, d) in enumerate(nodes):
            nid = int(nid); order[i] = nid; parent[nid] = int(pid); weight[nid] = float(w + "0" if w.endswith(".") else w)
            desc[nid] = [int(x) for x in d.split()]
        wn = np.zeros(len(words), np.int32)
        for wid, nid in words:
            wn[int(wid)] = int(nid)
        return ORBVocabulary(dict(k=head["k"], L=head["L"], scoring=head["scoringType"], weighting=head["weightingType"], parent=parent,
                                  weight=weight, desc=desc, node_order=order, word_node=wn), **kw)

    def size(self):
        return self._n_words

    def transform_features(self, desc, levelsup=4):
        """per descriptor: (word id, word weight, node id at level L - levelsup)  (ref :1218-1261)"""
        desc = np.ascontiguousarray(desc, np.uint8)
        if desc.ndim != 2 or desc.shape[1] != 32:
            raise ValueError("the vocabulary works on 32-byte descriptors (FORB::L)")
        n = len(desc)
        w = np.zeros(n, np.int32); wt = np.zeros(n, np.float64); nd = np.zeros(n, np.int32)
        _check(lib().mcs_bow_transform(self._h, _p(desc), n, levelsup, _p(w), _p(wt), _p(nd)))
        return w, wt, nd

    def transform(self, desc, levelsup=4):
        """transform(features, BowVector&, FeatureVector&, levelsup) (ref :1126-1194).
        -> (bow_words, bow_values, (fv_nodes, fv_offsets, fv_features))"""
        desc = np.ascontiguousarray(desc, np.uint8)
        if desc.ndim != 2 or (len(desc) and desc.shape[1] != 32):
            raise ValueError("the vocabulary works on 32-byte descriptors (FORB::L)")
        n = len(desc)
        bw = np.zeros(max(n, 1), np.int32); bv = np.zeros(max(n, 1), np.float64); nb = C.c_int32(0)
        fn = np.zeros(max(n, 1), np.int32); fo = np.zeros(n + 2, np.int32); nf = C.c_int32(0); ff = np.zeros(max(n, 1), np.int32)
        _check(lib().mcs_bow_vectors(self._h, _p(desc), n, levelsup, _p(bw), _p(bv), C.byref(nb), _p(fn), _p(fo), C.byref(nf), _p(ff)))
        k = nf.value
        return bw[:nb.value].copy(), bv[:nb.value].copy(), (fn[:k].copy(), fo[:k + 1].copy(), ff[:fo[k]].copy())

    def score(self, v1, v2):
        """score(BowVector, BowVector) with the vocabulary's scoring type; v = (words, values)."""
        w1 = np.ascontiguousarray(v1[0], np.int32); x1 = np.ascontiguousarray(v1[1], np.float64)
        w2 = np.ascontiguousarray(v2[0], np.int32); x2 = np.ascontiguousarray(v2[1], np.float64)
        s = C.c_double(0)
        _check(lib().mcs_bow_score(self._h, _p(w1), _p(x1), len(w1), _p(w2), _p(x2), len(w2), C.byref(s)))
        return s.value


class KeyFrameDatabase:
    """Mirror of cMultiKeyFrameDatabase (ref include/cMultiKeyFrameDatabase.h, src/cMultiKeyFrameDatabase.cpp): the inverted
    file over `voc`'s words and the per-key-frame query fields live on the GPU (mcs_kfdb_*).  Key frames are named by their
    mnId; bow = (words, values) as ORBVocabulary.transform returns them; covis = int64 [n, 10], row id = the ten best
    covisibility key frames of key frame id at query time (-1 = none).  The Detect* calls return int64 arrays of key-frame ids
    in the reference's order."""

    def __init__(self, voc: ORBVocabulary):
        self._voc = voc                      # the database reads the vocabulary's size and scoring type; keep it alive
        self._top = 0
        self._h = C.c_void_p()
        _check(lib().mcs_kfdb_create(voc._h, C.byref(self._h)))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().mcs_kfdb_destroy(self._h)
            self._h = None

    @staticmethod
    def _bow(bow):
        return np.ascontiguousarray(bow[0], np.int32), np.ascontiguousarray(bow[1], np.float64)

    def add(self, kf_id, bow):
        w, v = self._bow(bow)
        if len(w) != len(v):
            raise ValueError("BowVector words and values differ in length")
        _check(lib().mcs_kfdb_add(self._h, C.c_int64(kf_id), _p(w), _p(v), len(w)))
        self._top = max(self._top, int(kf_id) + 1)

    def erase(self, kf_id):
        _check(lib().mcs_kfdb_erase(self._h, C.c_int64(kf_id)))

    def clear(self):
        _check(lib().mcs_kfdb_clear(self._h))

    def _args(self, bow, covis):
        w, v = self._bow(bow)
        if len(w) != len(v):
            raise ValueError("BowVector words and values differ in length")
        cv = np.ascontiguousarray(np.zeros((0, 10), np.int64) if covis is None else covis, np.int64)
        if cv.ndim != 2 or cv.shape[1] != 10:
            raise ValueError("covis must be an int64 array [n, 10]")
        # every candidate is an added key frame or a neighbour named in covis, so this capacity always suffices
        out = np.zeros(max(self._top, int(cv.max()) + 1 if cv.size else 0, 1), np.int64)
        return w, v, cv, out

    def DetectLoopCandidates(self, kf_id, bow, connected, covis, minScore):
        w, v, cv, out = self._args(bow, covis)
        conn = np.ascontiguousarray(np.zeros(0) if connected is None else connected, np.int64)
        n = C.c_int32(0)
        _check(lib().mcs_kfdb_detect_loop_candidates(self._h, C.c_int64(kf_id), _p(w), _p(v), len(w), _p(conn), len(conn), _p(cv),
                                                     C.c_int64(len(cv)), C.c_double(minScore), _p(out), len(out), C.byref(n)))
        return out[:n.value].copy()

    def DetectRelocalisationCandidates(self, frame_id, bow, covis):
        w, v, cv, out = self._args(bow, covis)
        n = C.c_int32(0)
        _check(lib().mcs_kfdb_detect_relocalisation_candidates(self._h, C.c_int64(frame_id), _p(w), _p(v), len(w), _p(cv),
                                                               C.c_int64(len(cv)), _p(out), len(out), C.byref(n)))
        return out[:n.value].copy()
