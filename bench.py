#!/usr/bin/env python
"""bench.py -- Mfeatures/s (extract + match) of the B200 feature hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config {2,3,4}] [--frames F] [--impl reference] [--dump-outputs DIR]

--config 2 (default, the configuration BASELINE.json's metric is quoted on): a stream of 3-fisheye 754x480 multi-camera frames,
    8-level pyramid (scale 1.2), 2000 features per camera, mdBRIEF-256 with masks; every (frame, camera) is brute-force matched
    against the same camera of the previous frame (K best on the GPU + the greedy acceptance of SearchByBoW(KF,KF), also on
    the GPU).  N GPUs: every rank owns its own temporal chunk of the stream (weak scaling) and the ranks exchange their packed
    feature buffers with ONE ncclAllGather per step, issued by the library (mcs_allgather_features) on its own stream so that it
    overlaps the next step's extraction.
--config 3: synthetic 4-fisheye 1280x720 rig, one camera per GPU, 2000 features, allgather of the packed features, then
    SearchByProjection of the rank's camera frames against 50 000 map points (isInFrustum projection on the GPU, window search
    on the GPU, the order-dependent acceptance replayed on the host).
--config 4: synthetic 8-fisheye 1920x1080 rig, one camera per GPU, 4000 features, allgather, then brute-force Hamming of the
    rank's features against a 200 000-descriptor key-frame database resident on every GPU (query-sharded, DB replicated).

One step = one pass over one batch of F frames per GPU (synthetic, seeded).  `value` times the step with the inputs already
resident in HBM (CUDA events on the launching stream, max over ranks); `e2e` times the same work through the public API with
pinned HOST buffers, H2D and D2H inside the timed region.  `roofline` is the fused pyramid+blur+FAST kernel (K1): algorithmic
bytes per launch / CUDA-event time / measured HBM peak.  `cpu_baseline` / --impl reference: the reference's own extractor and
matcher (oracle/_ref/libmcs_ref.so, compiled from /root/reference where that exists) on the host cores over a bounded sample,
else the oracle port.

--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step returned to its caller as DIR/<name>.npy
(float32 / float64): every image's feature and match counts, and the keypoints, descriptors, descriptor masks and matches of a
fixed seeded sample of DUMP_IMAGES images.  The inputs are seeded, so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import json
import os
import pathlib
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))

NLEVELS = 8
DUMP_IMAGES = 32            # images of the last step whose features --dump-outputs writes (config 2: about 21 MB)
CONFIGS = {
    2: dict(n_cams=3, w=754, h=480, nfeatures=2000, frames=128, sharding="stream",
            workload="lafida-3cam-754x480-stream, 8 levels x1.2, 2000 feat/cam, mdBRIEF-256+masks, greedy brute-force match vs previous frame"),
    3: dict(n_cams=4, w=1280, h=720, nfeatures=2000, frames=8, sharding="camera", n_mappoints=50000,
            workload="synthetic-4cam-1280x720 rig, 1 cam/GPU, 8 levels x1.2, 2000 feat/cam, mdBRIEF-256+masks, allgather, SearchByProjection vs 50k map points"),
    4: dict(n_cams=8, w=1920, h=1080, nfeatures=4000, frames=8, sharding="camera", n_db=200000,
            workload="synthetic-8cam-1920x1080 rig, 1 cam/GPU, 8 levels x1.2, 4000 feat/cam, mdBRIEF-256+masks, allgather, brute force vs 200k-descriptor key-frame DB"),
}


def hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def rig_cams(cfg):
    from multicol_slam_b200 import synth
    base = synth.lafida_cams()
    if cfg["w"] == 754:
        return base[:cfg["n_cams"]]
    return [synth.scaled_cam(base[c % 3], cfg["w"], cfg["h"]) for c in range(cfg["n_cams"])]


def make_stream(cams, cam_ids, n_frames, seed0):
    """[F, len(cam_ids), H, W] uint8: per camera a sliding crop of one big seeded texture (real inter-frame motion)."""
    from multicol_slam_b200 import synth
    per_cam = [synth.texture_stream(cams[c], n_frames, seed=seed0 + c) for c in cam_ids]
    return np.ascontiguousarray(np.stack(per_cam, axis=1))


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def usable_cores():
    """Host threads this process may really use: min(affinity, cgroup CPU quota).  The GPU boxes expose 128 logical CPUs but
    cap the container at a 16-CPU quota (cpu.max = 1600000 100000); more threads than that only add throttling."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


# ---------------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own code where oracle/_ref travelled, else the oracle port
# ---------------------------------------------------------------------------------------------------------------------------
def _thread_map(fn, items, n_threads):
    out = [None] * len(items)
    nxt = [0]
    lock = threading.Lock()

    def run():
        while True:
            with lock:
                i = nxt[0]
                nxt[0] += 1
            if i >= len(items):
                return
            out[i] = fn(i, items[i])
    ths = [threading.Thread(target=run) for _ in range(max(1, min(n_threads, len(items))))]
    [t.start() for t in ths]
    [t.join() for t in ths]
    return out


def cpu_arm(cfg_id, cfg, cams, masks, images, n_threads, scene=None):
    """One pass of the config's hot path on the host over `images` [F, C, H, W] with n_threads threads.
    Returns (features, seconds, kind, what)."""
    import ref_mcs_api as ra
    nf = cfg["nfeatures"]
    F, Cn = images.shape[:2]
    if not ra.available():
        import oracle_api as oa
        oa.lib()
        t0 = time.perf_counter()
        if cfg_id == 2:
            nfeat, _ = oa.stream_mt(images, masks, cams, n_threads, nfeatures=nf, nlevels=NLEVELS)
        else:       # the port's extraction; matching as below is only available with the reference library
            per = _thread_map(lambda i, fc: len(oa.OracleExtractor(nfeatures=nf, do_dbrief=True, learn_masks=True).extract(
                images[fc[0], fc[1]], masks[fc[1]], cams[fc[1]])[0]), [(f, c) for f in range(F) for c in range(Cn)], n_threads)
            nfeat = sum(per)
        return nfeat, time.perf_counter() - t0, "port", "oracle/mcs_oracle.cpp (oracle/_ref not present)"
    import ref_match_api as rm
    import multicol_slam_b200.api as api           # array holders only
    ra.set_deterministic(False)                     # stock allocator: re-entrant, one extractor per thread
    local = threading.local()

    def extract(i, fc):
        if not hasattr(local, "ex"):
            local.ex = ra.RefExtractor(nfeatures=nf, do_dbrief=True, learn_masks=True)
        f, c = fc
        return local.ex.extract(images[f, c], masks[c], cams[c])
    t0 = time.perf_counter()
    jobs = [(f, c) for f in range(F) for c in range(Cn)]
    feats = _thread_map(extract, jobs, n_threads)
    nfeat = sum(len(k) for k, _, _ in feats)
    sf = [float(np.float32(1.2)) ** l for l in range(NLEVELS)]
    size = [(cfg["w"], cfg["h"])]
    if cfg_id == 2:         # SearchByBoW(KF, KF) of every (t, c) against (t-1, c): the reference's own all-pairs scan
        def match(i, fc):
            f, c = fc
            if f == 0:
                return 0
            (k1, d1, m1), (k2, d2, m2) = feats[f * Cn + c], feats[(f - 1) * Cn + c]
            F1 = api.Frame(k1, np.zeros(len(k1), np.int32), d1, m1, size, sf)
            F2 = api.Frame(k2, np.zeros(len(k2), np.int32), d2, m2, size, sf)
            n1, n2 = len(k1), len(k2)
            table = rm.MPTable(1, np.zeros((n1 + n2, 32), np.uint8))
            return rm.search_by_bow_kfkf(rm.KF(F1, [cams[c]], mp=np.arange(n1, dtype=np.int32)),
                                         rm.KF(F2, [cams[c]], mp=n1 + np.arange(n2, dtype=np.int32)), table, 0.9, True)[0]
        _thread_map(match, jobs, n_threads)
    elif cfg_id == 3:       # SearchByProjection(F, 50k map points, th = 3) per frame
        def match(i, fc):
            f, c = fc
            k, d, m = feats[i]
            Fr = api.Frame(k, np.zeros(len(k), np.int32), d, m, size, sf)
            v = scene["views"][f]
            table = rm.MPTable(1, scene["mp_desc"], dmask=scene["mp_dmask"], in_view=v[0], level=v[1], proj_x=v[2], proj_y=v[3], view_cos=v[4])
            return rm.search_by_projection(rm.KF(Fr, [cams[c]]), table, 3.0, 0.8, True)[0]
        _thread_map(match, jobs, n_threads)
    else:                   # config 4: brute force against the 200k database, queries split over the threads
        def match(i, fc):
            k, d, m = feats[i]
            n1, nd = len(k), len(scene["db"])
            F1 = api.Frame(k, np.zeros(n1, np.int32), d, m, size, sf)
            F2 = api.Frame(np.zeros(nd, api.KEYPOINT_DTYPE), np.zeros(nd, np.int32), scene["db"], scene["db_mask"], size, sf)
            table = rm.MPTable(1, np.zeros((n1 + nd, 32), np.uint8))
            return rm.search_by_bow_kfkf(rm.KF(F1, [cams[fc[1]]], mp=np.arange(n1, dtype=np.int32)),
                                         rm.KF(F2, [cams[fc[1]]], mp=n1 + np.arange(nd, dtype=np.int32)), table, 0.9, True)[0]
        _thread_map(match, jobs, n_threads)
    dt = time.perf_counter() - t0
    ra.set_deterministic(True)
    return nfeat, dt, "reference", "oracle/_ref/libmcs_ref.so: the reference's own mdBRIEFextractorOct + cORBmatcher compiled in place"


def make_scene(cfg_id, cfg, cams, cam_id, feats0, F, seed):
    """synthetic matching targets of configs 3 / 4 (SURVEY.md 8d), built from the descriptors of a first extracted frame"""
    rng = np.random.default_rng(seed)
    k0, d0, m0 = feats0

    def flips(src, kmax):
        out = src.copy()
        nb = rng.integers(0, kmax + 1, len(out))
        for i in np.flatnonzero(nb):
            for b in rng.choice(256, nb[i], replace=False):
                out[i, b // 8] ^= 1 << (b % 8)
        return out
    if cfg_id == 3:
        n = cfg["n_mappoints"]
        src = rng.integers(0, len(k0), n)
        # map points on a sphere shell around the rig; the F frame poses drift slowly
        v = rng.normal(size=(n, 3))
        world = v / np.linalg.norm(v, axis=1, keepdims=True) * rng.uniform(3.0, 9.0, (n, 1))
        normal = -world / np.linalg.norm(world, axis=1, keepdims=True)
        dist = np.linalg.norm(world, axis=1)
        poses = np.tile(np.eye(4), (F, 1, 1))
        poses[:, :3, 3] = np.cumsum(rng.normal(0, 0.01, (F, 3)), axis=0)
        return dict(world=world, normal=normal, min_d=dist * 0.5, max_d=dist * 2.0, poses=poses, mp_desc=flips(d0[src], 40), mp_dmask=m0[src].copy())
    n = cfg["n_db"]
    db = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    plant = rng.choice(n, len(k0), replace=False)
    db[plant] = flips(d0, 30)
    db_mask = (rng.random((n, 256)) < 0.85)
    db_mask = np.packbits(db_mask, axis=1, bitorder="little")
    return dict(db=db, db_mask=db_mask)


def run_reference(args, cfg_id, cfg):
    """--impl reference: the reference's CPU implementation of the path on the host cores, bounded sample per step."""
    from multicol_slam_b200 import synth
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cams = rig_cams(cfg)
    cam_ids = list(range(cfg["n_cams"])) if cfg_id == 2 else [0]
    masks = np.stack([synth.mirror_mask(c) for c in cams])
    cores = usable_cores()
    if cfg_id == 2:
        frames = max(2, min(max(args.ref_frames, 2 * cores // 3), 128))
    else:
        frames = 2
    images = make_stream(cams, cam_ids, frames, 1000)
    scene = None
    if cfg_id != 2:
        import ref_mcs_api as ra
        if not ra.available():
            print(json.dumps({"impl": "reference", "unavailable": "configs 3/4 need oracle/_ref (the reference's own matcher)"}))
            return
        f0 = ra.RefExtractor(nfeatures=cfg["nfeatures"], do_dbrief=True, learn_masks=True).extract(images[0, 0], masks[0], cams[0])
        scene = make_scene(cfg_id, cfg, cams, 0, f0, frames, 7)
        if cfg_id == 3:
            scene["views"] = host_views(cfg, cams[0], masks[0], scene, frames)
    nfeat, dt, kind, what = 0, 0.0, "", ""
    cpu_arm(cfg_id, cfg, cams, masks, images[:max(1, min(len(images), 2))], cores, scene)      # warms allocators / page faults
    for _ in range(args.steps):
        n, t, kind, what = cpu_arm(cfg_id, cfg, cams, masks, images, cores, scene)
        nfeat += n
        dt += t
    val = nfeat / dt / 1e6
    sample = f"{frames} frames x {len(cam_ids)} cams per step, {args.steps} steps, {cores} threads"
    print(json.dumps({"impl": "reference", "metric": "Mfeatures/s extract+match", "value": val, "unit": "Mfeatures/s",
                      "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                      "config": bench_config(cfg_id, cfg), "run": bench_run(cfg, frames, len(cam_ids), 1, sample=sample),
                      "cpu_baseline": {"value": val, "unit": "Mfeatures/s", "cores": cores, "logical_cpus": os.cpu_count(), "kind": kind,
                                       "what": what, "sample": sample},
                      "e2e": {"value": val, "unit": "Mfeatures/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def bench_config(cfg_id, cfg):
    """what is measured -- identical in the GPU arm and in the reference arm; how much of it one step covers is in `run`"""
    return {"workload": cfg["workload"], "baseline_config": cfg_id, "nfeatures": cfg["nfeatures"], "image": f"{cfg['w']}x{cfg['h']}",
            "rig_cameras": cfg["n_cams"], "pyramid": "8 levels x 1.2", "descriptor": "mdBRIEF-256 + masks"}


def bench_run(cfg, frames, cams_per_gpu, world, **extra):
    r = {"frames_per_step_per_gpu": frames, "images_per_step_per_gpu": frames * cams_per_gpu,
         "parallelism": (f"stream-sharded x{world}" if cfg["sharding"] == "stream" else f"camera-per-GPU x{world}") +
                        (", 1 ncclAllGather of the packed feature buffer per step (library call, own stream)" if world > 1 else "")}
    r.update(extra)
    return r


def host_views(cfg, cam, mask, scene, F):
    """isInFrustum fields of the 50k map points for the F frame poses of one camera, evaluated by the oracle's projection
    (CPU arm of config 3; the GPU arm uses mcs_project_mappoints)"""
    import oracle_api as oa
    sf = np.array([float(np.float32(1.2)) ** l for l in range(NLEVELS)])
    out = []
    for f in range(F):
        mt = scene["poses"][f]
        inv = np.linalg.inv(mt)
        iv, lv, px, py, vc = oa.project_mappoints(inv[None], mt[None], [cam], mask[None], scene["world"], scene["normal"], scene["min_d"],
                                                  scene["max_d"], sf)
        out.append((iv, lv, px, py, vc))
    return out


def dump_outputs(path, out, nmatches, matches12):
    """--dump-outputs: out = the packed feature views of the last timed step; nmatches [B] and matches12 (config 2 and 4: [B, cap]
    per image, config 3: one index per keypoint of the frame view) as the step's matcher returned them.  Rows past an image's
    feature count are not outputs (the buffer keeps whatever an earlier step left there) and are written as zeros / -1."""
    from multicol_slam_b200.ctypes_defs import KEYPOINT_DTYPE
    d = pathlib.Path(path)
    d.mkdir(parents=True, exist_ok=True)
    counts = out["counts"].cpu().numpy()
    B, cap = out["kps"].shape[:2]
    pick = np.sort(np.random.default_rng(0).choice(B, min(B, DUMP_IMAGES), replace=False))
    valid = (np.arange(cap)[None, :] < counts[pick, None])[..., None]
    kps = out["kps"].cpu().numpy()[pick].view(KEYPOINT_DTYPE)[..., 0]
    arrays = {"counts": counts, "nmatches": np.asarray(nmatches).reshape(-1), "sample_images": pick,
              "keypoints": np.where(valid, np.stack([kps[f].astype(np.float64) for f in KEYPOINT_DTYPE.names], -1), 0.0),
              "descriptors": np.where(valid, out["desc"].cpu().numpy()[pick], 0).astype(np.float32),
              "descriptor_masks": np.where(valid, out["dmask"].cpu().numpy()[pick], 0).astype(np.float32)}
    m12 = np.asarray(matches12)
    arrays["matches12"] = np.where(valid[..., 0], m12.reshape(B, cap)[pick], -1) if m12.size == B * cap else m12
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", np.asarray(a, np.float32 if a.dtype == np.float32 else np.float64))


# ---------------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4], help="BASELINE.json configuration (2 = headline)")
    ap.add_argument("--frames", type=int, default=0, help="multi-camera frames per step and per GPU (0 = the config's default)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-frames", type=int, default=8, help="frames per step of the CPU reference arm (config 2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    cfg_id, cfg = args.config, CONFIGS[args.config]
    if args.impl == "reference":
        return run_reference(args, cfg_id, cfg)

    import torch
    import torch.distributed as dist
    import multicol_slam_b200.api as api
    from multicol_slam_b200 import rig, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert api.device_count() > 0, "no sm_100 device"
    F = args.frames or cfg["frames"]
    W, H, NF = cfg["w"], cfg["h"], cfg["nfeatures"]
    cams = rig_cams(cfg)
    masks = np.stack([synth.mirror_mask(c) for c in cams])
    if cfg["sharding"] == "stream":          # every rank: all cameras, its own temporal chunk of the stream
        cam_ids = list(range(cfg["n_cams"]))
        images = make_stream(cams, cam_ids, F, 1000 + 97 * rank)                # [F, C, H, W]
    else:                                      # camera c -> GPU c mod G: this rank's camera of the rig
        assert world <= cfg["n_cams"], "more GPUs than cameras in the rig"
        cam_ids = [rank % cfg["n_cams"]]
        images = make_stream(cams, cam_ids, F, 1000)
    NC = len(cam_ids)
    B = F * NC
    coi = np.tile(np.asarray(cam_ids, np.int32), F)
    host_images = torch.from_numpy(images).pin_memory()
    PITCH = (W + 63) // 64 * 64                                                # 16-byte aligned rows: K1 stages by TMA
    dev_images = torch.zeros((B, H, PITCH), dtype=torch.uint8, device=dev)
    dev_images[:, :, :W] = host_images.to(dev, non_blocking=True).view(B, H, W)
    # L2 rule: a step must not find its inputs in the 126 MB L2 from the step before.  Config 2 streams 139 MB of images per step
    # (larger than L2 by itself); the small rig configs rotate through enough copies of their input that > 140 MB of other
    # input is read before a copy comes round again.
    in_bytes = B * H * PITCH
    n_rot = 1 if in_bytes > 130e6 else int(np.ceil(140e6 / in_bytes)) + 1
    rot_images = [dev_images] + [dev_images.clone() for _ in range(n_rot - 1)]

    ex = api.mdBRIEFextractorOct(nfeatures=NF, nlevels=NLEVELS, do_dBrief=True, learnMasks=True)
    cap, ds = ex.capacity, 32
    m = api.cORBmatcher(0.9, False, ds, True)
    K = int(os.environ.get("MCS_BENCH_K", "4"))      # candidates kept per query by M2 (the replay is exact for any K; K sets how often it rescans)
    pbytes = rig.packed_layout(B, cap, ds)[1]
    packed = [torch.zeros(pbytes, dtype=torch.uint8, device=dev) for _ in range(2)]       # double buffered: the gather of step i
    views = [ex.packed_views(p, B) for p in packed]                                       # overlaps the extraction of step i+1
    gathered = [torch.empty(world * pbytes, dtype=torch.uint8, device=dev) for _ in range(2)] if world > 1 else None
    comm = rig.Communicator(dev) if world > 1 else None
    stream, cstream, mstream = torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    ev_feat = [torch.cuda.Event() for _ in range(2)]
    ev_gath = [torch.cuda.Event() for _ in range(2)]
    ev_match = [torch.cuda.Event() for _ in range(2)]
    midx = torch.empty((B, cap, K), dtype=torch.int32, device=dev)
    mdist = torch.empty((B, cap, K), dtype=torch.int32, device=dev)
    m12 = torch.empty((B, cap), dtype=torch.int32, device=dev)
    nmat = torch.empty(B, dtype=torch.int32, device=dev)
    redo = torch.zeros(B, dtype=torch.int32, device=dev)
    m12b, nmatb = torch.empty_like(m12), torch.empty_like(nmat)
    sf = np.array([float(np.float32(1.2)) ** l for l in range(NLEVELS)])
    stats = {"matches": 0}
    last = {}               # matcher outputs of configs 3 / 4 in the last step (--dump-outputs)

    # matching targets of configs 3 / 4, built from the features of a first extraction
    scene = None
    if cfg_id != 2:
        with torch.cuda.stream(stream):
            o = ex.extract_batch_packed_device(dev_images, masks, cams, coi, packed[0], stream=stream, width=W)
        torch.cuda.synchronize(dev)
        n0 = int(o["counts"][0].item())
        f0 = (o["kps"][0, :n0].cpu().numpy().view(api.KEYPOINT_DTYPE).reshape(-1), o["desc"][0, :n0].cpu().numpy(), o["dmask"][0, :n0].cpu().numpy())
        scene = make_scene(cfg_id, cfg, cams, cam_ids[0], f0, F, 7)
        if cfg_id == 4:
            scene["db_t"] = torch.from_numpy(scene["db"]).to(dev)
            scene["dbm_t"] = torch.from_numpy(scene["db_mask"]).to(dev)
        else:
            scene["mtmc"] = np.ascontiguousarray(scene["poses"])
            scene["mtmc_inv"] = np.ascontiguousarray(np.stack([np.linalg.inv(p) for p in scene["poses"]]))
            scene["masks_f"] = np.ascontiguousarray(np.broadcast_to(masks[cam_ids[0]], (F,) + masks[cam_ids[0]].shape))
    h_feat = None
    if cfg_id == 3:         # host copies of the rank's own features for the projection search (window search + host replay)
        h_feat = dict(counts=torch.empty(B, dtype=torch.int32).pin_memory(), kps=torch.empty((B, cap, 7), dtype=torch.int32).pin_memory(),
                      desc=torch.empty((B, cap, ds), dtype=torch.uint8).pin_memory(), dmask=torch.empty((B, cap, ds), dtype=torch.uint8).pin_memory())

    def match_config3(v):
        t_m3 = time.perf_counter()
        for k in h_feat:
            h_feat[k].copy_(v[k], non_blocking=True)
        stream.synchronize()
        t_a = time.perf_counter()
        counts = h_feat["counts"].numpy()
        kps = h_feat["kps"].numpy().view(api.KEYPOINT_DTYPE).reshape(B, cap)
        # the F frames of this camera as the F "cameras" of one frame view: one projection launch, one window search, one replay
        keys = np.concatenate([kps[f, :counts[f]] for f in range(F)])
        key_cam = np.concatenate([np.full(counts[f], f, np.int32) for f in range(F)])
        desc = np.concatenate([h_feat["desc"].numpy()[f, :counts[f]] for f in range(F)])
        dmask = np.concatenate([h_feat["dmask"].numpy()[f, :counts[f]] for f in range(F)])
        Fr = api.Frame(keys, key_cam, desc, dmask, [(W, H)] * F, sf)
        t_b = time.perf_counter()
        iv, lv, px, py, vc = api.project_mappoints(scene["mtmc_inv"], scene["mtmc"], [cams[cam_ids[0]]] * F, scene["masks_f"], scene["world"],
                                                   scene["normal"], scene["min_d"], scene["max_d"], sf)
        t_c = time.perf_counter()
        mp = api.MapPoints(np.zeros(len(scene["world"]), np.uint8), iv, lv, px, py, vc, scene["mp_desc"], scene["mp_dmask"])
        mt = api.cORBmatcher(0.8, False, ds, True)
        n, last["matches12"] = mt.SearchByProjection(Fr, mp, 3.0)
        t_d = time.perf_counter()
        last["nmatches"] = [n]
        stats["matches"] = n
        stats["match_call_ms"] = (t_d - t_m3) * 1e3
        stats["parts_ms"] = {"wait_extract+d2h": (t_a - t_m3) * 1e3, "frame_view": (t_b - t_a) * 1e3, "mcs_project_mappoints": (t_c - t_b) * 1e3,
                             "mcs_search_by_projection": (t_d - t_c) * 1e3}

    def match_config4(v):
        t_m = time.perf_counter()
        counts = v["counts"].cpu().numpy()
        valid1 = (np.arange(cap)[None, :] < counts[:, None]).astype(np.uint8).reshape(-1)
        # every key frame of the batch against the database as its own SearchByBoW(KF1, KF2): independent "already matched" state
        # per frame, the K-best lists of all frames from one launch
        nms, last["matches12"] = api.match_bruteforce_batch_device(v["desc"].view(B * cap, ds), v["dmask"].view(B * cap, ds), valid1, np.arange(B + 1) * cap,
                                                   scene["db_t"], scene["dbm_t"], None, m.TH_LOW_, 0.9, stream=stream)
        last["nmatches"] = nms
        stats["matches"] = int(nms.sum())
        stats["match_call_ms"] = (time.perf_counter() - t_m) * 1e3      # includes waiting for this step's extraction (the counts read)

    step_no = [0]

    def step():
        i = step_no[0] & 1
        step_no[0] += 1
        if world > 1:
            stream.wait_event(ev_gath[i])                         # the gather that last read this buffer has finished
        stream.wait_event(ev_match[i])                            # ... and so has the matching of two steps ago
        v = ex.extract_batch_packed_device(rot_images[(step_no[0] - 1) % n_rot], masks, cams, coi, packed[i], stream=stream, width=W)
        ev_feat[i].record(stream)
        if world > 1:                                             # one ncclAllGather, on its own stream behind the features
            cstream.wait_event(ev_feat[i])
            comm.allgather(packed[i], gathered[i], cstream)
            ev_gath[i].record(cstream)
        if cfg_id == 2:
            # matching of step i on its own stream: the XU-bound popcount kernel and the latency-bound greedy replay (one CTA per
            # image, mostly a single warp walking the queries in order) share the SMs with the extraction of step i + 1
            mstream.wait_event(ev_feat[i])
            api.match_stream_greedy_device(v["desc"], v["dmask"], v["counts"], F, NC, m.TH_LOW_, 0.9, out=(m12, nmat), stream=mstream)
            ev_match[i].record(mstream)
        elif cfg_id == 3:
            match_config3(v)
        else:
            match_config4(v)
        return v

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    with torch.cuda.stream(stream):
        for _ in range(max(args.warmup, 3)):
            out = step()
        barrier()
        # ---- per-kernel timings (separate pass with event recording on; not part of the timed region) ----
        ex.set_profiling(True)
        k_ms = np.zeros(3)
        for _ in range(3):
            torch.cuda.synchronize(dev)                           # stage times without the overlapped matching of the step before
            out = step()
            torch.cuda.synchronize(dev)
            k_ms += np.array(ex.get_timings())
        k_ms /= 3
        ex.set_profiling(False)
        match_ms, replay_ms = None, None
        if cfg_id == 2:
            # the two kernels of mcs_match_stream_greedy_device timed apart (same bound, same K as the fused call uses)
            e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            e[0].record(stream)
            api.match_stream_greedy_device(out["desc"], out["dmask"], out["counts"], F, NC, m.TH_LOW_, 0.9, out=(m12, nmat), stream=stream)
            e[1].record(stream)
            api.match_stream_device(out["desc"], out["dmask"], out["counts"], F, NC, K=K, out=(midx, mdist), stream=stream)
            e[2].record(stream)
            api.match_stream_replay_device(midx, mdist, out["counts"], out["desc"], out["dmask"], F, NC, m.TH_LOW_, 0.9, out=(m12b, nmatb, redo), stream=stream)
            e[3].record(stream)
            torch.cuda.synchronize(dev)
            match_ms, replay_ms = e[0].elapsed_time(e[1]), None
            unbounded_ms = (e[1].elapsed_time(e[2]), e[2].elapsed_time(e[3]))
            assert torch.equal(m12, m12b) and torch.equal(nmat, nmatb), "bounded and unbounded K-best lists disagree on the greedy matches"
        # ---- timed region: exactly K steps, device resident ----
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            out = step()
        if world > 1:
            stream.wait_stream(cstream)                           # the last gathers belong to the timed region
        stream.wait_stream(mstream)                               # ... and so does the matching of the last step
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:          # before the e2e and roofline passes below reuse the buffers
        if cfg_id == 2:
            dump_outputs(args.dump_outputs, out, nmat.cpu().numpy(), m12.cpu().numpy())
        else:
            dump_outputs(args.dump_outputs, out, last["nmatches"], last["matches12"])
    feats_rank = int(out["counts"].sum().item())
    redo_n = int(redo.sum().item()) if cfg_id == 2 else 0
    matches_rank = int(nmat.sum().item()) if cfg_id == 2 else stats["matches"]
    t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
    feats = torch.tensor([feats_rank], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(feats, op=dist.ReduceOp.SUM)
    ms_per_step = t_ms.item() / args.steps
    value = feats.item() / (ms_per_step * 1e-3) / 1e6

    # ---- e2e: the public API with pinned HOST buffers, H2D + kernels + (allgather) + D2H inside the timed region ----
    from multicol_slam_b200.ctypes_defs import KEYPOINT_DTYPE
    e2e_steps = max(1, min(args.steps, 5))
    if cfg_id == 2:
        h_out = dict(kps=torch.empty((B, cap, 7), dtype=torch.int32).pin_memory(), desc=torch.empty((B, cap, ds), dtype=torch.uint8).pin_memory(),
                     dmask=torch.empty((B, cap, ds), dtype=torch.uint8).pin_memory(), counts=torch.empty(B, dtype=torch.int32).pin_memory(),
                     match_idx=torch.empty((B, cap, K), dtype=torch.int32).pin_memory(),
                     match_dist=torch.empty((B, cap, K), dtype=torch.int32).pin_memory())
        h_out.update(matches12=torch.empty((B, cap), dtype=torch.int32).pin_memory(), nmatches=torch.empty(B, dtype=torch.int32).pin_memory(),
                     redo=torch.empty(B, dtype=torch.int32).pin_memory())
        np_out = {k: v.numpy() for k, v in h_out.items()}
        np_out["kps"] = np_out["kps"].view(KEYPOINT_DTYPE).reshape(B, cap)
        himg = host_images.numpy()

        def e2e_step():
            # mcs_extract_match_stream_packed: chunked H2D | K1..K3 | K-best matching + greedy acceptance | D2H pipeline over host
            # buffers; at N > 1 the allgather of the packed buffer the call left on the GPU follows
            ex.extract_match_stream(himg, masks, cams, K=K, out=np_out, packed_t=packed[0], greedy=(m.TH_LOW_, 0.9))
            if world > 1:
                comm.allgather(packed[0], gathered[0], stream)
                stream.synchronize()
        h2d = int(himg.nbytes + masks.nbytes)
        d2h = int(sum(v.numel() * v.element_size() for v in h_out.values()))
        e2e_api = "mcs_extract_match_stream_packed (C ABI, pinned host buffers; K-best lists + greedy acceptance on the device)" + (" + mcs_allgather_features" if world > 1 else "")
    else:
        h_packed = torch.empty(pbytes, dtype=torch.uint8).pin_memory()

        def e2e_step():
            with torch.cuda.stream(stream):
                rot_images[step_no[0] % n_rot][:, :, :W].copy_(host_images.view(B, H, W), non_blocking=True)     # the buffer this step reads
                v = step()
                h_packed.copy_(packed[(step_no[0] - 1) & 1], non_blocking=True)
                if world > 1:
                    stream.wait_stream(cstream)
            stream.synchronize()
        h2d = int(host_images.numel() + masks.nbytes)
        d2h = int(pbytes)
        e2e_api = "pinned host images -> mcs_extract_batch_packed_device -> (mcs_allgather_features) -> config matcher -> packed features to the host"
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_val = feats.item() / (e2e_t.item() / e2e_steps) / 1e6
    if cfg_id == 2:
        assert int(np_out["counts"].sum()) == feats_rank, "e2e and device-resident runs disagree"
        assert int(np_out["nmatches"].sum()) == matches_rank, "e2e and device-resident greedy matches disagree"

    # ---- single-frame latency of the reference-shaped call: one multi-camera frame through mcs_extract_batch (host in/out) ----
    lat_ms, lat_graph = None, None
    if rank == 0 and cfg_id == 2:
        # the C-ABI call itself (arguments prepared once, as the C++ caller has them): pageable host buffers in and out
        import ctypes as C
        from multicol_slam_b200.ctypes_defs import KEYPOINT_DTYPE, Ocam
        two = [np.ascontiguousarray(host_images.numpy()[f]) for f in (0, 1)]
        cap1, ds1 = ex.info.capacity, ex.info.desc_size
        o_k, o_d = np.zeros((NC, cap1), KEYPOINT_DTYPE), np.zeros((NC, cap1, ds1), np.uint8)
        o_m, o_c = np.zeros((NC, cap1, ds1), np.uint8), np.zeros(NC, np.int32)
        ocs = (Ocam * NC)(*[api.as_ocam(c) for c in cams])
        coi1 = np.arange(NC, dtype=np.int32)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        def one_frame(img):
            rc = api.lib().mcs_extract_batch(ex._h, NC, vp(img), W, H, W, vp(masks), ocs, NC, vp(coi1), vp(o_k), vp(o_d), vp(o_m), vp(o_c), cap1)
            assert rc == 0, api.lib().mcs_last_error()
        for i in range(3):
            one_frame(two[i & 1])
        r0 = ex.graph_replays()
        t0 = time.perf_counter()
        for i in range(50):
            one_frame(two[i & 1])
        lat_ms = (time.perf_counter() - t0) / 50 * 1e3
        lat_graph = ex.graph_replays() - r0
    if rank == 0:
        # ---- roofline of K1 (fused pyramid + blur + FAST), algorithmic bytes per SURVEY 8d / DESIGN.md ----
        ex.extract_batch_packed_device(dev_images, masks, cams, coi, packed[0], stream=stream, width=W)
        torch.cuda.synchronize(dev)
        P = sum(int(ex.debug_read(l, 0).size) for l in range(NLEVELS))        # sum of pyramid pixels (1 120 256 at 754x480)
        n_raw = sum(len(ex.debug_read(l, 3, image_index=0)) for l in range(NLEVELS))
        alg_bytes_img = P + 8 * n_raw                                          # read L0 once + write L1..7 + 8 B / raw corner
        peak, peak_src = hbm_peak()
        achieved = alg_bytes_img * B / (k_ms[0] * 1e-3) / 1e9                  # all 8 level launches together
        achieved_blur = (alg_bytes_img + P) * B / (k_ms[0] * 1e-3) / 1e9       # counting the fused blurred output (SURVEY 8d: +P)
        traffic, traffic_note = None, "no committed ncu capture found"
        tp = ROOT / "profiles" / "k1_traffic.json"
        if tp.exists():        # DRAM bytes of K1 from the committed `ncu --set full` capture, per image; scaled to this batch
            tj = json.loads(tp.read_text())
            traffic = tj["dram_bytes_per_image"] * B / NLEVELS
            traffic_note = f"bytes per launch (average of the 8 level launches), from {tj['source']} ({tj.get('images', '?')} images in the capture)"
        roof = {"kernel": "pyr_fast_kernel (K1, 8 launches/step, one per level)", "bound": "hbm", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note,
                "achieved_counting_blurred_output": achieved_blur, "frac_counting_blurred_output": achieved_blur / peak,
                "algorithmic_bytes_per_launch_avg": alg_bytes_img * B / NLEVELS, "peak_source": peak_src,
                "algorithmic_bytes_per_camera_frame": alg_bytes_img, "ms_per_launch_avg": k_ms[0] / NLEVELS,
                "stage_ms": {"k1_pyr_blur_fast": k_ms[0], "k2_octree": k_ms[1], "k3_angle_describe": k_ms[2], "m2_match_greedy": match_ms}}
        n_feat = int(feats_rank)
        other = {"k3_describe_kernel": {"bound": "fp32 issue (tier 1) / FP64 (tiers 2, 3); see profiles/", "algorithmic_GB_per_s":
                                        n_feat * (845 + 51 * 51 + 28 + 64) / (k_ms[2] * 1e-3) / 1e9},
                 "k2_octree_kernel": {"bound": "latency (one CTA per image-level, serial passes)", "ms": k_ms[1]}}
        if cfg_id == 2 and match_ms:
            pairs = float((B - NC) if B > NC else 0) * NF * NF
            sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
            popc_rate = 148 * 16 * sm_mhz * 1e6                   # POPC issues on the XU pipe: 16 lanes / clk / SM (DESIGN.md section 7)
            # mcs_match_stream_greedy_device = K-best lists (entries beyond the relevance bound of the acceptance rule left out) +
            # greedy replay; timed next to it: the plain K-best lists and the replay over them
            other["m2_match_stream_greedy"] = {
                "bound": "integer issue: POPC on the XU pipe + LOP3 on the ALU pipe (lists); latency of the ordered walk (replay)", "ms": match_ms,
                "lists_ms": unbounded_ms[0], "replay_ms": unbounded_ms[1],
                "pair_distances_per_s": pairs / (unbounded_ms[0] * 1e-3), "popc_per_masked_pair": 9,
                "popc_issue_frac": pairs * 9 / (unbounded_ms[0] * 1e-3) / popc_rate,
                "algorithmic_GB_per_s": ((B - NC) * (64 * 2 * NF + 12 * NF)) / (unbounded_ms[0] * 1e-3) / 1e9}
        roof["other_stages"] = other
        cpu = None
        if not args.no_cpu_baseline:
            cores = usable_cores()
            if cfg_id == 2:
                cf = int(min(F, max(4, 2 * cores // NC)))
                sample_imgs = images[:cf]
                cscene = None
            else:
                cf = 2
                sample_imgs = images[:cf]
                cscene = dict(scene)
                if cfg_id == 3:
                    cscene["views"] = host_views(cfg, cams[cam_ids[0]], masks[cam_ids[0]], scene, cf)
            ccams = cams if cfg_id == 2 else [cams[cam_ids[0]]]
            cmasks = masks if cfg_id == 2 else masks[cam_ids[0]][None]
            cpu_arm(cfg_id, cfg, ccams, cmasks, sample_imgs[:2], cores, cscene)          # warm-up
            nf_c, dt_c, kind, what = cpu_arm(cfg_id, cfg, ccams, cmasks, sample_imgs, cores, cscene)
            cpu = {"value": nf_c / dt_c / 1e6, "unit": "Mfeatures/s", "cores": cores, "logical_cpus": os.cpu_count(), "kind": kind, "what": what,
                   "sample": f"{cf} frames x {len(ccams)} cams of the same workload, {dt_c:.1f} s wall on {cores} threads, after one warm-up pass"}
        launches = NLEVELS + 2 + (2 if cfg_id == 2 else 0)
        print(json.dumps({
            "metric": "Mfeatures/s extract+match", "value": value, "unit": "Mfeatures/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": bench_config(cfg_id, cfg),
            "run": bench_run(cfg, F, NC, world, features_per_step=int(feats.item()), matches_per_step_rank0=matches_rank, matcher_stats={k: v for k, v in stats.items() if k != 'matches'},
                             greedy_replay_redo_images=redo_n,
                             l2=(f"inputs {in_bytes / 1e6:.0f} MB per step, larger than the 126 MB L2" if n_rot == 1 else
                                 f"inputs {in_bytes / 1e6:.0f} MB per step, rotated through {n_rot} copies ({n_rot * in_bytes / 1e6:.0f} MB > 126 MB L2) so no step "
                                 f"finds its input cached") + f"; pyramid + blurred pyramid written and re-read within a step: {2 * P * B / 1e6:.0f} MB"),
            "e2e": {"value": e2e_val, "unit": "Mfeatures/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "api": e2e_api, "steps": e2e_steps},
            "gpu_launches": args.steps * launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
            "single_frame_latency_ms": {"value": lat_ms, "what": "one multi-camera frame through mcs_extract_batch (C ABI, pageable host buffers in and out), mean of 50 alternating frames", "cuda_graph_replays": lat_graph}}))
    if comm is not None:
        torch.cuda.synchronize(dev)
        comm.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
