"""Key-frame database benchmark: per-query time of DetectLoopCandidates / DetectRelocalisationCandidates on the GPU
(mcs_kfdb_*) and of the reference's own cMultiKeyFrameDatabase on the host cores (oracle/_ref/libkfdb_ref.so), on maps of
N = 250 / 1000 / 4000 key frames.

A key frame is a 3-camera Lafida frame, 2000 features per camera (mdBRIEF, learned masks), its BowVector from
ORBVocabulary.transform(levelsup 4) on the GPU with the shipped 6999-word vocabulary.  The trajectory first visits 0.7 N places,
then revisits earlier ones; a place's three images are crops of synth.texture_stream, so a revisit sees the images of the first
visit.  covis row i = the key frames at the same place, then the temporal neighbours (the ten best covisibility key frames).

Reported per map size:
  gpu      wall time of the synchronous C call per query (host clock around the call, which ends in a stream synchronise),
           and the summed device time of its kfdb_* kernels (torch.profiler, CUDA activities, in a separate pass);
  ref      wall time per query of the reference database on the host, over a sample of the same queries, run against a
           second GPU database fed the identical call sequence: the candidate lists must be identical (asserted);
  counts   from the shapes: inverted-file entries a query visits, key frames above minCommonWords (pairs scored) and merge
           steps of those scores (query words + key-frame words per pair).
Usage: python tools/kfdb_bench.py [--sizes 250,1000,4000] [--queries 50] [--ref-sample 10] [--out profiles/kfdb_bench_b200.json]"""
import argparse
import json
import pathlib
import subprocess
import sys
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))

import multicol_slam_b200.api as api  # noqa: E402
from multicol_slam_b200 import synth  # noqa: E402

PLACES_PER_TEXTURE = 500


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def place_bows(n_places, voc):
    """BowVector of every place: 3 cameras x 2000 features, the descriptors of the three cameras concatenated"""
    cams = synth.lafida_cams()
    masks = np.stack([synth.mirror_mask(c) for c in cams])
    ex = api.mdBRIEFextractorOct(nfeatures=2000, do_dBrief=True, learnMasks=True)
    out = []
    for t0 in range(0, n_places, PLACES_PER_TEXTURE):
        n = min(PLACES_PER_TEXTURE, n_places - t0)
        streams = [synth.texture_stream(cams[c], n, seed=1000 * c + t0 // PLACES_PER_TEXTURE) for c in range(3)]
        for b0 in range(0, n, 64):
            b1 = min(n, b0 + 64)
            imgs = np.concatenate([np.stack([streams[c][t] for c in range(3)]) for t in range(b0, b1)])
            coi = np.tile(np.arange(3, dtype=np.int32), b1 - b0)
            _, desc, _, counts = ex.extract_batch(imgs, masks, cams, coi)
            for k in range(b1 - b0):
                d = np.concatenate([desc[3 * k + c, :counts[3 * k + c]] for c in range(3)])
                out.append(voc.transform(d, 4)[:2])
    return out


def trajectory(n_kf):
    first = int(n_kf * 0.7)
    place = np.array([i if i < first else (i - first) * 3 % first for i in range(n_kf)])
    cv = -np.ones((n_kf, 10), np.int64)
    by_place = {}
    for i, p in enumerate(place):
        by_place.setdefault(int(p), []).append(i)
    for i in range(n_kf):
        same = [j for j in by_place[int(place[i])] if j != i]
        near = sorted((j for j in range(max(0, i - 6), min(n_kf, i + 7)) if j != i), key=lambda j: (abs(j - i), j))
        row = (same + [j for j in near if j not in same])[:10]
        cv[i, :len(row)] = row
    return place, first, cv


def queries(n_kf, n_q, seed):
    rng = np.random.default_rng(seed)
    return [(int(rng.integers(0, n_kf)), int(rng.integers(0, n_kf))) for _ in range(n_q)]


def counts(bows_of_kf, n_words, qs):
    """algorithmic counts from the shapes, per query: list entries visited, pairs scored, merge steps of those pairs"""
    n = len(bows_of_kf)
    occ = np.zeros((n, n_words), np.bool_)
    for i, (w, _) in enumerate(bows_of_kf):
        occ[i, w] = True
    list_len = occ.sum(0)
    out = []
    for q in qs:
        w = bows_of_kf[q][0]
        shared = occ[:, w].sum(1)
        scored = shared > int(shared.max() * 0.8)
        out.append((int(list_len[w].sum()), int(scored.sum()),
                    int(scored.sum() * len(w) + sum(len(bows_of_kf[j][0]) for j in np.nonzero(scored)[0]))))
    return np.array(out, np.float64).mean(0).tolist()


def kernel_time_per_query(db, cv, bows_of_kf, qs, qid0):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        for k, (q, f) in enumerate(qs):
            conn = [int(j) for j in cv[q] if j >= 0 and abs(j - q) <= 3]
            db.DetectLoopCandidates(q, bows_of_kf[q], conn, cv, 0.0)
            db.DetectRelocalisationCandidates(qid0 + k, bows_of_kf[f], cv)
    per = {}
    for e in prof.events():
        if e.device_type.name == "CUDA" and "kfdb_" in e.name:
            name = e.name.split("(")[0].replace("void ", "").replace("mcs::", "")
            us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            per[name] = per.get(name, 0.0) + us
    total_us = sum(per.values())
    return total_us / (2 * len(qs)), {k: v / (2 * len(qs)) for k, v in sorted(per.items())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="250,1000,4000")
    ap.add_argument("--queries", type=int, default=50)
    ap.add_argument("--ref-sample", type=int, default=10)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "kfdb_bench_b200.json"))
    a = ap.parse_args()
    if api.device_count() < 1:
        raise SystemExit("kfdb_bench needs a CUDA device")
    import ref_kfdb_api
    if not ref_kfdb_api.available():
        raise SystemExit("oracle/_ref/libkfdb_ref.so is missing (make -C oracle -f kfdb.mk ref where the reference sources are)")
    vz = np.load(ROOT / "tests" / "golden" / "voc_small_9_6.npz")
    voc = api.ORBVocabulary(vz)
    sizes = [int(s) for s in a.sizes.split(",")]
    res = {"gpu": gpu_info(), "vocabulary_words": voc.size(), "scoring": voc.scoring, "sizes": []}
    t = time.perf_counter()
    pbows = place_bows(int(max(sizes) * 0.7), voc)
    res["map_build_s"] = time.perf_counter() - t
    for n in sizes:
        place, first, cv = trajectory(n)
        kb = [pbows[int(p)] for p in place]
        db = api.KeyFrameDatabase(voc)
        t = time.perf_counter()
        for i in range(n):
            db.add(i, kb[i])
        add_ms = (time.perf_counter() - t) * 1e3 / n
        qs = queries(n, a.queries, seed=n)
        for q, f in qs[:5]:                                  # warm-up of every launch shape
            db.DetectRelocalisationCandidates(900_000 + q, kb[f], cv)
        loop_ms, reloc_ms, n_cand = [], [], []
        for k, (q, f) in enumerate(qs):
            conn = [int(j) for j in cv[q] if j >= 0 and abs(j - q) <= 3]
            t = time.perf_counter()
            c = db.DetectLoopCandidates(q, kb[q], conn, cv, 0.0)
            loop_ms.append((time.perf_counter() - t) * 1e3)
            t = time.perf_counter()
            r = db.DetectRelocalisationCandidates(1_000_000 + k, kb[f], cv)
            reloc_ms.append((time.perf_counter() - t) * 1e3)
            n_cand.append((len(c), len(r)))
        dev_us, per_kernel = kernel_time_per_query(db, cv, kb, qs[:20], 2_000_000)
        # reference arm: the same call sequence into the reference and into a fresh GPU database, lists compared
        ref, gdb = ref_kfdb_api.RefKeyFrameDatabase(voc.scoring, voc.weighting), api.KeyFrameDatabase(voc)
        for i in range(n):
            ref.add(i, kb[i]); gdb.add(i, kb[i])
        ref_loop, ref_reloc = [], []
        for k, (q, f) in enumerate(qs[:a.ref_sample]):
            conn = [int(j) for j in cv[q] if j >= 0 and abs(j - q) <= 3]
            t = time.perf_counter()
            rl = ref.DetectLoopCandidates(q, kb[q], conn, cv, 0.0)
            ref_loop.append((time.perf_counter() - t) * 1e3)
            t = time.perf_counter()
            rr = ref.DetectRelocalisationCandidates(1_000_000 + k, kb[f], cv)
            ref_reloc.append((time.perf_counter() - t) * 1e3)
            assert np.array_equal(rl, gdb.DetectLoopCandidates(q, kb[q], conn, cv, 0.0)), ("loop", n, k)
            assert np.array_equal(rr, gdb.DetectRelocalisationCandidates(1_000_000 + k, kb[f], cv)), ("reloc", n, k)
        visited, scored, merge = counts(kb, voc.size(), [q for q, _ in qs[:a.ref_sample]])
        row = {"n_keyframes": n, "places": first, "mean_bow_words": float(np.mean([len(b[0]) for b in kb])),
               "add_ms_per_keyframe": add_ms,
               "gpu_loop_ms": {"median": float(np.median(loop_ms)), "mean": float(np.mean(loop_ms))},
               "gpu_reloc_ms": {"median": float(np.median(reloc_ms)), "mean": float(np.mean(reloc_ms))},
               "gpu_kernel_us_per_query": dev_us, "gpu_kernel_us_per_query_by_kernel": per_kernel,
               "ref_loop_ms": {"median": float(np.median(ref_loop)), "mean": float(np.mean(ref_loop))},
               "ref_reloc_ms": {"median": float(np.median(ref_reloc)), "mean": float(np.mean(ref_reloc))},
               "ref_sample": a.ref_sample, "lists_identical": True,
               "mean_candidates_loop_reloc": np.mean(n_cand, 0).tolist(),
               "counts_per_query": {"list_entries_visited": visited, "pairs_scored": scored, "merge_steps": merge}}
        res["sizes"].append(row)
        print(json.dumps(row), flush=True)
    pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    pathlib.Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps({"gpu": res["gpu"], "out": a.out}))


if __name__ == "__main__":
    main()
