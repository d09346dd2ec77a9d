/*
 * mcs_b200.h -- C ABI of the B200-native MultiCol-SLAM feature hot path.
 *
 * One shared library (libmcs_b200.so) replaces the arithmetic behind
 *   mdBRIEFextractorOct::operator()            (ref include/mdBRIEFextractorOct.h:355-361,
 *                                               src/mdBRIEFextractorOct.cpp:1244-1337)
 *   cORBmatcher::SearchByProjection(F, MPs)    (ref src/cORBmatcher.cpp:67-166)
 *   cORBmatcher::SearchForInitialization       (ref src/cORBmatcher.cpp:579-726)
 *   cORBmatcher::SearchByBoW(KF, KF)           (ref src/cORBmatcher.cpp:885-966, all-pairs)
 *   DescriptorDistance64[Masked]               (ref src/cORBmatcher.cpp:2438-2474)
 *   cCamModelGeneral_::WorldToImg / ImgToWorld (ref src/cam_model_omni.cpp:49-67,146-161)
 *   CreateMirrorMask level 0                   (ref src/cam_model_omni.cpp:181-220)
 *
 * Plain pointers and sizes only; no C++/torch/OpenCV types cross this boundary.
 * Every function returns an int status (MCS_OK == 0) and never throws.
 * The C++ classes in include/mcs_shim.hpp adapt these entry points to the
 * reference's own class signatures (see INTEGRATION.md).
 *
 * Pointers named *_dev are CUDA device pointers on the extractor's device;
 * everything else is host memory owned by the caller.
 */
#ifndef MCS_B200_H
#define MCS_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCS_OK                0
#define MCS_ERR_INVALID      -1   /* bad argument (null pointer, size, ...)            */
#define MCS_ERR_UNSUPPORTED  -2   /* option of the reference that is not built (AGAST) */
#define MCS_ERR_CUDA         -3   /* CUDA runtime error; see mcs_last_error()          */
#define MCS_ERR_CAPACITY     -4   /* caller buffer too small                           */
#define MCS_ERR_NO_DEVICE    -5   /* no usable sm_100 device: there is NO CPU fallback */

#define MCS_MAX_LEVELS       16
#define MCS_FRAME_GRID_COLS  64   /* ref include/cMultiFrame.h:48 */
#define MCS_FRAME_GRID_ROWS  48   /* ref include/cMultiFrame.h:47 */

/* Scaramuzza/OCam interior orientation, the 17 doubles of cCamModelGeneral_
 * (ref include/cam_model_omni.h:47-110; YAML keys Camera.{c,d,e,u0,v0,a0..a4,pol0..pol11,Iw,Ih},
 * loaded zero-padded to 5 / 12 coefficients by src/cSystem.cpp:144-156). */
typedef struct mcs_ocam {
    double c, d, e, u0, v0;
    double pol[5];        /* forward polynomial  f(rho),   p_deg    == 5  */
    double inv_pol[12];   /* backward polynomial rho(theta), invP_deg == 12 */
    int32_t width, height;
    int32_t mirror_mask;  /* Camera.mirrorMask: 1 -> disc mask, 0 -> all ones */
    int32_t _pad;
} mcs_ocam;

/* Constructor arguments of mdBRIEFextractorOct, same order and defaults
 * (ref include/mdBRIEFextractorOct.h:340-352). */
typedef struct mcs_extractor_params {
    int32_t nfeatures;        /* 1000 */
    float   scale_factor;     /* 1.2f (kept as float: the reference widens the float) */
    int32_t nlevels;          /* 8 */
    int32_t edge_threshold;   /* 25 (the reference hard-codes EDGE_THRESHOLD = 25) */
    int32_t first_level;      /* 0, unused by the reference */
    int32_t score_type;       /* parsed, ignored by the reference (FAST score always) */
    int32_t patch_size;       /* 32, unused (PATCH_SIZE constant) */
    int32_t fast_threshold;   /* 20 */
    int32_t use_agast;        /* 0; 1 -> MCS_ERR_UNSUPPORTED */
    int32_t fast_agast_type;  /* 2 == FastFeatureDetector::TYPE_9_16 (only type built) */
    int32_t do_dbrief;        /* 0: ORB, 1: distorted BRIEF */
    int32_t learn_masks;      /* 1: mdBRIEF (descriptor + stability mask) */
    int32_t desc_size;        /* bytes: 16 / 32 / 64 */
} mcs_extractor_params;

/* Binary-compatible with cv::KeyPoint (28 bytes). */
typedef struct mcs_keypoint {
    float   x, y;
    float   size;
    float   angle;
    float   response;
    int32_t octave;
    int32_t class_id;
} mcs_keypoint;

typedef struct mcs_extractor_info {
    int32_t nlevels;
    int32_t capacity;                       /* nfeatures + 2*nlevels: max keypoints per image */
    int32_t desc_size;
    int32_t features_per_level[MCS_MAX_LEVELS];
    double  scale_factor[MCS_MAX_LEVELS];
    double  inv_scale_factor[MCS_MAX_LEVELS];
} mcs_extractor_info;

typedef struct mcs_extractor mcs_extractor;   /* opaque; one per (camera, thread), not re-entrant */

const char* mcs_last_error(void);             /* thread-local message of the last failure */
int  mcs_device_count(void);                  /* number of visible sm_100 devices (0 -> none) */
void mcs_params_default(mcs_extractor_params* p);

/* ---- camera model (C1) ------------------------------------------------------------------- */
/* Host-side scalar helpers with the reference's exact double arithmetic; callers (cMultiFrame
 * bearing rays, projection front-ends) use them per point.  The device copies live inside the
 * descriptor kernel. */
void mcs_cam_world_to_img(const mcs_ocam* cam, double x, double y, double z, double* u, double* v);
void mcs_cam_img_to_world(const mcs_ocam* cam, double u, double v, double* x, double* y, double* z);
/* level-0 mirror mask, h*w bytes, 255 inside the disc / 0 outside (or all 1 when mirror_mask==0) */
int  mcs_cam_mirror_mask(const mcs_ocam* cam, uint8_t* mask_out);

/* ---- extractor (E0..E9) ------------------------------------------------------------------ */
int  mcs_extractor_create(const mcs_extractor_params* p, mcs_extractor** out);
void mcs_extractor_destroy(mcs_extractor* ex);
int  mcs_extractor_get_info(const mcs_extractor* ex, mcs_extractor_info* info);

/* operator() for one image.  Host buffers, synchronous.
 *   mask: h x w bytes, mandatory (the reference throws on an empty mask);
 *   kps_out[capacity], desc_out[capacity*desc_size], dmask_out[capacity*desc_size] (may be NULL
 *   only when learn_masks==0; when given and learn_masks==0 it is zero-filled like the reference);
 *   *n_out = number of keypoints.  capacity must be >= info.capacity. */
int  mcs_extract(mcs_extractor* ex,
                 const uint8_t* image, int32_t width, int32_t height, int32_t stride,
                 const uint8_t* mask, int32_t mask_stride,
                 const mcs_ocam* cam,
                 mcs_keypoint* kps_out, uint8_t* desc_out, uint8_t* dmask_out,
                 int32_t capacity, int32_t* n_out);

/* Batched form: n_images images of identical size, image i seen by camera cam_of_image[i]
 * (index into cams[]/masks[]).  images: n_images*height*stride bytes; masks: n_cams*height*width.
 * Outputs are fixed-size slots of `capacity` entries per image.  Host buffers (pinned memory
 * recommended), H2D + kernels + D2H inside the call. */
int  mcs_extract_batch(mcs_extractor* ex, int32_t n_images,
                       const uint8_t* images, int32_t width, int32_t height, int32_t stride,
                       const uint8_t* masks, const mcs_ocam* cams, int32_t n_cams,
                       const int32_t* cam_of_image,
                       mcs_keypoint* kps_out, uint8_t* desc_out, uint8_t* dmask_out,
                       int32_t* counts_out, int32_t capacity);

/* Same, all image/output buffers resident in device memory; asynchronous on `stream`
 * (a cudaStream_t passed as void*; NULL = the extractor's own stream, then the call
 * synchronises before returning).  masks/cams/cam_of_image stay host pointers (tiny, cached
 * on the device by the extractor).  With a caller stream the capacity checks of the call (raw corner list, octree node table,
 * keypoint slots: MCS_ERR_CAPACITY) cannot be reported by the call itself: mcs_extractor_check_status does that afterwards. */
int  mcs_extract_batch_device(mcs_extractor* ex, int32_t n_images,
                              const uint8_t* images_dev, int32_t width, int32_t height, int32_t stride,
                              const uint8_t* masks, const mcs_ocam* cams, int32_t n_cams,
                              const int32_t* cam_of_image,
                              mcs_keypoint* kps_dev, uint8_t* desc_dev, uint8_t* dmask_dev,
                              int32_t* counts_dev, int32_t capacity, void* stream);

/* Stream form of the whole path: n_frames multi-camera frames (frame-major: image i = frame i/n_cams,
 * camera i%n_cams) are extracted, and every image is brute-force matched (bit-level Hamming, masked form when
 * learn_masks is set) against the same camera of the previous frame: K best (index, distance) per keypoint
 * slot, (-1, INT_MAX) where none / for frame 0.  match_idx/match_dist: [n_frames*n_cams*capacity*K].
 * Host buffers; H2D, all kernels and D2H happen inside the call. */
int  mcs_extract_match_stream(mcs_extractor* ex, int32_t n_frames, int32_t n_cams,
                              const uint8_t* images, int32_t width, int32_t height, int32_t stride,
                              const uint8_t* masks, const mcs_ocam* cams,
                              mcs_keypoint* kps_out, uint8_t* desc_out, uint8_t* dmask_out,
                              int32_t* counts_out, int32_t capacity,
                              int32_t K, int32_t* match_idx_out, int32_t* match_dist_out);

/* The stream call with two optional extras:
 *  - packed_dev (may be NULL): the features of the batch are also left in the caller's packed exchange buffer (device memory,
 *    mcs_packed_layout(n_frames*n_cams, capacity, descSize) bytes): K3 writes them there, the host copies are taken from there,
 *    and mcs_allgather_features can ship the buffer to the other GPUs of the rig right after the call;
 *  - matches12_out / nmatches_out / redo_out (all three or none): the greedy acceptance of SearchByBoW(KF1, KF2)
 *    (threshold th_low, ratio nnratio, every database keypoint used once; see mcs_match_stream_replay_device) evaluated on the
 *    device over each chunk's K-best lists; host arrays [n_images*capacity], [n_images], [n_images].  In this mode the lists
 *    returned in match_idx_out / match_dist_out hold only the entries that can influence the acceptance (distance below the
 *    relevance bound of mcs_match_stream_greedy_device); shorter lists are padded with (-1, INT_MAX). */
int  mcs_extract_match_stream_packed(mcs_extractor* ex, int32_t n_frames, int32_t n_cams,
                                     const uint8_t* images, int32_t width, int32_t height, int32_t stride,
                                     const uint8_t* masks, const mcs_ocam* cams,
                                     mcs_keypoint* kps_out, uint8_t* desc_out, uint8_t* dmask_out,
                                     int32_t* counts_out, int32_t capacity,
                                     int32_t K, int32_t* match_idx_out, int32_t* match_dist_out, void* packed_dev,
                                     int32_t th_low, double nnratio, int32_t* matches12_out, int32_t* nmatches_out, int32_t* redo_out);

/* Device-resident matching half of the stream form (descriptor slots as written by
 * mcs_extract_batch_device); asynchronous on `stream`. dmask_dev may be NULL (unmasked distance). */
int  mcs_match_stream_device(const uint8_t* desc_dev, const uint8_t* dmask_dev, const int32_t* counts_dev,
                             int32_t n_frames, int32_t n_cams, int32_t capacity, int32_t dim, int32_t K,
                             int32_t* match_idx_dev, int32_t* match_dist_dev, void* stream);

/* The greedy acceptance of SearchByBoW(KF1, KF2) (ref src/cORBmatcher.cpp:899-961: threshold, ratio test, every database
 * keypoint used once, queries in index order) over the K-best lists of mcs_match_stream_device, on the device and on the same
 * stream.  A query is decided from its list whenever the list provably contains the answer (two unmatched entries, or bounds
 * from the last list distance); otherwise the kernel rescans the previous image for that query, so the result equals the
 * reference's sequential loop for every K >= 1.  matches12_dev [n_images*capacity] = matched slot of the previous frame's image
 * or -1, nmatches_dev [n_images]; redo_dev [n_images] is always 0 (kept for callers that check it).  desc_dev / dmask_dev: the
 * descriptor slots the lists were computed from (dmask_dev NULL = unmasked). */
int  mcs_match_stream_replay_device(const int32_t* match_idx_dev, const int32_t* match_dist_dev, const int32_t* counts_dev,
                                    const uint8_t* desc_dev, const uint8_t* dmask_dev,
                                    int32_t n_frames, int32_t n_cams, int32_t capacity, int32_t dim, int32_t K, int32_t th_low, double nnratio,
                                    int32_t* matches12_dev, int32_t* nmatches_dev, int32_t* redo_dev, void* stream);

/* Both steps as one call -- the operation cLoopClosing / cTracking actually want from a brute-force match (SearchByBoW(KF1, KF2)'s
 * acceptance rule, ref src/cORBmatcher.cpp:885-966, of every image against the same camera's image one frame earlier): K-best
 * lists in scratch memory of the stream's pool, then the greedy replay.  Because th_low and nnratio are known to the list kernel
 * here, entries that cannot influence any decision (distance >= the smallest b with (th_low - 1) < nnratio * b) are left out of
 * the lists, so a list shorter than K proves that every relevant entry is in it and the replay rescans less often; the matches
 * are the same as mcs_match_stream_device + mcs_match_stream_replay_device give for any K. */
int  mcs_match_stream_greedy_device(const uint8_t* desc_dev, const uint8_t* dmask_dev, const int32_t* counts_dev,
                                    int32_t n_frames, int32_t n_cams, int32_t capacity, int32_t dim, int32_t th_low, double nnratio,
                                    int32_t* matches12_dev, int32_t* nmatches_dev, void* stream);

/* Per-stage device timings of the LAST extract call, measured with CUDA events on the launching stream when
 * profiling is enabled: ms[0] = K1 (pyramid+blur+FAST, all levels), ms[1] = K2 octree, ms[2] = K3 describe.
 * mcs_extractor_set_profiling(ex, 1) turns the event recording on (off by default). */
int  mcs_extractor_set_profiling(mcs_extractor* ex, int32_t enable);
int  mcs_extractor_get_timings(mcs_extractor* ex, float* ms3);

/* Diagnostics of the descriptor kernel (K3): the distorted patterns are evaluated by the cheapest of three tiers whose error
 * bound still decides every rounding of the reference (fp32 relative to the keypoint / FP64 polynomial / exact operation
 * sequence, multicol_slam_b200/csrc/describe_kernel.cu).  enable != 0 switches counting on for the following extract calls
 * (one atomic per pattern: not for timed runs); counts4 (may be NULL) receives the patterns decided since then by
 * [0] tier 1, [1] tier 1 after the FP64 repair of its near-tie points, [2] tier 2, [3] tier 3. */
int  mcs_extractor_tier_stats(mcs_extractor* ex, int32_t enable, int64_t* counts4);

/* Overflow report of the LAST asynchronous extract call (mcs_extract_batch_device / ..._packed_device on a caller stream):
 * synchronises `stream` (the stream that call ran on; NULL = the extractor's own) and returns MCS_ERR_CAPACITY if a raw corner
 * list, the octree node table or the keypoint slots were too small for some image (results are truncated then), MCS_OK otherwise. */
int  mcs_extractor_check_status(mcs_extractor* ex, void* stream);

/* The per-camera table behind tiers 1 and 2 of the descriptor kernel, as the host builds it (no GPU needed): one row of
 * *row_doubles doubles per integer radius i of the undistorted plane, R(r) = rho(atan(-z / r)) the radial distortion function of
 * cam (ref src/cam_model_omni.cpp:49-67):
 *   [0..1]  tau offset / scale and [2..11] the degree-9 polynomial of R on [i - 22.5, i + 22.5]            (tier 2; NaN = disabled)
 *   [12] R(i), [13] q0, [14..16] q1..q5 as floats: R(i + s) - R(i) = s' q(s'), s' = s / 32, [17] 1.0 = usable (tier 1, s-form)
 *   [18] G(c_i), [19..22] a0..a7 as floats: G(c_i + hw_i t) - G(c_i) = t P(t), G(m) = R(sqrt m) / sqrt m, c_i = i^2 + 22.5^2,
 *           hw_i = 45 i, [23] 1.0 = usable                                                                  (tier 1, m-form)
 * rows_out (may be NULL to query the sizes) receives min(*n_rows, max_rows) rows.  Exists so that the tables can be checked
 * against the camera model independently of the kernel (tests/test_distort_table_cpu.py). */
int  mcs_cam_distort_table(const mcs_ocam* cam, double* rows_out, int32_t max_rows, int32_t* n_rows, int32_t* row_doubles);

/* mcs_extract_batch / mcs_extract with at most 16 images (the per-frame call of cMultiFrame's constructor, ref
 * src/cMultiFrame.cpp:128-139) stage through pinned buffers owned by the extractor, and once a call repeats the previous one's
 * geometry, camera table, camera models and masks the whole copy-in / K1..K3 / copy-out sequence is ONE cudaGraphLaunch.
 * *n receives how many calls were served that way (diagnostics; tests assert the shortcut is taken and changes nothing). */
int  mcs_extractor_graph_replays(mcs_extractor* ex, int64_t* n);

/* Introspection for the parity tests: copy intermediate device buffers of the LAST extract call
 * (image 0 of the batch unless image_index is given) back to the host.
 *   what: 0 = unblurred level (w*h bytes), 1 = blurred level, 2 = mask level,
 *         3 = raw corners of the level as int32 triples (x, y, score) in reference order.
 *   *w_out,*h_out = level size (for what==3: *w_out = number of corners, *h_out = 3). */
int  mcs_extractor_debug_read(mcs_extractor* ex, int32_t image_index, int32_t level, int32_t what,
                              void* out, size_t out_bytes, int32_t* w_out, int32_t* h_out);

/* ---- Hamming distance (M0) --------------------------------------------------------------- */
int  mcs_descriptor_distance64(const uint64_t* a, const uint64_t* b, int32_t dim);
int  mcs_descriptor_distance64_masked(const uint64_t* a, const uint64_t* b,
                                      const uint64_t* mask_a, const uint64_t* mask_b, int32_t dim);

/* ---- brute force (M2 kernel) ------------------------------------------------------------- */
/* For every query q: the K smallest (distance, index) pairs over the nd database descriptors that
 * are not flagged in db_skip (nd bytes, may be NULL), ordered by (distance, index) ascending.
 * Distances are the reference's bit-level popcounts (masked form when qmask/dmask != NULL).
 * Output: topk_idx[nq*K] (-1 = none), topk_dist[nq*K].  Host buffers.  nd < 2^21 per call (MCS_ERR_UNSUPPORTED beyond: split the database). */
int  mcs_hamming_topk(const uint8_t* q, const uint8_t* qmask, int32_t nq,
                      const uint8_t* d, const uint8_t* dmask, int32_t nd,
                      const uint8_t* db_skip, int32_t dim, int32_t K,
                      int32_t* topk_idx, int32_t* topk_dist);
int  mcs_hamming_topk_device(const uint8_t* q_dev, const uint8_t* qmask_dev, int32_t nq,
                             const uint8_t* d_dev, const uint8_t* dmask_dev, int32_t nd,
                             const uint8_t* db_skip_dev, int32_t dim, int32_t K,
                             int32_t* topk_idx_dev, int32_t* topk_dist_dev, void* stream);

/* cORBmatcher::SearchByBoW(KF1, KF2, matches12) semantics (ref :885-966): all-pairs scan,
 * best/second best, `best < th_low`, `best < nnratio*second`, every KF2 entry used at most once,
 * queries visited in index order.  valid1/valid2: 1 where the keypoint carries a good map point
 * (NULL = all valid).  matches12[nq] = matched database index or -1.  Returns via *nmatches. */
int  mcs_match_bruteforce(const uint8_t* q, const uint8_t* qmask, const uint8_t* valid1, int32_t nq,
                          const uint8_t* d, const uint8_t* dmask, const uint8_t* valid2, int32_t nd,
                          int32_t dim, int32_t th_low, double nnratio,
                          int32_t* matches12, int32_t* nmatches);
/* Same with query and database descriptors (and masks) resident in device memory -- e.g. the descriptor section of a packed
 * feature buffer against a key-frame database that stays on the GPU; valid1 / valid2 / matches12 / nmatches are host memory.
 * Runs on `stream` and returns when the result is complete. */
int  mcs_match_bruteforce_device(const uint8_t* q_dev, const uint8_t* qmask_dev, const uint8_t* valid1, int32_t nq,
                                 const uint8_t* d_dev, const uint8_t* dmask_dev, const uint8_t* valid2, int32_t nd,
                                 int32_t dim, int32_t th_low, double nnratio, int32_t* matches12, int32_t* nmatches, void* stream);
/* Several query sets against ONE database in one call -- the batched key frames of the loop-closure path (BASELINE config 4:
 * every key frame of a batch against the key-frame database).  seg_start[0..n_seg] delimits the sets inside q_dev; each set is
 * matched exactly as a separate mcs_match_bruteforce_device call would match it (its own "database entry already used" state,
 * as between separate SearchByBoW(KF1, KF2) calls, ref src/cORBmatcher.cpp:885-966), but the K-best lists of all sets come from
 * one kernel launch.  matches12 [seg_start[n_seg]], nmatches [n_seg]. */
int  mcs_match_bruteforce_batch_device(const uint8_t* q_dev, const uint8_t* qmask_dev, const uint8_t* valid1,
                                       const int32_t* seg_start, int32_t n_seg,
                                       const uint8_t* d_dev, const uint8_t* dmask_dev, const uint8_t* valid2, int32_t nd,
                                       int32_t dim, int32_t th_low, double nnratio, int32_t* matches12, int32_t* nmatches, void* stream);

/* Diagnostics: K-best launches the last mcs_match_bruteforce[_batch][_device] call of this thread needed.  Always 1 since the
 * ordered acceptance runs on the device (queries whose list is used up are rescanned inside the replay kernel). */
int  mcs_last_bruteforce_rounds(void);


/* cORBmatcher::SearchForTriangulationRaw(KF1, KF2, ...) (ref src/cORBmatcher.cpp:968-1156): all-pairs scan, same camera only,
 * over the keypoints that carry NO map point (free1/free2 != 0); per query the candidates with distance <= th_low are
 * ordered by (distance, index), and the first one within cvRound(2*best) whose bearing rays satisfy the epipolar constraint
 * CheckDistEpipolarLine(ray1, ray2, E[cam][cam], epi_thresh) (ref src/misc.cpp:53-69) is matched; every KF2 keypoint is used
 * at most once, queries are visited in index order.  rays: [n*3] doubles; E: [n_cams*n_cams*9] row-major 3x3 (ComputeE).
 * matches12[n1] = KF2 index or -1. */
int  mcs_search_for_triangulation(const uint8_t* desc1, const uint8_t* mask1, const int32_t* cam1, const uint8_t* free1,
                                  const double* rays1, int32_t n1,
                                  const uint8_t* desc2, const uint8_t* mask2, const int32_t* cam2, const uint8_t* free2,
                                  const double* rays2, int32_t n2,
                                  int32_t dim, int32_t th_low, const double* E, int32_t n_cams, double epi_thresh,
                                  int32_t* matches12, int32_t* nmatches);

/* ---- multi-camera frame view + grid window search (G1, M1, M3) ---------------------------- */
/* Flat view of the fields of cMultiFrame the matchers read (ref include/cMultiFrame.h:90-175).
 * Keypoints are in the contiguous (camera-major) order of src/cMultiFrame.cpp:168-184. */
typedef struct mcs_frame_view {
    int32_t n_cams;
    int32_t n_keys;                 /* totalN */
    const mcs_keypoint* keys;       /* [n_keys] contiguous index order (mvKeys) */
    const int32_t* key_cam;         /* [n_keys] keypoint_to_cam */
    const uint8_t* desc;            /* [n_keys*dim] descriptor rows in contiguous index order */
    const uint8_t* dmask;           /* [n_keys*dim] or NULL */
    const int32_t* cam_width;       /* [n_cams] mnMaxX - mnMinX */
    const int32_t* cam_height;      /* [n_cams] */
    int32_t dim;                    /* descriptor bytes */
    int32_t n_levels;
    const double* scale_factors;    /* [n_levels] mvScaleFactors */
} mcs_frame_view;

/* Per-frame epilogue of the cMultiFrame constructor on the GPU (SURVEY 8f "next" row 3; ref src/cMultiFrame.cpp:143-184):
 * bearing rays camModel.ImgToWorld(pt) of every keypoint ([n_keys*3] doubles, bit-identical to the host evaluation: only
 * + - * / sqrt) and the 64x48 grid of PosInGrid (:342-353) as CSR over (cam, ix, iy): cell_start [n_cams*64*48 + 1],
 * cell_items [n_keys] (first *n_in_grid valid), ascending keypoint index inside a cell.  keys/key_cam as in mcs_frame_view
 * (cam_width/height are taken from cams[]).  Host buffers.  The window searches build their grid with the same kernel. */
int  mcs_frame_prepare(const mcs_keypoint* keys, const int32_t* key_cam, int32_t n_keys, const mcs_ocam* cams, int32_t n_cams,
                       double* rays_out, int32_t* cell_start_out, int32_t* cell_items_out, int32_t* n_in_grid);

/* One window query: GetFeaturesInArea(cam, x, y, r, min_level, max_level)
 * (ref src/cMultiFrame.cpp:272-340) followed by Hamming distance to every candidate. */
typedef struct mcs_window_query {
    int32_t cam;
    int32_t min_level, max_level;   /* -1,-1 = no level filter */
    int32_t desc_index;             /* row of the query descriptor in the query descriptor array */
    double  x, y, r;
} mcs_window_query;

/* Candidate lists in the reference's visiting order (cell-x outer, cell-y inner, insertion
 * order inside a cell).  cand_idx/cand_dist: [nq*max_cand]; cand_count[nq] holds the TRUE number
 * of candidates (may exceed max_cand: then only the first max_cand are stored and the call
 * returns MCS_ERR_CAPACITY so the caller can retry with a larger max_cand). */
int  mcs_window_search(const mcs_frame_view* frame,
                       const mcs_window_query* queries, int32_t nq,
                       const uint8_t* qdesc, const uint8_t* qmask,
                       int32_t max_cand,
                       int32_t* cand_idx, int32_t* cand_dist, int32_t* cand_count);

/* cORBmatcher::SearchByProjection(F, vpMapPoints, th) (ref :67-166).
 * Map points as parallel arrays: for map point i and camera c, entry i*n_cams+c.
 *   mp_bad[nmp]; in_view[nmp*n_cams]; level[..]; proj_x[..], proj_y[..]; view_cos[..];
 *   mp_desc[nmp*dim] (+ mp_dmask).
 * frame_mp[n_keys]: in/out, index of the map point assigned to each keypoint (-1 = none) --
 * the flat image of F.mvpMapPoints.  having_masks selects the masked distance. */
typedef struct mcs_mappoint_view {
    int32_t n_points;
    const uint8_t* bad;
    const uint8_t* in_view;
    const int32_t* level;
    const double*  proj_x;
    const double*  proj_y;
    const double*  view_cos;
    const uint8_t* desc;
    const uint8_t* dmask;
} mcs_mappoint_view;

int  mcs_search_by_projection(const mcs_frame_view* frame, const mcs_mappoint_view* mps,
                              double th, double nnratio, int32_t th_high, int32_t having_masks,
                              int32_t* frame_mp, int32_t* nmatches);

/* ---- projection front-end of SearchByProjection (SURVEY 8f "next" row 2) ------------------------ */
/* cMultiFrame::isInFrustum(cam, pMP, .) for every (map point, camera) (ref src/cMultiFrame.cpp:218-270) with
 * cMultiCamSys_::WorldToCamHom_fast (ref src/cam_system_omni.cpp:92-112) and isPointInMirrorMask
 * (ref src/cam_model_omni.cpp:163-178): fills exactly the arrays mcs_mappoint_view / mcs_search_by_projection consume.
 *   mtmc_inv, mtmc: [n_cams*16] row-major 4x4 (MtMc_inv[c] and Get_MtMc(c)); masks: n_cams level-0 mirror masks (h*w each);
 *   world_pos, normal: [n_points*3]; min_dist, max_dist: [n_points] (Get{Min,Max}DistanceInvariance);
 *   outputs indexed [point*n_cams + cam].  Host buffers.  Integer outputs (in_view, level) are exact; the projections go
 *   through atan(), so they agree with a CPU evaluation to ~1e-13 px. */
int  mcs_project_mappoints(int32_t n_cams, const double* mtmc_inv, const double* mtmc, const mcs_ocam* cams,
                           const uint8_t* masks, int32_t n_points, const double* world_pos, const double* normal,
                           const double* min_dist, const double* max_dist, const double* scale_factors, int32_t n_levels,
                           uint8_t* in_view, int32_t* level, double* proj_x, double* proj_y, double* view_cos);

/* Generic projection-window search: the shape shared by the remaining cORBmatcher searches (SURVEY 8a row M4).
 * Queries are visited in order; for each one the candidates of GetFeaturesInArea(cam, x, y, r, min_level, max_level)
 * that are not yet taken (assigned[idx] >= 0) are scanned in the reference's order, best / second best are tracked
 * with strict `<`, and the best candidate is accepted by `rule`:
 *   MCS_RULE_RATIO        best <= second*nnratio && best <= threshold   WindowSearch (ref src/cORBmatcher.cpp:420),
 *                                                                       SearchByProjection(F1,F2,win,..) (:556-558)
 *   MCS_RULE_BEST         best <= threshold                             SearchByProjection(Current, Last, th) (:2070)
 *   MCS_RULE_LEVEL_RATIO  best <= threshold && !(bestLevel == secondLevel && best > nnratio*second)
 *                                                                       SearchByProjection(F, MapPoints, th) (:151-158)
 *   MCS_RULE_BEST_FREE    best <= threshold, candidates are NOT skipped when taken and nothing is marked: the per-query
 *                         answer is written to assigned[q] (best index or -1; `assigned` is then an output of nq entries).
 *                         This is the matching core of Fuse(pKF, curKF, ..) (:1326-1366), Fuse(pKF, Scw, ..) (:1620-1660) and
 *                         SearchBySim3 (:1793-1830, :1869-1906): their level filter {l-1, l} goes into the query.
 *   MCS_RULE_FIRST_FREE   Fuse(pKF, vpMapPoints, th) (:1420-1568, the overload cLocalMapping calls at src/cLocalMapping.cpp:450)
 *                         as the reference really behaves: it computes the descriptor distance and DISCARDS it (:1506-1514, `dist`
 *                         stays 0), so the first candidate of the window that passes the level filter wins with distance
 *                         0 <= threshold.  Stateless like MCS_RULE_BEST_FREE: assigned[q] = that candidate or -1.
 *   MCS_RULE_SCW          SearchByProjection(pKF, Scw, vpPoints, vpMatched, th) (:2265-2392) as written: taken candidates
 *                         (vpMatched[idx], i.e. assigned[idx] >= 0) are skipped; the descriptor compared for candidate idx of a
 *                         query of camera c is ROW idx OF CAMERA c's MATRIX -- the contiguous keypoint id used as a per-camera row
 *                         (:2367, :2372) -- i.e. contiguous keypoint first(c) + idx; candidates whose row lies beyond camera c's own
 *                         rows (where the reference reads past the matrix: undefined) are dropped; accepted when
 *                         best <= threshold && bestIdx > 0 (:2385, keypoint 0 can never be matched).  Needs camera-major keypoints.
 * On acceptance assigned[bestIdx] = query_tag[q] (tags must be >= 0).  The caller builds the queries (projection
 * front-end, "bad"/duplicate filters of the reference loops) and owns `assigned` (in/out, [n_keys], -1 = free). */
#define MCS_RULE_RATIO        0
#define MCS_RULE_BEST         1
#define MCS_RULE_LEVEL_RATIO  2
#define MCS_RULE_BEST_FREE    3
#define MCS_RULE_FIRST_FREE   4
#define MCS_RULE_SCW          5
int  mcs_search_windows(const mcs_frame_view* frame, const mcs_window_query* queries, int32_t nq,
                        const uint8_t* qdesc, const uint8_t* qmask, const int32_t* query_tag,
                        int32_t rule, double nnratio, int32_t threshold, int32_t* assigned, int32_t* nmatches);

/* cORBmatcher::SearchForInitialization(F1, F2, vbPrevMatched, vnMatches12, windowSize)
 * (ref :579-726, checkOrientation is compile-time false: include/cORBmatcher.h:40).
 * prev_matched[2*n1] in/out (x,y doubles); matches12[n1] out. */
int  mcs_search_for_initialization(const mcs_frame_view* f1, const mcs_frame_view* f2,
                                   double* prev_matched, int32_t window_size,
                                   double nnratio, int32_t th_low, int32_t having_masks,
                                   int32_t* matches12, int32_t* nmatches);

/* ---- bag of words: ORBVocabulary::transform and the feature-vector guided search (SURVEY 8f, rank 4) ------- */
/* The vocabulary tree of DBoW2::TemplatedVocabulary<FORB::TDescriptor, FORB> (ref include/cORBVocabulary.h:34,
 * ThirdParty/DBoW2/DBoW2/TemplatedVocabulary.h) as flat arrays.  Node 0 is the root; parent[0] is ignored.
 * descriptors: n_nodes x 32 bytes (FORB::L = 32; row 0 unused).  weight[i]: node weight (word weight for leaves).
 * node_order: the n_nodes-1 non-root node ids in the order the reference's load() appends them to their parent's
 * children (ref :1596-1608 / :1382-1421); NULL = ascending id.  word_node[w] = node id of word w.
 * scoring: 0 L1_NORM, 1 L2_NORM, 2 CHI_SQUARE, 3 KL, 4 BHATTACHARYYA, 5 DOT_PRODUCT; weighting: 0 TF_IDF, 1 TF, 2 IDF,
 * 3 BINARY (ref ThirdParty/DBoW2/DBoW2/BowVector.h:36-59). */
typedef struct mcs_vocabulary mcs_vocabulary;
int  mcs_vocabulary_create(int32_t k, int32_t L, int32_t scoring, int32_t weighting, int32_t n_nodes,
                           const int32_t* parent, const double* weight, const uint8_t* descriptors,
                           const int32_t* node_order, int32_t n_words, const int32_t* word_node,
                           mcs_vocabulary** out);
void mcs_vocabulary_destroy(mcs_vocabulary* voc);

/* transform(feature, word_id, weight, &nid, levelsup) for n descriptors of 32 bytes (ref :1218-1261): the tree
 * descent on the GPU, one 16-lane group per descriptor, FORB::distance (ref FORB.cpp:84-104), first minimum wins.
 * node_id[i] = ancestor at level L - levelsup (0 when that level is <= 0).  The reference leaves nid indeterminate
 * when the leaf is shallower than that level; this library returns the leaf's node id there.  Any output may be NULL. */
int  mcs_bow_transform(const mcs_vocabulary* voc, const uint8_t* desc, int32_t n, int32_t levelsup,
                       int32_t* word_id, double* weight, int32_t* node_id);

/* transform(features, BowVector&, FeatureVector&, levelsup) (ref :1126-1194; call sites src/cMultiFrame.cpp:356-363,
 * src/cMultiKeyFrame.cpp:105-114).  desc = the frame's descriptors of all cameras concatenated in camera order
 * (cConverter::toDescriptorVector, ref src/cConverter.cpp:58-66).
 * BowVector: bow_words/bow_values[<= n] ascending word id (std::map order), *n_bow entries, weights accumulated in
 * feature order and normalised as the scoring type asks.
 * FeatureVector: CSR -- fv_nodes[<= n] ascending node id, fv_offsets[*n_fv + 1], fv_features[<= n] (ascending feature
 * index inside a node). */
int  mcs_bow_vectors(const mcs_vocabulary* voc, const uint8_t* desc, int32_t n, int32_t levelsup,
                     int32_t* bow_words, double* bow_values, int32_t* n_bow,
                     int32_t* fv_nodes, int32_t* fv_offsets, int32_t* n_fv, int32_t* fv_features);

/* ORBVocabulary::score(v1, v2) with the vocabulary's scoring type (ref ScoringObject.cpp:23-313); host arithmetic. */
int  mcs_bow_score(const mcs_vocabulary* voc, const int32_t* words1, const double* values1, int32_t n1,
                   const int32_t* words2, const double* values2, int32_t n2, double* score);

/* cORBmatcher::SearchByBoW(cMultiKeyFrame*, cMultiFrame&, vpMapPointMatches) (ref src/cORBmatcher.cpp:179-324; call site
 * src/cTracking.cpp:1177): for every vocabulary node both feature vectors hold, each key-frame keypoint that carries a
 * good map point (valid1) looks for its best / second best among the frame keypoints of that node that are still
 * unmatched; accepted if best <= th_low and best < nnratio * second.  Distances for all (node, keypoint) groups are
 * computed on the GPU, the order-dependent bookkeeping is replayed on the host.  desc1/desc2: n x dim rows in the
 * concatenated keypoint order the feature vectors index; masks NULL = unmasked.  match_of_2[n2] = key-frame keypoint
 * index or -1.  checkOrientation is compile-time false in the reference (include/cORBmatcher.h:40). */
int  mcs_search_by_bow(const uint8_t* desc1, const uint8_t* mask1, const uint8_t* valid1, int32_t n1,
                       const int32_t* fv1_nodes, const int32_t* fv1_offsets, int32_t n_fv1, const int32_t* fv1_features,
                       const uint8_t* desc2, const uint8_t* mask2, int32_t n2,
                       const int32_t* fv2_nodes, const int32_t* fv2_offsets, int32_t n_fv2, const int32_t* fv2_features,
                       int32_t dim, int32_t th_low, double nnratio, int32_t* match_of_2, int32_t* nmatches);

/* ---- key-frame database: loop and relocalisation candidates (ref src/cMultiKeyFrameDatabase.cpp) ------------------------ */
/* cMultiKeyFrameDatabase(voc) (ref :36-40).  The inverted file, the BowVectors given to add() and the per-key-frame query
 * fields live on the device that is current at creation; every call checks that it still is (MCS_ERR_INVALID otherwise).
 * The entry points are serialised by one internal mutex (the reference shares the database between the tracking and the
 * loop-closing threads).  KL scoring (type 3): MCS_ERR_UNSUPPORTED (a device log() need not round like the host's; the other
 * five types use + - * / sqrt |.| only and reproduce mcs_bow_score bit for bit).
 * Key-frame ids are cMultiKeyFrame::mnId: non-negative, below 2^30 here (MCS_ERR_UNSUPPORTED beyond: the per-key-frame fields
 * mnLoopQuery / mnLoopWords / mLoopScore / mnRelocQuery / mnRelocWords / mRelocScore are arrays indexed by id).  Those fields
 * start at 0 (0.0 for the scores; the reference leaves all but the two query ids uninitialised, src/cMultiKeyFrame.cpp:44-45),
 * outlive erase() and clear() and carry from one query to the next, as on the reference's key frames.
 * A BowVector is (words ascending, strictly, each < voc size; values), as mcs_bow_vectors returns it; MCS_ERR_INVALID otherwise. */
typedef struct mcs_keyframe_db mcs_keyframe_db;
int  mcs_kfdb_create(const mcs_vocabulary* voc, mcs_keyframe_db** out);
void mcs_kfdb_destroy(mcs_keyframe_db* db);
/* add(pKF) (ref :43-50): appends kf_id to the list of every word of its BowVector, after the entries already there; a second add
 * of the same id appends it again (it then counts twice).  The BowVector is kept as pKF->mBowVec for scoring and erase. */
int  mcs_kfdb_add(mcs_keyframe_db* db, int64_t kf_id, const int32_t* bow_words, const double* bow_values, int32_t n_bow);
/* erase(pKF) (ref :52-73): removes the first (oldest) entry of kf_id from the list of every word of its latest BowVector.
 * An id that was never added: MCS_OK, nothing changes. */
int  mcs_kfdb_erase(mcs_keyframe_db* db, int64_t kf_id);
/* clear() (ref :75-79): empties every list; the per-key-frame fields and stored BowVectors stay. */
int  mcs_kfdb_clear(mcs_keyframe_db* db);
/* DetectLoopCandidates(pKF, minScore) (ref :82-215; call site src/cLoopClosing.cpp:155) and DetectRelocalisationCandidates(F)
 * (ref :217-327; call site src/cTracking.cpp:1134).
 * kf_id / frame_id: pKF->mnId / F->mnId (non-negative); bow: pKF->mBowVec / F->mBowVec.
 * connected[n_connected]: pKF->GetConnectedKeyFrames() (never listed; their mnLoopWords are still reset and counted, ref :102-111).
 * covis: row id = GetBestCovisibilityKeyFrames(10) of key frame id as the reference reads it at query time, covis[id*10 + j],
 * -1 = none, rows for ids 0..n_covis_rows-1 (missing rows: no neighbours).  Entries must be -1 or an id.
 * candidates: key-frame ids in the reference's order (first encounter: query words ascending, each list in add order; pBestKF
 * deduplicated keeping the first).  MCS_ERR_CAPACITY with *n_candidates = the required count when `capacity` is too small;
 * the query has run all the same (its effect on the per-key-frame fields stays, as in the reference), so a retry is a new
 * query.  A capacity of 1 + the largest id added or named in covis always suffices.
 * Relocalisation reads a neighbour's mRelocScore whenever mnRelocQuery == F->mnId (ref :293), also when this query did not
 * score it: the value is then the one of the last query that did (0.0 if none). */
int  mcs_kfdb_detect_loop_candidates(mcs_keyframe_db* db, int64_t kf_id, const int32_t* bow_words, const double* bow_values,
                                     int32_t n_bow, const int64_t* connected, int32_t n_connected, const int64_t* covis,
                                     int64_t n_covis_rows, double min_score, int64_t* candidates, int32_t capacity,
                                     int32_t* n_candidates);
int  mcs_kfdb_detect_relocalisation_candidates(mcs_keyframe_db* db, int64_t frame_id, const int32_t* bow_words,
                                               const double* bow_values, int32_t n_bow, const int64_t* covis,
                                               int64_t n_covis_rows, int64_t* candidates, int32_t capacity,
                                               int32_t* n_candidates);

/* ---- multi-GPU: one camera (or stream chunk) per GPU, ONE allgather of the packed feature buffer (SURVEY 8e) -------------- */
/* Packed feature buffer of a batch of n_images images: the four output arrays of the batched extractor in one allocation,
 *   [ counts int32[n_images] | mcs_keypoint[n_images][capacity] | desc u8[n_images][capacity][dim] | dmask u8[n_images][capacity][dim] ]
 * every section on a 256-byte boundary.  offsets4 (may be NULL) receives the four byte offsets; returns the total size.  It is
 * the only layout that travels between GPUs: K3 writes it in place, the allgather moves it, the matchers read it in place. */
size_t mcs_packed_layout(int32_t n_images, int32_t capacity, int32_t dim, size_t* offsets4);
size_t mcs_slot_bytes(int32_t capacity, int32_t dim);     /* == mcs_packed_layout(1, capacity, dim, NULL): one camera of a rig */

/* mcs_extract_batch_device with the four outputs laid out as above inside packed_dev (device memory, mcs_packed_layout bytes). */
int  mcs_extract_batch_packed_device(mcs_extractor* ex, int32_t n_images,
                                     const uint8_t* images_dev, int32_t width, int32_t height, int32_t stride,
                                     const uint8_t* masks, const mcs_ocam* cams, int32_t n_cams, const int32_t* cam_of_image,
                                     void* packed_dev, int32_t capacity, void* stream);

/* Communicator of the rig's GPUs: one process per GPU.  Rank 0 draws the 128-byte rendezvous token (ncclGetUniqueId) and the host
 * program hands it to the other ranks by whatever it already has (MPI, torch.distributed, a socket); every rank then calls
 * mcs_comm_create on its current CUDA device (collective; ncclCommInitRank).  NCCL is loaded at run time: the copy the process
 * already carries (e.g. PyTorch's) or the system libnccl.so.2; MCS_ERR_UNSUPPORTED when there is none. */
typedef struct mcs_comm mcs_comm;
int  mcs_comm_unique_id(uint8_t* id128);
int  mcs_comm_create(const uint8_t* id128, int32_t rank, int32_t world, mcs_comm** out);
void mcs_comm_destroy(mcs_comm* comm);
int  mcs_comm_info(const mcs_comm* comm, int32_t* rank, int32_t* world, int32_t* nccl_version);

/* The single exchange of the path, the device-side counterpart of cMultiFrame's camera-order concatenation (ref
 * src/cMultiFrame.cpp:168-184): every rank contributes its packed buffer (`bytes` identical on all ranks) and receives
 * world * bytes in rank order in gathered_dev.  One ncclAllGather on `stream` (a cudaStream_t as void*), asynchronous: issue it
 * right behind the extraction on the same stream, or on a second stream behind an event to overlap it with the next batch. */
int  mcs_allgather_features(mcs_comm* comm, const void* packed_dev, size_t bytes, void* gathered_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MCS_B200_H */
