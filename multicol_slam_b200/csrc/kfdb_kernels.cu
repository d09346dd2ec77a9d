// kfdb_kernels.cu -- key-frame database (ref src/cMultiKeyFrameDatabase.cpp:36-330) on the device.
//   kfdb_add_kernel / kfdb_erase_kernel       : add(pKF) appends one entry per word (:43-50); erase(pKF) tombstones the oldest
//                                                live entry of pKF in each of its words (:52-73).
//   kfdb_live_count_kernel / kfdb_compact_kernel : segment rebuild when a word's segment is full (host-driven, rare).
//   one detection (:80-215 DetectLoopCandidates, :217-327 DetectRelocalisationCandidates) is six launches:
//   kfdb_init_kernel       : clears the per-query scratch.
//   kfdb_visit_kernel      : one warp per query word walks that word's segment: words counter + first-encounter key per key frame.
//   kfdb_update_kernel     : replays the per-key-frame state machine of the walk (mnXQuery / mnXWords) from those counts.
//   kfdb_score_kernel      : one warp per key frame above minCommonWords: ORBVocabulary::score, terms in parallel, summed in
//                            ascending word order (the same double operations as mcs_bow_score, so the same bits).
//   kfdb_accumulate_kernel : covisibility sum over the ten best neighbours, reading the state the reference reads.
//   kfdb_select_kernel     : one block: bestAccScore, the 0.75 cut, pBestKF dedup by first occurrence, ordering by first encounter.
#include "kfdb_kernels.h"

namespace mcs {

namespace {
constexpr unsigned kFull = 0xFFFFFFFFu;
constexpr int kSelectThreads = 1024;

__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v = min(v, __shfl_xor_sync(kFull, v, o));
    return v;
}
}  // namespace

__global__ void __launch_bounds__(256) kfdb_add_kernel(KfdbFile f, const int* __restrict__ words, int n, int kf, long long seq) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int w = words[k];                     // distinct words: no two threads touch the same segment
    const int len = f.seg_len[w], p = f.seg_off[w] + len;
    f.ent_kf[p] = kf;
    f.ent_seq[p] = seq;
    f.seg_len[w] = len + 1;
}

__global__ void __launch_bounds__(256) kfdb_erase_kernel(KfdbFile f, const int* __restrict__ words, int n, int kf) {
    const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (k >= n) return;
    const int w = words[k], o = f.seg_off[w], len = f.seg_len[w];
    unsigned long long oldest = kKeyNone;       // the list's first occurrence = smallest add sequence among kf's live entries
    for (int e = lane; e < len; e += 32)
        if (f.ent_kf[o + e] == kf) oldest = min(oldest, (unsigned long long)f.ent_seq[o + e]);
    oldest = warp_min_u64(oldest);
    if (oldest == kKeyNone) return;
    for (int e = lane; e < len; e += 32)
        if (f.ent_kf[o + e] == kf && (unsigned long long)f.ent_seq[o + e] == oldest) f.ent_kf[o + e] = -1;
}

__global__ void __launch_bounds__(256) kfdb_live_count_kernel(KfdbFile f, int n_words, int* __restrict__ live) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n_words) return;
    const int o = f.seg_off[w], len = f.seg_len[w];
    int c = 0;
    for (int e = lane; e < len; e += 32) c += f.ent_kf[o + e] >= 0;
#pragma unroll
    for (int s = 16; s; s >>= 1) c += __shfl_xor_sync(kFull, c, s);
    if (lane == 0) live[w] = c;
}

__global__ void __launch_bounds__(256) kfdb_compact_kernel(KfdbFile f, int n_words, const int* __restrict__ new_off,
                                                           int* __restrict__ new_kf, long long* __restrict__ new_seq) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n_words) return;
    const int o = f.seg_off[w], len = f.seg_len[w], no = new_off[w];
    int base = 0;
    for (int e0 = 0; e0 < len; e0 += 32) {
        const int e = e0 + lane;
        const int kf = e < len ? f.ent_kf[o + e] : -1;
        const unsigned m = __ballot_sync(kFull, kf >= 0);
        if (kf >= 0) {
            const int p = no + base + __popc(m & ((1u << lane) - 1));
            new_kf[p] = kf;
            new_seq[p] = f.ent_seq[o + e];
        }
        base += __popc(m);
    }
    if (lane == 0) f.seg_len[w] = base;
}

__global__ void __launch_bounds__(256) kfdb_init_kernel(KfdbQuery q, int n_words) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < q.n_ids) { q.cnt[i] = 0; q.key[i] = kKeyNone; q.status[i] = 0; q.win[i] = kKeyNone; }
    if (i < n_words) q.qpos[i] = -1;
    if (i == 0) *q.max_words = 0;
}

// ref :93-111 / :226-240: every live entry of a query word is one encounter (pKFi->mnXWords++); the first encounter of a key
// frame is its smallest (query word index, add sequence).
__global__ void __launch_bounds__(256) kfdb_visit_kernel(KfdbFile f, KfdbQuery q) {
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (i >= q.n_q) return;
    const int w = q.q_words[i];
    if (lane == 0) q.qpos[w] = i;
    const int o = f.seg_off[w], len = f.seg_len[w];
    for (int e = lane; e < len; e += 32) {
        const int kf = f.ent_kf[o + e];
        if (kf < 0) continue;
        atomicAdd(q.cnt + kf, 1);
        atomicMin(q.key + kf, ((unsigned long long)i << kKeySeqBits) | (unsigned long long)f.ent_seq[o + e]);
    }
}

// The walk's per-encounter rule, folded over a key frame's c encounters:
//   already stamped with this query id  -> words += c, not listed (it was listed by an earlier query with the same id)
//   loop query, connected key frame     -> reset and incremented on every encounter: words = 1, stamp unchanged (:102-111)
//   otherwise                           -> words = c, stamped, listed at its first encounter
__global__ void __launch_bounds__(256) kfdb_update_kernel(KfdbQuery q) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= q.n_ids) return;
    const int c = q.cnt[j];
    if (c == 0) return;
    if (q.st_query[j] == q.id) {
        q.st_words[j] += c;
    } else if (q.loop && ((q.connected[j >> 5] >> (j & 31)) & 1u)) {
        q.st_words[j] = 1;
    } else {
        q.st_words[j] = c;
        q.st_query[j] = q.id;
        q.status[j] = 1;
        atomicMax(q.max_words, c);
    }
}

__device__ __forceinline__ int min_common_words(const KfdbQuery& q) {
    return static_cast<int>((double)*q.max_words * 0.8);               // ref :128 / :252
}

// ref :132-149 / :257-269 with ScoringObject.cpp:23-313 for every type but KL (rejected at create)
__global__ void __launch_bounds__(256) kfdb_score_kernel(KfdbQuery q, KfdbBows b, int scoring) {
    const int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (j >= q.n_ids || q.status[j] != 1 || q.st_words[j] <= min_common_words(q)) return;
    __shared__ double terms[8][32];                         // per warp: the common-word terms of one chunk, in word order
    double* tw = terms[threadIdx.x >> 5];
    const long long off = b.bow_off[j];
    const int n = b.bow_n[j];
    double acc = 0;
    for (int base = 0; base < n; base += 32) {
        const int k = base + lane;
        double t = 0;
        bool has = false;
        if (k < n) {
            const int qi = q.qpos[b.bow_w[off + k]];
            if (qi >= 0) {
                const double x = q.q_values[qi], y = b.bow_v[off + k];
                has = true;
                if (scoring == 0) t = fabs(x - y) - fabs(x) - fabs(y);
                else if (scoring == 1 || scoring == 5) t = x * y;
                else if (scoring == 2) { has = x + y != 0.0; if (has) t = x * y / (x + y); }
                else t = sqrt(x * y);
            }
        }
        // common words in ascending word order, added one by one by lane 0: the host merge's order of additions
        const unsigned m = __ballot_sync(kFull, has);
        if (has) tw[__popc(m & ((1u << lane) - 1))] = t;
        __syncwarp();
        if (lane == 0)
            for (int i = 0, c = __popc(m); i < c; ++i) acc += tw[i];
        __syncwarp();
    }
    if (lane) return;
    if (scoring == 0) acc = -acc / 2.0;
    else if (scoring == 1) acc = acc >= 1 ? 1.0 : 1.0 - sqrt(1.0 - acc);
    else if (scoring == 2) acc = 2. * acc;
    q.st_score[j] = acc;
    if (!q.loop || acc >= q.min_score) { q.status[j] = 2; q.sc[j] = acc; }
}

// ref :157-181 / :276-299
__global__ void __launch_bounds__(256) kfdb_accumulate_kernel(KfdbQuery q) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= q.n_ids || q.status[j] != 2) return;
    const int minc = min_common_words(q);
    const double s = q.sc[j];
    double best = s, acc = s;
    int best_kf = j;
    if (j < q.n_covis_rows)
        for (int k = 0; k < 10; ++k) {
            const int nb = q.covis[(size_t)j * 10 + k];
            if (nb < 0 || q.st_query[nb] != q.id || (q.loop && q.st_words[nb] <= minc)) continue;
            const double s2 = q.st_score[nb];               // the reloc test reads no words count: possibly a stale score
            acc += s2;
            if (s2 > best) { best_kf = nb; best = s2; }
        }
    q.acc[j] = acc;
    q.best[j] = best_kf;
}

// ref :183-212 / :301-324.  The survivors of the cut, in first-encounter order, deduplicated on pBestKF keeping the first: for each
// pBestKF the survivor with the smallest key wins; the winners are then sorted by key (bitonic, in global memory, one block).
__global__ void __launch_bounds__(kSelectThreads) kfdb_select_kernel(KfdbQuery q) {
    __shared__ double red[kSelectThreads / 32];
    __shared__ int n_out;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    double m = q.loop ? q.min_score : 0.0;                 // bestAccScore
    for (int j = tid; j < q.n_ids; j += kSelectThreads)
        if (q.status[j] == 2 && q.acc[j] > m) m = q.acc[j];
#pragma unroll
    for (int o = 16; o; o >>= 1) { const double v = __shfl_xor_sync(kFull, m, o); if (v > m) m = v; }
    if (lane == 0) red[wid] = m;
    if (tid == 0) n_out = 0;
    __syncthreads();
    if (tid == 0) {
        double b = red[0];
        for (int k = 1; k < kSelectThreads / 32; ++k) if (red[k] > b) b = red[k];
        red[0] = b;
    }
    __syncthreads();
    const double cut = 0.75 * red[0];
    for (int j = tid; j < q.n_ids; j += kSelectThreads)
        if (q.status[j] == 2 && q.acc[j] > cut) atomicMin(q.win + q.best[j], q.key[j]);
    __syncthreads();
    for (int j = tid; j < q.n_ids; j += kSelectThreads)
        if (q.status[j] == 2 && q.acc[j] > cut && __ldcg(q.win + q.best[j]) == q.key[j]) {
            const int p = atomicAdd(&n_out, 1);
            q.sort_key[p] = q.key[j];
            q.sort_val[p] = q.best[j];
        }
    __syncthreads();
    const int n = n_out;
    int P = 1;
    while (P < n) P <<= 1;
    for (int i = n + tid; i < P; i += kSelectThreads) q.sort_key[i] = kKeyNone;
    __syncthreads();
    for (int k = 2; k <= P; k <<= 1)
        for (int s = k >> 1; s > 0; s >>= 1) {
            for (int i = tid; i < P; i += kSelectThreads) {
                const int l = i ^ s;
                if (l <= i) continue;
                const unsigned long long a = q.sort_key[i], c = q.sort_key[l];
                if ((a > c) == ((i & k) == 0)) {
                    q.sort_key[i] = c; q.sort_key[l] = a;
                    const int v = q.sort_val[i]; q.sort_val[i] = q.sort_val[l]; q.sort_val[l] = v;
                }
            }
            __syncthreads();
        }
    if (tid == 0) q.out[0] = n;
    for (int i = tid; i < n; i += kSelectThreads) q.out[1 + i] = q.sort_val[i];
}

static unsigned blocks_for(long long threads) { return (unsigned)((threads + 255) / 256); }

cudaError_t launch_kfdb_add(KfdbFile f, const int* words, int n, int kf, long long seq, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    kfdb_add_kernel<<<blocks_for(n), 256, 0, st>>>(f, words, n, kf, seq);
    return cudaGetLastError();
}

cudaError_t launch_kfdb_erase(KfdbFile f, const int* words, int n, int kf, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    kfdb_erase_kernel<<<blocks_for((long long)n * 32), 256, 0, st>>>(f, words, n, kf);
    return cudaGetLastError();
}

cudaError_t launch_kfdb_live_count(KfdbFile f, int n_words, int* live, cudaStream_t st) {
    kfdb_live_count_kernel<<<blocks_for((long long)n_words * 32), 256, 0, st>>>(f, n_words, live);
    return cudaGetLastError();
}

cudaError_t launch_kfdb_compact(KfdbFile f, int n_words, const int* new_off, int* new_kf, long long* new_seq, cudaStream_t st) {
    kfdb_compact_kernel<<<blocks_for((long long)n_words * 32), 256, 0, st>>>(f, n_words, new_off, new_kf, new_seq);
    return cudaGetLastError();
}

cudaError_t launch_kfdb_query(const KfdbFile& f, const KfdbBows& b, const KfdbQuery& q, int n_words, int scoring, cudaStream_t st) {
    kfdb_init_kernel<<<blocks_for(q.n_ids > n_words ? q.n_ids : n_words), 256, 0, st>>>(q, n_words);
    if (q.n_q > 0) kfdb_visit_kernel<<<blocks_for((long long)q.n_q * 32), 256, 0, st>>>(f, q);
    if (q.n_ids > 0) {
        kfdb_update_kernel<<<blocks_for(q.n_ids), 256, 0, st>>>(q);
        kfdb_score_kernel<<<blocks_for((long long)q.n_ids * 32), 256, 0, st>>>(q, b, scoring);
        kfdb_accumulate_kernel<<<blocks_for(q.n_ids), 256, 0, st>>>(q);
    }
    kfdb_select_kernel<<<1, kSelectThreads, 0, st>>>(q);
    return cudaGetLastError();
}

}  // namespace mcs
