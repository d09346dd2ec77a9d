// kfdb_kernels.h -- device side of the key-frame database (kfdb_kernels.cu, host layer mcs_kfdb_api.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace mcs {

// first-encounter key of an inverted-file entry: query word index << kKeySeqBits | add sequence.  Ordering key frames by their
// smallest key reproduces the reference's visit order (query words ascending, each word's list in add order).
constexpr int kKeySeqBits = 40;
constexpr unsigned long long kKeyNone = ~0ull;

// Inverted file: word w owns entries [seg_off[w], seg_off[w] + seg_len[w]) of ent_kf / ent_seq; ent_kf = -1 is a tombstone.
struct KfdbFile {
    const int* seg_off;
    int* seg_len;
    int* ent_kf;
    long long* ent_seq;
};

// BowVectors stored at add time: key frame id's words / values are bow_w / bow_v [bow_off[id], bow_off[id] + bow_n[id]).
struct KfdbBows {
    const int* bow_w;
    const double* bow_v;
    const long long* bow_off;
    const int* bow_n;
};

// one detection: the per-key-frame fields of the reference (mnLoopQuery / mnLoopWords / mLoopScore or the Reloc triple) and the
// per-query scratch, all indexed by key-frame id < n_ids.
struct KfdbQuery {
    long long id;                 // pKF->mnId / F->mnId
    int loop;                     // 1: DetectLoopCandidates, 0: DetectRelocalisationCandidates
    double min_score;             // loop only
    const int* q_words;           // query BowVector
    const double* q_values;
    int n_q;
    const unsigned* connected;    // loop only: bitmap over ids
    const int* covis;             // [n_covis_rows][10], -1 = none
    int n_covis_rows;
    int n_ids;
    long long* st_query;          // persistent state
    int* st_words;
    double* st_score;
    int* qpos;                    // [voc size]: index of word w in the query, -1 if absent
    int* cnt;                     // scratch [n_ids]
    unsigned long long* key;
    unsigned char* status;        // 1 listed, 2 scored and kept
    double* sc;
    double* acc;
    int* best;
    unsigned long long* win;      // [n_ids] by pBestKF: smallest key among survivors naming it
    unsigned long long* sort_key; // [sort_cap]
    int* sort_val;
    int sort_cap;                 // power of two >= n_ids
    int* max_words;               // scalar
    int* out;                     // [1 + n_ids]: count, then candidate ids in order
};

cudaError_t launch_kfdb_add(KfdbFile f, const int* words, int n, int kf, long long seq, cudaStream_t st);
cudaError_t launch_kfdb_erase(KfdbFile f, const int* words, int n, int kf, cudaStream_t st);
cudaError_t launch_kfdb_live_count(KfdbFile f, int n_words, int* live, cudaStream_t st);
cudaError_t launch_kfdb_compact(KfdbFile f, int n_words, const int* new_off, int* new_kf, long long* new_seq, cudaStream_t st);
cudaError_t launch_kfdb_query(const KfdbFile& f, const KfdbBows& b, const KfdbQuery& q, int n_words, int scoring, cudaStream_t st);

}  // namespace mcs
