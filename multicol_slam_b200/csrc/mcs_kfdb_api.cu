// mcs_kfdb_api.cu -- C ABI of the key-frame database (include/mcs_b200.h), cMultiKeyFrameDatabase of the reference
// (src/cMultiKeyFrameDatabase.cpp).  The inverted file, the stored BowVectors and the per-key-frame query state live on the
// device (kfdb_kernels.cu); the host validates arguments, tracks segment fill levels and drives the launches.
#include <algorithm>
#include <climits>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "../../include/mcs_b200.h"
#include "kfdb_kernels.h"
#include "vocabulary.h"

using namespace mcs;

void mcs_set_error_(const std::string& msg);   // mcs_api.cu

namespace {

int kfail(int code, const std::string& msg) { mcs_set_error_(msg); return code; }

int cuda_code(cudaError_t e) { return e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? MCS_ERR_NO_DEVICE : MCS_ERR_CUDA; }

#define KCK(expr)                                                                                                   \
    do {                                                                                                            \
        cudaError_t e__ = (expr);                                                                                   \
        if (e__ != cudaSuccess) {                                                                                   \
            cudaGetLastError();                                                                                     \
            return kfail(cuda_code(e__), std::string(#expr) + ": " + cudaGetErrorString(e__));                     \
        }                                                                                                           \
    } while (0)

constexpr int kMinSegment = 8;                 // initial entries per word
constexpr long long kMaxIds = 1ll << 30;       // key-frame / neighbour ids: the state arrays are indexed by id
constexpr long long kMaxSeq = 1ll << kKeySeqBits;

// device buffer owned by the database; resize() keeps the first `keep` bytes and zero-fills the rest
struct DBuf {
    void* p = nullptr;
    size_t bytes = 0;
    DBuf() = default;
    DBuf(const DBuf&) = delete;
    DBuf& operator=(const DBuf&) = delete;
    ~DBuf() { if (p) cudaFree(p); }
    cudaError_t resize(size_t nb, size_t keep, cudaStream_t st) {
        void* q = nullptr;
        cudaError_t e = cudaMalloc(&q, std::max<size_t>(nb, 8));
        if (e == cudaSuccess) e = cudaMemsetAsync(q, 0, std::max<size_t>(nb, 8), st);
        keep = std::min(keep, std::min(nb, bytes));
        if (e == cudaSuccess && keep) e = cudaMemcpyAsync(q, p, keep, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { if (q) cudaFree(q); return e; }
        swap_in(q, nb);
        return cudaSuccess;
    }
    void swap_in(void* q, size_t nb) { if (p) cudaFree(p); p = q; bytes = nb; }
    template <typename T> T* as() const { return (T*)p; }
};

struct PinBuf {   // page-locked staging for the per-query upload and download
    void* p = nullptr;
    size_t bytes = 0;
    ~PinBuf() { if (p) cudaFreeHost(p); }
    cudaError_t reserve(size_t nb) {
        if (nb <= bytes) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; bytes = 0;
        nb = std::max<size_t>(nb, 2 * bytes);
        cudaError_t e = cudaHostAlloc(&p, nb, cudaHostAllocDefault);
        if (e == cudaSuccess) bytes = nb;
        return e;
    }
};

size_t align8(size_t x) { return (x + 7) & ~(size_t)7; }

int check_bow(const int32_t* words, const double* values, int32_t n, int n_voc) {
    if (n < 0) return kfail(MCS_ERR_INVALID, "negative BowVector size");
    if (n > 0 && (!words || !values)) return kfail(MCS_ERR_INVALID, "null BowVector");
    for (int i = 0; i < n; ++i) {
        if (words[i] < 0 || words[i] >= n_voc) return kfail(MCS_ERR_INVALID, "BowVector word id out of the vocabulary");
        if (i > 0 && words[i] <= words[i - 1]) return kfail(MCS_ERR_INVALID, "BowVector word ids must be strictly ascending");
    }
    return MCS_OK;
}

int check_id(int64_t id, const char* what) {
    if (id < 0) return kfail(MCS_ERR_INVALID, std::string(what) + " must be non-negative");
    if (id >= kMaxIds) return kfail(MCS_ERR_UNSUPPORTED, std::string(what) + " >= 2^30 (per-key-frame state is indexed by id)");
    return MCS_OK;
}

}  // namespace

struct mcs_keyframe_db {
    std::mutex mu;                             // the reference's database is shared by the tracking and loop-closing threads
    int device = 0, scoring = 0, n_words = 0;
    cudaStream_t st = nullptr;
    // inverted file: host mirror of each word's segment offset, capacity and fill (entries appended, tombstones included)
    std::vector<long long> off;
    std::vector<int> cap, used;
    long long ent_cap = 0, tombs = 0, n_used = 0;
    long long seq = 0;                         // add sequence: position in the reference's std::list order
    DBuf d_off, d_len, d_kf, d_seq, d_live;
    // BowVectors stored at add time (the latest add of an id, as pKF->mBowVec)
    DBuf d_bw, d_bv;
    long long pool_used = 0, pool_cap = 0;
    std::vector<long long> bow_off;
    std::vector<int> bow_n;
    std::vector<uint8_t> bow_known;
    DBuf d_boff, d_bn;
    // per key-frame state and per-query scratch, indexed by id < n_ids <= ids_cap
    long long n_ids = 0, ids_cap = 0;
    DBuf loop_q, loop_w, loop_s, reloc_q, reloc_w, reloc_s;
    DBuf cnt, key, status, sc, acc, best, win, sort_key, sort_val, out, qpos, max_words, upload;
    PinBuf h_up, h_out;

    ~mcs_keyframe_db() { if (st) cudaStreamDestroy(st); }

    KfdbFile file() const { return KfdbFile{d_off.as<int>(), d_len.as<int>(), d_kf.as<int>(), d_seq.as<long long>()}; }

    int ensure_ids(long long need) {
        if (need <= ids_cap) { n_ids = std::max(n_ids, need); return MCS_OK; }
        long long nc = 256;
        while (nc < need) nc <<= 1;
        const size_t o = (size_t)ids_cap, n = (size_t)nc;
        DBuf* keep8[] = {&loop_q, &loop_s, &reloc_q, &reloc_s, &d_boff};
        for (DBuf* b : keep8) KCK(b->resize(n * 8, o * 8, st));
        DBuf* keep4[] = {&loop_w, &reloc_w, &d_bn};
        for (DBuf* b : keep4) KCK(b->resize(n * 4, o * 4, st));
        DBuf* s8[] = {&key, &sc, &acc, &win, &sort_key};
        for (DBuf* b : s8) KCK(b->resize(n * 8, 0, st));
        DBuf* s4[] = {&cnt, &best, &sort_val};
        for (DBuf* b : s4) KCK(b->resize(n * 4, 0, st));
        KCK(status.resize(n, 0, st));
        KCK(out.resize((n + 1) * 4, 0, st));
        bow_off.resize(n, 0); bow_n.resize(n, 0); bow_known.resize(n, 0);
        ids_cap = nc;
        n_ids = need;
        return MCS_OK;
    }

    // one device pass: drop tombstones and give every word 2 x its live entries + kMinSegment of room
    int rebuild() {
        const int V = n_words;
        KCK(launch_kfdb_live_count(file(), V, d_live.as<int>(), st));
        std::vector<int> live(V);
        KCK(cudaMemcpyAsync(live.data(), d_live.p, (size_t)V * 4, cudaMemcpyDeviceToHost, st));
        KCK(cudaStreamSynchronize(st));
        std::vector<long long> noff(V);
        std::vector<int> ncap(V), noff32(V);
        long long tot = 0, nlive = 0;
        for (int w = 0; w < V; ++w) {
            ncap[w] = 2 * live[w] + kMinSegment;
            noff[w] = tot; tot += ncap[w]; nlive += live[w];
        }
        if (tot > INT_MAX) return kfail(MCS_ERR_UNSUPPORTED, "inverted file beyond 2^31 entries");
        for (int w = 0; w < V; ++w) noff32[w] = (int)noff[w];
        DBuf nkf, nseq, noffd;
        KCK(nkf.resize((size_t)tot * 4, 0, st));
        KCK(nseq.resize((size_t)tot * 8, 0, st));
        KCK(noffd.resize((size_t)V * 4, 0, st));
        KCK(cudaMemcpyAsync(noffd.p, noff32.data(), (size_t)V * 4, cudaMemcpyHostToDevice, st));
        KCK(launch_kfdb_compact(file(), V, noffd.as<int>(), nkf.as<int>(), nseq.as<long long>(), st));
        KCK(cudaStreamSynchronize(st));
        d_kf.swap_in(nkf.p, nkf.bytes); nkf.p = nullptr;
        d_seq.swap_in(nseq.p, nseq.bytes); nseq.p = nullptr;
        d_off.swap_in(noffd.p, noffd.bytes); noffd.p = nullptr;
        off = noff; cap = ncap; used = live;
        ent_cap = tot; n_used = nlive; tombs = 0;
        return MCS_OK;
    }

    int check_device() {
        int cur = -1;
        KCK(cudaGetDevice(&cur));
        if (cur != device) return kfail(MCS_ERR_INVALID, "key-frame database was created on another CUDA device than the current one");
        return MCS_OK;
    }
};

extern "C" {

int mcs_kfdb_create(const mcs_vocabulary* voc, mcs_keyframe_db** out) {
    if (!out) return kfail(MCS_ERR_INVALID, "null argument");
    *out = nullptr;
    if (!voc) return kfail(MCS_ERR_INVALID, "null argument");
    if (voc->scoring == 3)
        return kfail(MCS_ERR_UNSUPPORTED, "KL scoring: a device log() is not guaranteed to round like the host's (DESIGN.md section 8)");
    if (voc->n_words >= (1 << (64 - kKeySeqBits - 1))) return kfail(MCS_ERR_UNSUPPORTED, "vocabulary beyond 2^23 words");
    int ndev = 0;
    KCK(cudaGetDeviceCount(&ndev));
    if (ndev == 0) return kfail(MCS_ERR_NO_DEVICE, "no CUDA device");
    int cur = -1;
    KCK(cudaGetDevice(&cur));
    if (cur != voc->device) return kfail(MCS_ERR_INVALID, "vocabulary was created on another CUDA device than the current one");
    mcs_keyframe_db* db = new mcs_keyframe_db();
    db->device = cur; db->scoring = voc->scoring; db->n_words = voc->n_words;
    const int V = voc->n_words;
    auto init = [&]() -> int {
        KCK(cudaStreamCreateWithFlags(&db->st, cudaStreamNonBlocking));
        db->cap.assign(V, kMinSegment); db->used.assign(V, 0); db->off.resize(V);
        std::vector<int> off32(V);
        for (int w = 0; w < V; ++w) { db->off[w] = (long long)w * kMinSegment; off32[w] = w * kMinSegment; }
        db->ent_cap = (long long)V * kMinSegment;
        KCK(db->d_off.resize((size_t)V * 4, 0, db->st));
        KCK(cudaMemcpyAsync(db->d_off.p, off32.data(), (size_t)V * 4, cudaMemcpyHostToDevice, db->st));
        KCK(db->d_len.resize((size_t)V * 4, 0, db->st));
        KCK(db->d_live.resize((size_t)V * 4, 0, db->st));
        KCK(db->qpos.resize((size_t)V * 4, 0, db->st));
        KCK(db->d_kf.resize((size_t)db->ent_cap * 4, 0, db->st));
        KCK(db->d_seq.resize((size_t)db->ent_cap * 8, 0, db->st));
        KCK(db->max_words.resize(8, 0, db->st));
        KCK(cudaStreamSynchronize(db->st));
        return MCS_OK;
    };
    const int rc = init();
    if (rc) { delete db; return rc; }
    *out = db;
    return MCS_OK;
}

void mcs_kfdb_destroy(mcs_keyframe_db* db) { delete db; }

int mcs_kfdb_add(mcs_keyframe_db* db, int64_t kf_id, const int32_t* bow_words, const double* bow_values, int32_t n_bow) {
    if (!db) return kfail(MCS_ERR_INVALID, "null argument");
    int rc = check_id(kf_id, "key-frame id");
    if (!rc) rc = check_bow(bow_words, bow_values, n_bow, db->n_words);
    if (rc) return rc;
    std::lock_guard<std::mutex> lock(db->mu);
    if ((rc = db->check_device())) return rc;
    if (db->seq + 1 >= kMaxSeq) return kfail(MCS_ERR_UNSUPPORTED, "more than 2^40 add calls");
    if ((rc = db->ensure_ids(kf_id + 1))) return rc;
    bool full = false;
    for (int i = 0; i < n_bow && !full; ++i) full = db->used[bow_words[i]] >= db->cap[bow_words[i]];
    if (full && (rc = db->rebuild())) return rc;
    if (db->pool_used + n_bow > db->pool_cap) {
        const long long nc = std::max(db->pool_cap * 2, db->pool_used + n_bow + 4096);
        KCK(db->d_bw.resize((size_t)nc * 4, (size_t)db->pool_used * 4, db->st));
        KCK(db->d_bv.resize((size_t)nc * 8, (size_t)db->pool_used * 8, db->st));
        db->pool_cap = nc;
    }
    const long long po = db->pool_used;
    if (n_bow > 0) {
        KCK(cudaMemcpyAsync(db->d_bw.as<int>() + po, bow_words, (size_t)n_bow * 4, cudaMemcpyHostToDevice, db->st));
        KCK(cudaMemcpyAsync(db->d_bv.as<double>() + po, bow_values, (size_t)n_bow * 8, cudaMemcpyHostToDevice, db->st));
    }
    db->bow_off[kf_id] = po; db->bow_n[kf_id] = n_bow; db->bow_known[kf_id] = 1;
    KCK(cudaMemcpyAsync(db->d_boff.as<long long>() + kf_id, &db->bow_off[kf_id], 8, cudaMemcpyHostToDevice, db->st));
    KCK(cudaMemcpyAsync(db->d_bn.as<int>() + kf_id, &db->bow_n[kf_id], 4, cudaMemcpyHostToDevice, db->st));
    KCK(launch_kfdb_add(db->file(), db->d_bw.as<int>() + po, n_bow, (int)kf_id, db->seq, db->st));
    KCK(cudaStreamSynchronize(db->st));
    for (int i = 0; i < n_bow; ++i) ++db->used[bow_words[i]];
    db->pool_used += n_bow;
    db->n_used += n_bow;
    ++db->seq;
    return MCS_OK;
}

int mcs_kfdb_erase(mcs_keyframe_db* db, int64_t kf_id) {
    if (!db) return kfail(MCS_ERR_INVALID, "null argument");
    int rc = check_id(kf_id, "key-frame id");
    if (rc) return rc;
    std::lock_guard<std::mutex> lock(db->mu);
    if ((rc = db->check_device())) return rc;
    if (kf_id >= db->n_ids || !db->bow_known[kf_id] || db->bow_n[kf_id] == 0) return MCS_OK;   // nothing to remove (ref :52-73)
    const int n = db->bow_n[kf_id];
    KCK(launch_kfdb_erase(db->file(), db->d_bw.as<int>() + db->bow_off[kf_id], n, (int)kf_id, db->st));
    KCK(cudaStreamSynchronize(db->st));
    db->tombs += n;                            // an upper bound: a word may hold no live entry of kf_id any more
    if (db->tombs > 4096 && 2 * db->tombs > db->n_used) return db->rebuild();
    return MCS_OK;
}

int mcs_kfdb_clear(mcs_keyframe_db* db) {
    if (!db) return kfail(MCS_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lock(db->mu);
    int rc = db->check_device();
    if (rc) return rc;
    KCK(cudaMemsetAsync(db->d_len.p, 0, (size_t)db->n_words * 4, db->st));
    KCK(cudaStreamSynchronize(db->st));
    std::fill(db->used.begin(), db->used.end(), 0);
    db->tombs = 0; db->n_used = 0;
    return MCS_OK;
}

static int kfdb_detect(mcs_keyframe_db* db, bool loop, int64_t qid, const int32_t* bow_words, const double* bow_values, int32_t n_bow,
                       const int64_t* connected, int32_t n_connected, const int64_t* covis, int64_t n_covis_rows, double min_score,
                       int64_t* candidates, int32_t capacity, int32_t* n_candidates) {
    if (!db || !n_candidates) return kfail(MCS_ERR_INVALID, "null argument");
    *n_candidates = 0;
    if (capacity < 0 || (capacity > 0 && !candidates)) return kfail(MCS_ERR_INVALID, "bad candidate buffer");
    if (qid < 0) return kfail(MCS_ERR_INVALID, "query id must be non-negative");
    int rc = check_bow(bow_words, bow_values, n_bow, db->n_words);
    if (rc) return rc;
    if (n_connected < 0 || (n_connected > 0 && !connected)) return kfail(MCS_ERR_INVALID, "bad connected key-frame list");
    for (int i = 0; i < n_connected; ++i) if (connected[i] < 0) return kfail(MCS_ERR_INVALID, "connected key-frame ids must be non-negative");
    if (n_covis_rows < 0 || (n_covis_rows > 0 && !covis)) return kfail(MCS_ERR_INVALID, "bad covisibility rows");
    for (long long i = 0; i < n_covis_rows * 10; ++i)
        if (covis[i] < -1 || covis[i] >= kMaxIds) return kfail(MCS_ERR_INVALID, "covisibility entries must be -1 or a key-frame id");
    std::lock_guard<std::mutex> lock(db->mu);
    if ((rc = db->check_device())) return rc;
    if (db->n_ids == 0) return MCS_OK;         // nothing was ever added: no word is shared
    // only rows of ids that can be candidates are read; their neighbours get state slots (initial values if never touched)
    const long long rows = std::min<long long>(n_covis_rows, db->n_ids);
    long long need = 0;
    for (long long i = 0; i < rows * 10; ++i) need = std::max<long long>(need, covis[i] + 1);
    if ((rc = db->ensure_ids(need))) return rc;
    const int n = (int)db->n_ids, nmap = (n + 31) / 32;
    // one upload: query words | query values | connected bitmap | covisibility rows (int32)
    const size_t o_val = align8((size_t)n_bow * 4), o_con = o_val + (size_t)n_bow * 8, o_cov = align8(o_con + (size_t)nmap * 4);
    const size_t up_bytes = o_cov + (size_t)rows * 40;
    KCK(db->h_up.reserve(up_bytes));
    if (db->upload.bytes < up_bytes) KCK(db->upload.resize(std::max(up_bytes, 2 * db->upload.bytes), 0, db->st));
    char* h = (char*)db->h_up.p;
    if (n_bow > 0) { std::memcpy(h, bow_words, (size_t)n_bow * 4); std::memcpy(h + o_val, bow_values, (size_t)n_bow * 8); }
    unsigned* bits = (unsigned*)(h + o_con);
    std::memset(bits, 0, (size_t)nmap * 4);
    if (loop) for (int i = 0; i < n_connected; ++i) if (connected[i] < n) bits[connected[i] >> 5] |= 1u << (connected[i] & 31);
    int* cv = (int*)(h + o_cov);
    for (long long i = 0; i < rows * 10; ++i) cv[i] = (int)covis[i];
    KCK(cudaMemcpyAsync(db->upload.p, h, up_bytes, cudaMemcpyHostToDevice, db->st));
    char* d = (char*)db->upload.p;
    KfdbQuery q{};
    q.id = qid; q.loop = loop; q.min_score = min_score;
    q.q_words = (const int*)d; q.q_values = (const double*)(d + o_val); q.n_q = n_bow;
    q.connected = (const unsigned*)(d + o_con); q.covis = (const int*)(d + o_cov); q.n_covis_rows = (int)rows;
    q.n_ids = n;
    q.st_query = (loop ? db->loop_q : db->reloc_q).as<long long>();
    q.st_words = (loop ? db->loop_w : db->reloc_w).as<int>();
    q.st_score = (loop ? db->loop_s : db->reloc_s).as<double>();
    q.qpos = db->qpos.as<int>(); q.cnt = db->cnt.as<int>(); q.key = db->key.as<unsigned long long>();
    q.status = db->status.as<unsigned char>(); q.sc = db->sc.as<double>(); q.acc = db->acc.as<double>(); q.best = db->best.as<int>();
    q.win = db->win.as<unsigned long long>(); q.sort_key = db->sort_key.as<unsigned long long>(); q.sort_val = db->sort_val.as<int>();
    q.sort_cap = (int)db->ids_cap; q.max_words = db->max_words.as<int>(); q.out = db->out.as<int>();
    const KfdbBows b{db->d_bw.as<int>(), db->d_bv.as<double>(), db->d_boff.as<long long>(), db->d_bn.as<int>()};
    KCK(launch_kfdb_query(db->file(), b, q, db->n_words, db->scoring, db->st));
    const size_t down = 1 + (size_t)std::min<long long>(capacity, n);
    KCK(db->h_out.reserve(down * 4));
    KCK(cudaMemcpyAsync(db->h_out.p, db->out.p, down * 4, cudaMemcpyDeviceToHost, db->st));
    KCK(cudaStreamSynchronize(db->st));
    const int* res = (const int*)db->h_out.p;
    *n_candidates = res[0];
    if (res[0] > capacity) return kfail(MCS_ERR_CAPACITY, "candidate buffer too small: *n_candidates holds the required count");
    for (int i = 0; i < res[0]; ++i) candidates[i] = res[1 + i];
    return MCS_OK;
}

int mcs_kfdb_detect_loop_candidates(mcs_keyframe_db* db, int64_t kf_id, const int32_t* bow_words, const double* bow_values,
                                    int32_t n_bow, const int64_t* connected, int32_t n_connected, const int64_t* covis,
                                    int64_t n_covis_rows, double min_score, int64_t* candidates, int32_t capacity,
                                    int32_t* n_candidates) {
    return kfdb_detect(db, true, kf_id, bow_words, bow_values, n_bow, connected, n_connected, covis, n_covis_rows, min_score,
                       candidates, capacity, n_candidates);
}

int mcs_kfdb_detect_relocalisation_candidates(mcs_keyframe_db* db, int64_t frame_id, const int32_t* bow_words,
                                              const double* bow_values, int32_t n_bow, const int64_t* covis,
                                              int64_t n_covis_rows, int64_t* candidates, int32_t capacity,
                                              int32_t* n_candidates) {
    return kfdb_detect(db, false, frame_id, bow_words, bow_values, n_bow, nullptr, 0, covis, n_covis_rows, 0.0, candidates,
                       capacity, n_candidates);
}

}  // extern "C"
