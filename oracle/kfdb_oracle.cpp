/*
 * kfdb_oracle.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Scalar CPU restatement of the reference's key-frame database (src/cMultiKeyFrameDatabase.cpp, paths relative to the original
 * project), the parity checker of the GPU database (mcs_kfdb_*) for tests/ and __graft_entry__.smoke().  Nothing under
 * multicol_slam_b200/ may call into this file.  Pinned against the reference's own database compiled in place
 * (oracle/_ref/libkfdb_ref.so, recipe oracle/kfdb.mk) through tests/golden/kfdb_ref.npz (tests/test_kfdb_cpu.py).
 * Scores come from the oracle's DBoW2 restatement, mcso_bow_score of libmcs_oracle.so (pinned by tests/test_bow_cpu.py).
 *
 * Build: oracle/kfdb.mk (g++ -O2 -std=c++17 -ffp-contract=off, linked against libmcs_oracle.so).
 */
#include <algorithm>
#include <list>
#include <utility>
#include <vector>

extern "C" {

double mcso_bow_score(int scoring, const int* w1, const double* v1, int n1, const int* w2, const double* v2, int n2);   // mcs_oracle.cpp

// ---- key-frame database: cMultiKeyFrameDatabase, src/cMultiKeyFrameDatabase.cpp ------------------------------------------
// A literal restatement over std::list, as the reference keeps it.  Key frames are stand-ins indexed by id that carry the
// fields the database reads and writes (include/cMultiKeyFrame.h:176-204); the fields the reference leaves uninitialised
// (src/cMultiKeyFrame.cpp:44-45 sets only the two query ids) start at 0 here, as in the product.
namespace {
struct OKF {
    std::vector<int> w;                  // mBowVec (words ascending) ...
    std::vector<double> v;               // ... and values
    long long loopQuery = 0, relocQuery = 0;
    int loopWords = 0, relocWords = 0;
    double loopScore = 0.0, relocScore = 0.0;
};
struct OKFDB {
    int scoring = 0;
    std::vector<std::list<int>> inv;     // mvInvertedFile
    std::vector<OKF> kf;
    OKF& at(long long id) { if ((size_t)id >= kf.size()) kf.resize((size_t)id + 1); return kf[(size_t)id]; }
};
}  // namespace

void* mcso_kfdb_create(int n_words, int scoring) {             // :36-40
    OKFDB* db = new OKFDB();
    db->scoring = scoring;
    db->inv.resize((size_t)n_words);
    return db;
}
void mcso_kfdb_destroy(void* h) { delete (OKFDB*)h; }

void mcso_kfdb_add(void* h, long long id, const int* w, const double* v, int n) {   // :43-50
    OKFDB* db = (OKFDB*)h;
    OKF& k = db->at(id);
    k.w.assign(w, w + n); k.v.assign(v, v + n);
    for (int i = 0; i < n; ++i) db->inv[(size_t)w[i]].push_back((int)id);
}

void mcso_kfdb_erase(void* h, long long id) {                  // :52-73
    OKFDB* db = (OKFDB*)h;
    if ((size_t)id >= db->kf.size()) return;
    for (int word : db->kf[(size_t)id].w) {
        std::list<int>& l = db->inv[(size_t)word];
        for (auto it = l.begin(); it != l.end(); ++it)
            if (*it == id) { l.erase(it); break; }
    }
}

void mcso_kfdb_clear(void* h) {                                // :75-79
    OKFDB* db = (OKFDB*)h;
    const size_t n = db->inv.size();
    db->inv.clear(); db->inv.resize(n);
}

// DetectLoopCandidates (:82-215, loop = 1) and DetectRelocalisationCandidates (:217-327, loop = 0).  covis row id = the ten best
// covisibility key frames of id (-1 = none), rows 0..n_rows-1.  Returns the candidate count; writes at most cap ids.
int mcso_kfdb_detect(void* h, int loop, long long qid, const int* qw, const double* qv, int nq, const long long* connected,
                     int n_connected, const long long* covis, long long n_rows, double minScore, long long* out, int cap) {
    OKFDB* db = (OKFDB*)h;
    std::vector<long long> conn(connected, connected + (loop ? n_connected : 0));
    std::sort(conn.begin(), conn.end());
    auto isConnected = [&](int id) { return std::binary_search(conn.begin(), conn.end(), (long long)id); };
    auto Q = [&](OKF& k) -> long long& { return loop ? k.loopQuery : k.relocQuery; };
    auto W = [&](OKF& k) -> int& { return loop ? k.loopWords : k.relocWords; };
    auto S = [&](OKF& k) -> double& { return loop ? k.loopScore : k.relocScore; };
    std::list<int> lKFsSharingWords;
    for (int i = 0; i < nq; ++i)                                     // :93-111 / :226-240
        for (int id : db->inv[(size_t)qw[i]]) {
            OKF& k = db->at(id);
            if (Q(k) != qid) {
                W(k) = 0;
                if (!loop || !isConnected(id)) { Q(k) = qid; lKFsSharingWords.push_back(id); }
            }
            W(k)++;
        }
    if (lKFsSharingWords.empty()) return 0;
    int maxCommonWords = 0;                                          // :121-126 / :246-251
    for (int id : lKFsSharingWords) maxCommonWords = std::max(maxCommonWords, W(db->at(id)));
    const int minCommonWords = static_cast<int>((double)maxCommonWords * 0.8);
    std::list<std::pair<double, int>> lScoreAndMatch;
    for (int id : lKFsSharingWords) {                                // :132-149 / :257-269
        OKF& k = db->at(id);
        if (W(k) > minCommonWords) {
            const double si = mcso_bow_score(db->scoring, qw, qv, nq, k.w.data(), k.v.data(), (int)k.w.size());
            S(k) = si;
            if (!loop || si >= minScore) lScoreAndMatch.push_back(std::make_pair(si, id));
        }
    }
    if (lScoreAndMatch.empty()) return 0;
    std::list<std::pair<double, int>> lAccScoreAndMatch;
    double bestAccScore = loop ? minScore : 0;
    for (auto& sm : lScoreAndMatch) {                                // :157-181 / :276-299
        double bestScore = sm.first, accScore = sm.first;
        int pBestKF = sm.second;
        if (sm.second < n_rows)
            for (int j = 0; j < 10; ++j) {
                const long long nb = covis[(size_t)sm.second * 10 + j];
                if (nb < 0) continue;
                OKF& k2 = db->at(nb);
                if (Q(k2) != qid || (loop && W(k2) <= minCommonWords)) continue;
                accScore += S(k2);
                if (S(k2) > bestScore) { pBestKF = (int)nb; bestScore = S(k2); }
            }
        lAccScoreAndMatch.push_back(std::make_pair(accScore, pBestKF));
        if (accScore > bestAccScore) bestAccScore = accScore;
    }
    const double minScoreToRetain = 0.75 * bestAccScore;             // :183-212 / :301-324
    std::vector<int> seen;
    int n = 0;
    for (auto& am : lAccScoreAndMatch)
        if (am.first > minScoreToRetain && std::find(seen.begin(), seen.end(), am.second) == seen.end()) {
            seen.push_back(am.second);
            if (n < cap) out[n] = am.second;
            ++n;
        }
    return n;
}

}  // extern "C"
