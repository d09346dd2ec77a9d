// mcs_bow_api.cu -- C ABI of the bag-of-words row (include/mcs_b200.h): vocabulary object, transform, score,
// feature-vector guided SearchByBoW.  Tree descent and group distances run on the GPU (bow_kernels.cu); the
// std::map bookkeeping of DBoW2 and the matcher's order-dependent greedy rule are replayed on the host.
#include <algorithm>
#include <cfloat>
#include <climits>
#include <cmath>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "../../include/mcs_b200.h"
#include "kernels.h"
#include "dev_scratch.h"
#include "vocabulary.h"

using namespace mcs;

void mcs_set_error_(const std::string& msg);   // mcs_api.cu

namespace {

int bfail(int code, const std::string& msg) { mcs_set_error_(msg); return code; }

#define BCK(expr)                                                                                      \
    do {                                                                                               \
        cudaError_t e__ = (expr);                                                                      \
        if (e__ != cudaSuccess) {                                                                      \
            cudaGetLastError();                                                                        \
            return bfail(e__ == cudaErrorNoDevice || e__ == cudaErrorInsufficientDriver ? MCS_ERR_NO_DEVICE : MCS_ERR_CUDA, \
                         std::string(#expr) + ": " + cudaGetErrorString(e__));                         \
        }                                                                                              \
    } while (0)


}  // namespace


extern "C" {

int mcs_vocabulary_create(int32_t k, int32_t L, int32_t scoring, int32_t weighting, int32_t n_nodes, const int32_t* parent,
                          const double* weight, const uint8_t* descriptors, const int32_t* node_order, int32_t n_words,
                          const int32_t* word_node, mcs_vocabulary** out) {
    if (!out) return bfail(MCS_ERR_INVALID, "null argument");
    *out = nullptr;
    if (!parent || !weight || !descriptors || !word_node) return bfail(MCS_ERR_INVALID, "null argument");
    if (n_nodes < 2 || n_words < 1 || k < 1 || L < 1) return bfail(MCS_ERR_INVALID, "empty vocabulary");
    if (scoring < 0 || scoring > 5 || weighting < 0 || weighting > 3) return bfail(MCS_ERR_INVALID, "unknown scoring / weighting type");
    // children in the reference's push_back order (ref TemplatedVocabulary.h:1596-1608)
    std::vector<int> cnt(n_nodes + 1, 0), ids(n_nodes - 1), won(n_nodes, -1);
    std::vector<uint8_t> seen(n_nodes, 0);
    for (int i = 0; i + 1 < n_nodes; ++i) {
        const int nid = node_order ? node_order[i] : i + 1;
        if (nid < 1 || nid >= n_nodes || seen[nid]) return bfail(MCS_ERR_INVALID, "node_order is not a permutation of 1..n_nodes-1");
        seen[nid] = 1;
        const int pid = parent[nid];
        if (pid < 0 || pid >= n_nodes || pid == nid) return bfail(MCS_ERR_INVALID, "parent id out of range");
        ++cnt[pid + 1];
    }
    for (int i = 0; i < n_nodes; ++i)
        if (cnt[i + 1] > 65535) return bfail(MCS_ERR_UNSUPPORTED, "more than 65535 children under one node (the descent packs the child position in 16 bits)");
    for (int i = 0; i < n_nodes; ++i) cnt[i + 1] += cnt[i];
    if (cnt[1] == 0) return bfail(MCS_ERR_INVALID, "the root has no children");
    std::vector<int> cur(cnt.begin(), cnt.end() - 1);
    for (int i = 0; i + 1 < n_nodes; ++i) {
        const int nid = node_order ? node_order[i] : i + 1;
        ids[cur[parent[nid]]++] = nid;
    }
    for (int i = 1; i < n_nodes; ++i) {                  // every node must hang under the root: walk up at most n_nodes steps
        int a = i, steps = 0;
        while (a != 0 && steps <= n_nodes) { a = parent[a]; ++steps; }
        if (a != 0) return bfail(MCS_ERR_INVALID, "parent links contain a cycle");
    }
    for (int w = 0; w < n_words; ++w) {
        const int nid = word_node[w];
        if (nid < 1 || nid >= n_nodes || cnt[nid + 1] != cnt[nid]) return bfail(MCS_ERR_INVALID, "word_node must name leaves");
        won[nid] = w;
    }
    for (int i = 1; i < n_nodes; ++i)
        if (cnt[i + 1] == cnt[i] && won[i] < 0) return bfail(MCS_ERR_INVALID, "a leaf has no word id");
    int ndev = 0;
    BCK(cudaGetDeviceCount(&ndev));
    if (ndev == 0) return bfail(MCS_ERR_NO_DEVICE, "no CUDA device");
    mcs_vocabulary* v = new mcs_vocabulary();
    v->k = k; v->L = L; v->scoring = scoring; v->weighting = weighting; v->n_nodes = n_nodes; v->n_words = n_words;
    cudaError_t e = cudaGetDevice(&v->device);
    if (e == cudaSuccess) e = v->child_off.alloc((size_t)(n_nodes + 1) * 4);
    if (e == cudaSuccess) e = v->child_ids.alloc((size_t)(n_nodes - 1) * 4);
    if (e == cudaSuccess) e = v->desc.alloc((size_t)n_nodes * 32);
    if (e == cudaSuccess) e = v->word_of_node.alloc((size_t)n_nodes * 4);
    if (e == cudaSuccess) e = v->weight.alloc((size_t)n_nodes * 8);
    if (e == cudaSuccess) e = cudaMemcpy(v->child_off.p, cnt.data(), (size_t)(n_nodes + 1) * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(v->child_ids.p, ids.data(), (size_t)(n_nodes - 1) * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(v->desc.p, descriptors, (size_t)n_nodes * 32, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(v->word_of_node.p, won.data(), (size_t)n_nodes * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(v->weight.p, weight, (size_t)n_nodes * 8, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        delete v;
        cudaGetLastError();
        return bfail(e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? MCS_ERR_NO_DEVICE : MCS_ERR_CUDA,
                     std::string("vocabulary upload: ") + cudaGetErrorString(e));
    }
    v->view = VocabularyDev{v->child_off.as<int>(), v->child_ids.as<int>(), v->desc.as<uint4>(), v->word_of_node.as<int>(),
                            v->weight.as<double>(), n_nodes, L};
    *out = v;
    return MCS_OK;
}

void mcs_vocabulary_destroy(mcs_vocabulary* voc) { delete voc; }

int mcs_bow_transform(const mcs_vocabulary* voc, const uint8_t* desc, int32_t n, int32_t levelsup, int32_t* word_id, double* weight,
                      int32_t* node_id) {
    if (!voc || (n > 0 && !desc)) return bfail(MCS_ERR_INVALID, "null argument");
    if (n <= 0) return MCS_OK;
    {   // the tree lives on the device that was current when the vocabulary was created: a call from a thread whose current
        // device differs would hand the kernel foreign pointers
        int cur = -1;
        BCK(cudaGetDevice(&cur));
        if (cur != voc->device) return bfail(MCS_ERR_INVALID, "vocabulary was created on another CUDA device than the current one");
    }
    Dev dd, dw, dwt, dn;
    BCK(dd.alloc((size_t)n * 32)); BCK(dw.alloc((size_t)n * 4)); BCK(dwt.alloc((size_t)n * 8)); BCK(dn.alloc((size_t)n * 4));
    BCK(cudaMemcpy(dd.p, desc, (size_t)n * 32, cudaMemcpyHostToDevice));
    BCK(launch_bow_descend(voc->view, dd.as<uint8_t>(), n, levelsup, dw.as<int>(), dwt.as<double>(), dn.as<int>(), nullptr));
    if (word_id) BCK(cudaMemcpy(word_id, dw.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
    if (weight) BCK(cudaMemcpy(weight, dwt.p, (size_t)n * 8, cudaMemcpyDeviceToHost));
    if (node_id) BCK(cudaMemcpy(node_id, dn.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
    BCK(cudaDeviceSynchronize());
    return MCS_OK;
}

int mcs_bow_vectors(const mcs_vocabulary* voc, const uint8_t* desc, int32_t n, int32_t levelsup, int32_t* bow_words,
                    double* bow_values, int32_t* n_bow, int32_t* fv_nodes, int32_t* fv_offsets, int32_t* n_fv, int32_t* fv_features) {
    if (!voc || !n_bow || !n_fv || !fv_offsets) return bfail(MCS_ERR_INVALID, "null argument");
    *n_bow = 0; *n_fv = 0; fv_offsets[0] = 0;
    if (n <= 0) return MCS_OK;
    if (!bow_words || !bow_values || !fv_nodes || !fv_features) return bfail(MCS_ERR_INVALID, "null argument");
    std::vector<int> word(n), node(n);
    std::vector<double> wt(n);
    const int rc = mcs_bow_transform(voc, desc, n, levelsup, word.data(), wt.data(), node.data());
    if (rc) return rc;
    // features whose word is not stopped (w > 0), ref :1157-1161
    std::vector<int> live;
    live.reserve(n);
    for (int i = 0; i < n; ++i) if (wt[i] > 0) live.push_back(i);
    // BowVector = std::map<WordId, WordValue>: ascending word id; addWeight adds in feature order, addIfNotExist keeps the
    // first weight (ref BowVector.cpp:34-59)
    const bool accumulate = voc->weighting == 0 || voc->weighting == 1;        // TF_IDF, TF
    const bool must = voc->scoring != 5, l2 = voc->scoring == 1;               // mustNormalize (ref ScoringObject.h:74-89)
    std::vector<int> order(live);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return word[a] < word[b]; });
    int nb = 0;
    for (size_t s = 0; s < order.size();) {
        size_t e = s;
        double sum = wt[order[s]];
        for (e = s + 1; e < order.size() && word[order[e]] == word[order[s]]; ++e)
            if (accumulate) sum += wt[order[e]];
        bow_words[nb] = word[order[s]]; bow_values[nb] = sum; ++nb;
        s = e;
    }
    if (accumulate && nb > 0 && !must) {                                       // ref :1165-1171
        const double nd = (double)nb;
        for (int i = 0; i < nb; ++i) bow_values[i] /= nd;
    }
    if (must) {                                                                // BowVector::normalize (ref BowVector.cpp:63-87)
        double norm = 0.0;
        if (!l2) for (int i = 0; i < nb; ++i) norm += std::fabs(bow_values[i]);
        else { for (int i = 0; i < nb; ++i) norm += bow_values[i] * bow_values[i]; norm = std::sqrt(norm); }
        if (norm > 0.0) for (int i = 0; i < nb; ++i) bow_values[i] /= norm;
    }
    *n_bow = nb;
    // FeatureVector = std::map<NodeId, vector<unsigned>>: ascending node id, features in insertion (= index) order
    order = live;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return node[a] < node[b]; });
    int nf = 0;
    for (size_t s = 0; s < order.size(); ++s) {
        if (s == 0 || node[order[s]] != node[order[s - 1]]) { fv_nodes[nf] = node[order[s]]; fv_offsets[nf] = (int)s; ++nf; }
        fv_features[s] = order[s];
    }
    fv_offsets[nf] = (int)order.size();
    *n_fv = nf;
    return MCS_OK;
}

int mcs_bow_score(const mcs_vocabulary* voc, const int32_t* w1, const double* v1, int32_t n1, const int32_t* w2, const double* v2,
                  int32_t n2, double* score_out) {
    if (!voc || !score_out || (n1 > 0 && (!w1 || !v1)) || (n2 > 0 && (!w2 || !v2))) return bfail(MCS_ERR_INVALID, "null argument");
    const int kind = voc->scoring;
    const double log_eps = std::log(DBL_EPSILON);                              // GeneralScoring::LOG_EPS (ref ScoringObject.cpp:18)
    double acc = 0;
    int i = 0, j = 0;
    // the reference walks both std::maps with lower_bound jumps; on sorted arrays that is a merge over the common words
    while (i < n1 && j < n2) {
        if (w1[i] < w2[j]) {
            if (kind == 3) acc += v1[i] * (std::log(v1[i]) - log_eps);         // KL: words only v1 holds (ref :196-200)
            ++i;
        } else if (w2[j] < w1[i]) {
            ++j;
        } else {
            const double a = v1[i], b = v2[j];
            if (kind == 0) acc += std::fabs(a - b) - std::fabs(a) - std::fabs(b);
            else if (kind == 1 || kind == 5) acc += a * b;
            else if (kind == 2) { if (a + b != 0.0) acc += a * b / (a + b); }
            else if (kind == 3) { if (a != 0 && b != 0) acc += a * std::log(a / b); }
            else acc += std::sqrt(a * b);
            ++i; ++j;
        }
    }
    if (kind == 0) acc = -acc / 2.0;
    else if (kind == 1) acc = acc >= 1 ? 1.0 : 1.0 - std::sqrt(1.0 - acc);
    else if (kind == 2) acc = 2. * acc;
    else if (kind == 3) for (; i < n1; ++i) if (v1[i] != 0) acc += v1[i] * (std::log(v1[i]) - log_eps);
    *score_out = acc;
    return MCS_OK;
}

int mcs_search_by_bow(const uint8_t* desc1, const uint8_t* mask1, const uint8_t* valid1, int32_t n1, const int32_t* fv1_nodes,
                      const int32_t* fv1_offsets, int32_t n_fv1, const int32_t* fv1_features, const uint8_t* desc2, const uint8_t* mask2,
                      int32_t n2, const int32_t* fv2_nodes, const int32_t* fv2_offsets, int32_t n_fv2, const int32_t* fv2_features,
                      int32_t dim, int32_t th_low, double nnratio, int32_t* match_of_2, int32_t* nmatches) {
    if (!match_of_2 || !nmatches) return bfail(MCS_ERR_INVALID, "null argument");
    if (dim != 16 && dim != 32 && dim != 64) return bfail(MCS_ERR_INVALID, "dim must be 16, 32 or 64");
    *nmatches = 0;
    for (int i = 0; i < n2; ++i) match_of_2[i] = -1;
    if (n1 <= 0 || n2 <= 0 || n_fv1 <= 0 || n_fv2 <= 0) return MCS_OK;
    if (!desc1 || !desc2 || !fv1_nodes || !fv1_offsets || !fv1_features || !fv2_nodes || !fv2_offsets || !fv2_features)
        return bfail(MCS_ERR_INVALID, "null argument");
    // feature vectors are std::map<NodeId, vector<unsigned>> in the reference: node ids strictly ascending, CSR offsets monotone
    for (int side = 0; side < 2; ++side) {
        const int32_t* nodes = side ? fv2_nodes : fv1_nodes;
        const int32_t* off = side ? fv2_offsets : fv1_offsets;
        const int n = side ? n_fv2 : n_fv1;
        if (off[0] < 0) return bfail(MCS_ERR_INVALID, "feature-vector offsets must start at >= 0");
        for (int i = 0; i < n; ++i) {
            if (off[i + 1] < off[i]) return bfail(MCS_ERR_INVALID, "feature-vector offsets must be non-decreasing");
            if (i > 0 && nodes[i] <= nodes[i - 1]) return bfail(MCS_ERR_INVALID, "feature-vector node ids must be strictly ascending");
        }
    }
    const int nf1 = fv1_offsets[n_fv1], nf2 = fv2_offsets[n_fv2];
    for (int i = fv1_offsets[0]; i < nf1; ++i) if (fv1_features[i] < 0 || fv1_features[i] >= n1) return bfail(MCS_ERR_INVALID, "feature index out of range");
    for (int i = fv2_offsets[0]; i < nf2; ++i) if (fv2_features[i] < 0 || fv2_features[i] >= n2) return bfail(MCS_ERR_INVALID, "feature index out of range");
    const bool masked = mask1 && mask2;
    // queries in the reference's visiting order: common nodes ascending, key-frame keypoints in list order (ref :199-217)
    std::vector<GroupQuery> qs;
    for (int a = 0, b = 0; a < n_fv1 && b < n_fv2;) {
        if (fv1_nodes[a] < fv2_nodes[b]) ++a;
        else if (fv2_nodes[b] < fv1_nodes[a]) ++b;
        else {
            const int cs = fv2_offsets[b], cc = fv2_offsets[b + 1] - cs;
            for (int ia = fv1_offsets[a]; ia < fv1_offsets[a + 1]; ++ia) {
                const int i1 = fv1_features[ia];
                if (valid1 && !valid1[i1]) continue;                           // no map point / bad map point (ref :212-216)
                if (cc > 0) qs.push_back(GroupQuery{i1, cs, cc, 0});
            }
            ++a; ++b;
        }
    }
    if (qs.empty()) return MCS_OK;
    Dev d1, m1, d2, m2, dc;
    BCK(d1.alloc((size_t)n1 * dim)); BCK(d2.alloc((size_t)n2 * dim)); BCK(dc.alloc((size_t)nf2 * 4));
    BCK(cudaMemcpy(d1.p, desc1, (size_t)n1 * dim, cudaMemcpyHostToDevice));
    BCK(cudaMemcpy(d2.p, desc2, (size_t)n2 * dim, cudaMemcpyHostToDevice));
    BCK(cudaMemcpy(dc.p, fv2_features, (size_t)nf2 * 4, cudaMemcpyHostToDevice));
    if (masked) {
        BCK(m1.alloc((size_t)n1 * dim)); BCK(m2.alloc((size_t)n2 * dim));
        BCK(cudaMemcpy(m1.p, mask1, (size_t)n1 * dim, cudaMemcpyHostToDevice));
        BCK(cudaMemcpy(m2.p, mask2, (size_t)n2 * dim, cudaMemcpyHostToDevice));
    }
    // distance lists go through a bounded staging buffer: consecutive queries are cut into chunks of <= kChunk distances
    const size_t kChunk = (size_t)8 << 20;
    size_t biggest = 0;
    for (size_t s = 0; s < qs.size();) {
        size_t tot = 0, e = s;
        while (e < qs.size() && (e == s || tot + qs[e].cand_count <= kChunk)) { tot += qs[e].cand_count; ++e; }
        biggest = std::max(biggest, tot);
        s = e;
    }
    Dev dq, dout;
    BCK(dq.alloc(qs.size() * sizeof(GroupQuery))); BCK(dout.alloc(biggest * 4));
    std::vector<int> dist(biggest);
    int nm = 0;
    for (size_t s = 0; s < qs.size();) {
        size_t tot = 0, e = s;
        while (e < qs.size() && (e == s || tot + qs[e].cand_count <= kChunk)) { qs[e].out_off = (int)tot; tot += qs[e].cand_count; ++e; }
        BCK(cudaMemcpy(dq.as<GroupQuery>() + s, qs.data() + s, (e - s) * sizeof(GroupQuery), cudaMemcpyHostToDevice));
        BCK(launch_group_distance(dq.as<GroupQuery>() + s, (int)(e - s), d1.as<uint8_t>(), masked ? m1.as<uint8_t>() : nullptr,
                                  d2.as<uint8_t>(), masked ? m2.as<uint8_t>() : nullptr, dc.as<int>(), dim, dout.as<int>(), nullptr));
        BCK(cudaMemcpy(dist.data(), dout.p, tot * 4, cudaMemcpyDeviceToHost));
        // host: the reference's sequential scan over the GPU distances (ref :226-279)
        for (size_t qi = s; qi < e; ++qi) {
            const GroupQuery& q = qs[qi];
            int best1 = INT_MAX, best2 = INT_MAX, bestIdx = -1;
            const int* dl = dist.data() + q.out_off;
            for (int j = 0; j < q.cand_count; ++j) {
                const int i2 = fv2_features[q.cand_start + j];
                if (match_of_2[i2] >= 0) continue;
                const int d = dl[j];
                if (d < best1) { best2 = best1; best1 = d; bestIdx = i2; }
                else if (d < best2) best2 = d;
            }
            if (best1 <= th_low && (double)best1 < nnratio * (double)best2) { match_of_2[bestIdx] = q.feature; ++nm; }
        }
        s = e;
    }
    *nmatches = nm;
    return MCS_OK;
}

}  // extern "C"
