// C entry points around the REFERENCE's own cMultiKeyFrameDatabase (src/cMultiKeyFrameDatabase.cpp compiled in place by
// oracle/kfdb.mk target `ref`, against ref_kfdb/stub_kfdb.h).  The stand-in key frames live as long as the handle, so their
// query fields persist from call to call as on the reference's key frames.  TEST INFRASTRUCTURE, never linked into the product.
#include <cstdint>
#include <memory>
#include <vector>

#include "cMultiKeyFrameDatabase.h"

using namespace MultiColSLAM;

namespace {
struct RefKfdb {
	ORBVocabulary voc;
	std::unique_ptr<cMultiKeyFrameDatabase> db;
	std::vector<std::unique_ptr<cMultiKeyFrame>> kfs;
	cMultiKeyFrame* kf(long long id)
	{
		while ((long long)kfs.size() <= id) {
			kfs.emplace_back(new cMultiKeyFrame());
			kfs.back()->mnId = kfs.size() - 1;
		}
		return kfs[(size_t)id].get();
	}
};

DBoW2::BowVector bow_of(const int32_t* w, const double* v, int n)
{
	DBoW2::BowVector b;
	for (int i = 0; i < n; ++i) b.insert(b.end(), std::make_pair((DBoW2::WordId)w[i], v[i]));
	return b;
}
}  // namespace

extern "C" {

// ORBVocabulary from the text layout, types set as oracle/ref_dbow2/wrap.cpp does; cMultiKeyFrameDatabase(voc)
void* refkfdb_create(const char* voc_txt, int scoring, int weighting)
{
	RefKfdb* r = new RefKfdb();
	if (!r->voc.loadFromTextFile(voc_txt)) { delete r; return nullptr; }
	r->voc.setScoringType((DBoW2::ScoringType)scoring);
	r->voc.setWeightingType((DBoW2::WeightingType)weighting);
	r->db.reset(new cMultiKeyFrameDatabase(r->voc));
	return r;
}
void refkfdb_free(void* h) { delete (RefKfdb*)h; }

void refkfdb_add(void* h, long long id, const int32_t* w, const double* v, int n)
{
	RefKfdb* r = (RefKfdb*)h;
	cMultiKeyFrame* k = r->kf(id);
	k->mBowVec = bow_of(w, v, n);
	r->db->add(k);
}
void refkfdb_erase(void* h, long long id) { RefKfdb* r = (RefKfdb*)h; r->db->erase(r->kf(id)); }
void refkfdb_clear(void* h) { ((RefKfdb*)h)->db->clear(); }

// loop = 1: DetectLoopCandidates(pKF, minScore) with pKF = a key frame of id qid carrying the given BowVector and connected set;
// loop = 0: DetectRelocalisationCandidates(F) with F->mnId = qid.  covis rows as in include/mcs_b200.h.  Returns the count.
int refkfdb_detect(void* h, int loop, long long qid, const int32_t* w, const double* v, int n, const long long* connected,
                   int n_connected, const long long* covis, long long n_rows, double min_score, long long* out, int cap)
{
	RefKfdb* r = (RefKfdb*)h;
	long long top = n_rows;
	for (long long i = 0; i < n_rows * 10; ++i) top = std::max(top, covis[i] + 1);
	if (top > 0) r->kf(top - 1);
	for (size_t id = 0; id < r->kfs.size(); ++id) {
		r->kfs[id]->covis.clear();
		if ((long long)id < n_rows)
			for (int j = 0; j < 10; ++j)
				if (covis[id * 10 + j] >= 0) r->kfs[id]->covis.push_back(r->kf(covis[id * 10 + j]));
	}
	std::vector<cMultiKeyFrame*> res;
	if (loop) {
		cMultiKeyFrame q;                         // pKF: only mnId, mBowVec and GetConnectedKeyFrames() are read
		q.mnId = (long unsigned int)qid;
		q.mBowVec = bow_of(w, v, n);
		for (int i = 0; i < n_connected; ++i) q.connected.insert(r->kf(connected[i]));
		res = r->db->DetectLoopCandidates(&q, min_score);
	} else {
		cMultiFrame f;
		f.mnId = (long unsigned int)qid;
		f.mBowVec = bow_of(w, v, n);
		res = r->db->DetectRelocalisationCandidates(&f);
	}
	for (size_t i = 0; i < res.size() && (int)i < cap; ++i) out[i] = (long long)res[i]->mnId;
	return (int)res.size();
}

}  // extern "C"
