// stub_kfdb.h -- data-only stand-ins for cMultiKeyFrame / cMultiFrame as src/cMultiKeyFrameDatabase.cpp reads them, so that the
// reference's key-frame database compiles WHERE IT LIES without the rest of the system.   TEST INFRASTRUCTURE (oracle/kfdb.mk
// target `ref` -> oracle/_ref/libkfdb_ref.so).
//
// Force-included (-include) ahead of the reference's headers; it pre-defines the include guards of include/cMultiKeyFrame.h and
// include/cMultiFrame.h, so those two files are skipped.  Everything else is the reference's own code:
// cMultiKeyFrameDatabase.{h,cpp}, cORBVocabulary.h and the vendored DBoW2.  The classes carry the fields the database touches,
// under the reference's names and types (include/cMultiKeyFrame.h:176-204, include/cMultiFrame.h:119), filled by wrap.cpp.
// The reference initialises only mnLoopQuery / mnRelocQuery (src/cMultiKeyFrame.cpp:44-45); the other four fields start at 0
// here, the value the library defines for them.
#pragma once
#define MULTIKEYFRAME_H
#define MULTIFRAME_H

#include <set>
#include <vector>

#include "DBoW2/DBoW2/BowVector.h"

namespace MultiColSLAM
{
class cMultiKeyFrame
{
public:
	long unsigned int mnId = 0;
	long unsigned int mnLoopQuery = 0;
	int mnLoopWords = 0;
	double mLoopScore = 0.0;
	long unsigned int mnRelocQuery = 0;
	int mnRelocWords = 0;
	double mRelocScore = 0.0;
	DBoW2::BowVector mBowVec;

	std::set<cMultiKeyFrame*> connected;          // GetConnectedKeyFrames() at query time
	std::vector<cMultiKeyFrame*> covis;           // GetBestCovisibilityKeyFrames(10) at query time, best first

	std::set<cMultiKeyFrame*> GetConnectedKeyFrames() { return connected; }
	std::vector<cMultiKeyFrame*> GetBestCovisibilityKeyFrames(const int& N)
	{
		return std::vector<cMultiKeyFrame*>(covis.begin(), covis.begin() + std::min<size_t>(covis.size(), (size_t)N));
	}
};

class cMultiFrame
{
public:
	long unsigned int mnId = 0;
	DBoW2::BowVector mBowVec;
};
}  // namespace MultiColSLAM
