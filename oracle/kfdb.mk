# Key-frame database test infrastructure, built after oracle/Makefile (which writes libmcs_oracle.so and _ref/voc_small_9_6.txt):
#   libkfdb_oracle.so     restatement of cMultiKeyFrameDatabase (kfdb_oracle.cpp), scores from libmcs_oracle.so
#   _ref/libkfdb_ref.so   the REFERENCE's own key-frame database (src/cMultiKeyFrameDatabase.cpp) with its vendored DBoW2, compiled
#                         where it lies against data-only stand-ins of cMultiKeyFrame / cMultiFrame (ref_kfdb/stub_kfdb.h,
#                         force-included); built only where the reference sources exist, git-ignored like the rest of _ref.
# usage: make -C oracle -f kfdb.mk
CXX = g++
CXXFLAGS ?= -O2 -std=c++17 -ffp-contract=off -fPIC -Wall -Wno-unused-function -pthread
REF ?= /root/reference
DBOW := $(REF)/ThirdParty/DBoW2
all: libkfdb_oracle.so ref
libkfdb_oracle.so: kfdb_oracle.cpp libmcs_oracle.so
	$(CXX) $(CXXFLAGS) -shared -o $@ kfdb_oracle.cpp -L. -lmcs_oracle -Wl,-rpath,'$$ORIGIN'
ref:
	@if [ -f $(REF)/src/cMultiKeyFrameDatabase.cpp ] && [ -d $(DBOW) ]; then mkdir -p _ref && \
	  $(CXX) -O2 -std=c++11 -fPIC -shared -w -ffp-contract=off -Iref_dbow2/stub -I$(REF)/include -I$(REF)/ThirdParty -I$(DBOW) \
	    -include ref_kfdb/stub_kfdb.h ref_kfdb/wrap.cpp $(REF)/src/cMultiKeyFrameDatabase.cpp $(DBOW)/DBoW2/BowVector.cpp \
	    $(DBOW)/DBoW2/FeatureVector.cpp $(DBOW)/DBoW2/FORB.cpp $(DBOW)/DBoW2/ScoringObject.cpp $(DBOW)/DUtils/Random.cpp \
	    $(DBOW)/DUtils/Timestamp.cpp -Wl,--no-undefined -o _ref/libkfdb_ref.so; \
	else echo "oracle: $(REF) not present, keeping prebuilt _ref/libkfdb_ref.so (if any)"; fi
clean:
	rm -f libkfdb_oracle.so
.PHONY: all ref clean
