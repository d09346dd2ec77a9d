// vocabulary.h -- the vocabulary object behind the C ABI's opaque mcs_vocabulary (created in mcs_bow_api.cu, also read by the
// key-frame database in mcs_kfdb_api.cu for its size, scoring type and device).
#pragma once
#include "kernels.h"
#include "dev_scratch.h"

struct mcs_vocabulary {
    int k = 0, L = 0, scoring = 0, weighting = 0, n_nodes = 0, n_words = 0, device = 0;
    mcs::Dev child_off, child_ids, desc, word_of_node, weight;
    mcs::VocabularyDev view{};
};
