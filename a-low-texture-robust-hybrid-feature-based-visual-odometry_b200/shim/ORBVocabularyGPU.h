// Device side of Frame::ComputeBoW (reference src/Frame.cc:1692-1699): the one call it makes,
//
//     mpORBvocabulary->transform(vCurrentDesc, mBowVec, mFeatVec, 4);
//
// i.e. DBoW2::TemplatedVocabulary<FORB::TDescriptor, FORB>::transform(features, BowVector&, FeatureVector&, levelsup)
// (Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1137-1206, 1228-1270), with the same signature and results:
//
//     #include "shim/ORBVocabularyGPU.h"
//     hvo_shim::BowTransformerT<ORBVocabulary> bow(*mpORBvocabulary);         // once, after the vocabulary is loaded
//     bow.transform(vCurrentDesc, mBowVec, mFeatVec, 4);                       // instead of mpORBvocabulary->transform(...)
//
// The vocabulary object stays the reference's own (loading, scoring, the key-frame database keep using it); the constructor reads its tree
// (m_nodes, m_L: protected members, reached through a derived accessor, no change to DBoW2) once and hands it to the device as arrays
// (hvo_bow_set_vocabulary).  transform() descends the tree on the GPU (hvo_bow_transform: one warp per descriptor), and fills the two
// std::map-derived outputs in ascending key order (hvo_shim::fill), which is the order the reference's own insertions produce; BowVector
// values are the reference's doubles bit for bit (accumulated and L1-normalised in its order).  TF-IDF / L1 is what ORB-SLAM2's vocabulary
// uses (ORBvoc.txt header); other weighting / scoring types are refused at construction.
//
// A frame integration that extracts with hvo_frame_* / hvo_seq_* gets the same vectors from the frame call instead (INTEGRATION.md §5):
//
//     hvo_shim::VocabularyArrays<ORBVocabulary> va(*mpORBvocabulary);            // the same arrays, read once
//     hvo_frame_set_vocabulary(frame_handle, va.n_nodes(), va.child_start.data(), va.child_ids.data(), va.desc.data(), va.weight.data(),
//                              va.word.data(), va.levels, 4);
//     ...  hvo_frame_extract_batch_bow(frame_handle, gray, depth, n, &out, &bow);
//     hvo_shim::fill(&bow_words[f * cap], &bow_values[f * cap], bow_counts[f], &fv_order[f * cap], fv_counts[f], &node_of[f * cap],
//                    mBowVec, mFeatVec);                                       // frame f; Frame::ComputeBoW then finds mBowVec filled
#ifndef HVO_SHIM_ORBVOCABULARYGPU_H
#define HVO_SHIM_ORBVOCABULARYGPU_H

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <utility>
#include <vector>

#include "hvo_capi.h"

namespace hvo_shim {

// The vocabulary tree of the reference's own object (m_nodes, m_L) as the arrays hvo_bow_set_vocabulary / hvo_frame_set_vocabulary take.
template <class TVoc>
struct VocabularyArrays {
    std::vector<int32_t> child_start, child_ids, word;
    std::vector<uint8_t> desc;
    std::vector<double> weight;
    int levels = 0;

    explicit VocabularyArrays(const TVoc& voc) {
        const auto& nodes = voc.*(Access::nodes());
        levels = voc.*(Access::levels());
        const int n = (int)nodes.size();
        child_start.assign(n + 1, 0);
        word.assign(n, -1);
        desc.assign((size_t)n * 32, 0);
        weight.assign(n, 0.0);
        for (int i = 0; i < n; ++i) {
            for (size_t c = 0; c < nodes[i].children.size(); ++c) child_ids.push_back((int32_t)nodes[i].children[c]);
            child_start[i + 1] = (int32_t)child_ids.size();
            if (!nodes[i].descriptor.empty()) std::memcpy(&desc[(size_t)i * 32], nodes[i].descriptor.template ptr<uint8_t>(), 32);
            weight[i] = nodes[i].weight;
            if (i != 0 && nodes[i].isLeaf()) word[i] = (int32_t)nodes[i].word_id;
        }
    }
    int n_nodes() const { return (int)weight.size(); }

private:
    // m_nodes / m_L are protected in TemplatedVocabulary (TemplatedVocabulary.h:417-439); a derived class may form pointers to them
    struct Access : public TVoc {
        static auto nodes() -> decltype(&Access::m_nodes) { return &Access::m_nodes; }
        static auto levels() -> decltype(&Access::m_L) { return &Access::m_L; }
    };
};

// One frame's rows of hvo_bow_transform / hvo_frame_bow_outputs -> the reference's BowVector and FeatureVector (types deduced), as
// TemplatedVocabulary::transform leaves them: words[0 .. nwords) ascending with their values; fv_order[0 .. nfv) sorted by (node_of, feature).
template <class BowVector, class FeatureVector>
void fill(const int32_t* words, const double* values, int nwords, const int32_t* fv_order, int nfv, const int32_t* node_of, BowVector& v,
          FeatureVector& fv) {
    v.clear();
    fv.clear();
    typedef typename BowVector::key_type WordId;
    typedef typename BowVector::mapped_type WordValue;
    typedef typename FeatureVector::key_type NodeId;
    for (int k = 0; k < nwords; ++k) v.insert(v.end(), std::make_pair((WordId)words[k], (WordValue)values[k]));   // ascending word id
    for (int k = 0; k < nfv; ++k) {                                                                                 // ascending (node, feature)
        const NodeId nid = (NodeId)node_of[fv_order[k]];
        typename FeatureVector::iterator it = fv.end();
        if (fv.empty() || (--it)->first != nid) it = fv.insert(fv.end(), std::make_pair(nid, typename FeatureVector::mapped_type()));
        it->second.push_back((unsigned int)fv_order[k]);
    }
}

template <class TVoc>
class BowTransformerT {
public:
    explicit BowTransformerT(const TVoc& voc, int device = 0) : h_(nullptr), ok_(false) {
        if (hvo_bow_create(device, &h_) != HVO_OK) { std::fprintf(stderr, "BowTransformer: %s\n", hvo_last_error()); return; }
        const VocabularyArrays<TVoc> a(voc);
        const int n = a.n_nodes();
        ok_ = n > 0 && hvo_bow_set_vocabulary(h_, n, a.child_start.data(), a.child_ids.empty() ? nullptr : a.child_ids.data(), a.desc.data(),
                                              a.weight.data(), a.word.data(), a.levels) == HVO_OK;
        if (!ok_) std::fprintf(stderr, "BowTransformer: %s\n", n > 0 ? hvo_last_error() : "empty vocabulary");
    }
    ~BowTransformerT() { hvo_bow_destroy(h_); }
    BowTransformerT(const BowTransformerT&) = delete;
    BowTransformerT& operator=(const BowTransformerT&) = delete;
    bool valid() const { return ok_; }

    // TemplatedVocabulary::transform(features, v, fv, levelsup); BowVector / FeatureVector are the reference's own types (deduced)
    template <class BowVector, class FeatureVector>
    void transform(const std::vector<cv::Mat>& features, BowVector& v, FeatureVector& fv, int levelsup) const {
        v.clear();
        fv.clear();
        const int n = (int)features.size();
        if (!ok_ || n == 0) return;
        std::vector<uint8_t> desc((size_t)n * 32);
        for (int i = 0; i < n; ++i) std::memcpy(&desc[(size_t)i * 32], features[i].template ptr<uint8_t>(), 32);
        const int32_t offsets[2] = {0, n};
        std::vector<int32_t> node_of(n), words(n), order(n);
        std::vector<double> values(n);
        int32_t nwords = 0, nfeat = 0;
        if (hvo_bow_transform(h_, desc.data(), offsets, 1, levelsup, nullptr, node_of.data(), &nwords, words.data(), values.data(), order.data(), &nfeat) !=
            HVO_OK) {
            std::fprintf(stderr, "BowTransformer: %s\n", hvo_last_error());
            return;
        }
        fill(words.data(), values.data(), nwords, order.data(), nfeat, node_of.data(), v, fv);
    }

private:
    hvo_bow* h_;
    bool ok_;
};

}  // namespace hvo_shim

#endif
