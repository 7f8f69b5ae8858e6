// Test driver: hvo_shim::fill (shim/ORBVocabularyGPU.h) turns one frame's BoW rows of the frame call into the reference's BowVector /
// FeatureVector, and hvo_shim::VocabularyArrays reads a vocabulary object's tree.  Host code only: runs without a GPU.
//   in.bin : int32 magic, nframes, cap ; per frame int32 bow_count, fv_count ; then [n][cap] int32 bow_words, [n][cap] double bow_values,
//            [n][cap] int32 fv_order, [n][cap] int32 node_of
//   out.bin: per frame int32 nwords, (uint32 word, double value) pairs in map order, int32 nnodes, per node uint32 node, int32 k, k uint32
//            features; then the arrays VocabularyArrays reads from a small fixed tree: int32 n, L, child_start [n+1], nchild, child_ids,
//            word [n], weight [n], desc [n][32]
#include <cstdint>
#include <cstdio>
#include <map>
#include <vector>

#include <opencv2/core/core.hpp>

#include "DBoW2/FeatureVector.h"
#include "ORBVocabularyGPU.h"

typedef std::map<unsigned int, double> BowVector;   // DBoW2::BowVector is a std::map<WordId, WordValue> (BowVector.h)

// The members of DBoW2::TemplatedVocabulary that VocabularyArrays reads (protected there as well).
class TinyVocabulary {
public:
    TinyVocabulary() {
        // root 0 -> {1, 2}; 1 -> {3, 4, 5}; 2 is a leaf (uneven depth); the leaves 2..5 are the words 0..3
        const int children[6][3] = {{1, 2, -1}, {3, 4, 5}, {-1, -1, -1}, {-1, -1, -1}, {-1, -1, -1}, {-1, -1, -1}};
        const int words[6] = {0, 0, 0, 1, 2, 3};
        m_nodes.resize(6);
        for (int i = 0; i < 6; ++i) {
            for (int c = 0; c < 3; ++c) if (children[i][c] >= 0) m_nodes[i].children.push_back((unsigned)children[i][c]);
            m_nodes[i].weight = i == 4 ? 0.0 : 0.25 * i;   // node 4: a stopped word
            m_nodes[i].word_id = (unsigned)words[i];
            if (i > 0) {
                m_nodes[i].descriptor = cv::Mat(1, 32, CV_8U);
                for (int b = 0; b < 32; ++b) m_nodes[i].descriptor.ptr<uint8_t>()[b] = (uint8_t)(7 * i + b);
            }
        }
        m_L = 2;
    }

protected:
    struct Node {
        std::vector<unsigned> children;
        cv::Mat descriptor;
        double weight = 0;
        unsigned word_id = 0;
        bool isLeaf() const { return children.empty(); }
    };
    std::vector<Node> m_nodes;
    int m_L = 0;
};

int main(int argc, char** argv) {
    if (argc != 3) { std::fprintf(stderr, "usage: shim_bow_fill in.bin out.bin\n"); return 2; }
    FILE* fi = std::fopen(argv[1], "rb");
    FILE* fo = std::fopen(argv[2], "wb");
    if (!fi || !fo) return 2;
    int32_t hdr[3];
    if (std::fread(hdr, 4, 3, fi) != 3 || hdr[0] != 0x46424f57) return 3;
    const int n = hdr[1], cap = hdr[2];
    const size_t rows = (size_t)n * cap;
    std::vector<int32_t> counts(2 * (size_t)n), words(rows), order(rows), node_of(rows);
    std::vector<double> values(rows);
    if (std::fread(counts.data(), 4, counts.size(), fi) != counts.size() || std::fread(words.data(), 4, rows, fi) != rows ||
        std::fread(values.data(), 8, rows, fi) != rows || std::fread(order.data(), 4, rows, fi) != rows || std::fread(node_of.data(), 4, rows, fi) != rows)
        return 4;
    std::fclose(fi);

    for (int f = 0; f < n; ++f) {
        const size_t o = (size_t)f * cap;
        BowVector v;
        DBoW2::FeatureVector fv;
        v[12345] = 1.0;          // fill replaces whatever the vectors held
        fv.addFeature(777, 1);
        hvo_shim::fill(&words[o], &values[o], counts[2 * f], &order[o], counts[2 * f + 1], &node_of[o], v, fv);
        const int32_t nw = (int32_t)v.size();
        std::fwrite(&nw, 4, 1, fo);
        for (const auto& e : v) { std::fwrite(&e.first, 4, 1, fo); std::fwrite(&e.second, 8, 1, fo); }
        const int32_t nn = (int32_t)fv.size();
        std::fwrite(&nn, 4, 1, fo);
        for (const auto& e : fv) {
            const int32_t k = (int32_t)e.second.size();
            std::fwrite(&e.first, 4, 1, fo);
            std::fwrite(&k, 4, 1, fo);
            std::fwrite(e.second.data(), 4, k, fo);
        }
    }

    const hvo_shim::VocabularyArrays<TinyVocabulary> a{TinyVocabulary()};
    const int32_t head[2] = {a.n_nodes(), a.levels}, nchild = (int32_t)a.child_ids.size();
    std::fwrite(head, 4, 2, fo);
    std::fwrite(a.child_start.data(), 4, a.child_start.size(), fo);
    std::fwrite(&nchild, 4, 1, fo);
    std::fwrite(a.child_ids.data(), 4, a.child_ids.size(), fo);
    std::fwrite(a.word.data(), 4, a.word.size(), fo);
    std::fwrite(a.weight.data(), 8, a.weight.size(), fo);
    std::fwrite(a.desc.data(), 1, a.desc.size(), fo);
    std::fclose(fo);
    return 0;
}
