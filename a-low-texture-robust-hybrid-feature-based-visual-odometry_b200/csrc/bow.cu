// Bag-of-words transform for sm_100a: Frame::ComputeBoW (reference src/Frame.cc:1692-1699) =
// DBoW2::TemplatedVocabulary<FORB::TDescriptor, FORB>::transform(features, BowVector&, FeatureVector&, levelsup = 4)
// (Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1137-1206, single-feature descent :1228-1270, FORB::distance FORB.cpp:81-101,
// BowVector::addWeight / normalize BowVector.cpp:33-83, FeatureVector::addFeature FeatureVector.cpp) for the vocabulary ORB-SLAM2 uses:
// TF-IDF weights, L1 scoring (so the vector is L1-normalised at the end).
//
//   k_bow_descend   one tile of T = 8, 16 or 32 lanes per descriptor (the smallest that holds the vocabulary's largest branching
//                   factor; wider nodes are scored T children at a time): at every level the children of the current node are scored
//                   (8 x __popc per lane), the first child of minimum distance wins (strict '<' in child order, as in the reference),
//                   until a leaf; the node passed at level L - levelsup is kept for the FeatureVector
//   k_bow_frame     one CTA per frame: (word, feature) keys sorted in shared memory; one thread per distinct word accumulates its
//                   weights in feature order (value = w; value += w ...: the additions BowVector::addWeight performs), words are
//                   compacted in ascending order (std::map order), one thread sums |value| in that order (BowVector::normalize L1)
//                   and every value is divided by the norm; a second sort by (node, feature) gives the FeatureVector order
// All floating point is double, one rounding per operation, in the reference's order: the vectors are bit-identical.
//
// Both kernels serve two layouts of the descriptor rows (BowRows): the compact one of hvo_bow_transform (frame f = rows offsets[f] ..
// offsets[f+1]) and the frame handle's (frame f = rows f * orb_capacity .., kp_counts[f] of them, the counts read on the device).  Rows
// at or past a frame's count are neither read nor written.
#include <algorithm>
#include <climits>
#include <new>

#include "hvo_common.cuh"

namespace hvo {

static const int kBowMaxFeatures = 4096;   // per frame (shared-memory sort)

// frame f = rows base(f) .. base(f) + count(f) of the per-row arrays
struct BowRows {
    const int* offsets;   // compact layout: base = offsets[f], count = offsets[f+1] - offsets[f]
    const int* counts;    // otherwise: base = f * stride, count = counts[f]
    int stride;
    __device__ __forceinline__ int base(int f) const { return offsets ? offsets[f] : f * stride; }
    __device__ __forceinline__ int count(int f) const { return offsets ? offsets[f + 1] - offsets[f] : counts[f]; }
    __device__ __forceinline__ bool valid(int i) const { return offsets || i % stride < counts[i / stride]; }   // i < total
};

template <int T>
__global__ void __launch_bounds__(128) k_bow_descend(const uint4* __restrict__ desc, BowRows rows, int total, const int* __restrict__ child_start,
                                                     const int* __restrict__ child_ids, const uint4* __restrict__ node_desc,
                                                     const double* __restrict__ node_weight, const int* __restrict__ node_word, int nid_level,
                                                     int* __restrict__ word_of, int* __restrict__ node_of, double* __restrict__ weight_of) {
    const int i = (int)(((long long)blockIdx.x * 128 + threadIdx.x) / T), lane = threadIdx.x & (T - 1);
    if (i >= total || !rows.valid(i)) return;   // the whole tile leaves together
    const unsigned tile = T == 32 ? 0xffffffffu : ((1u << T) - 1u) << (threadIdx.x & 31 & ~(T - 1));
    const uint4 qa = desc[2 * (size_t)i], qb = desc[2 * (size_t)i + 1];
    int cur = 0, level = 0, nid = 0;   // nid stays the root when nid_level <= 0 (TemplatedVocabulary.h:1240)
    while (true) {
        const int b = child_start[cur], e = child_start[cur + 1];
        if (b == e) break;             // leaf
        ++level;
        unsigned best = 0xffffffffu;   // (distance << 16 | position among the children): the minimum is the first child of least distance,
                                       // whatever the tile width
        for (int base = b; base < e; base += T) {
            const int c = base + lane;
            unsigned key = 0xffffffffu;
            if (c < e) {
                const int id = child_ids[c];
                const uint4 da = node_desc[2 * id], db = node_desc[2 * id + 1];
                const int d = __popc(qa.x ^ da.x) + __popc(qa.y ^ da.y) + __popc(qa.z ^ da.z) + __popc(qa.w ^ da.w) + __popc(qb.x ^ db.x) +
                              __popc(qb.y ^ db.y) + __popc(qb.z ^ db.z) + __popc(qb.w ^ db.w);
                key = ((unsigned)d << 16) | (unsigned)(c - b);
            }
            best = min(best, __reduce_min_sync(tile, key));
        }
        cur = child_ids[b + (int)(best & 0xffffu)];
        if (level == nid_level) nid = cur;
    }
    if (lane == 0) {
        const double w = node_weight[cur];
        word_of[i] = w > 0 ? node_word[cur] : -1;   // "if(w > 0) // not stopped"
        node_of[i] = nid;
        weight_of[i] = w;
    }
}

__device__ __forceinline__ void bow_bitonic_sort(unsigned long long* key, int N) {   // N = power of two, all threads of the CTA
    for (int k = 2; k <= N; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = threadIdx.x; t < N; t += blockDim.x) {
                const int p = t ^ j;
                if (p > t) {
                    const unsigned long long a = key[t], b = key[p];
                    const bool up = (t & k) == 0;
                    if ((a > b) == up) { key[t] = b; key[p] = a; }
                }
            }
            __syncthreads();
        }
}

__global__ void __launch_bounds__(256) k_bow_frame(BowRows rows, const int* __restrict__ word_of, const int* __restrict__ node_of,
                                                   const double* __restrict__ weight_of, int* __restrict__ bow_counts, int* __restrict__ bow_words,
                                                   double* __restrict__ bow_values, int* __restrict__ fv_order, int* __restrict__ fv_counts) {
    extern __shared__ unsigned long long key[];   // [N]
    __shared__ int s_scan[256];
    __shared__ int s_total;
    __shared__ double s_norm;
    const int f = blockIdx.x, tid = threadIdx.x;
    const int base = rows.base(f), n = rows.count(f);
    int N = 1;
    while (N < n) N <<= 1;
    // ---- BowVector: sort by (word, feature); stopped features go to the end ----
    for (int t = tid; t < N; t += 256) {
        unsigned long long k = ~0ull;
        if (t < n && word_of[base + t] >= 0) k = ((unsigned long long)(unsigned)word_of[base + t] << 32) | (unsigned)t;
        key[t] = k;
    }
    __syncthreads();
    bow_bitonic_sort(key, N);
    // heads of the runs of equal words, compacted in ascending word order
    const int per = (N + 255) / 256;               // consecutive elements per thread
    int heads = 0;
    for (int t = tid * per; t < min((tid + 1) * per, N); ++t) {
        const unsigned long long k = key[t];
        if (k != ~0ull && (t == 0 || (key[t - 1] >> 32) != (k >> 32))) ++heads;
    }
    s_scan[tid] = heads;
    __syncthreads();
    if (tid == 0) {
        int acc = 0;
        for (int t = 0; t < 256; ++t) { const int v = s_scan[t]; s_scan[t] = acc; acc += v; }
        s_total = acc;
    }
    __syncthreads();
    int out = s_scan[tid];
    for (int t = tid * per; t < min((tid + 1) * per, N); ++t) {
        const unsigned long long k = key[t];
        if (k != ~0ull && (t == 0 || (key[t - 1] >> 32) != (k >> 32))) {
            const unsigned word = (unsigned)(k >> 32);
            double v = weight_of[base + (int)(k & 0xffffffffu)];                      // insert(id, w)
            for (int u = t + 1; u < N && (key[u] >> 32) == word; ++u) v = __dadd_rn(v, weight_of[base + (int)(key[u] & 0xffffffffu)]);  // += w, in feature order
            bow_words[base + out] = (int)word;
            bow_values[base + out] = v;
            ++out;
        }
    }
    __syncthreads();
    const int nw = s_total;
    if (tid == 0) {   // BowVector::normalize(L1): the sum runs over the map in key order
        double norm = 0.0;
        for (int t = 0; t < nw; ++t) norm = __dadd_rn(norm, fabs(bow_values[base + t]));
        s_norm = norm;
        bow_counts[f] = nw;
    }
    __syncthreads();
    const double norm = s_norm;
    if (norm > 0.0)
        for (int t = tid; t < nw; t += 256) bow_values[base + t] = __ddiv_rn(bow_values[base + t], norm);
    __syncthreads();
    // ---- FeatureVector: (node, feature) ascending over the features that were not stopped ----
    for (int t = tid; t < N; t += 256) {
        unsigned long long k = ~0ull;
        if (t < n && word_of[base + t] >= 0) k = ((unsigned long long)(unsigned)node_of[base + t] << 32) | (unsigned)t;
        key[t] = k;
    }
    __syncthreads();
    bow_bitonic_sort(key, N);
    int cnt = 0;
    for (int t = tid; t < n; t += 256) {
        const unsigned long long k = key[t];
        fv_order[base + t] = k == ~0ull ? -1 : (int)(k & 0xffffffffu);
        cnt += k != ~0ull;
    }
    s_scan[tid] = cnt;
    __syncthreads();
    if (tid == 0) {
        int acc = 0;
        for (int t = 0; t < 256; ++t) acc += s_scan[t];
        fv_counts[f] = acc;
    }
}

}  // namespace hvo

using namespace hvo;

struct hvo_bow {
    int device = 0;
    cudaStream_t stream = nullptr;
    int n_nodes = 0, levels = 0;
    int tile = 32;   // lanes per descriptor in k_bow_descend: 8, 16 or 32 (the largest branching factor, capped at 32)
    int *d_child_start = nullptr, *d_child_ids = nullptr, *d_node_word = nullptr;
    uint8_t* d_node_desc = nullptr;
    double* d_node_weight = nullptr;
    // per call
    int cap = 0, fcap = 0;
    uint8_t* d_desc = nullptr;
    int *d_offsets = nullptr, *d_word = nullptr, *d_node = nullptr, *d_bow_counts = nullptr, *d_bow_words = nullptr, *d_fv = nullptr, *d_fv_counts = nullptr;
    double *d_weight = nullptr, *d_bow_values = nullptr;
    int last_launches = 0;
};

template <class T>
static int bgrow(T*& p, size_t count) {
    if (p) cudaFree(p);
    p = nullptr;
    if (cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T)) != cudaSuccess) { set_error("cudaMalloc: %s", cudaGetErrorString(cudaGetLastError())); return HVO_ERR_CUDA; }
    return HVO_OK;
}

extern "C" {

int hvo_bow_create(int device, hvo_bow** out) {
    HVO_CHECK_ARG(out, "null out");
    *out = nullptr;
    int ndev = 0;
    HVO_CUDA(cudaGetDeviceCount(&ndev));
    if (ndev < 1) { set_error("no CUDA device: libhvofront has no CPU fallback"); return HVO_ERR_CUDA; }
    HVO_CHECK_ARG(device >= 0 && device < ndev, "device index out of range");
    hvo_bow* h = new (std::nothrow) hvo_bow();
    if (!h) { set_error("out of host memory"); return HVO_ERR_ARG; }
    h->device = device;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = create_stream(&h->stream);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_bow_frame, cudaFuncAttributeMaxDynamicSharedMemorySize, kBowMaxFeatures * 8);
    if (e != cudaSuccess) { set_error("hvo_bow_create: %s", cudaGetErrorString(e)); hvo_bow_destroy(h); return HVO_ERR_CUDA; }
    *out = h;
    return HVO_OK;
}

void hvo_bow_destroy(hvo_bow* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    void* bufs[] = {h->d_child_start, h->d_child_ids, h->d_node_word, h->d_node_desc, h->d_node_weight, h->d_desc, h->d_offsets, h->d_word, h->d_node,
                    h->d_bow_counts, h->d_bow_words, h->d_fv, h->d_fv_counts, h->d_weight, h->d_bow_values};
    for (void* b : bufs) if (b) cudaFree(b);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int hvo_bow_set_vocabulary(hvo_bow* h, int n_nodes, const int32_t* child_start, const int32_t* child_ids, const uint8_t* node_desc,
                           const double* node_weight, const int32_t* node_word, int depth_levels) {
    HVO_CHECK_ARG(h && child_start && child_ids && node_desc && node_weight && node_word, "null argument");
    HVO_CHECK_ARG(n_nodes >= 1 && depth_levels >= 1, "empty vocabulary");
    HVO_CHECK_ARG(child_start[0] == 0, "child_start[0] must be 0");
    const int nchild = child_start[n_nodes];
    int max_children = 0;
    for (int i = 0; i < n_nodes; ++i) {
        HVO_CHECK_ARG(child_start[i + 1] >= child_start[i], "child_start must be non-decreasing");
        HVO_CHECK_ARG(child_start[i + 1] - child_start[i] < 65536, "too many children in one node");
        max_children = std::max(max_children, child_start[i + 1] - child_start[i]);
    }
    for (int i = 0; i < nchild; ++i) HVO_CHECK_ARG(child_ids[i] > 0 && child_ids[i] < n_nodes, "child id out of range");
    HVO_CUDA(cudaSetDevice(h->device));
    int st;
    if ((st = bgrow(h->d_child_start, (size_t)n_nodes + 1)) || (st = bgrow(h->d_child_ids, nchild)) || (st = bgrow(h->d_node_word, n_nodes)) ||
        (st = bgrow(h->d_node_desc, (size_t)n_nodes * 32)) || (st = bgrow(h->d_node_weight, n_nodes)))
        return st;
    cudaStream_t s = h->stream;
    HVO_CUDA(cudaMemcpyAsync(h->d_child_start, child_start, ((size_t)n_nodes + 1) * 4, cudaMemcpyHostToDevice, s));
    if (nchild) HVO_CUDA(cudaMemcpyAsync(h->d_child_ids, child_ids, (size_t)nchild * 4, cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(h->d_node_word, node_word, (size_t)n_nodes * 4, cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(h->d_node_desc, node_desc, (size_t)n_nodes * 32, cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(h->d_node_weight, node_weight, (size_t)n_nodes * 8, cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaStreamSynchronize(s));
    h->n_nodes = n_nodes; h->levels = depth_levels;
    h->tile = max_children <= 8 ? 8 : max_children <= 16 ? 16 : 32;
    return HVO_OK;
}

static int bow_reserve(hvo_bow* h, int total, int nframes) {
    int st;
    if (total > h->cap) {
        const int cap = std::max(total, 4096);
        if ((st = bgrow(h->d_desc, (size_t)cap * 32)) || (st = bgrow(h->d_word, cap)) || (st = bgrow(h->d_node, cap)) || (st = bgrow(h->d_weight, cap)) ||
            (st = bgrow(h->d_bow_words, cap)) || (st = bgrow(h->d_bow_values, cap)) || (st = bgrow(h->d_fv, cap)))
            return st;
        h->cap = cap;
    }
    if (nframes > h->fcap) {
        const int cap = std::max(nframes, 64);
        if ((st = bgrow(h->d_offsets, (size_t)cap + 1)) || (st = bgrow(h->d_bow_counts, cap)) || (st = bgrow(h->d_fv_counts, cap))) return st;
        h->fcap = cap;
    }
    return HVO_OK;
}

// The two kernels on `nframes` frames laid out as `rows` (`total` rows, at most `max_rows` per frame), asynchronous on `s`.
static int bow_launch(const hvo_bow* h, cudaStream_t s, const uint8_t* d_desc, BowRows rows, int total, int nframes, int max_rows, int levelsup,
                      int* word_of, int* node_of, double* weight_of, int* bow_counts, int* bow_words, double* bow_values, int* fv_order, int* fv_counts) {
    const uint4* q = reinterpret_cast<const uint4*>(d_desc);
    const uint4* nd = reinterpret_cast<const uint4*>(h->d_node_desc);
    const int nid_level = h->levels - levelsup;
    const unsigned blocks = (unsigned)(((long long)total * h->tile + 127) / 128);
#define HVO_BOW_DESCEND(T) k_bow_descend<T><<<blocks, 128, 0, s>>>(q, rows, total, h->d_child_start, h->d_child_ids, nd, h->d_node_weight, \
                                                                   h->d_node_word, nid_level, word_of, node_of, weight_of)
    if (h->tile == 8) HVO_BOW_DESCEND(8);
    else if (h->tile == 16) HVO_BOW_DESCEND(16);
    else HVO_BOW_DESCEND(32);
#undef HVO_BOW_DESCEND
    int N = 1;
    while (N < max_rows) N <<= 1;
    k_bow_frame<<<nframes, 256, (size_t)N * 8, s>>>(rows, word_of, node_of, weight_of, bow_counts, bow_words, bow_values, fv_order, fv_counts);
    HVO_CUDA(cudaGetLastError());
    return HVO_OK;
}

static int bow_run(hvo_bow* h, const uint8_t* d_desc, int total, int nframes, const int32_t* offsets, int levelsup) {
    cudaStream_t s = h->stream;
    int maxn = 0;
    for (int f = 0; f < nframes; ++f) maxn = std::max(maxn, offsets[f + 1] - offsets[f]);
    HVO_CHECK_ARG(maxn <= kBowMaxFeatures, "more than 4096 features in one frame");
    HVO_CUDA(cudaMemcpyAsync(h->d_offsets, offsets, ((size_t)nframes + 1) * 4, cudaMemcpyHostToDevice, s));
    const int st = bow_launch(h, s, d_desc, BowRows{h->d_offsets, nullptr, 0}, total, nframes, maxn, levelsup, h->d_word, h->d_node, h->d_weight,
                              h->d_bow_counts, h->d_bow_words, h->d_bow_values, h->d_fv, h->d_fv_counts);
    h->last_launches = 2;
    return st;
}

int hvo_bow_transform(hvo_bow* h, const uint8_t* desc, const int32_t* offsets, int nframes, int levelsup, int32_t* word_of, int32_t* node_of,
                      int32_t* bow_counts, int32_t* bow_words, double* bow_values, int32_t* fv_order, int32_t* fv_counts) {
    HVO_CHECK_ARG(h && offsets && bow_counts && bow_words && bow_values, "null argument");
    HVO_CHECK_ARG(h->n_nodes > 0, "no vocabulary (hvo_bow_set_vocabulary)");
    if (nframes <= 0) return HVO_OK;
    HVO_CHECK_ARG(offsets[0] == 0, "offsets[0] must be 0");
    for (int f = 0; f < nframes; ++f) HVO_CHECK_ARG(offsets[f + 1] >= offsets[f], "offsets must be non-decreasing");
    const int total = offsets[nframes];
    for (int f = 0; f < nframes; ++f) { bow_counts[f] = 0; if (fv_counts) fv_counts[f] = 0; }
    if (total == 0) return HVO_OK;
    HVO_CHECK_ARG(desc, "null descriptors");
    HVO_CUDA(cudaSetDevice(h->device));
    int st = bow_reserve(h, total, nframes);
    if (st != HVO_OK) return st;
    cudaStream_t s = h->stream;
    HVO_CUDA(cudaMemcpyAsync(h->d_desc, desc, (size_t)total * 32, cudaMemcpyHostToDevice, s));
    st = bow_run(h, h->d_desc, total, nframes, offsets, levelsup);
    if (st != HVO_OK) return st;
    if (word_of) HVO_CUDA(cudaMemcpyAsync(word_of, h->d_word, (size_t)total * 4, cudaMemcpyDeviceToHost, s));
    if (node_of) HVO_CUDA(cudaMemcpyAsync(node_of, h->d_node, (size_t)total * 4, cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaMemcpyAsync(bow_counts, h->d_bow_counts, (size_t)nframes * 4, cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaMemcpyAsync(bow_words, h->d_bow_words, (size_t)total * 4, cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaMemcpyAsync(bow_values, h->d_bow_values, (size_t)total * 8, cudaMemcpyDeviceToHost, s));
    if (fv_order) HVO_CUDA(cudaMemcpyAsync(fv_order, h->d_fv, (size_t)total * 4, cudaMemcpyDeviceToHost, s));
    if (fv_counts) HVO_CUDA(cudaMemcpyAsync(fv_counts, h->d_fv_counts, (size_t)nframes * 4, cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaStreamSynchronize(s));
    return HVO_OK;
}

int hvo_bow_last_launches(const hvo_bow* h) { return h ? h->last_launches : 0; }

}  // extern "C"

namespace hvo {

// The frame handle's layout: frame f = rows f * stride .., d_counts[f] of them (device), every output [nframes][stride] or [nframes].
int bow_frame_launch(hvo_bow* h, cudaStream_t s, const uint8_t* d_desc, const int32_t* d_counts, int nframes, int stride, int levelsup,
                     double* d_weight, const hvo_frame_bow_outputs* o) {
    HVO_CHECK_ARG(stride <= kBowMaxFeatures, "more than 4096 features in one frame");
    return bow_launch(h, s, d_desc, BowRows{nullptr, d_counts, stride}, nframes * stride, nframes, stride, levelsup, o->word_of, o->node_of, d_weight,
                      o->bow_counts, o->bow_words, o->bow_values, o->fv_order, o->fv_counts);
}
int bow_max_features() { return kBowMaxFeatures; }

}  // namespace hvo
