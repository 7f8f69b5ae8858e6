// Plane extraction (PEAC / agglomerative hierarchical clustering) for sm_100a.
// Replaces PlaneDetection::readDepthImage + runPlaneDetection (reference src/PlaneExtractor.cpp:26-66) and the
// ahc::PlaneFitter they drive (include/peac/AHCPlaneFitter.hpp, AHCPlaneSeg.hpp, AHCParamSet.hpp).
//
//   k_plane_blocks   depth back-projection fused with the 10x10-block plane seeds: validity (missing data, right/down
//                    depth discontinuity), the nine second-order sums, centre, PCA normal, MSE.  The point cloud
//                    (7.4 MB / frame in the reference) is never materialised.  One thread per block walks its 100 pixels
//                    in the reference's row-major order, so the double-precision sums are bit-identical.
//   k_plane_ahc      the graph part, one CTA per frame (frames are independent, a batch fills the machine): initial
//                    edges, min-MSE agglomerative merging (heap + disjoint set in shared memory, neighbour sets as a
//                    bit matrix, merge candidates evaluated one per lane with a 3x3 Jacobi eigen-solve each), block
//                    erosion, the ordered pixel flood fill (8 queue entries x 4 neighbours per warp step, same-pixel
//                    hits applied in queue order), the last merge and the final relabelling.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <new>

#include "hvo_common.cuh"

namespace hvo {

struct BlockOut {  // 96 bytes per block
    double s[9];   // sx sy sz sxx syy szz sxy syz sxz
    int N, queued; // queued: mse < T_mse(INIT) && !nouse
    double mse;
};

struct PlaneCam { double factor, fx, fy, cx, cy, rfx, rfy; };  // rfx = RN(1 / fx), rfy = RN(1 / fy)

// a / b for a divisor b that is fixed per handle, with r = RN(1 / b): q = RN(a r) is a faithful quotient, the remainder
// a - b q is exact in one FMA, and RN(q + rem r) is the correctly rounded a / b (Markstein's theorem; it needs a b whose
// significand is not all ones, true for focal lengths that come from floats, and no over / underflow).  Three dependent
// operations instead of the ~20 of a general double division, bit-identical to it.
__device__ __forceinline__ double div_by_const(double a, double b, double r) {
    const double q = __dmul_rn(a, r);
    const double rem = __fma_rn(-q, b, a);
    return __fma_rn(rem, r, q);
}

// Smallest eigenpair of a symmetric positive semi-definite 3x3 matrix (a covariance) with + - * / sqrt only, so the CPU
// oracle and the CUDA kernels produce bit-identical results: Newton's iteration on the characteristic polynomial
// p(x) = det(K - xI) = -x^3 + c2 x^2 - c1 x + c0 from x = 0 (p is convex and decreasing on (-inf, lambda_min], so the
// iterates approach lambda_min monotonically), then the eigenvector as the largest of the three row cross products
// of K - lambda I.  Accuracy on plane covariances: |d lambda| <= 2e-12 lambda_max, direction error < 1e-7 rad.
__host__ __device__ inline double eig33_lambda_min(double a, double b, double c, double d, double e, double f) {
    const double c2 = a + b + c;
    const double c1 = (a * b - d * d) + (a * c - e * e) + (b * c - f * f);
    const double c0 = a * (b * c - f * f) - d * (d * c - f * e) + e * (d * f - b * e);
    double x = 0, prev = INFINITY;
    for (int k = 0; k < 40; ++k) {
        const double p = ((-x + c2) * x - c1) * x + c0;
        const double dp = (-3 * x + 2 * c2) * x - c1;
        if (dp == 0) break;
        const double dx = p / dp, adx = fabs(dx);
        if (k >= 2 && adx >= prev) break;  // rounding floor reached
        x -= dx;
        prev = adx;
        if (adx <= 1e-16 * c2) break;
    }
    return x;
}
__host__ __device__ inline void eig33_vector(double a, double b, double c, double d, double e, double f, double x, double v[3]) {
    const double r0[3] = {a - x, d, e}, r1[3] = {d, b - x, f}, r2[3] = {e, f, c - x};
    const double u0[3] = {r0[1] * r1[2] - r0[2] * r1[1], r0[2] * r1[0] - r0[0] * r1[2], r0[0] * r1[1] - r0[1] * r1[0]};
    const double u1[3] = {r0[1] * r2[2] - r0[2] * r2[1], r0[2] * r2[0] - r0[0] * r2[2], r0[0] * r2[1] - r0[1] * r2[0]};
    const double u2[3] = {r1[1] * r2[2] - r1[2] * r2[1], r1[2] * r2[0] - r1[0] * r2[2], r1[0] * r2[1] - r1[1] * r2[0]};
    const double n0 = u0[0] * u0[0] + u0[1] * u0[1] + u0[2] * u0[2];
    const double n1 = u1[0] * u1[0] + u1[1] * u1[1] + u1[2] * u1[2];
    const double n2 = u2[0] * u2[0] + u2[1] * u2[1] + u2[2] * u2[2];
    const double* u = u0;
    double n = n0;
    if (n1 > n) { u = u1; n = n1; }
    if (n2 > n) { u = u2; n = n2; }
    if (n > 0) {
        const double s = sqrt(n);
        v[0] = u[0] / s; v[1] = u[1] / s; v[2] = u[2] / s;
    } else {
        v[0] = 0; v[1] = 0; v[2] = 1;
    }
}
__host__ __device__ inline void eig33_smallest(const double K[3][3], double& lam, double v[3]) {
    lam = eig33_lambda_min(K[0][0], K[1][1], K[2][2], K[0][1], K[0][2], K[1][2]);
    eig33_vector(K[0][0], K[1][1], K[2][2], K[0][1], K[0][2], K[1][2], lam, v);
}

// Stats::compute (AHCPlaneSeg.hpp:125-163), split so that the merge loop can rank candidates by MSE (eigenvalue only) and
// compute the eigenvector for the winner alone.  K6 = {Kxx, Kyy, Kzz, Kxy, Kxz, Kyz}; same operations in the same order as
// stats_compute, so the two routes are bit-identical.
__host__ __device__ inline void stats_cov(const double s[9], int N, double K6[6]) {
    const double sc = 1.0 / N;
    K6[0] = s[3] - s[0] * s[0] * sc; K6[3] = s[6] - s[0] * s[1] * sc; K6[4] = s[8] - s[0] * s[2] * sc;
    K6[1] = s[4] - s[1] * s[1] * sc; K6[5] = s[7] - s[1] * s[2] * sc;
    K6[2] = s[5] - s[2] * s[2] * sc;
}
__host__ __device__ inline double stats_mse(const double s[9], int N, double K6[6], double& lam) {
    const double sc = 1.0 / N;
    stats_cov(s, N, K6);
    lam = eig33_lambda_min(K6[0], K6[1], K6[2], K6[3], K6[4], K6[5]);
    return lam * sc;
}
__host__ __device__ inline void stats_finish(const double s[9], int N, const double K6[6], double lam, double center[3], double normal[3]) {
    const double sc = 1.0 / N;
    center[0] = s[0] * sc; center[1] = s[1] * sc; center[2] = s[2] * sc;
    double v[3];
    eig33_vector(K6[0], K6[1], K6[2], K6[3], K6[4], K6[5], lam, v);
    const double sgn = (v[0] * center[0] + v[1] * center[1] + v[2] * center[2] <= 0) ? 1.0 : -1.0;
    normal[0] = sgn * v[0]; normal[1] = sgn * v[1]; normal[2] = sgn * v[2];
}
__host__ __device__ inline void stats_compute(const double s[9], int N, double center[3], double normal[3], double& mse, double& curv) {
    double K6[6], lam;
    mse = stats_mse(s, N, K6, lam);
    stats_finish(s, N, K6, lam, center, normal);
    curv = lam / (K6[0] + K6[1] + K6[2]);
}

__global__ void __launch_bounds__(128) k_plane_blocks(const uint16_t* __restrict__ depth, int w, int h, PlaneCam cam, int Nw, int Nh,
                                                      BlockOut* __restrict__ out) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x, f = blockIdx.y;
    if (b >= Nw * Nh) return;
    const int by = b / Nw, bx = b - by * Nw;
    const uint16_t* D = depth + (long long)f * w * h;
    double s[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    int N = 0;
    bool valid = true;
    for (int ic = 0; ic < 10 && valid; ++ic) {
        const int i = by * 10 + ic;
        for (int jc = 0; jc < 10; ++jc) {
            const int j = bx * 10 + jc;
            const double z = (double)D[(long long)i * w + j] * cam.factor;
            if (z == 0) { valid = false; break; }                       // INIT_STRICT: one missing pixel rejects the block
            const double tdz = 0.04 * fabs(z) + 0.02;                   // ParamSet::T_dz
            if (j + 1 < w) { const double zn = (double)D[(long long)i * w + j + 1] * cam.factor; if (zn != 0 && fabs(z - zn) > tdz) { valid = false; break; } }
            if (i + 1 < h) { const double zn = (double)D[(long long)(i + 1) * w + j] * cam.factor; if (zn != 0 && fabs(z - zn) > tdz) { valid = false; break; } }
            const double x = div_by_const(((double)j - cam.cx) * z, cam.fx, cam.rfx), y = div_by_const(((double)i - cam.cy) * z, cam.fy, cam.rfy);
            s[0] += x; s[1] += y; s[2] += z;
            s[3] += x * x; s[4] += y * y; s[5] += z * z;
            s[6] += x * y; s[7] += y * z; s[8] += x * z;
            ++N;
        }
    }
    BlockOut o;
    if (!valid) { N = 0; for (int k = 0; k < 9; ++k) s[k] = 0; }
    for (int k = 0; k < 9; ++k) o.s[k] = s[k];
    o.N = N;
    o.queued = 0;
    o.mse = 0;
    if (N >= 4) {
        double c[3], n[3], mse, curv;
        stats_compute(s, N, c, n, mse, curv);
        const double t = 1.6e-6 * c[2] * c[2] + 5;  // ParamSet::T_mse(P_INIT): pow(depthSigma*z*z + stdTol_init, 2)
        o.mse = mse;
        o.queued = (mse < t * t) ? 1 : 0;
    }
    out[(long long)f * Nw * Nh + b] = o;
}

// --------------------------------------------------------------------------------------------------------------------
// k_plane_ahc: the graph part of ahc::PlaneFitter::run, one CTA (4 warps) per frame.
//
// Node slots == block ids (creation order of the initial nodes == block scan order).  A merged node takes over the slot
// of the popped node p (p is out of the heap by then, its partner stays in the heap as a `nouse` tombstone, exactly like
// the reference's lazy deletion), so no slot beyond the initial Nb is ever needed.  `key` keeps the creation order
// (reference: pointer / id order of std::set iteration, only consulted on exact MSE ties).  The neighbour sets are rows
// of an Nb x Nb bit matrix in global memory: set union = OR of two rows, erase/insert = one bit.
// The heap reproduces std::priority_queue (libstdc++ push_heap / pop_heap sift order) on mse.
// --------------------------------------------------------------------------------------------------------------------
struct __align__(16) NodeG { double s[9]; double center[3]; double normal[3]; int N; int rid; };  // 128 bytes

#ifndef HVO_AHC_MINBLOCKS
#define HVO_AHC_MINBLOCKS 15  /* resident k_plane_cluster warps per SM the register budget is sized for */
#endif
static const int kMinSupport = 3000, kAhcThreads = 128;
static const int kRowW = 9;  // neighbour-matrix row words per lane: up to 9 * 32 * 32 = 9216 blocks (1280x720)
// beyond that: up to 24 * 32 * 32 = 24576 blocks (1920x1200).  Node ids, keys (< 2 Nb + max_ext), union-log halves and the
// disjoint set stay below 2^16 there, and a heap entry keeps 15 id bits + 17 key bits.
static const int kRowWL = 24;
#define AHC_TH_MERGE 0.50000000000000011   /* cos(pi/180*60) as computed by std::cos */
#define AHC_TH_REFINE 0.86602540378443871  /* cos(pi/180*30) */

struct AhcArgs {
    const uint16_t* depth;   // [B][h][w]
    const BlockOut* blocks;  // [B][Nb]
    NodeG* nodes;            // [B][Nb]
    uint32_t* adj;           // [B][Nb][nw]   (zeroed before launch)
    uint16_t* key;           // [B][Nb]
    double* cand;            // [B][Nb]
    uint32_t* ulog;          // [B][Nb]  union log of the first clustering
    uint16_t* cnode;         // [B][Nb]  node of candidate i
    uint32_t* queue;         // [B][qcap]
    int32_t* membership;     // [B][h*w]   working membershipImg, final labels on exit
    uint8_t* membership8;    // [B][h*w]   optional compact copy of the final labels (255 = no plane)
    double* planes7;         // [B][planes_stride][7]
    int32_t* n_planes;       // [B]
    int32_t* status;         // [B]  0 ok, 1 refinement queue overflow
    long long* cycles;       // [B][4] SM clock cycles: first clustering, erosion + seeds, flood fill, last merge + relabel
    // state handed from kernel to kernel (per frame)
    double* g_mse;           // [B][Nb]
    uint16_t* g_ds;          // [B][2 Nb]   disjoint-set parent, size
    uint32_t* g_nouse;       // [B][nw]
    int16_t* g_blkmap;       // [B][Nb]
    uint16_t* g_ext;         // [B][max_ext]
    uint8_t* g_isvalid;      // [B][max_ext]
    double* g_pl;            // [B][max_ext][7]
    int* g_ctl;              // [B][8]: 0 n_ext, 1 next key
    int w, h, Nw, Nh, nw, qcap, max_ext, planes_stride;
    PlaneCam cam;
    double th_merge, th_refine;
};

__device__ __forceinline__ double ahc_t_ang_init(double z) {  // ParamSet::T_ang(P_INIT, z), AHCParamSet.hpp:99-115
    const double z_near = 500, z_far = 4000, a_near = M_PI / 180.0 * 15.0, a_far = M_PI / 180.0 * 90.0;
    double cz = fmax(z, z_near);
    cz = fmin(cz, z_far);
    const double factor = (a_far - a_near) / (z_far - z_near);
    return cos(factor * cz + a_near - factor * z_near);
}


struct AhcS {  // working set of the clustering kernels (shared memory unless noted)
    double* mse;        // [Nb]  global: exact MSE of every node
    uint32_t* heap;     // [hcap] heap entries (see heap_entry)
    uint32_t idmask;    // low bits of a heap entry that hold the node id
    int idbits;
    uint16_t* stage;    // [32]  the neighbours evaluated in the current round (one per lane)
    uint16_t* parent;   // [Nb]  disjoint set (k_plane_cluster: overlays the heap once it has drained)
    uint16_t* ssize;    // [Nb]
    uint32_t* nouse;    // [ceil(Nb/32)]
    uint16_t* ext;      // [max_ext]
    uint16_t* ext2;     // [max_ext]
    int16_t* plidmap;   // [max_ext]
    uint8_t* isvalid;   // [max_ext]
    int* ctl;           // [8]: 0 heap size, 1 next key, 2 n_ext, 3 n_ext2, 5 union-log length
    uint32_t* ulog;     // global [Nb]: k_plane_cluster logs DisjointSet::Union(x, y) as x | y << 16 and replays the log afterwards
    uint16_t* cnode;    // global [Nb]: node of candidate i (read back only on an exact MSE tie)
};

// Heap entries are one 32-bit word: a monotone quantisation of the MSE (5 exponent bits covering [2^-24, 2^8), the
// remaining bits mantissa; everything below maps to the smallest key, everything above to the largest) with the node id
// in the low `idbits` bits.  Two entries whose keys differ compare as plain unsigned integers; equal keys fall back to the
// exact double MSEs in global memory, so the order is exactly the reference's whatever the quantiser does.  Both children
// of a slot sit in one aligned 8-byte word (the array starts at an address = 4 mod 8).
__device__ __forceinline__ uint32_t heap_entry(const AhcS& S, int v, double mv) {
    const long long b = __double_as_longlong(mv);
    const int e = (int)(b >> 52) - (1023 - 24);  // negative values have a negative exponent field here
    const int mbits = 27 - S.idbits;
    uint32_t key;
    if (e < 0) key = 0u;
    else if (e >= 32) key = (1u << (mbits + 5)) - 1u;
    else key = ((uint32_t)e << mbits) | (uint32_t)((b & 0xfffffffffffffLL) >> (52 - mbits));
    return (key << S.idbits) | (uint32_t)v;
}
#ifdef HVO_AHC_PROF
__device__ int g_less_calls, g_less_ties, g_pops;
#endif
__device__ __forceinline__ bool heap_less(const AhcS& S, uint32_t ea, uint32_t eb) {
#ifdef HVO_AHC_PROF
    ++g_less_calls;
#endif
    if ((ea ^ eb) & ~S.idmask) return ea < eb;
#ifdef HVO_AHC_PROF
    ++g_less_ties;
#endif
    return S.mse[ea & S.idmask] < S.mse[eb & S.idmask];
}
__device__ __forceinline__ void heap_push(AhcS& S, int v, double mv) {  // std::push_heap with comp(a, b) = mse[b] < mse[a]; mv == S.mse[v]
    int hole = S.ctl[0]++;
    const uint32_t ev = heap_entry(S, v, mv);
    while (hole > 0) {
        const int parent = (hole - 1) >> 1;
        const uint32_t ep = S.heap[parent];
        if (!heap_less(S, ev, ep)) break;
        S.heap[hole] = ep;
        hole = parent;
    }
    S.heap[hole] = ev;
}
__device__ __forceinline__ int heap_pop(AhcS& S) {  // std::pop_heap + pop_back
    const int top = (int)(S.heap[0] & S.idmask);
    const int len = --S.ctl[0];  // elements remaining
    if (len == 0) return top;
    const uint32_t ev = S.heap[len];
    int hole = 0, child = 0;
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        const uint2 lr = *reinterpret_cast<const uint2*>(S.heap + child - 1);  // left = child - 1, right = child
        if (heap_less(S, lr.x, lr.y)) { S.heap[hole] = lr.x; --child; }  // comp(first[child], first[child-1])
        else S.heap[hole] = lr.y;
        hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        S.heap[hole] = S.heap[child - 1];
        hole = child - 1;
    }
    while (hole > 0) {  // __push_heap(first, hole, 0, value)
        const int parent = (hole - 1) >> 1;
        const uint32_t ep = S.heap[parent];
        if (!heap_less(S, ev, ep)) break;
        S.heap[hole] = ep;
        hole = parent;
    }
    S.heap[hole] = ev;
    return top;
}
__device__ __forceinline__ int ds_find(const uint16_t* parent, int x) {
    while (parent[x] != x) x = parent[x];
    return x;
}
__device__ __forceinline__ void ds_union(AhcS& S, int x, int y) {  // DisjointSet::Union (union by size, ties keep x's root)
    const int xr = ds_find(S.parent, x), yr = ds_find(S.parent, y);
    if (xr == yr) return;
    if (S.ssize[xr] < S.ssize[yr]) { S.parent[xr] = (uint16_t)yr; S.ssize[yr] = (uint16_t)(S.ssize[yr] + S.ssize[xr]); }
    else { S.parent[yr] = (uint16_t)xr; S.ssize[xr] = (uint16_t)(S.ssize[xr] + S.ssize[yr]); }
}
__device__ __forceinline__ bool nouse_get(const AhcS& S, int i) { return (S.nouse[i >> 5] >> (i & 31)) & 1u; }

// PlaneFitter::ahCluster (AHCPlaneFitter.hpp:983-1189).  Warp-collective (warp 0); extracted planes appended to out[].
// kLogUnions: the disjoint set is not resident (its shared memory is the heap's); unions are logged and replayed later.
#ifdef HVO_AHC_PROF
#define AHC_T(k) { const long long t_ = clock64(); prof[k] += t_ - tl; tl = t_; }
#else
#define AHC_T(k)
#endif
template <bool kLogUnions, int RW>
__device__ void ahc_cluster(const AhcArgs& A, AhcS& S, NodeG* nodes, uint32_t* adj, uint16_t* key, double* cand, uint16_t* out,
                            int* n_out, int lane) {
    const int nw = A.nw;
#ifdef HVO_AHC_PROF
    long long prof[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tl = clock64();
#endif
    while (true) {
        int p = -1;
        if (lane == 0) {
            while (S.ctl[0] > 0) { const int q = heap_pop(S); if (!nouse_get(S, q)) { p = q; break; } }
        }
        p = __shfl_sync(0xffffffffu, p, 0);
        AHC_T(0)
        if (p < 0) break;
        uint32_t* rowp = adj + (size_t)p * nw;
        // row p of the neighbour matrix -> registers (one round trip); neighbour i (ascending slot order) = i-th set bit
        uint32_t rw[RW], rem[RW];
        int pos[RW];
#pragma unroll
        for (int k = 0; k < RW; ++k) { const int wi = k * 32 + lane; rw[k] = (wi < nw) ? rowp[wi] : 0u; }
        const NodeG P = nodes[p];
        int cnt = 0;
#pragma unroll
        for (int k = 0; k < RW; ++k) {
            rem[k] = rw[k]; pos[k] = 0;
            if (k * 32 >= nw) continue;
            const int c = __popc(rw[k]);
            int pre = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int n = __shfl_up_sync(0xffffffffu, pre, o); if (lane >= o) pre += n; }
            const int total = __shfl_sync(0xffffffffu, pre, 31);
            pos[k] = cnt + pre - c;
            cnt += total;
        }
        AHC_T(1)
        // candidate merges: MSE of p + nb for every neighbour with |n_p . n_nb| >= similarityTh_merge, 32 neighbours per
        // round.  Only the eigenvalue is needed to rank them; each lane keeps the sums of its own best candidate and the
        // winning lane finishes the node (eigenvector) alone.
        double bm_l = INFINITY, blam = 0, ms[9];
        int bi_l = -1, mN = 0, mrid = 0, qrid = 0, bnode = -1, nmin_l = 0;
        for (int base = 0; base < cnt; base += 32) {
#pragma unroll
            for (int k = 0; k < RW; ++k) {
                if (k * 32 >= nw) continue;
                while (rem[k] && pos[k] < base + 32) {
                    const int b = __ffs(rem[k]) - 1;
                    rem[k] &= rem[k] - 1;
                    S.stage[pos[k] - base] = (uint16_t)((k * 32 + lane) * 32 + b);
                    ++pos[k];
                }
            }
            __syncwarp();
            const int i = base + lane;
            if (i < cnt) {
                const int q = S.stage[lane];
                const NodeG Q = nodes[q];
                const double sim = fabs(P.normal[0] * Q.normal[0] + P.normal[1] * Q.normal[1] + P.normal[2] * Q.normal[2]);
                double m = INFINITY;
                if (!(sim < A.th_merge)) {
                    double s[9], K6[6], lam;
#pragma unroll
                    for (int k = 0; k < 9; ++k) s[k] = P.s[k] + Q.s[k];
                    m = stats_mse(s, P.N + Q.N, K6, lam);
                    if (!(m == m)) m = INFINITY;  // NaN never wins a `>` comparison in the reference either
                    if (m < bm_l) {
                        bm_l = m; blam = lam; bi_l = i; nmin_l = 1; mN = P.N + Q.N; mrid = P.N >= Q.N ? P.rid : Q.rid;
                        qrid = Q.rid; bnode = q;
#pragma unroll
                        for (int k = 0; k < 9; ++k) ms[k] = s[k];
                    } else if (m == bm_l && m < INFINITY) {
                        ++nmin_l;
                    }
                }
                cand[i] = m;  // only read back on an exact tie
                S.cnode[i] = (uint16_t)q;
            }
            __syncwarp();
        }
        double bm = bm_l;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) bm = fmin(bm, __shfl_xor_sync(0xffffffffu, bm, o));
        AHC_T(2)
        int best_i = -1;
        if (bm < INFINITY) {
            const unsigned holders = __ballot_sync(0xffffffffu, bm_l == bm);
            int ties = (bm_l == bm) ? nmin_l : 0;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) ties += __shfl_xor_sync(0xffffffffu, ties, o);
            if (ties == 1) {
                best_i = __shfl_sync(0xffffffffu, bi_l, __ffs(holders) - 1);
            } else {
                // exact MSE tie: the reference folds in set order (creation order) and replaces the incumbent only if
                // incumbent.N < candidate.mse (sic, AHCPlaneFitter.hpp:1045)
                __syncwarp();
                if (lane == 0) {
                    int inc = -1;
                    unsigned last_key = 0;
                    for (int t = 0; t < ties; ++t) {
                        int pick = -1;
                        unsigned pk = 0xffffffffu;
                        for (int i = 0; i < cnt; ++i) {
                            if (cand[i] != bm) continue;
                            const unsigned k = key[S.cnode[i]];
                            if ((t == 0 || k > last_key) && k < pk) { pk = k; pick = i; }
                        }
                        last_key = pk;
                        if (inc < 0 || (double)(P.N + nodes[S.cnode[inc]].N) < bm) inc = pick;
                    }
                    best_i = inc;
                }
                best_i = __shfl_sync(0xffffffffu, best_i, 0);
            }
        }
        const int owner = best_i & 31;  // the lane that evaluated candidate best_i
        int nb = -1;
        bool merged = false;
        double K6[6];
        if (best_i >= 0) {
            if (lane == owner) {
                if (bi_l != best_i) {  // only after an exact tie inside this lane's own candidates
                    bnode = S.cnode[best_i];
                    const NodeG Q = nodes[bnode];
#pragma unroll
                    for (int k = 0; k < 9; ++k) ms[k] = P.s[k] + Q.s[k];
                    mN = P.N + Q.N;
                    mrid = P.N >= Q.N ? P.rid : Q.rid;
                    qrid = Q.rid;
                    bm_l = stats_mse(ms, mN, K6, blam);
                } else {
                    stats_cov(ms, mN, K6);  // same bits as the ranking pass
                }
                const double cz = ms[2] * (1.0 / mN);
                const double t = 1.6e-6 * cz * cz + 8;  // ParamSet::T_mse(P_MERGING)
                merged = bm_l < t * t;
            }
            merged = __shfl_sync(0xffffffffu, (int)merged, owner) != 0;
            nb = __shfl_sync(0xffffffffu, bnode, owner);
        }
        AHC_T(3)
        if (merged) {
            uint32_t* rownb = adj + (size_t)nb * nw;
            // row[p] = (row[p] | row[nb]) \ {p, nb};  row[nb] = {};  every neighbour x of the merged node: erase nb, insert p.
            // The row of nb is requested first; the owner finishes the merged node while it is in flight.
            uint32_t rn[RW];
#pragma unroll
            for (int k = 0; k < RW; ++k) { const int wi = k * 32 + lane; rn[k] = (wi < nw) ? rownb[wi] : 0u; }
            double mv = 0;
            if (lane == owner) {
                NodeG M;
#pragma unroll
                for (int k = 0; k < 9; ++k) M.s[k] = ms[k];
                stats_finish(ms, mN, K6, blam, M.center, M.normal);
                M.N = mN; M.rid = mrid;
                nodes[p] = M;
                S.mse[p] = bm_l;
                mv = bm_l;
                key[p] = (uint16_t)S.ctl[1]++;
                S.nouse[nb >> 5] |= 1u << (nb & 31);
                if (kLogUnions) S.ulog[S.ctl[5]++] = (uint32_t)P.rid | ((uint32_t)qrid << 16);
                else ds_union(S, P.rid, qrid);
            }
#pragma unroll
            for (int k = 0; k < RW; ++k) {
                const int wi = k * 32 + lane;
                if (wi >= nw) break;
                uint32_t v = rw[k] | rn[k];
                if (wi == (p >> 5)) v &= ~(1u << (p & 31));
                if (wi == (nb >> 5)) v &= ~(1u << (nb & 31));
                rowp[wi] = v;
                rownb[wi] = 0u;
                while (v) {
                    const int x = wi * 32 + __ffs(v) - 1;
                    v &= v - 1;
                    uint32_t* rx = adj + (size_t)x * nw;
                    atomicAnd(&rx[nb >> 5], ~(1u << (nb & 31)));
                    atomicOr(&rx[p >> 5], 1u << (p & 31));
                }
            }
            mv = __shfl_sync(0xffffffffu, mv, owner);
            __syncwarp();
            AHC_T(4)
            if (lane == 0) heap_push(S, p, mv);
            __syncwarp();
            AHC_T(5)
        } else {
            if (lane == 0 && P.N >= kMinSupport) out[(*n_out)++] = (uint16_t)p;
#pragma unroll
            for (int k = 0; k < RW; ++k) {  // disconnectAllNbs
                const int wi = k * 32 + lane;
                if (wi >= nw) break;
                uint32_t v = rw[k];
                while (v) {
                    const int x = wi * 32 + __ffs(v) - 1;
                    v &= v - 1;
                    atomicAnd(&adj[(size_t)x * nw + (p >> 5)], ~(1u << (p & 31)));
                }
                rowp[wi] = 0u;
            }
        }
        __syncwarp();
        // the next node to be popped is known now (heap top): pull its neighbour row and its record towards L1 while
        // lane 0 runs the next pop's sift loop (one 128-byte line per lane covers rows of up to 1024 words, kRowWL uses 768)
        if (S.ctl[0] > 0) {
            const int q = (int)(S.heap[0] & S.idmask);
            const char* rq = (const char*)(adj + (size_t)q * nw);
            if (lane * 128 < nw * 4) asm volatile("prefetch.global.L1 [%0];" ::"l"(rq + lane * 128));
            if (lane == 31) asm volatile("prefetch.global.L1 [%0];" ::"l"((const char*)(nodes + q)));
        }
        AHC_T(6)
    }
#ifdef HVO_AHC_PROF
    if (lane == 0 && kLogUnions) { for (int k = 0; k < 7; ++k) printf("ahc prof[%d] = %lld\n", k, prof[k]); printf("less calls %d ties %d\n", g_less_calls, g_less_ties); }
#endif
    // extractedPlanes sorted by N descending (std::sort on <= 16 elements is an insertion sort; kept stable beyond that)
    if (lane == 0) {
        const int n = *n_out;
        for (int i = 1; i < n; ++i) {
            const uint16_t v = out[i];
            const int vn = nodes[v].N;
            int j = i - 1;
            while (j >= 0 && nodes[out[j]].N < vn) { out[j + 1] = out[j]; --j; }
            out[j + 1] = v;
        }
    }
    __syncwarp();
}

// shared memory of k_plane_cluster: the heap spans every block; the disjoint set reuses the heap's bytes once it has drained
__host__ __device__ inline size_t ahc_cluster_smem_bytes(int Nb, int max_ext) {
    return (size_t)((Nb + 31) / 32) * 4 + 32 + 8 + (size_t)Nb * 4 + 64 + (size_t)max_ext * 7 + 16;
}
__device__ __forceinline__ void ahc_cluster_smem_views(unsigned char* p, int Nb, int max_ext, AhcS& S) {
    S.nouse = (uint32_t*)p; p += (size_t)((Nb + 31) / 32) * 4;
    S.ctl = (int*)p; p += 8 * 4;
    p += (((size_t)p & 7) == 4) ? 0 : 4;  // heap base = 4 mod 8
    S.heap = (uint32_t*)p; S.parent = (uint16_t*)p; S.ssize = S.parent + Nb; p += (size_t)Nb * 4;
    p += 4;
    S.stage = (uint16_t*)p; p += 64;
    S.ext = (uint16_t*)p; p += (size_t)max_ext * 2;
    S.ext2 = (uint16_t*)p; p += (size_t)max_ext * 2;
    S.plidmap = (int16_t*)p; p += (size_t)max_ext * 2;
    S.isvalid = (uint8_t*)p;
    S.idbits = 32 - __clz(Nb - 1);
    S.idmask = (1u << S.idbits) - 1u;
}
// shared memory of k_plane_merge: a heap of at most max_ext planes, the disjoint set resident
__host__ __device__ inline size_t ahc_merge_smem_bytes(int Nb, int max_ext) {
    return (size_t)((Nb + 31) / 32) * 4 + 32 + 8 + (size_t)max_ext * 4 + 8 + (size_t)Nb * 4 + 64 + (size_t)max_ext * 7 + 16;
}
__device__ __forceinline__ void ahc_merge_smem_views(unsigned char* p, int Nb, int max_ext, AhcS& S) {
    S.nouse = (uint32_t*)p; p += (size_t)((Nb + 31) / 32) * 4;
    S.ctl = (int*)p; p += 8 * 4;
    p += (((size_t)p & 7) == 4) ? 0 : 4;  // heap base = 4 mod 8
    S.heap = (uint32_t*)p; p += (size_t)max_ext * 4;
    p += (((size_t)p & 3) ? 4 - ((size_t)p & 3) : 0);
    S.parent = (uint16_t*)p; p += (size_t)Nb * 2;
    S.ssize = (uint16_t*)p; p += (size_t)Nb * 2;
    S.stage = (uint16_t*)p; p += 64;
    S.ext = (uint16_t*)p; p += (size_t)max_ext * 2;
    S.ext2 = (uint16_t*)p; p += (size_t)max_ext * 2;
    S.plidmap = (int16_t*)p; p += (size_t)max_ext * 2;
    S.isvalid = (uint8_t*)p;
    S.idbits = 32 - __clz(Nb - 1);
    S.idmask = (1u << S.idbits) - 1u;
}

// ---- kernel 1 of the graph stage: initial graph + first clustering + block erosion.  One warp per frame. ----
template <int RW>
__global__ void __launch_bounds__(32, HVO_AHC_MINBLOCKS) k_plane_cluster(AhcArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int f = blockIdx.x, lane = threadIdx.x;
    const int Nw = A.Nw, Nh = A.Nh, Nb = Nw * Nh;
    AhcS S;
    ahc_cluster_smem_views(smem_raw, Nb, A.max_ext, S);
    S.mse = A.g_mse + (size_t)f * Nb;
    S.ulog = A.ulog + (size_t)f * Nb;
    S.cnode = A.cnode + (size_t)f * Nb;
    const BlockOut* blocks = A.blocks + (size_t)f * Nb;
    NodeG* nodes = A.nodes + (size_t)f * Nb;
    uint32_t* adj = A.adj + (size_t)f * Nb * A.nw;
    uint16_t* key = A.key + (size_t)f * Nb;
    double* cand = A.cand + (size_t)f * Nb;
    const long long t_start = clock64();
    for (int i = lane; i < (Nb + 31) / 32; i += 32) S.nouse[i] = 0u;
    for (int i = lane; i < A.max_ext; i += 32) S.isvalid[i] = 0;
    if (lane == 0) { S.ctl[0] = 0; S.ctl[1] = Nb; S.ctl[2] = 0; S.ctl[3] = 0; S.ctl[5] = 0; A.status[f] = 0; }
    __syncwarp();
    // ---- initial graph nodes (AHCPlaneFitter.hpp:786-826), pushed in block order ----
    for (int b0 = 0; b0 < Nb; b0 += 32) {
        const int b = b0 + lane;
        double m = INFINITY;
        bool queued = false;
        if (b < Nb) {
            const BlockOut o = blocks[b];
            key[b] = (uint16_t)b;
            queued = o.queued != 0;
            if (queued) {
                NodeG n;
                double curv;
#pragma unroll
                for (int k = 0; k < 9; ++k) n.s[k] = o.s[k];
                n.N = o.N; n.rid = b;
                stats_compute(n.s, n.N, n.center, n.normal, m, curv);
                nodes[b] = n;
            }
            S.mse[b] = m;
        }
        unsigned qm = __ballot_sync(0xffffffffu, queued);
        while (qm) {
            const int j = __ffs(qm) - 1;
            qm &= qm - 1;
            const double mj = __shfl_sync(0xffffffffu, m, j);
            if (lane == 0) heap_push(S, b0 + j, mj);
        }
        __syncwarp();
    }
    // ---- edges (AHCPlaneFitter.hpp:896-954): rows, then columns ----
    for (int i = lane; i < Nh; i += 32)
        for (int j = 1; j < Nw; j += 2) {
            const int c = i * Nw + j;
            if (!blocks[c - 1].queued) { --j; continue; }
            if (!blocks[c].queued) continue;
            if (j < Nw - 1 && !blocks[c + 1].queued) { ++j; continue; }
            const double th = ahc_t_ang_init(nodes[c].center[2]);
            const double* n0 = nodes[c - 1].normal;
            const double* n1 = (j < Nw - 1) ? nodes[c + 1].normal : nodes[c].normal;
            if (fabs(n0[0] * n1[0] + n0[1] * n1[1] + n0[2] * n1[2]) >= th) {
                atomicOr(&adj[(size_t)c * A.nw + ((c - 1) >> 5)], 1u << ((c - 1) & 31));
                atomicOr(&adj[(size_t)(c - 1) * A.nw + (c >> 5)], 1u << (c & 31));
                if (j < Nw - 1) {
                    atomicOr(&adj[(size_t)c * A.nw + ((c + 1) >> 5)], 1u << ((c + 1) & 31));
                    atomicOr(&adj[(size_t)(c + 1) * A.nw + (c >> 5)], 1u << (c & 31));
                }
            } else {
                --j;
            }
        }
    __syncwarp();
    for (int j = lane; j < Nw; j += 32)
        for (int i = 1; i < Nh; i += 2) {
            const int c = i * Nw + j;
            if (!blocks[c - Nw].queued) { --i; continue; }
            if (!blocks[c].queued) continue;
            if (i < Nh - 1 && !blocks[c + Nw].queued) { ++i; continue; }
            const double th = ahc_t_ang_init(nodes[c].center[2]);
            const double* n0 = nodes[c - Nw].normal;
            const double* n1 = (i < Nh - 1) ? nodes[c + Nw].normal : nodes[c].normal;
            if (fabs(n0[0] * n1[0] + n0[1] * n1[1] + n0[2] * n1[2]) >= th) {
                atomicOr(&adj[(size_t)c * A.nw + ((c - Nw) >> 5)], 1u << ((c - Nw) & 31));
                atomicOr(&adj[(size_t)(c - Nw) * A.nw + (c >> 5)], 1u << (c & 31));
                if (i < Nh - 1) {
                    atomicOr(&adj[(size_t)c * A.nw + ((c + Nw) >> 5)], 1u << ((c + Nw) & 31));
                    atomicOr(&adj[(size_t)(c + Nw) * A.nw + (c >> 5)], 1u << (c & 31));
                }
            } else {
                --i;
            }
        }
    __syncwarp();
    ahc_cluster<true, RW>(A, S, nodes, adj, key, cand, S.ext, &S.ctl[2], lane);
    const int ne = S.ctl[2];
    // ---- the heap has drained: its bytes now hold the disjoint set; replay the logged unions in order ----
    for (int b = lane; b < Nb; b += 32) { S.parent[b] = (uint16_t)b; S.ssize[b] = 1; }
    __syncwarp();
    if (lane == 0) {
        const int nu = S.ctl[5];
        uint32_t u = nu > 0 ? S.ulog[0] : 0u;
        for (int i = 0; i < nu; ++i) {
            const uint32_t un = (i + 1 < nu) ? S.ulog[i + 1] : 0u;
            ds_union(S, (int)(u & 0xffffu), (int)(u >> 16));
            u = un;
        }
    }
    __syncwarp();
    // ---- hand the disjoint set over, then flatten it in place: parent[b] becomes the set id of block b (concurrent
    // pointer jumping is safe: a chain read meets either the old parent or the root, both lead to the same root) ----
    uint16_t* g_ds = A.g_ds + (size_t)f * 2 * Nb;
    for (int b = lane; b < Nb; b += 32) { g_ds[b] = S.parent[b]; g_ds[Nb + b] = S.ssize[b]; }
    __syncwarp();
    for (int b = lane; b < Nb; b += 32) { const int r = ds_find(S.parent, b); if (r != b) S.parent[b] = (uint16_t)r; }
    __syncwarp();
    // ---- refineDetails: findBlockMembership (AHCPlaneFitter.hpp:485-587), block part ----
    const uint16_t* setids = S.parent;
    int16_t* g_blkmap = A.g_blkmap + (size_t)f * Nb;
    for (int b = lane; b < Nb; b += 32) {
        const int i = b / Nw, j = b - i * Nw, setid = setids[b];
        int bm = -1;
        if ((int)S.ssize[setid] * 100 >= kMinSupport) {
            bool same = true;
            if (j > 0 && setids[b - 1] != setid) same = false;
            if (j < Nw - 1 && setids[b + 1] != setid) same = false;
            if (i > 0 && setids[b - Nw] != setid) same = false;
            if (i < Nh - 1 && setids[b + Nw] != setid) same = false;  // ERODE_ALL_BORDER
            int plid = 0;  // std::map::operator[] yields 0 for an unknown set id (reference quirk)
            for (int e = 0; e < ne; ++e) if (nodes[S.ext[e]].rid == setid) { plid = e; break; }
            if (same && plid < ne) { bm = plid; S.isvalid[plid] = 1; }
        }
        g_blkmap[b] = (int16_t)bm;
    }
    __syncwarp();
    // ---- hand the rest of the state over ----
    for (int i = lane; i < A.nw; i += 32) A.g_nouse[(size_t)f * A.nw + i] = S.nouse[i];
    for (int i = lane; i < ne; i += 32) {
        const NodeG* n = nodes + S.ext[i];
        double* o = A.g_pl + ((size_t)f * A.max_ext + i) * 7;
        o[0] = n->normal[0]; o[1] = n->normal[1]; o[2] = n->normal[2];
        o[3] = n->center[0]; o[4] = n->center[1]; o[5] = n->center[2];
        o[6] = S.mse[S.ext[i]];
        A.g_ext[(size_t)f * A.max_ext + i] = S.ext[i];
    }
    for (int i = lane; i < A.max_ext; i += 32) A.g_isvalid[(size_t)f * A.max_ext + i] = S.isvalid[i];
    if (lane == 0) {
        A.g_ctl[8 * f + 0] = ne; A.g_ctl[8 * f + 1] = S.ctl[1];
        A.cycles[4 * (size_t)f + 0] = clock64() - t_start;
    }
}

// ---- kernel 2: membership image, refinement seeds and the ordered pixel flood fill.  One CTA of 256 per frame. ----
// A step takes up to 256 consecutive queue entries, one per thread, each with its 4 neighbour visits (1024 visits in
// flight per step).  A visit reads only the state of the pixel it visits, so visits of one step are independent except
// where two of them hit the same pixel: those are applied in queue order by a hash-bucket tournament (a visit goes when it
// is the lowest pending visit of its bucket; equal pixels share a bucket, so the earlier one always went before).
// The reference's distance map is not stored: for a pixel outside the member blocks it always equals the distance to the
// plane the pixel is currently labelled with (FLT_MAX while unlabelled), which is recomputed when needed.
#ifndef HVO_FLOOD_THREADS
#define HVO_FLOOD_THREADS 256
#endif
// a refinement queue entry is pixel | plane << kQPixBits: 22 pixel bits (1920x1200 = 2.3 M pixels), 10 plane bits (max_ext <= 821)
static const int kQPixBits = 22;
static const uint32_t kQPixMask = (1u << kQPixBits) - 1u;
// visits per step = 4 * threads; a visit's rank inside the step takes kFloodPosBits bits of the tournament word, 4 buckets per visit
static const int kFloodThreads = HVO_FLOOD_THREADS;
static const int kFloodPosBits = kFloodThreads == 128 ? 9 : (kFloodThreads == 256 ? 10 : (kFloodThreads == 512 ? 11 : 12));
// Two hash tables of 2 buckets per visit each: a visit goes when it holds the bucket of its pixel in EITHER table.  Visits of one pixel
// share their bucket in both tables, so only the earliest pending one can hold either; a visit of another pixel blocks it falsely only if it
// collides in both (a few percent instead of ~ 20 % with one table of the same total size): 4.2 -> fewer tournament rounds per step.
static const int kFloodBuckets = 4 << kFloodPosBits, kFloodHashShift = 32 - (kFloodPosBits + 1);
static_assert(kFloodThreads == 128 || kFloodThreads == 256 || kFloodThreads == 512 || kFloodThreads == 1024, "flood CTA size");

struct FloodPix { double px, py, z; };
// (double)v for a 16-bit value without the conversion pipe: 2^52 + v is exact, subtracting 2^52 gives v
__device__ __forceinline__ double u16_to_double(uint16_t v) { return __hiloint2double(0x43300000, (int)v) - 4503599627370496.0; }
__device__ __forceinline__ bool flood_point(const AhcArgs& A, const uint16_t* D, int cIdx, int cx, int cy, FloodPix& P) {
    P.z = (double)D[cIdx] * A.cam.factor;
    if (P.z == 0) return false;
    P.px = div_by_const(((double)cx - A.cam.cx) * P.z, A.cam.fx, A.cam.rfx);
    P.py = div_by_const(((double)cy - A.cam.cy) * P.z, A.cam.fy, A.cam.rfy);
    return true;
}
__device__ __forceinline__ float flood_dist(const double* p, const FloodPix& P) {
    return (float)fabs(p[0] * (P.px - p[3]) + p[1] * (P.py - p[4]) + p[2] * (P.z - p[5]));
}

// 64 registers x 256 threads: four frames per SM.  More resident frames (register cap 5..8 CTAs, measured) only slow the
// kernel down: its steps are bound by the scattered 32-byte sector traffic of the membership / depth images.
#ifndef HVO_FLOOD_MINBLOCKS
#define HVO_FLOOD_MINBLOCKS (1024 / HVO_FLOOD_THREADS)
#endif
__global__ void __launch_bounds__(kFloodThreads, HVO_FLOOD_MINBLOCKS) k_plane_flood(AhcArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ unsigned s_bucket[kFloodBuckets];
    __shared__ int s_wsum[kFloodThreads / 32];
    __shared__ int s_head, s_tail, s_overflow;
    const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int Nw = A.Nw, Nh = A.Nh, Nb = Nw * Nh, W = A.w, H = A.h, npix = W * H;
    double* pl = (double*)smem_raw;                                   // [max_ext][8]: normal, center, mse, 9 mse + 1e-5
    int16_t* blkmap = (int16_t*)(smem_raw + (size_t)A.max_ext * 64);  // [Nb]
    uint16_t* ext = (uint16_t*)(blkmap + Nb);                         // [max_ext]
    const uint16_t* D = A.depth + (size_t)f * npix;
    uint32_t* adj = A.adj + (size_t)f * Nb * A.nw;
    uint32_t* queue = A.queue + (size_t)f * A.qcap;
    int32_t* mem = A.membership + (size_t)f * npix;
    const long long t_start = clock64();
    const int ne = A.g_ctl[8 * f + 0];
    for (int i = tid; i < ne; i += kFloodThreads) {
        const double* g = A.g_pl + ((size_t)f * A.max_ext + i) * 7;
        double* p = pl + 8 * i;
#pragma unroll
        for (int k = 0; k < 7; ++k) p[k] = g[k];
        p[7] = 9 * g[6] + 1e-5;
        ext[i] = A.g_ext[(size_t)f * A.max_ext + i];
    }
    for (int b = tid; b < Nb; b += kFloodThreads) blkmap[b] = A.g_blkmap[(size_t)f * Nb + b];
    for (int i = tid; i < kFloodBuckets; i += kFloodThreads) s_bucket[i] = 0u;
    if (tid == 0) { s_head = 0; s_tail = 0; s_overflow = 0; }
    __syncthreads();
    // membershipImg: block label inside eroded member blocks, -1 elsewhere
    for (int y = wid; y < H; y += kFloodThreads / 32) {
        const int by = y / 10;
        for (int x = lane; x < W; x += 32) {
            const int bx = x / 10;
            mem[(size_t)y * W + x] = (by < Nh && bx < Nw) ? (int)blkmap[by * Nw + bx] : -1;
        }
    }
    // refinement seeds, in block scan order (AHCPlaneFitter.hpp:545-583)
    if (wid == 0) {
        int tail = 0;
        for (int b0 = 0; b0 < Nb; b0 += 32) {
            const int b = b0 + lane;
            int c0 = 0, c1 = 0, i = 0, j = 0, me = -1;
            if (b < Nb) {
                i = b / Nw; j = b - i * Nw; me = blkmap[b];
                if (me < 0) { c0 = (i > 0 && blkmap[b - Nw] >= 0); c1 = (j > 0 && blkmap[b - 1] >= 0); }
                else { c0 = (i > 0 && blkmap[b - Nw] != me); c1 = (j > 0 && blkmap[b - 1] != me); }
            }
            const int c = 9 * (c0 + c1);
            int pre = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int n = __shfl_up_sync(0xffffffffu, pre, o); if (lane >= o) pre += n; }
            const int total = __shfl_sync(0xffffffffu, pre, 31);
            int pos = tail + pre - c;
            if (c && pos + c <= A.qcap) {
                if (me < 0) {
                    if (c0) { const uint32_t u = (uint32_t)blkmap[b - Nw] << kQPixBits; const int sp = (i * 10 - 1) * W + j * 10; for (int k = 1; k < 10; ++k) queue[pos++] = (uint32_t)(sp + k) | u; }
                    if (c1) { const uint32_t l = (uint32_t)blkmap[b - 1] << kQPixBits; const int sp = (i * 10) * W + j * 10 - 1; for (int k = 0; k < 9; ++k) queue[pos++] = (uint32_t)(sp + k * W) | l; }
                } else {
                    const uint32_t u = (uint32_t)me << kQPixBits;
                    const int sp = (i * 10) * W + j * 10;
                    if (c0) for (int k = 0; k < 9; ++k) queue[pos++] = (uint32_t)(sp + k) | u;
                    if (c1) for (int k = 1; k < 10; ++k) queue[pos++] = (uint32_t)(sp + k * W) | u;
                }
            }
            tail += total;
        }
        if (lane == 0) { if (tail > A.qcap) { s_overflow = 1; tail = 0; } s_tail = tail; }
    }
    __syncthreads();
    const long long t_seeds = clock64();
    // ---- floodFill (AHCPlaneFitter.hpp:428-476): FIFO over (pixel, plane) seeds ----
#ifdef HVO_FLOOD_PROF
    int st_steps = 0, st_rounds = 0; long long st_t0 = 0, st_load = 0, st_tour = 0, st_comp = 0;
#endif
    unsigned tag = 1;
    uint32_t q_next = 0;      // queue entry of the next step, fetched one step ahead when it already exists
    bool have_next = false;
    while (true) {
        const int head = s_head, tail = s_tail;
        if (head >= tail) break;
        const int nbat = min(kFloodThreads, tail - head);
#ifdef HVO_FLOOD_PROF
        ++st_steps; st_t0 = clock64();
#endif
        const bool have = tid < nbat;
        const uint32_t q = have ? (have_next ? q_next : queue[head + tid]) : 0u;
        have_next = head + nbat + tid < tail;
        if (have_next) q_next = queue[head + nbat + tid];
        const int plid = (int)(q >> kQPixBits);
        int cI[4], trail0[4];
        int cxs[4] = {0, 0, 0, 0}, cys[4] = {0, 0, 0, 0};
        uint16_t z16[4] = {0, 0, 0, 0};
        float cdist[4];
        unsigned okm = 0, pend = 0, pushm = 0;  // bit d: visit d passes the plane test / is pending / pushes a new seed
        if (have) {
            const int sIdx = (int)(q & kQPixMask);
            const int sy = sIdx / W, sx = sIdx - sy * W;
            // valid4 order: left, right, up, down
            cI[0] = sx > 0 ? sIdx - 1 : -1;
            cI[1] = sx < W - 1 ? sIdx + 1 : -1;
            cI[2] = sy > 0 ? sIdx - W : -1;
            cI[3] = sy < H - 1 ? sIdx + W : -1;
            cxs[0] = sx - 1; cxs[1] = sx + 1; cxs[2] = sx; cxs[3] = sx;
            cys[0] = sy; cys[1] = sy; cys[2] = sy - 1; cys[3] = sy + 1;
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                if (cI[d] >= 0) {
                    const int by = cys[d] / 10, bx = cxs[d] / 10;
                    if (by < Nh && bx < Nw && blkmap[by * Nw + bx] >= 0) cI[d] = -1;  // inside an eroded member block
                }
                trail0[d] = 0; z16[d] = 0;
                if (cI[d] >= 0) { trail0[d] = mem[cI[d]]; z16[d] = D[cI[d]]; pend |= 1u << d; }  // speculative: exact for round 1
            }
            const double* p = pl + 8 * plid;
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                cdist[d] = -1.f;
                if (cI[d] >= 0) {
                    const double z = u16_to_double(z16[d]) * A.cam.factor;
                    if (z != 0) {
                        FloodPix P;
                        P.z = z;
                        P.px = div_by_const(((double)cxs[d] - A.cam.cx) * z, A.cam.fx, A.cam.rfx);
                        P.py = div_by_const(((double)cys[d] - A.cam.cy) * z, A.cam.fy, A.cam.rfy);
                        cdist[d] = flood_dist(p, P);
                        if ((double)cdist[d] * (double)cdist[d] < p[7]) okm |= 1u << d;
                    }
                }
            }
        } else {
#pragma unroll
            for (int d = 0; d < 4; ++d) { cI[d] = -1; trail0[d] = 0; cdist[d] = -1.f; }
        }
#ifdef HVO_FLOOD_PROF
        { const long long t = clock64(); st_load += t - st_t0; st_t0 = t; }
#endif
        bool first = true;
        while (__syncthreads_or(pend != 0)) {
#ifdef HVO_FLOOD_PROF
            ++st_rounds;
#endif
#pragma unroll
            for (int d = 0; d < 4; ++d)
                if (pend & (1u << d)) {
                    const unsigned key = (tag << kFloodPosBits) | (unsigned)((1 << kFloodPosBits) - 1 - (tid * 4 + d));
                    atomicMax(&s_bucket[((unsigned)cI[d] * 2654435761u) >> kFloodHashShift], key);
                    atomicMax(&s_bucket[(kFloodBuckets / 2) + (((unsigned)cI[d] * 2246822519u) >> kFloodHashShift)], key);
                }
            __syncthreads();
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                if (!(pend & (1u << d))) continue;
                const unsigned key = (tag << kFloodPosBits) | (unsigned)((1 << kFloodPosBits) - 1 - (tid * 4 + d));
                if (s_bucket[((unsigned)cI[d] * 2654435761u) >> kFloodHashShift] != key &&
                    s_bucket[(kFloodBuckets / 2) + (((unsigned)cI[d] * 2246822519u) >> kFloodHashShift)] != key) continue;
                pend &= ~(1u << d);
                const int cIdx = cI[d];
                const int trail = first ? trail0[d] : mem[cIdx];
                if (trail > -6 && !(trail >= 0 && trail == plid)) {
                    if (okm & (1u << d)) {
                        float od = 3.402823466e+38f;
                        if (trail >= 0) {
                            const double *a = pl + 8 * plid, *b = pl + 8 * trail;
                            if (fabs(a[0] * b[0] + a[1] * b[1] + a[2] * b[2]) >= A.th_refine) {  // connect(planes)
                                const int na = ext[trail], nbn = ext[plid];
                                atomicOr(&adj[(size_t)na * A.nw + (nbn >> 5)], 1u << (nbn & 31));
                                atomicOr(&adj[(size_t)nbn * A.nw + (na >> 5)], 1u << (na & 31));
                            }
                            FloodPix P;   // okm implies a valid depth; the pixel's depth is still in a register
                            P.z = u16_to_double(z16[d]) * A.cam.factor;
                            P.px = div_by_const(((double)cxs[d] - A.cam.cx) * P.z, A.cam.fx, A.cam.rfx);
                            P.py = div_by_const(((double)cys[d] - A.cam.cy) * P.z, A.cam.fy, A.cam.rfy);
                            od = flood_dist(b, P);  // == distMap[cIdx]: the distance stored when the pixel took label `trail`
                        }
                        if (cdist[d] < od) { mem[cIdx] = plid; pushm |= 1u << d; }
                        else if (trail < 0) mem[cIdx] = trail - 1;
                    } else if (trail < 0) {
                        mem[cIdx] = trail - 1;
                    }
                }
            }
            first = false;
            ++tag;
        }
#ifdef HVO_FLOOD_PROF
        { const long long t = clock64(); st_tour += t - st_t0; st_t0 = t; }
#endif
        // append the new seeds in (entry, neighbour) order
        const int mine = __popc(pushm);
        int pre = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int n = __shfl_up_sync(0xffffffffu, pre, o); if (lane >= o) pre += n; }
        if (lane == 31) s_wsum[wid] = pre;
        __syncthreads();
        int base = 0, total = 0;
#pragma unroll
        for (int w = 0; w < kFloodThreads / 32; ++w) { const int v = s_wsum[w]; if (w < wid) base += v; total += v; }
        if (mine) {
            int pos = tail + base + pre - mine;
#pragma unroll
            for (int d = 0; d < 4; ++d)
                if (pushm & (1u << d)) { if (pos < A.qcap) queue[pos] = (uint32_t)cI[d] | ((uint32_t)plid << kQPixBits); ++pos; }
        }
        __syncthreads();
        if (tid == 0) {
            int nt = tail + total;
            if (nt > A.qcap) { s_overflow = 1; nt = A.qcap; }
            s_tail = nt; s_head = head + nbat;
        }
        __syncthreads();
#ifdef HVO_FLOOD_PROF
        { const long long t = clock64(); st_comp += t - st_t0; }
#endif
    }
#ifdef HVO_FLOOD_PROF
    if (tid == 0 && f == 0) printf("flood: steps %d rounds %d tail %d load %lld tour %lld comp %lld\n", st_steps, st_rounds, s_tail, st_load, st_tour, st_comp);
#endif
    if (tid == 0) {
        if (s_overflow) A.status[f] = 1;
        A.cycles[4 * (size_t)f + 1] = t_seeds - t_start;
        A.cycles[4 * (size_t)f + 2] = clock64() - t_seeds;
    }
}

// ---- kernel 3: last merge among the refined planes (AHCPlaneFitter.hpp:317-371) + final labels ----
template <int RW>
__global__ void __launch_bounds__(kAhcThreads) k_plane_merge(AhcArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int Nb = A.Nw * A.Nh;
    AhcS S;
    ahc_merge_smem_views(smem_raw, Nb, A.max_ext, S);
    S.mse = A.g_mse + (size_t)f * Nb;
    S.ulog = nullptr;
    S.cnode = A.cnode + (size_t)f * Nb;
    NodeG* nodes = A.nodes + (size_t)f * Nb;
    uint32_t* adj = A.adj + (size_t)f * Nb * A.nw;
    uint16_t* key = A.key + (size_t)f * Nb;
    double* cand = A.cand + (size_t)f * Nb;
    const long long t_start = clock64();
    const int ne = A.g_ctl[8 * f + 0];
    for (int b = tid; b < Nb; b += kAhcThreads) {
        S.parent[b] = A.g_ds[(size_t)f * 2 * Nb + b];
        S.ssize[b] = A.g_ds[(size_t)f * 2 * Nb + Nb + b];
    }
    for (int i = tid; i < A.nw; i += kAhcThreads) S.nouse[i] = A.g_nouse[(size_t)f * A.nw + i];
    for (int i = tid; i < A.max_ext; i += kAhcThreads) {
        S.isvalid[i] = A.g_isvalid[(size_t)f * A.max_ext + i];
        S.ext[i] = i < ne ? A.g_ext[(size_t)f * A.max_ext + i] : 0;
        S.plidmap[i] = -1;
    }
    if (tid == 0) { S.ctl[0] = 0; S.ctl[1] = A.g_ctl[8 * f + 1]; S.ctl[3] = 0; }
    __syncthreads();
    if (wid == 0) {
        if (lane == 0)
            for (int i = 0; i < ne; ++i) if (S.isvalid[i]) heap_push(S, S.ext[i], S.mse[S.ext[i]]);
        __syncwarp();
        ahc_cluster<false, RW>(A, S, nodes, adj, key, cand, S.ext2, &S.ctl[3], lane);
        const int ne2 = S.ctl[3];
        for (int i = lane; i < ne; i += 32) {
            int m = -1;
            if (S.isvalid[i]) {
                const int r = ds_find(S.parent, nodes[S.ext[i]].rid);
                for (int j = 0; j < ne2; ++j) if (nodes[S.ext2[j]].rid == r) { m = j; break; }
            }
            S.plidmap[i] = (int16_t)m;
        }
        for (int i = lane; i < ne2 && i < A.planes_stride; i += 32) {
            const NodeG* n = nodes + S.ext2[i];
            double* o = A.planes7 + ((size_t)f * A.planes_stride + i) * 7;
            o[0] = n->normal[0]; o[1] = n->normal[1]; o[2] = n->normal[2];
            o[3] = n->center[0]; o[4] = n->center[1]; o[5] = n->center[2];
            o[6] = (double)n->N;
        }
        if (lane == 0) A.n_planes[f] = ne2;
    }
    __syncthreads();
    // the refined-plane -> final-plane map goes to global memory (the block map's storage is free after the flood fill);
    // k_plane_relabel applies it to the pixels with the whole machine instead of this one CTA
    for (int i = tid; i < A.max_ext; i += kAhcThreads) A.g_blkmap[(size_t)f * Nb + i] = S.plidmap[i];
    if (tid == 0) A.cycles[4 * (size_t)f + 3] = clock64() - t_start;
}

// ---- kernel 4: final labels.  membership[i] = plidmap[membership[i]] (or -1), optionally also as one byte per pixel ----
__device__ __forceinline__ int relabel_one(const int16_t* __restrict__ map, int plid) { return plid >= 0 ? (int)map[plid] : -1; }
__device__ __forceinline__ uint32_t label_byte(int lab) { return (uint32_t)(lab < 0 || lab > 254 ? 255 : lab); }
__global__ void __launch_bounds__(256) k_plane_relabel(AhcArgs A) {
    const int f = blockIdx.y, npix = A.w * A.h, Nb = A.Nw * A.Nh;
    const int16_t* map = A.g_blkmap + (size_t)f * Nb;
    int32_t* mem = A.membership + (size_t)f * npix;
    uint8_t* m8 = A.membership8 ? A.membership8 + (size_t)f * npix : nullptr;
    const bool vec = (npix & 3) == 0 && (reinterpret_cast<uintptr_t>(A.membership) & 15) == 0 && (reinterpret_cast<uintptr_t>(A.membership8) & 3) == 0;
    const int i4 = blockIdx.x * 256 + threadIdx.x;
    if (vec) {
        if (4 * i4 >= npix) return;
        int4 v = reinterpret_cast<int4*>(mem)[i4];
        v.x = relabel_one(map, v.x); v.y = relabel_one(map, v.y); v.z = relabel_one(map, v.z); v.w = relabel_one(map, v.w);
        reinterpret_cast<int4*>(mem)[i4] = v;
        if (m8) reinterpret_cast<uint32_t*>(m8)[i4] = label_byte(v.x) | (label_byte(v.y) << 8) | (label_byte(v.z) << 16) | (label_byte(v.w) << 24);
    } else {
        for (int i = 4 * i4; i < min(4 * i4 + 4, npix); ++i) {
            const int lab = relabel_one(map, mem[i]);
            mem[i] = lab;
            if (m8) m8[i] = (uint8_t)label_byte(lab);
        }
    }
}

}  // namespace hvo

using namespace hvo;

struct hvo_plane {
    int device = 0, width = 0, height = 0, max_batch = 0, Nw = 0, Nh = 0, nw = 0, qcap = 0, max_ext = 0;
    size_t ahc_smem = 0, merge_smem = 0;
    PlaneCam cam;
    cudaStream_t stream = nullptr;
    cudaEvent_t tev[2] = {nullptr, nullptr};
    uint16_t* d_depth = nullptr;
    BlockOut* d_blocks = nullptr;
    BlockOut* h_blocks = nullptr;  // pinned, one frame (inspection)
    NodeG* d_nodes = nullptr;
    uint32_t* d_adj = nullptr;
    uint16_t* d_key = nullptr;
    double* d_cand = nullptr;
    uint32_t* d_ulog = nullptr;
    uint16_t* d_cnode = nullptr;
    uint32_t* d_queue = nullptr;
    int32_t* d_mem = nullptr;
    double* d_planes = nullptr;  // [B][max_ext][7]
    int32_t *d_nplanes = nullptr, *d_status = nullptr;
    long long* d_cycles = nullptr;
    double *d_gmse = nullptr, *d_gpl = nullptr;
    uint16_t *d_gds = nullptr, *d_gext = nullptr;
    uint32_t* d_gnouse = nullptr;
    int16_t* d_gblkmap = nullptr;
    uint8_t* d_gisvalid = nullptr;
    int* d_gctl = nullptr;
    size_t flood_smem = 0;
    int32_t* h_status = nullptr;  // pinned [B]
    int last_launches = 0;
};

namespace hvo {
cudaStream_t plane_stream(hvo_plane* h) { return h->stream; }  // internal: frame.cu chains the stages on events
const int32_t* plane_status(hvo_plane* h) { return h->d_status; }    // internal: per frame, != 0 = refinement queue overflow
}

extern "C" {

int hvo_plane_create(const hvo_plane_params* p, int width, int height, int max_batch, int device, hvo_plane** out) {
    HVO_CHECK_ARG(out, "null out");
    *out = nullptr;
    HVO_CHECK_ARG(p, "null params");
    HVO_CHECK_ARG(width >= 20 && height >= 20 && width <= 8192 && height <= 8192, "image size out of range");
    HVO_CHECK_ARG((long long)width * height <= (1 << kQPixBits), "image too large for the 22-bit pixel index of the refinement queue");
    HVO_CHECK_ARG(max_batch >= 1, "max_batch < 1");
    HVO_CHECK_ARG(p->fx != 0 && p->fy != 0, "fx / fy must be non-zero");
    int ndev = 0;
    HVO_CUDA(cudaGetDeviceCount(&ndev));
    if (ndev < 1) { set_error("no CUDA device: libhvofront has no CPU fallback"); return HVO_ERR_CUDA; }
    HVO_CHECK_ARG(device >= 0 && device < ndev, "device index out of range");
    hvo_plane* h = new (std::nothrow) hvo_plane();
    if (!h) { set_error("out of host memory"); return HVO_ERR_ARG; }
    h->device = device; h->width = width; h->height = height; h->max_batch = max_batch;
    h->Nw = width / 10; h->Nh = height / 10;
    const int Nb = h->Nw * h->Nh;
    if (Nb > kRowWL * 1024) { delete h; set_error("bad argument: too many 10x10 blocks (max 24576, e.g. 1920x1200)"); return HVO_ERR_ARG; }
    h->nw = (Nb + 31) / 32;
    h->qcap = 2 * width * height;
    // test aid: a smaller refinement queue, to provoke HVO_ERR_OVERFLOW
    if (const char* e = getenv("HVO_DEBUG_PLANE_QCAP")) h->qcap = std::max(64, std::min(h->qcap, atoi(e)));
    h->max_ext = Nb * 100 / kMinSupport + 2;   // <= 821 < 2^(32 - kQPixBits)
    h->cam.factor = (double)p->depth_factor; h->cam.fx = (double)p->fx; h->cam.fy = (double)p->fy;
    h->cam.rfx = 1.0 / h->cam.fx; h->cam.rfy = 1.0 / h->cam.fy;
    h->cam.cx = (double)p->cx; h->cam.cy = (double)p->cy;
    h->ahc_smem = ahc_cluster_smem_bytes(Nb, h->max_ext);
    h->merge_smem = ahc_merge_smem_bytes(Nb, h->max_ext);
    int st = HVO_OK;
    do {
#define HVO_TRY(call) if ((call) != cudaSuccess) { set_error("%s: %s", #call, cudaGetErrorString(cudaGetLastError())); st = HVO_ERR_CUDA; break; }
        HVO_TRY(cudaSetDevice(device));
        if (h->ahc_smem > 220 * 1024) { set_error("image too large: the plane graph does not fit shared memory"); st = HVO_ERR_ARG; break; }
        h->flood_smem = (size_t)h->max_ext * 64 + (size_t)Nb * 2 + (size_t)h->max_ext * 2 + 16;
        // the attribute is per function (shared by all handles on the device, whatever their image size): only ever raise it, or a
        // smaller handle created later would make the larger one's launches fail
        static size_t s_smem_max[64][3] = {};
        size_t sm[3] = {h->ahc_smem, h->merge_smem, h->flood_smem};
        if (device < 64)
            for (int k = 0; k < 3; ++k) sm[k] = std::max(s_smem_max[device][k], sm[k]);
        HVO_TRY(cudaFuncSetAttribute(k_plane_cluster<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm[0]));
        HVO_TRY(cudaFuncSetAttribute(k_plane_cluster<kRowW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm[0]));
        HVO_TRY(cudaFuncSetAttribute(k_plane_cluster<kRowWL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm[0]));
        HVO_TRY(cudaFuncSetAttribute(k_plane_merge<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm[1]));
        HVO_TRY(cudaFuncSetAttribute(k_plane_merge<kRowW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm[1]));
        HVO_TRY(cudaFuncSetAttribute(k_plane_merge<kRowWL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm[1]));
        HVO_TRY(cudaFuncSetAttribute(k_plane_flood, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm[2]));
        if (device < 64)   // recorded once every attribute holds it
            for (int k = 0; k < 3; ++k) s_smem_max[device][k] = sm[k];
        pin_carveout(k_plane_blocks); pin_carveout(k_plane_cluster<3>); pin_carveout(k_plane_cluster<kRowW>);
        pin_carveout(k_plane_flood); pin_carveout(k_plane_merge<3>); pin_carveout(k_plane_merge<kRowW>);
        pin_carveout(k_plane_cluster<kRowWL>); pin_carveout(k_plane_merge<kRowWL>);
        HVO_TRY(create_stream(&h->stream));
        HVO_TRY(cudaEventCreate(&h->tev[0]));
        HVO_TRY(cudaEventCreate(&h->tev[1]));
        const size_t B = (size_t)max_batch, px = (size_t)width * height;
        HVO_TRY(cudaMalloc(&h->d_depth, B * px * 2));
        HVO_TRY(cudaMalloc(&h->d_blocks, B * Nb * sizeof(BlockOut)));
        HVO_TRY(cudaMallocHost(&h->h_blocks, (size_t)Nb * sizeof(BlockOut)));
        HVO_TRY(cudaMalloc(&h->d_nodes, B * Nb * sizeof(NodeG)));
        HVO_TRY(cudaMalloc(&h->d_adj, B * Nb * h->nw * sizeof(uint32_t)));
        HVO_TRY(cudaMalloc(&h->d_key, B * Nb * sizeof(uint16_t)));
        HVO_TRY(cudaMalloc(&h->d_cand, B * Nb * sizeof(double)));
        HVO_TRY(cudaMalloc(&h->d_ulog, B * Nb * sizeof(uint32_t)));
        HVO_TRY(cudaMalloc(&h->d_cnode, B * Nb * sizeof(uint16_t)));
        HVO_TRY(cudaMalloc(&h->d_queue, B * (size_t)h->qcap * sizeof(uint32_t)));
        HVO_TRY(cudaMalloc(&h->d_mem, B * px * sizeof(int32_t)));
        HVO_TRY(cudaMalloc(&h->d_planes, B * (size_t)h->max_ext * 7 * sizeof(double)));
        HVO_TRY(cudaMalloc(&h->d_nplanes, B * sizeof(int32_t)));
        HVO_TRY(cudaMalloc(&h->d_status, B * sizeof(int32_t)));
        HVO_TRY(cudaMalloc(&h->d_cycles, B * 4 * sizeof(long long)));
        HVO_TRY(cudaMalloc(&h->d_gmse, B * Nb * sizeof(double)));
        HVO_TRY(cudaMalloc(&h->d_gds, B * 2 * Nb * sizeof(uint16_t)));
        HVO_TRY(cudaMalloc(&h->d_gnouse, B * h->nw * sizeof(uint32_t)));
        HVO_TRY(cudaMalloc(&h->d_gblkmap, B * Nb * sizeof(int16_t)));
        HVO_TRY(cudaMalloc(&h->d_gext, B * (size_t)h->max_ext * sizeof(uint16_t)));
        HVO_TRY(cudaMalloc(&h->d_gisvalid, B * (size_t)h->max_ext));
        HVO_TRY(cudaMalloc(&h->d_gpl, B * (size_t)h->max_ext * 7 * sizeof(double)));
        HVO_TRY(cudaMalloc(&h->d_gctl, B * 8 * sizeof(int)));
        HVO_TRY(cudaMallocHost(&h->h_status, B * sizeof(int32_t)));
#undef HVO_TRY
    } while (0);
    if (st != HVO_OK) { hvo_plane_destroy(h); return st; }
    *out = h;
    return HVO_OK;
}

void hvo_plane_destroy(hvo_plane* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    void* bufs[] = {h->d_depth, h->d_blocks, h->d_nodes, h->d_adj, h->d_key, h->d_cand, h->d_ulog, h->d_cnode, h->d_queue, h->d_mem, h->d_planes,
                    h->d_nplanes, h->d_status, h->d_cycles, h->d_gmse, h->d_gds, h->d_gnouse, h->d_gblkmap, h->d_gext, h->d_gisvalid,
                    h->d_gpl, h->d_gctl};
    for (void* b : bufs) if (b) cudaFree(b);
    if (h->h_blocks) cudaFreeHost(h->h_blocks);
    if (h->h_status) cudaFreeHost(h->h_status);
    for (auto& e : h->tev) if (e) cudaEventDestroy(e);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

static int plane_blocks_launch(hvo_plane* h, const uint16_t* d_depth, int nframes) {
    const int nb = h->Nw * h->Nh;
    timeline_mark(h->stream, "k_plane_blocks");
    k_plane_blocks<<<dim3(div_up(nb, 128), nframes), 128, 0, h->stream>>>(d_depth, h->width, h->height, h->cam, h->Nw, h->Nh, h->d_blocks);
    HVO_CUDA(cudaGetLastError());
    return HVO_OK;
}

// blocks + graph stage on device-resident depth; results into d_nplanes / d_planes7 ([n][planes_stride][7]) / d_membership
static int plane_detect_launch(hvo_plane* h, const uint16_t* d_depth, int nframes, int32_t* d_nplanes, double* d_planes7, int planes_stride,
                               int32_t* d_membership, uint8_t* d_membership8 = nullptr) {
    int st = plane_blocks_launch(h, d_depth, nframes);
    if (st != HVO_OK) return st;
    const int Nb = h->Nw * h->Nh;
    HVO_CUDA(cudaMemsetAsync(h->d_adj, 0, (size_t)nframes * Nb * h->nw * sizeof(uint32_t), h->stream));
    AhcArgs A;
    A.depth = d_depth; A.blocks = h->d_blocks; A.nodes = h->d_nodes; A.adj = h->d_adj; A.key = h->d_key; A.cand = h->d_cand; A.ulog = h->d_ulog; A.cnode = h->d_cnode;
    A.queue = h->d_queue; A.membership = d_membership; A.membership8 = d_membership8; A.planes7 = d_planes7; A.n_planes = d_nplanes;
    A.status = h->d_status; A.cycles = h->d_cycles;
    A.w = h->width; A.h = h->height; A.Nw = h->Nw; A.Nh = h->Nh; A.nw = h->nw; A.qcap = h->qcap; A.max_ext = h->max_ext;
    A.planes_stride = planes_stride; A.cam = h->cam;
    A.th_merge = std::cos(M_PI / 180.0 * 60.0);   // ParamSet::similarityTh_merge
    A.th_refine = std::cos(M_PI / 180.0 * 30.0);  // ParamSet::similarityTh_refine
    A.g_mse = h->d_gmse; A.g_ds = h->d_gds; A.g_nouse = h->d_gnouse; A.g_blkmap = h->d_gblkmap; A.g_ext = h->d_gext;
    A.g_isvalid = h->d_gisvalid; A.g_pl = h->d_gpl; A.g_ctl = h->d_gctl;
    // row words per lane: 3 up to 3072 blocks (640x480), kRowW up to 9216 (1280x720), kRowWL beyond
    const int rw = h->nw <= 3 * 32 ? 3 : (h->nw <= kRowW * 32 ? kRowW : kRowWL);
    timeline_mark(h->stream, rw == kRowWL ? "k_plane_cluster<24>" : "k_plane_cluster");
    if (rw == 3) k_plane_cluster<3><<<nframes, 32, h->ahc_smem, h->stream>>>(A);
    else if (rw == kRowW) k_plane_cluster<kRowW><<<nframes, 32, h->ahc_smem, h->stream>>>(A);
    else k_plane_cluster<kRowWL><<<nframes, 32, h->ahc_smem, h->stream>>>(A);
    timeline_mark(h->stream, "k_plane_flood");
    k_plane_flood<<<nframes, kFloodThreads, h->flood_smem, h->stream>>>(A);
    timeline_mark(h->stream, rw == kRowWL ? "k_plane_merge<24>" : "k_plane_merge");
    if (rw == 3) k_plane_merge<3><<<nframes, kAhcThreads, h->merge_smem, h->stream>>>(A);
    else if (rw == kRowW) k_plane_merge<kRowW><<<nframes, kAhcThreads, h->merge_smem, h->stream>>>(A);
    else k_plane_merge<kRowWL><<<nframes, kAhcThreads, h->merge_smem, h->stream>>>(A);
    timeline_mark(h->stream, "k_plane_relabel");
    k_plane_relabel<<<dim3(div_up(div_up(h->width * h->height, 4), 256), nframes), 256, 0, h->stream>>>(A);
    HVO_CUDA(cudaGetLastError());
    h->last_launches = 6;
    return HVO_OK;
}

/* device-only leg: block statistics of nframes device-resident depth images (inspection / roofline of k_plane_blocks) */
int hvo_plane_blocks_device(hvo_plane* h, const uint16_t* d_depth, int nframes) {
    HVO_CHECK_ARG(h && d_depth, "null argument");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch, "nframes out of range for this handle");
    HVO_CUDA(cudaSetDevice(h->device));
    return plane_blocks_launch(h, d_depth, nframes);
}

int hvo_plane_get_blocks(hvo_plane* h, int frame, double* out9) {
    HVO_CHECK_ARG(h && out9, "null argument");
    HVO_CHECK_ARG(frame >= 0 && frame < h->max_batch, "frame out of range");
    HVO_CUDA(cudaSetDevice(h->device));
    const int nb = h->Nw * h->Nh;
    HVO_CUDA(cudaMemcpyAsync(h->h_blocks, h->d_blocks + (size_t)frame * nb, (size_t)nb * sizeof(BlockOut), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    for (int b = 0; b < nb; ++b) {
        const BlockOut& o = h->h_blocks[b];
        double* r = out9 + 9 * (size_t)b;
        r[0] = o.queued; r[1] = o.N;
        if (o.N >= 4) {
            double c[3], n[3], mse, curv;
            stats_compute(o.s, o.N, c, n, mse, curv);
            for (int k = 0; k < 3; ++k) { r[2 + k] = c[k]; r[5 + k] = n[k]; }
            r[8] = o.mse;
        } else {
            for (int k = 2; k < 8; ++k) r[k] = 0;
            r[8] = std::numeric_limits<double>::quiet_NaN();
        }
    }
    return HVO_OK;
}

int hvo_plane_detect_batch_device(hvo_plane* h, const uint16_t* d_depth16, int nframes, int32_t* d_n_planes, double* d_planes7,
                                  int max_planes, int32_t* d_membership) {
    HVO_CHECK_ARG(h && d_depth16 && d_n_planes && d_planes7 && d_membership, "null argument");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch && max_planes >= 1, "nframes / max_planes out of range");
    HVO_CUDA(cudaSetDevice(h->device));
    return plane_detect_launch(h, d_depth16, nframes, d_n_planes, d_planes7, max_planes, d_membership);
}

int hvo_plane_detect_batch_device_u8(hvo_plane* h, const uint16_t* d_depth16, int nframes, int32_t* d_n_planes, double* d_planes7,
                                     int max_planes, int32_t* d_membership, uint8_t* d_membership8) {
    HVO_CHECK_ARG(h && d_depth16 && d_n_planes && d_planes7 && d_membership && d_membership8, "null argument");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch && max_planes >= 1, "nframes / max_planes out of range");
    HVO_CUDA(cudaSetDevice(h->device));
    return plane_detect_launch(h, d_depth16, nframes, d_n_planes, d_planes7, max_planes, d_membership, d_membership8);
}

int hvo_plane_detect_batch(hvo_plane* h, const uint16_t* depth16, int nframes, int32_t* n_planes, double* planes7, int max_planes,
                           int32_t* membership) {
    HVO_CHECK_ARG(h && depth16 && n_planes && planes7 && membership, "null argument");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch && max_planes >= 1, "nframes / max_planes out of range");
    HVO_CUDA(cudaSetDevice(h->device));
    const size_t px = (size_t)h->width * h->height, n = (size_t)nframes;
    HVO_CUDA(cudaMemcpyAsync(h->d_depth, depth16, n * px * 2, cudaMemcpyHostToDevice, h->stream));
    int st = plane_detect_launch(h, h->d_depth, nframes, h->d_nplanes, h->d_planes, h->max_ext, h->d_mem);
    if (st != HVO_OK) return st;
    HVO_CUDA(cudaMemcpyAsync(n_planes, h->d_nplanes, n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaMemcpyAsync(h->h_status, h->d_status, n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    const int cp = max_planes < h->max_ext ? max_planes : h->max_ext;
    HVO_CUDA(cudaMemcpy2DAsync(planes7, (size_t)max_planes * 56, h->d_planes, (size_t)h->max_ext * 56, (size_t)cp * 56, n,
                               cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaMemcpyAsync(membership, h->d_mem, n * px * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    for (int f = 0; f < nframes; ++f)
        if (h->h_status[f] != 0) { set_error("plane refinement queue overflow in frame %d", f); return HVO_ERR_OVERFLOW; }
    return HVO_OK;
}

int hvo_plane_detect(hvo_plane* h, const uint16_t* depth16, int32_t* n_planes, double* planes7, int max_planes, int32_t* membership) {
    return hvo_plane_detect_batch(h, depth16, 1, n_planes, planes7, max_planes, membership);
}

int hvo_plane_last_launches(const hvo_plane* h) { return h ? h->last_launches : 0; }

int hvo_plane_get_phase_cycles(hvo_plane* h, int frame, int64_t* out4) {
    HVO_CHECK_ARG(h && out4, "null argument");
    HVO_CHECK_ARG(frame >= 0 && frame < h->max_batch, "frame out of range");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaMemcpyAsync(out4, h->d_cycles + 4 * (size_t)frame, 4 * sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return HVO_OK;
}

int hvo_plane_sync(hvo_plane* h) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return HVO_OK;
}
int hvo_plane_timer_start(hvo_plane* h) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[0], h->stream));
    return HVO_OK;
}
int hvo_plane_timer_stop(hvo_plane* h, float* ms_out) {
    HVO_CHECK_ARG(h && ms_out, "null argument");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[1], h->stream));
    HVO_CUDA(cudaEventSynchronize(h->tev[1]));
    HVO_CUDA(cudaEventElapsedTime(ms_out, h->tev[0], h->tev[1]));
    return HVO_OK;
}

}  // extern "C"
