// Windowed (projection) matching for sm_100a: the frame grid and the greedy best / second-best search inside it.
//
// Replaces, for one frame at a time (tracking is sequential; SURVEY §8e "replicas only"):
//   Frame::AssignFeaturesToGrid / PosInGrid         reference src/Frame.cc:832-847, 1680-1690
//   Frame::GetFeaturesInArea                        src/Frame.cc:1502-1555
//   ORBmatcher::SearchByProjection(F, MapPoints)    src/ORBmatcher.cc:45-132          (mode 0)
//   ORBmatcher::SearchByProjection(Cur, Last / KF)  src/ORBmatcher.cc:1353-1497, 1499-1628   (mode 1, matching part)
//
//   k_proj_grid    one CTA per frame: cell of every keypoint (round), histogram, exclusive scan, scatter, per-cell index sort, so a
//                  cell lists its keypoints in index order exactly like the reference's push_back loop (hvo_proj_set_frame: one
//                  frame; the frame pipeline: every frame of a call, hvo_frame_grid_outputs)
//   k_proj_round   one warp per query: the cells of the window in the reference's order (ix outer, iy inner; the iy run of
//                  one ix is contiguous in memory), 32 candidates at a time: level / window / right-coordinate filters and
//                  8 x __popc per lane, then the reference's sequential best / second update over the surviving lanes
//
// The reference assignment is greedy: a keypoint taken by an earlier query (whose map point has observations) is skipped by
// later ones.  That order dependence is resolved exactly by iterating to the fixed point: every round all queries search in
// parallel, treating a keypoint as claimed iff the smallest query index that chose it in the previous round is lower than
// their own; queries 0..r are final after round r+1, and a round that changes no choice proves the fixed point, which is
// the sequential result.  Conflicts are rare, so this takes two or three rounds.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstring>
#include <new>

#include "hvo_common.cuh"

namespace hvo {

static const int kGridCols = 64, kGridRows = 48, kGridCells = kGridCols * kGridRows;

struct ProjKey { float x, y; int octave; float uright; };  // 16 bytes per keypoint
struct ProjQuery { float u, v, r; int min_level, max_level; float ur; int claims; int pad; };  // hvo_proj_query
struct GridGeom { float min_x, min_y, inv_w, inv_h; };

// Frame::PosInGrid (Frame.cc:1680-1690): the cell (ix * 48 + iy) of an undistorted keypoint, -1 outside the grid
__device__ __forceinline__ int pos_in_grid(const GridGeom& g, float x, float y) {
    const int px = (int)roundf(__fmul_rn(__fsub_rn(x, g.min_x), g.inv_w)), py = (int)roundf(__fmul_rn(__fsub_rn(y, g.min_y), g.inv_h));
    return (px >= 0 && px < kGridCols && py >= 0 && py < kGridRows) ? px * kGridRows + py : -1;
}

// One CTA per frame: frame f = keypoint rows [f * stride, + n_f), n_f = counts ? counts[f] : n.  Outputs of frame f: cell_start
// [3073] (exclusive scan; NULL in the frame pipeline) or cell_count [f][3072]; cell_items [f][stride] (the first sum(counts) entries
// written); pk [n] ProjKey rows (NULL in the frame pipeline).
template <class Item>
__global__ void __launch_bounds__(1024) k_proj_grid(const hvo_keypoint* __restrict__ keys, const float* __restrict__ uright, int n,
                                                    const int32_t* __restrict__ counts, int stride, GridGeom g, ProjKey* __restrict__ pk,
                                                    int* __restrict__ cell_start, uint16_t* __restrict__ cell_count, Item* __restrict__ cell_items) {
    __shared__ int s_cnt[kGridCells];
    __shared__ int s_part[32];
    const int tid = threadIdx.x, f = blockIdx.x;
    if (counts) n = min(counts[f], stride);
    keys += (size_t)f * stride;
    cell_items += (size_t)f * stride;
    for (int c = tid; c < kGridCells; c += 1024) s_cnt[c] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += 1024) {
        const hvo_keypoint k = keys[i];
        if (pk) {
            ProjKey p;
            p.x = k.x; p.y = k.y; p.octave = k.octave; p.uright = uright ? uright[i] : -1.f;
            pk[i] = p;
        }
        const int c = pos_in_grid(g, k.x, k.y);
        if (c >= 0) atomicAdd(&s_cnt[c], 1);
    }
    __syncthreads();
    // exclusive scan of the 3072 counts: 3 per thread
    int v[3], start[3], sum = 0;
#pragma unroll
    for (int k = 0; k < 3; ++k) { v[k] = s_cnt[tid * 3 + k]; sum += v[k]; }
    int base = block_exclusive_scan3(sum, s_part);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int c = tid * 3 + k;
        if (cell_start) cell_start[c] = base;
        if (cell_count) cell_count[(size_t)f * kGridCells + c] = (uint16_t)v[k];
        start[k] = s_cnt[c] = base;
        base += v[k];
    }
    if (cell_start && tid == 1023) cell_start[kGridCells] = base;
    __syncthreads();
    for (int i = tid; i < n; i += 1024) {
        const hvo_keypoint k = keys[i];
        const int c = pos_in_grid(g, k.x, k.y);
        if (c >= 0) cell_items[atomicAdd(&s_cnt[c], 1)] = (Item)i;
    }
    __syncthreads();
    // a cell lists its keypoints in index order (reference: push_back in the i loop)
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int b = start[k], e = b + v[k];
        for (int i = b + 1; i < e; ++i) {
            const Item x = cell_items[i];
            int j = i - 1;
            while (j >= b && cell_items[j] > x) { cell_items[j + 1] = cell_items[j]; --j; }
            cell_items[j + 1] = x;
        }
    }
}

static GridGeom grid_geom(float min_x, float min_y, float max_x, float max_y) {
    GridGeom g;
    g.min_x = min_x; g.min_y = min_y;
    g.inv_w = (float)kGridCols / (max_x - min_x);   // Frame.cc:419-420
    g.inv_h = (float)kGridRows / (max_y - min_y);
    return g;
}

// The frame pipeline's point grids (hvo_frame_grid_outputs): nframes frames of `stride` keypoint rows, counts on the device.
int proj_grid_frames_launch(cudaStream_t s, const hvo_keypoint* d_kps, const int32_t* d_counts, int nframes, int stride, float min_x, float min_y,
                            float max_x, float max_y, uint16_t* d_cell_count, uint16_t* d_cell_items) {
    k_proj_grid<uint16_t><<<nframes, 1024, 0, s>>>(d_kps, nullptr, 0, d_counts, stride, grid_geom(min_x, min_y, max_x, max_y), nullptr, nullptr,
                                                   d_cell_count, d_cell_items);
    HVO_CUDA(cudaGetLastError());
    return HVO_OK;
}

struct ProjWindow { int x0, x1, y0, y1; bool empty; };
__device__ __forceinline__ ProjWindow proj_window(const GridGeom& g, float x, float y, float r) {  // Frame.cc:1507-1521
    ProjWindow w;
    w.empty = true;
    w.x0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(__fsub_rn(x, g.min_x), r), g.inv_w)));
    w.x1 = min(kGridCols - 1, (int)ceilf(__fmul_rn(__fadd_rn(__fsub_rn(x, g.min_x), r), g.inv_w)));
    w.y0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(__fsub_rn(y, g.min_y), r), g.inv_h)));
    w.y1 = min(kGridRows - 1, (int)ceilf(__fmul_rn(__fadd_rn(__fsub_rn(y, g.min_y), r), g.inv_h)));
    if (w.x0 >= kGridCols || w.x1 < 0 || w.y0 >= kGridRows || w.y1 < 0) return w;
    w.empty = false;
    return w;
}
__device__ __forceinline__ bool proj_in_area(const ProjKey& p, float x, float y, float r, int minLevel, int maxLevel) {
    if (minLevel > 0 || maxLevel >= 0) {
        if (p.octave < minLevel) return false;
        if (maxLevel >= 0 && p.octave > maxLevel) return false;
    }
    return fabsf(__fsub_rn(p.x, x)) < r && fabsf(__fsub_rn(p.y, y)) < r;
}

// Frame::GetFeaturesInArea for one window (inspection / parity of the candidate order).  One warp.
__global__ void __launch_bounds__(32) k_proj_area(const ProjKey* __restrict__ pk, const int* __restrict__ cell_start,
                                                  const int* __restrict__ cell_items, GridGeom g, float x, float y, float r, int minLevel,
                                                  int maxLevel, int* __restrict__ out, int cap, int* __restrict__ n_out) {
    const int lane = threadIdx.x;
    const ProjWindow w = proj_window(g, x, y, r);
    int cnt = 0;
    if (!w.empty)
        for (int ix = w.x0; ix <= w.x1; ++ix) {
            const int b = cell_start[ix * kGridRows + w.y0], e = cell_start[ix * kGridRows + w.y1 + 1];
            for (int base = b; base < e; base += 32) {
                const int i = base + lane;
                int id = -1;
                bool ok = false;
                if (i < e) { id = cell_items[i]; ok = proj_in_area(pk[id], x, y, r, minLevel, maxLevel); }
                const unsigned m = __ballot_sync(0xffffffffu, ok);
                if (ok) { const int o = cnt + __popc(m & ((1u << lane) - 1u)); if (o < cap) out[o] = id; }
                cnt += __popc(m);
            }
        }
    if (lane == 0) *n_out = cnt;
}

__global__ void __launch_bounds__(128) k_proj_round(const ProjKey* __restrict__ pk, const uint4* __restrict__ desc,
                                                    const int* __restrict__ cell_start, const int* __restrict__ cell_items, GridGeom g,
                                                    const ProjQuery* __restrict__ qs, const uint4* __restrict__ qdesc, int nq,
                                                    const int* __restrict__ claim_prev, int* __restrict__ claim_next, int mode, int th_dist,
                                                    float nnratio, const float* __restrict__ inv_sigma2, int* __restrict__ choice,
                                                    int* __restrict__ choice_dist, int* __restrict__ changed) {
    const int k = (blockIdx.x * 128 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (k >= nq) return;
    const ProjQuery q = qs[k];
    const uint4 qa = qdesc[2 * k], qb = qdesc[2 * k + 1];
    const ProjWindow w = proj_window(g, q.u, q.v, q.r);
    int bestDist = 256, bestLevel = -1, bestDist2 = 256, bestLevel2 = -1, bestIdx = -1;
    if (!w.empty)
        for (int ix = w.x0; ix <= w.x1; ++ix) {
            const int b = cell_start[ix * kGridRows + w.y0], e = cell_start[ix * kGridRows + w.y1 + 1];
            for (int base = b; base < e; base += 32) {
                const int i = base + lane;
                int id = -1, dist = 256, oct = 0;
                bool ok = false;
                if (i < e) {
                    id = cell_items[i];
                    const ProjKey p = pk[id];
                    oct = p.octave;
                    ok = proj_in_area(p, q.u, q.v, q.r, q.min_level, q.max_level);
                    if (mode == 2) {  // ORBmatcher::Fuse (ORBmatcher.cc:914-944): chi-square gate on the reprojection error, nothing is claimed
                        if (ok) {
                            const float ex = __fsub_rn(q.u, p.x), ey = __fsub_rn(q.v, p.y);
                            float e2 = __fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey));
                            double lim = 5.99;
                            if (p.uright >= 0) { const float er = __fsub_rn(q.ur, p.uright); e2 = __fadd_rn(e2, __fmul_rn(er, er)); lim = 7.8; }
                            ok = !((double)__fmul_rn(e2, inv_sigma2[oct]) > lim);
                        }
                    } else {
                        ok = ok && !(claim_prev[id] < k);
                        if (ok && p.uright > 0) ok = !(fabsf(__fsub_rn(q.ur, p.uright)) > q.r);
                    }
                    if (ok) {
                        const uint4 da = desc[2 * id], db = desc[2 * id + 1];
                        dist = __popc(qa.x ^ da.x) + __popc(qa.y ^ da.y) + __popc(qa.z ^ da.z) + __popc(qa.w ^ da.w) +
                               __popc(qb.x ^ db.x) + __popc(qb.y ^ db.y) + __popc(qb.z ^ db.z) + __popc(qb.w ^ db.w);
                    }
                }
                unsigned m = __ballot_sync(0xffffffffu, ok);
                while (m) {  // the reference's update, candidate by candidate (ORBmatcher.cc:104-117)
                    const int j = __ffs(m) - 1;
                    m &= m - 1;
                    const int d = __shfl_sync(0xffffffffu, dist, j), l = __shfl_sync(0xffffffffu, oct, j), c = __shfl_sync(0xffffffffu, id, j);
                    if (d < bestDist) { bestDist2 = bestDist; bestDist = d; bestLevel2 = bestLevel; bestLevel = l; bestIdx = c; }
                    else if (d < bestDist2) { bestLevel2 = l; bestDist2 = d; }
                }
            }
        }
    int pick = -1;
    if (bestDist <= th_dist && !(mode == 0 && bestLevel == bestLevel2 && (float)bestDist > __fmul_rn(nnratio, (float)bestDist2))) pick = bestIdx;
    if (lane == 0) {
        if (choice[k] != pick) { choice[k] = pick; *changed = 1; }
        choice_dist[k] = pick >= 0 ? bestDist : 256;
        if (pick >= 0 && q.claims && mode != 2) atomicMin(&claim_next[pick], k);
    }
}

__global__ void k_proj_claim_init(const uint8_t* __restrict__ claimed, int n, int* __restrict__ a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = (claimed && claimed[i]) ? -1 : INT_MAX;
}
__global__ void k_proj_fill(int* __restrict__ a, int n, int v) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = v;
}

// generic candidate lists: one warp per query, candidates in the caller's order, strict '<' updates
__global__ void __launch_bounds__(128) k_match_candidates(const uint4* __restrict__ q, int nq, const uint4* __restrict__ t,
                                                          const int* __restrict__ off, const int* __restrict__ cand, int4* __restrict__ best4) {
    const int k = (blockIdx.x * 128 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (k >= nq) return;
    const uint4 qa = q[2 * k], qb = q[2 * k + 1];
    int d0 = 256, i0 = -1, d1 = 256, i1 = -1;
    const int b = off[k], e = off[k + 1];
    for (int base = b; base < e; base += 32) {
        const int i = base + lane;
        int id = -1, dist = 256;
        if (i < e) {
            id = cand[i];
            const uint4 da = t[2 * id], db = t[2 * id + 1];
            dist = __popc(qa.x ^ da.x) + __popc(qa.y ^ da.y) + __popc(qa.z ^ da.z) + __popc(qa.w ^ da.w) + __popc(qb.x ^ db.x) +
                   __popc(qb.y ^ db.y) + __popc(qb.z ^ db.z) + __popc(qb.w ^ db.w);
        }
        const int cnt = min(32, e - base);
        for (int j = 0; j < cnt; ++j) {
            const int d = __shfl_sync(0xffffffffu, dist, j), c = __shfl_sync(0xffffffffu, id, j);
            if (d < d0) { d1 = d0; i1 = i0; d0 = d; i0 = c; }
            else if (d < d1) { d1 = d; i1 = c; }
        }
    }
    if (lane == 0) best4[k] = make_int4(i0, d0, i1, d1);
}

// Greedy search over caller-given candidate lists (ORBmatcher::SearchByBoW, src/ORBmatcher.cc:197-251): query k skips train
// rows already assigned to an earlier query (vpMapPointMatches[realIdxF] != NULL), keeps best / second with strict '<', and
// takes the best when best <= th_dist and (float)best < nnratio * (float)second.  One round of the fixed-point iteration.
__global__ void __launch_bounds__(128) k_cand_round(const uint4* __restrict__ q, int nq, const uint4* __restrict__ t, const int* __restrict__ off,
                                                    const int* __restrict__ cand, const int* __restrict__ claim_prev, int* __restrict__ claim_next,
                                                    int th_dist, float nnratio, int* __restrict__ choice, int* __restrict__ choice_dist,
                                                    int* __restrict__ changed) {
    const int k = (blockIdx.x * 128 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (k >= nq) return;
    const uint4 qa = q[2 * k], qb = q[2 * k + 1];
    int d0 = 256, i0 = -1, d1 = 256;
    const int b = off[k], e = off[k + 1];
    for (int base = b; base < e; base += 32) {
        const int i = base + lane;
        int id = -1, dist = 256;
        bool ok = false;
        if (i < e) {
            id = cand[i];
            ok = !(claim_prev[id] < k);
            if (ok) {
                const uint4 da = t[2 * id], db = t[2 * id + 1];
                dist = __popc(qa.x ^ da.x) + __popc(qa.y ^ da.y) + __popc(qa.z ^ da.z) + __popc(qa.w ^ da.w) + __popc(qb.x ^ db.x) +
                       __popc(qb.y ^ db.y) + __popc(qb.z ^ db.z) + __popc(qb.w ^ db.w);
            }
        }
        unsigned m = __ballot_sync(0xffffffffu, ok);
        while (m) {
            const int j = __ffs(m) - 1;
            m &= m - 1;
            const int d = __shfl_sync(0xffffffffu, dist, j), c = __shfl_sync(0xffffffffu, id, j);
            if (d < d0) { d1 = d0; d0 = d; i0 = c; }
            else if (d < d1) d1 = d;
        }
    }
    const int pick = (i0 >= 0 && d0 <= th_dist && (float)d0 < __fmul_rn(nnratio, (float)d1)) ? i0 : -1;
    if (lane == 0) {
        if (choice[k] != pick) { choice[k] = pick; *changed = 1; }
        choice_dist[k] = pick >= 0 ? d0 : 256;
        if (pick >= 0) atomicMin(&claim_next[pick], k);
    }
}

// ORBmatcher::SearchForTriangulation (src/ORBmatcher.cc:668-836): candidates of a query = the second key frame's features of the
// same vocabulary node, in list order; a candidate passes when it holds no map point, satisfies the stereo-only rule, has
// dist <= TH_LOW, lies away from the epipole (monocular pair) and close to the epipolar line (CheckDistEpipolarLine, :143-160);
// among the passing candidates `dist <= bestDist` keeps the LAST one of the minimum distance.  Queries are independent
// (this reference never sets vbMatched2).
struct TriParams { float F[9]; float ex, ey; int only_stereo, th_low; };

__global__ void __launch_bounds__(128) k_tri_search(const uint4* __restrict__ qdesc, const hvo_keypoint* __restrict__ qkeys,
                                                    const uint8_t* __restrict__ qstereo, int nq, const uint4* __restrict__ tdesc,
                                                    const hvo_keypoint* __restrict__ tkeys, const uint8_t* __restrict__ tflags,
                                                    const int* __restrict__ off, const int* __restrict__ cand, TriParams P,
                                                    const float* __restrict__ scale_factors, const float* __restrict__ level_sigma2,
                                                    int* __restrict__ match_idx, int* __restrict__ match_dist) {
    const int k = (blockIdx.x * 128 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (k >= nq) return;
    const uint4 qa = qdesc[2 * k], qb = qdesc[2 * k + 1];
    const hvo_keypoint kp1 = qkeys[k];
    const bool stereo1 = qstereo[k] != 0;
    // epipolar line l = x1' F12
    const float a = __fadd_rn(__fadd_rn(__fmul_rn(kp1.x, P.F[0]), __fmul_rn(kp1.y, P.F[3])), P.F[6]);
    const float b = __fadd_rn(__fadd_rn(__fmul_rn(kp1.x, P.F[1]), __fmul_rn(kp1.y, P.F[4])), P.F[7]);
    const float c = __fadd_rn(__fadd_rn(__fmul_rn(kp1.x, P.F[2]), __fmul_rn(kp1.y, P.F[5])), P.F[8]);
    const float den = __fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b));
    int bestDist = P.th_low, bestIdx = -1;
    const bool skip_query = P.only_stereo && !stereo1;
    const int beg = off[k], end = skip_query ? beg : off[k + 1];
    for (int base = beg; base < end; base += 32) {
        const int i = base + lane;
        int id = -1, dist = 256;
        bool ok = false;
        if (i < end) {
            id = cand[i];
            const uint8_t fl = tflags[id];  // bit 0: holds a map point, bit 1: has a right coordinate
            const bool stereo2 = (fl & 2) != 0;
            ok = !(fl & 1) && !(P.only_stereo && !stereo2);
            if (ok) {
                const uint4 da = tdesc[2 * id], db = tdesc[2 * id + 1];
                dist = __popc(qa.x ^ da.x) + __popc(qa.y ^ da.y) + __popc(qa.z ^ da.z) + __popc(qa.w ^ da.w) + __popc(qb.x ^ db.x) +
                       __popc(qb.y ^ db.y) + __popc(qb.z ^ db.z) + __popc(qb.w ^ db.w);
                ok = dist <= P.th_low;
            }
            if (ok) {
                const hvo_keypoint kp2 = tkeys[id];
                if (!stereo1 && !stereo2) {
                    const float dx = __fsub_rn(P.ex, kp2.x), dy = __fsub_rn(P.ey, kp2.y);
                    if (__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)) < __fmul_rn(100.f, scale_factors[kp2.octave])) ok = false;
                }
                if (ok) {
                    if (den == 0) ok = false;
                    else {
                        const float num = __fadd_rn(__fadd_rn(__fmul_rn(a, kp2.x), __fmul_rn(b, kp2.y)), c);
                        const float dsqr = __fdiv_rn(__fmul_rn(num, num), den);
                        ok = (double)dsqr < 3.84 * (double)level_sigma2[kp2.octave];
                    }
                }
            }
        }
        unsigned m = __ballot_sync(0xffffffffu, ok);
        while (m) {
            const int j = __ffs(m) - 1;
            m &= m - 1;
            const int d = __shfl_sync(0xffffffffu, dist, j), cidx = __shfl_sync(0xffffffffu, id, j);
            if (!(d > bestDist)) { bestDist = d; bestIdx = cidx; }
        }
    }
    if (lane == 0) { match_idx[k] = bestIdx; match_dist[k] = bestIdx >= 0 ? bestDist : 256; }
}

}  // namespace hvo

using namespace hvo;


// ---- Frame::isInFrustum(MapPoint*, viewingCosLimit)  (src/Frame.cc:1371-1436) --------------------------------------------------
// One thread per map point.  The arithmetic follows the reference's cv::Mat expressions as OpenCV evaluates them for CV_32F:
//   mRcw * P + mtcw      cv::gemm 3x3 * 3x1: float products summed in k order, then (float)(double(t) + double(c))
//   cv::norm(PO)         sqrt of the sum of squares accumulated in double, in order
//   PO.dot(Pn) / dist    products accumulated in double, in order, divided in double
// everything else in float, one rounding per operation.  PredictScale compares the ratio with host-made thresholds.
struct FrustumCam { float R[9], t[3], O[3], fx, fy, cx, cy, bf, min_x, min_y, max_x, max_y; int n_levels; };
struct MapPt { float pos[3], normal[3], min_dist, max_dist; };           // hvo_map_point
struct TrackPt { float u, v, ur; int level; float view_cos; int in_view; };  // hvo_track_point

__device__ __forceinline__ float gemm_row3(const float* r, float x, float y, float z, float c) {
    const float t = __fadd_rn(__fadd_rn(__fmul_rn(r[0], x), __fmul_rn(r[1], y)), __fmul_rn(r[2], z));
    return (float)((double)t + (double)c);
}
__device__ __forceinline__ TrackPt frustum_point(const FrustumCam& c, const MapPt& m, float cos_limit, const float* __restrict__ thr) {
    TrackPt o;
    o.u = o.v = o.ur = 0.f; o.level = 0; o.view_cos = 0.f; o.in_view = 0;
    const float X = gemm_row3(c.R + 0, m.pos[0], m.pos[1], m.pos[2], c.t[0]);
    const float Y = gemm_row3(c.R + 3, m.pos[0], m.pos[1], m.pos[2], c.t[1]);
    const float Z = gemm_row3(c.R + 6, m.pos[0], m.pos[1], m.pos[2], c.t[2]);
    if (Z < 0.0f) return o;
    const float invz = __fdiv_rn(1.0f, Z);
    const float u = __fadd_rn(__fmul_rn(__fmul_rn(c.fx, X), invz), c.cx);
    const float v = __fadd_rn(__fmul_rn(__fmul_rn(c.fy, Y), invz), c.cy);
    if (u < c.min_x || u > c.max_x) return o;
    if (v < c.min_y || v > c.max_y) return o;
    const float px = __fsub_rn(m.pos[0], c.O[0]), py = __fsub_rn(m.pos[1], c.O[1]), pz = __fsub_rn(m.pos[2], c.O[2]);
    const double n2 = __dadd_rn(__dadd_rn(__dmul_rn((double)px, (double)px), __dmul_rn((double)py, (double)py)), __dmul_rn((double)pz, (double)pz));
    const float dist = (float)sqrt(n2);
    if (dist < __fmul_rn(0.8f, m.min_dist) || dist > __fmul_rn(1.2f, m.max_dist)) return o;   // Get{Min,Max}DistanceInvariance
    const double dot = __dadd_rn(__dadd_rn(__dmul_rn((double)px, (double)m.normal[0]), __dmul_rn((double)py, (double)m.normal[1])),
                                 __dmul_rn((double)pz, (double)m.normal[2]));
    const float view_cos = (float)(dot / (double)dist);
    if (view_cos < cos_limit) return o;
    const float ratio = __fdiv_rn(m.max_dist, dist);
    int level = 0;
    for (int k = 0; k < c.n_levels - 1; ++k) level += ratio >= thr[k];
    o.u = u; o.v = v; o.ur = __fsub_rn(u, __fmul_rn(c.bf, invz)); o.level = level; o.view_cos = view_cos; o.in_view = 1;
    return o;
}

// mode: bit 0 = write TrackPt, bit 1 = write the search query (ORBmatcher::SearchByProjection(F, vpMapPoints, th), :58-71)
__global__ void __launch_bounds__(128) k_frustum_points(FrustumCam c, const MapPt* __restrict__ pts, const uint8_t* __restrict__ skip,
                                                        const uint8_t* __restrict__ claims, int n, float cos_limit,
                                                        const float* __restrict__ thr, float th, const float* __restrict__ scale_factors,
                                                        TrackPt* __restrict__ track, ProjQuery* __restrict__ qs, int* __restrict__ n_in_view) {
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= n) return;
    TrackPt o;
    o.u = o.v = o.ur = 0.f; o.level = 0; o.view_cos = 0.f; o.in_view = 0;
    if (!(skip && skip[i])) o = frustum_point(c, pts[i], cos_limit, thr);
    if (track) track[i] = o;
    if (qs) {
        ProjQuery q;
        if (o.in_view) {
            float r = ((double)o.view_cos > 0.998) ? 2.5f : 4.0f;      // RadiusByViewingCos, ORBmatcher.cc:134-140
            if (th != 1.0f) r = __fmul_rn(r, th);
            q.u = o.u; q.v = o.v; q.r = __fmul_rn(r, scale_factors[o.level]);
            q.min_level = o.level - 1; q.max_level = o.level; q.ur = o.ur; q.claims = claims ? (claims[i] != 0) : 1; q.pad = 0;
        } else {   // not searched: an empty window
            q.u = -1e30f; q.v = -1e30f; q.r = -1.f; q.min_level = 0; q.max_level = 0; q.ur = 0.f; q.claims = 0; q.pad = 0;
        }
        qs[i] = q;
    }
    if (n_in_view && o.in_view) atomicAdd(n_in_view, 1);
}

// ---- ORBmatcher::SearchForInitialization (src/ORBmatcher.cc:412-497) ------------------------------------------------------------
// The loop is sequential through vMatchedDistance / vnMatches21 (a later query may take a keypoint over and un-match an earlier one),
// and it only runs for the monocular initialisation: one warp walks the queries in order, 32 candidates of the window at a time.
__global__ void __launch_bounds__(32) k_init_search(const ProjKey* __restrict__ pk, const uint4* __restrict__ desc, const int* __restrict__ cell_start,
                                                    const int* __restrict__ cell_items, GridGeom g, int n2, const float2* __restrict__ prev,
                                                    const int* __restrict__ octave1, const uint4* __restrict__ desc1, int n1, float window,
                                                    int th_dist, float nnratio, int* __restrict__ matched_dist, int* __restrict__ matches21,
                                                    int* __restrict__ matches12, int* __restrict__ accepted12, int* __restrict__ n_matches) {
    const int lane = threadIdx.x;
    for (int i = lane; i < n2; i += 32) { matched_dist[i] = INT_MAX; matches21[i] = -1; }
    for (int i = lane; i < n1; i += 32) { matches12[i] = -1; accepted12[i] = -1; }
    __syncwarp();
    for (int i1 = 0; i1 < n1; ++i1) {
        if (octave1[i1] > 0) continue;
        const float2 c = prev[i1];
        const ProjWindow w = proj_window(g, c.x, c.y, window);
        if (w.empty) continue;
        const uint4 qa = desc1[2 * i1], qb = desc1[2 * i1 + 1];
        int bestDist = INT_MAX, bestDist2 = INT_MAX, bestIdx2 = -1;
        for (int ix = w.x0; ix <= w.x1; ++ix) {
            const int b = cell_start[ix * kGridRows + w.y0], e = cell_start[ix * kGridRows + w.y1 + 1];
            for (int base = b; base < e; base += 32) {
                const int i = base + lane;
                int id = -1, dist = 256;
                bool ok = false;
                if (i < e) {
                    id = cell_items[i];
                    ok = proj_in_area(pk[id], c.x, c.y, window, 0, 0);
                    if (ok) {
                        const uint4 da = desc[2 * id], db = desc[2 * id + 1];
                        dist = __popc(qa.x ^ da.x) + __popc(qa.y ^ da.y) + __popc(qa.z ^ da.z) + __popc(qa.w ^ da.w) +
                               __popc(qb.x ^ db.x) + __popc(qb.y ^ db.y) + __popc(qb.z ^ db.z) + __popc(qb.w ^ db.w);
                        ok = !(matched_dist[id] <= dist);
                    }
                }
                unsigned m = __ballot_sync(0xffffffffu, ok);
                while (m) {
                    const int j = __ffs(m) - 1;
                    m &= m - 1;
                    const int d = __shfl_sync(0xffffffffu, dist, j), cidx = __shfl_sync(0xffffffffu, id, j);
                    if (d < bestDist) { bestDist2 = bestDist; bestDist = d; bestIdx2 = cidx; }
                    else if (d < bestDist2) bestDist2 = d;
                }
            }
        }
        if (bestDist <= th_dist && (float)bestDist < __fmul_rn((float)bestDist2, nnratio)) {
            if (lane == 0) {
                const int old = matches21[bestIdx2];
                if (old >= 0) matches12[old] = -1;       // a taken-over keypoint un-matches its previous owner
                matches12[i1] = bestIdx2;
                accepted12[i1] = bestIdx2;
                matches21[bestIdx2] = i1;
                matched_dist[bestIdx2] = bestDist;
            }
        }
        __syncwarp();
    }
    // nmatches = accepted - taken over = entries of matches12 that survive
    int cnt = 0;
    for (int i = lane; i < n1; i += 32) cnt += matches12[i] >= 0;
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) *n_matches = cnt;
}

struct hvo_proj {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t tev[2] = {nullptr, nullptr};
    int n = 0, kcap = 0, qcap = 0, ccap = 0;
    GridGeom g{0, 0, 0, 0};    // geometry the cells were built with (Frame::AssignFeaturesToGrid)
    GridGeom gw{0, 0, 0, 0};   // geometry of the window lookups: = g, or with KeyFrame's integer origin (hvo_proj_set_window_origin)
    hvo_keypoint* d_keys = nullptr;
    float* d_uright = nullptr;
    uint8_t* d_desc = nullptr;
    ProjKey* d_pk = nullptr;
    int *d_cell_start = nullptr, *d_cell_items = nullptr;
    uint8_t* d_claimed = nullptr;
    int *d_claim0 = nullptr, *d_claim_a = nullptr, *d_claim_b = nullptr;
    ProjQuery* d_q = nullptr;
    uint8_t* d_qdesc = nullptr;
    int *d_choice = nullptr, *d_cdist = nullptr, *d_flag = nullptr, *d_area = nullptr;
    int* h_flag = nullptr;  // pinned [2]
    int *d_off = nullptr, *d_cand = nullptr;
    int4* d_best4 = nullptr;
    float* d_inv_sigma2 = nullptr;  // [64] mvInvLevelSigma2 (mode 2)
    bool has_sigma = false;
    // local-map projection (isInFrustum + search) and SearchForInitialization
    float* d_thr = nullptr;         // [64] PredictScale thresholds, [64..128) scale factors
    float thr_log = 0.f; int thr_levels = 0;
    MapPt* d_pts = nullptr; TrackPt* d_track = nullptr; uint8_t *d_skip = nullptr, *d_claims = nullptr;
    int pcap = 0;
    int *d_m21 = nullptr, *d_mdist = nullptr; int icap = 0;
    int last_rounds = 0, last_launches = 0;
};

#define HVO_TRYB(call) do { if ((call) != cudaSuccess) { set_error("%s: %s", #call, cudaGetErrorString(cudaGetLastError())); return HVO_ERR_CUDA; } } while (0)

template <class T>
static int grow(T*& p, size_t count) {
    if (p) cudaFree(p);
    p = nullptr;
    HVO_TRYB(cudaMalloc(&p, count * sizeof(T)));
    return HVO_OK;
}

static int proj_reserve_keys(hvo_proj* h, int n) {
    if (n <= h->kcap) return HVO_OK;
    const int cap = std::max(n, 2048);
    int st;
    if ((st = grow(h->d_keys, cap)) || (st = grow(h->d_uright, cap)) || (st = grow(h->d_desc, (size_t)cap * 32)) || (st = grow(h->d_pk, cap)) ||
        (st = grow(h->d_cell_items, cap)) || (st = grow(h->d_claimed, cap)) || (st = grow(h->d_claim0, cap)) ||
        (st = grow(h->d_claim_a, cap)) || (st = grow(h->d_claim_b, cap)) || (st = grow(h->d_area, cap)))
        return st;
    h->kcap = cap;
    return HVO_OK;
}
static int proj_reserve_queries(hvo_proj* h, int nq) {
    if (nq <= h->qcap) return HVO_OK;
    const int cap = std::max(nq, 2048);
    int st;
    if ((st = grow(h->d_q, cap)) || (st = grow(h->d_qdesc, (size_t)cap * 32)) || (st = grow(h->d_choice, cap)) || (st = grow(h->d_cdist, cap)) ||
        (st = grow(h->d_off, (size_t)cap + 1)) || (st = grow(h->d_best4, cap)))
        return st;
    h->qcap = cap;
    return HVO_OK;
}

extern "C" {

int hvo_proj_create(int device, hvo_proj** out) {
    HVO_CHECK_ARG(out, "null out");
    *out = nullptr;
    int ndev = 0;
    HVO_CUDA(cudaGetDeviceCount(&ndev));
    if (ndev < 1) { set_error("no CUDA device: libhvofront has no CPU fallback"); return HVO_ERR_CUDA; }
    HVO_CHECK_ARG(device >= 0 && device < ndev, "device index out of range");
    hvo_proj* h = new (std::nothrow) hvo_proj();
    if (!h) { set_error("out of host memory"); return HVO_ERR_ARG; }
    h->device = device;
    int st = HVO_OK;
    do {
#define HVO_TRY(call) if ((call) != cudaSuccess) { set_error("%s: %s", #call, cudaGetErrorString(cudaGetLastError())); st = HVO_ERR_CUDA; break; }
        HVO_TRY(cudaSetDevice(device));
        HVO_TRY(create_stream(&h->stream));
        HVO_TRY(cudaEventCreate(&h->tev[0]));
        HVO_TRY(cudaEventCreate(&h->tev[1]));
        HVO_TRY(cudaMalloc(&h->d_cell_start, (kGridCells + 1) * sizeof(int)));
        HVO_TRY(cudaMalloc(&h->d_flag, 2 * sizeof(int)));
        HVO_TRY(cudaMalloc(&h->d_inv_sigma2, 64 * sizeof(float)));
        HVO_TRY(cudaMalloc(&h->d_thr, 128 * sizeof(float)));
        HVO_TRY(cudaMallocHost(&h->h_flag, 2 * sizeof(int)));
#undef HVO_TRY
    } while (0);
    if (st != HVO_OK) { hvo_proj_destroy(h); return st; }
    *out = h;
    return HVO_OK;
}

void hvo_proj_destroy(hvo_proj* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    void* bufs[] = {h->d_keys, h->d_uright, h->d_desc, h->d_pk, h->d_cell_start, h->d_cell_items, h->d_claimed, h->d_claim0,
                    h->d_claim_a, h->d_claim_b, h->d_q, h->d_qdesc, h->d_choice, h->d_cdist, h->d_flag, h->d_area, h->d_off, h->d_cand, h->d_best4,
                    h->d_inv_sigma2, h->d_thr, h->d_pts, h->d_track, h->d_skip, h->d_claims, h->d_m21, h->d_mdist};
    for (void* b : bufs) if (b) cudaFree(b);
    if (h->h_flag) cudaFreeHost(h->h_flag);
    for (auto& e : h->tev) if (e) cudaEventDestroy(e);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int hvo_proj_set_frame(hvo_proj* h, const hvo_keypoint* keys_un, const float* uright, const uint8_t* desc, int n, float min_x, float min_y,
                       float max_x, float max_y) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CHECK_ARG(n >= 0 && (n == 0 || (keys_un && desc)), "null keypoints / descriptors");
    HVO_CHECK_ARG(max_x > min_x && max_y > min_y, "empty image bounds");
    HVO_CUDA(cudaSetDevice(h->device));
    int st = proj_reserve_keys(h, n);
    if (st != HVO_OK) return st;
    h->n = n;
    h->g = grid_geom(min_x, min_y, max_x, max_y);
    h->gw = h->g;
    if (n > 0) {
        HVO_CUDA(cudaMemcpyAsync(h->d_keys, keys_un, (size_t)n * sizeof(hvo_keypoint), cudaMemcpyHostToDevice, h->stream));
        if (uright) HVO_CUDA(cudaMemcpyAsync(h->d_uright, uright, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
        HVO_CUDA(cudaMemcpyAsync(h->d_desc, desc, (size_t)n * 32, cudaMemcpyHostToDevice, h->stream));
    }
    k_proj_grid<int><<<1, 1024, 0, h->stream>>>(h->d_keys, uright ? h->d_uright : nullptr, n, nullptr, 0, h->g, h->d_pk, h->d_cell_start, nullptr,
                                                 h->d_cell_items);
    HVO_CUDA(cudaGetLastError());
    h->last_launches = 1;
    return HVO_OK;
}

int hvo_proj_set_window_origin(hvo_proj* h, float min_x, float min_y) {
    HVO_CHECK_ARG(h, "null handle");
    h->gw.min_x = min_x; h->gw.min_y = min_y;   // cells stay as built (h->g); inv_w / inv_h are the frame's (KeyFrame copies them, KeyFrame.cc:47-48)
    return HVO_OK;
}

int hvo_proj_get_grid(hvo_proj* h, int32_t* cell_start, int32_t* cell_items) {
    HVO_CHECK_ARG(h && cell_start && cell_items, "null argument");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaMemcpyAsync(cell_start, h->d_cell_start, (kGridCells + 1) * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    const int m = cell_start[kGridCells];
    if (m > 0) HVO_CUDA(cudaMemcpyAsync(cell_items, h->d_cell_items, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return HVO_OK;
}

int hvo_proj_features_in_area(hvo_proj* h, float x, float y, float r, int min_level, int max_level, int32_t* out, int capacity, int* n_out) {
    HVO_CHECK_ARG(h && out && n_out, "null argument");
    HVO_CHECK_ARG(capacity >= 1, "capacity < 1");
    HVO_CUDA(cudaSetDevice(h->device));
    *n_out = 0;
    if (h->n == 0) return HVO_OK;
    k_proj_area<<<1, 32, 0, h->stream>>>(h->d_pk, h->d_cell_start, h->d_cell_items, h->gw, x, y, r, min_level, max_level, h->d_area, h->kcap,
                                          h->d_flag);
    HVO_CUDA(cudaGetLastError());
    HVO_CUDA(cudaMemcpyAsync(h->h_flag, h->d_flag, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    const int cnt = h->h_flag[0];
    const int cp = std::min(cnt, capacity);
    if (cp > 0) HVO_CUDA(cudaMemcpyAsync(out, h->d_area, (size_t)cp * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    *n_out = cnt;
    return HVO_OK;
}

// the fixed-point rounds over nq device-resident queries (h->d_q, h->d_qdesc); results copied to the host arrays
static int proj_run_rounds(hvo_proj* h, int nq, const uint8_t* claimed, int mode, int th_dist, float nnratio, int32_t* match_idx, int32_t* match_dist,
                           int* n_matches, int launches) {
    cudaStream_t s = h->stream;
    if (claimed) HVO_CUDA(cudaMemcpyAsync(h->d_claimed, claimed, (size_t)h->n, cudaMemcpyHostToDevice, s));
    const int nb = div_up(h->n, 256);
    k_proj_claim_init<<<nb, 256, 0, s>>>(claimed ? h->d_claimed : nullptr, h->n, h->d_claim0);
    HVO_CUDA(cudaMemcpyAsync(h->d_claim_a, h->d_claim0, (size_t)h->n * sizeof(int), cudaMemcpyDeviceToDevice, s));
    k_proj_fill<<<div_up(nq, 256), 256, 0, s>>>(h->d_choice, nq, -2);
    launches += 2;
    int rounds = 0;
    int *prev = h->d_claim_a, *next = h->d_claim_b;
    while (true) {
        HVO_CUDA(cudaMemcpyAsync(next, h->d_claim0, (size_t)h->n * sizeof(int), cudaMemcpyDeviceToDevice, s));
        HVO_CUDA(cudaMemsetAsync(h->d_flag, 0, sizeof(int), s));
        k_proj_round<<<div_up(nq * 32, 128), 128, 0, s>>>(h->d_pk, reinterpret_cast<const uint4*>(h->d_desc), h->d_cell_start, h->d_cell_items,
                                                          h->gw, h->d_q, reinterpret_cast<const uint4*>(h->d_qdesc), nq, prev, next, mode, th_dist,
                                                          nnratio, h->d_inv_sigma2, h->d_choice, h->d_cdist, h->d_flag);
        HVO_CUDA(cudaGetLastError());
        HVO_CUDA(cudaMemcpyAsync(h->h_flag, h->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
        HVO_CUDA(cudaStreamSynchronize(s));
        ++launches; ++rounds;
        if (!h->h_flag[0]) break;        // no choice changed: fixed point == the reference's sequential assignment
        if (rounds > nq + 1) { set_error("projection search did not reach its fixed point"); return HVO_ERR_CUDA; }
        std::swap(prev, next);
    }
    h->last_rounds = rounds; h->last_launches = launches;
    HVO_CUDA(cudaMemcpyAsync(match_idx, h->d_choice, (size_t)nq * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (match_dist) HVO_CUDA(cudaMemcpyAsync(match_dist, h->d_cdist, (size_t)nq * sizeof(int), cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaStreamSynchronize(s));
    if (n_matches) { int c = 0; for (int i = 0; i < nq; ++i) c += match_idx[i] >= 0; *n_matches = c; }
    return HVO_OK;
}

int hvo_proj_search(hvo_proj* h, const hvo_proj_query* queries, const uint8_t* qdesc, int nq, const uint8_t* claimed, int mode, int th_dist,
                    float nnratio, int32_t* match_idx, int32_t* match_dist, int* n_matches) {
    HVO_CHECK_ARG(h && match_idx, "null argument");
    HVO_CHECK_ARG(mode >= 0 && mode <= 2, "mode must be 0 (best + second, level ratio), 1 (best only) or 2 (Fuse: reprojection gate)");
    HVO_CHECK_ARG(mode != 2 || (h->has_sigma && !claimed), "mode 2 needs hvo_proj_set_level_sigma and takes no claimed array");
    if (n_matches) *n_matches = 0;
    if (nq <= 0) return HVO_OK;
    HVO_CHECK_ARG(queries && qdesc, "null queries");
    if (h->n == 0) {
        for (int i = 0; i < nq; ++i) { match_idx[i] = -1; if (match_dist) match_dist[i] = 256; }
        return HVO_OK;
    }
    HVO_CUDA(cudaSetDevice(h->device));
    int st = proj_reserve_queries(h, nq);
    if (st != HVO_OK) return st;
    cudaStream_t s = h->stream;
    HVO_CUDA(cudaMemcpyAsync(h->d_q, queries, (size_t)nq * sizeof(ProjQuery), cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(h->d_qdesc, qdesc, (size_t)nq * 32, cudaMemcpyHostToDevice, s));
    return proj_run_rounds(h, nq, claimed, mode, th_dist, nnratio, match_idx, match_dist, n_matches, 0);
}

// ---- isInFrustum over a batch of map points, alone or in front of the search ----
static float predict_scale_host(float ratio, float log_scale_factor) { return std::ceil(std::log(ratio) / log_scale_factor); }  // float logf, float division

int hvo_predict_scale_thresholds(float log_scale_factor, int lo, int n, float* thresholds) {
    HVO_CHECK_ARG(thresholds && n >= 0 && log_scale_factor > 0.f, "null thresholds / non-positive log scale factor");
    for (int k = 0; k < n; ++k) {
        // smallest positive float r with ceil(logf(r) / L) > lo + k; bit patterns of positive floats are ordered like their values
        const float want = (float)(lo + k);
        uint32_t a = 0x00800000u, b = 0x7f800000u;   // predicate false at a (log of the smallest normal is hugely negative), true at +inf
        while (b - a > 1) {
            const uint32_t mid = a + (b - a) / 2;
            float r; std::memcpy(&r, &mid, 4);
            if (predict_scale_host(r, log_scale_factor) > want) b = mid; else a = mid;
        }
        std::memcpy(&thresholds[k], &b, 4);
    }
    return HVO_OK;
}

static int proj_reserve_points(hvo_proj* h, int n) {
    if (n <= h->pcap) return HVO_OK;
    const int cap = std::max(n, 4096);
    int st;
    if ((st = grow(h->d_pts, cap)) || (st = grow(h->d_track, cap)) || (st = grow(h->d_skip, cap)) || (st = grow(h->d_claims, cap))) return st;
    h->pcap = cap;
    return HVO_OK;
}
static int proj_set_thresholds(hvo_proj* h, const hvo_frustum_cam* cam) {
    HVO_CHECK_ARG(cam->n_levels >= 1 && cam->n_levels <= 64, "n_levels must be in [1, 64]");
    if (h->thr_log == cam->log_scale_factor && h->thr_levels == cam->n_levels) return HVO_OK;
    float thr[64];
    int st = hvo_predict_scale_thresholds(cam->log_scale_factor, 0, cam->n_levels - 1, thr);
    if (st != HVO_OK) return st;
    HVO_CUDA(cudaMemcpyAsync(h->d_thr, thr, sizeof(float) * (size_t)(cam->n_levels - 1), cudaMemcpyHostToDevice, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));   // thr lives on this stack frame
    h->thr_log = cam->log_scale_factor; h->thr_levels = cam->n_levels;
    return HVO_OK;
}
static FrustumCam make_cam(const hvo_frustum_cam* cam) {
    FrustumCam c;
    for (int i = 0; i < 9; ++i) c.R[i] = cam->Rcw[i];
    for (int i = 0; i < 3; ++i) { c.t[i] = cam->tcw[i]; c.O[i] = cam->Ow[i]; }
    c.fx = cam->fx; c.fy = cam->fy; c.cx = cam->cx; c.cy = cam->cy; c.bf = cam->bf;
    c.min_x = cam->min_x; c.min_y = cam->min_y; c.max_x = cam->max_x; c.max_y = cam->max_y; c.n_levels = cam->n_levels;
    return c;
}

int hvo_proj_frustum_points(hvo_proj* h, const hvo_frustum_cam* cam, const hvo_map_point* pts, int n, float viewing_cos_limit, hvo_track_point* out) {
    HVO_CHECK_ARG(h && cam && out, "null argument");
    if (n <= 0) return HVO_OK;
    HVO_CHECK_ARG(pts, "null map points");
    HVO_CUDA(cudaSetDevice(h->device));
    int st = proj_reserve_points(h, n);
    if (st != HVO_OK || (st = proj_set_thresholds(h, cam)) != HVO_OK) return st;
    cudaStream_t s = h->stream;
    HVO_CUDA(cudaMemcpyAsync(h->d_pts, pts, (size_t)n * sizeof(MapPt), cudaMemcpyHostToDevice, s));
    k_frustum_points<<<div_up(n, 128), 128, 0, s>>>(make_cam(cam), h->d_pts, nullptr, nullptr, n, viewing_cos_limit, h->d_thr, 1.f, nullptr, h->d_track,
                                                    nullptr, nullptr);
    HVO_CUDA(cudaGetLastError());
    HVO_CUDA(cudaMemcpyAsync(out, h->d_track, (size_t)n * sizeof(TrackPt), cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaStreamSynchronize(s));
    h->last_launches = 1;
    return HVO_OK;
}

int hvo_proj_search_local_map(hvo_proj* h, const hvo_frustum_cam* cam, const hvo_map_point* pts, const uint8_t* pdesc, const uint8_t* skip,
                              const uint8_t* claims, int n, float viewing_cos_limit, float th, const float* scale_factors, const uint8_t* claimed,
                              int th_dist, float nnratio, hvo_track_point* track, int32_t* match_idx, int32_t* match_dist, int* n_in_view,
                              int* n_matches) {
    HVO_CHECK_ARG(h && cam && match_idx && scale_factors, "null argument");
    if (n_matches) *n_matches = 0;
    if (n_in_view) *n_in_view = 0;
    if (n <= 0) return HVO_OK;
    HVO_CHECK_ARG(pts && pdesc, "null map points / descriptors");
    HVO_CUDA(cudaSetDevice(h->device));
    int st = proj_reserve_points(h, n);
    if (st != HVO_OK || (st = proj_reserve_queries(h, n)) != HVO_OK || (st = proj_set_thresholds(h, cam)) != HVO_OK) return st;
    cudaStream_t s = h->stream;
    HVO_CUDA(cudaMemcpyAsync(h->d_pts, pts, (size_t)n * sizeof(MapPt), cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(h->d_qdesc, pdesc, (size_t)n * 32, cudaMemcpyHostToDevice, s));
    if (skip) HVO_CUDA(cudaMemcpyAsync(h->d_skip, skip, (size_t)n, cudaMemcpyHostToDevice, s));
    if (claims) HVO_CUDA(cudaMemcpyAsync(h->d_claims, claims, (size_t)n, cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(h->d_thr + 64, scale_factors, sizeof(float) * (size_t)cam->n_levels, cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemsetAsync(h->d_flag + 1, 0, sizeof(int), s));
    k_frustum_points<<<div_up(n, 128), 128, 0, s>>>(make_cam(cam), h->d_pts, skip ? h->d_skip : nullptr, claims ? h->d_claims : nullptr, n,
                                                    viewing_cos_limit, h->d_thr, th, h->d_thr + 64, h->d_track, h->d_q, h->d_flag + 1);
    HVO_CUDA(cudaGetLastError());
    if (track) HVO_CUDA(cudaMemcpyAsync(track, h->d_track, (size_t)n * sizeof(TrackPt), cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaMemcpyAsync(h->h_flag + 1, h->d_flag + 1, sizeof(int), cudaMemcpyDeviceToHost, s));
    if (h->n == 0) {
        HVO_CUDA(cudaStreamSynchronize(s));
        for (int i = 0; i < n; ++i) { match_idx[i] = -1; if (match_dist) match_dist[i] = 256; }
        if (n_in_view) *n_in_view = h->h_flag[1];
        return HVO_OK;
    }
    st = proj_run_rounds(h, n, claimed, 0, th_dist, nnratio, match_idx, match_dist, n_matches, 1);
    if (st == HVO_OK && n_in_view) *n_in_view = h->h_flag[1];
    return st;
}

int hvo_proj_search_initialization(hvo_proj* h, const float* prev_matched_xy, const int32_t* octave1, const uint8_t* desc1, int n1, int window_size,
                                   int th_dist, float nnratio, int32_t* matches12, int32_t* accepted12, int* n_matches) {
    HVO_CHECK_ARG(h && matches12, "null argument");
    if (n_matches) *n_matches = 0;
    if (n1 <= 0) return HVO_OK;
    HVO_CHECK_ARG(prev_matched_xy && octave1 && desc1, "null queries");
    if (h->n == 0) {
        for (int i = 0; i < n1; ++i) { matches12[i] = -1; if (accepted12) accepted12[i] = -1; }
        return HVO_OK;
    }
    HVO_CUDA(cudaSetDevice(h->device));
    int st = proj_reserve_queries(h, n1);
    if (st != HVO_OK) return st;
    if (h->n > h->icap) {
        const int cap = std::max(h->n, 2048);
        if ((st = grow(h->d_m21, cap)) || (st = grow(h->d_mdist, cap))) return st;
        h->icap = cap;
    }
    cudaStream_t s = h->stream;
    // query staging reuses the search buffers: d_q holds the window centres (8 B each), d_off the octaves, d_choice / d_cdist the results
    HVO_CUDA(cudaMemcpyAsync(h->d_q, prev_matched_xy, (size_t)n1 * 2 * sizeof(float), cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(h->d_off, octave1, (size_t)n1 * sizeof(int), cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(h->d_qdesc, desc1, (size_t)n1 * 32, cudaMemcpyHostToDevice, s));
    k_init_search<<<1, 32, 0, s>>>(h->d_pk, reinterpret_cast<const uint4*>(h->d_desc), h->d_cell_start, h->d_cell_items, h->g, h->n,
                                   reinterpret_cast<const float2*>(h->d_q), h->d_off, reinterpret_cast<const uint4*>(h->d_qdesc), n1, (float)window_size,
                                   th_dist, nnratio, h->d_mdist, h->d_m21, h->d_choice, h->d_cdist, h->d_flag);
    HVO_CUDA(cudaGetLastError());
    HVO_CUDA(cudaMemcpyAsync(matches12, h->d_choice, (size_t)n1 * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (accepted12) HVO_CUDA(cudaMemcpyAsync(accepted12, h->d_cdist, (size_t)n1 * sizeof(int), cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaMemcpyAsync(h->h_flag, h->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaStreamSynchronize(s));
    if (n_matches) *n_matches = h->h_flag[0];
    h->last_launches = 1; h->last_rounds = 1;
    return HVO_OK;
}

int hvo_proj_set_level_sigma(hvo_proj* h, const float* inv_level_sigma2, int nlevels) {
    HVO_CHECK_ARG(h && inv_level_sigma2, "null argument");
    HVO_CHECK_ARG(nlevels >= 1 && nlevels <= 64, "nlevels out of range (1..64)");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaMemcpyAsync(h->d_inv_sigma2, inv_level_sigma2, (size_t)nlevels * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    h->has_sigma = true;
    return HVO_OK;
}

int hvo_proj_last_rounds(const hvo_proj* h) { return h ? h->last_rounds : 0; }
int hvo_proj_last_launches(const hvo_proj* h) { return h ? h->last_launches : 0; }

int hvo_proj_match_candidates(hvo_proj* h, const uint8_t* q, int nq, const uint8_t* t, int nt, const int32_t* offsets, const int32_t* cand,
                              int32_t* best4) {
    HVO_CHECK_ARG(h && best4, "null argument");
    if (nq <= 0) return HVO_OK;
    HVO_CHECK_ARG(q && offsets, "null argument");
    const int total = offsets[nq];
    HVO_CHECK_ARG(total >= 0 && (total == 0 || (cand && t && nt > 0)), "candidate lists without a train set");
    HVO_CUDA(cudaSetDevice(h->device));
    int st = proj_reserve_queries(h, nq);
    if (st == HVO_OK) st = proj_reserve_keys(h, nt);
    if (st != HVO_OK) return st;
    if (total > h->ccap) {
        if ((st = grow(h->d_cand, (size_t)std::max(total, 4096)))) return st;
        h->ccap = std::max(total, 4096);
    }
    cudaStream_t s = h->stream;
    HVO_CUDA(cudaMemcpyAsync(h->d_qdesc, q, (size_t)nq * 32, cudaMemcpyHostToDevice, s));
    if (nt > 0) HVO_CUDA(cudaMemcpyAsync(h->d_desc, t, (size_t)nt * 32, cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(h->d_off, offsets, ((size_t)nq + 1) * sizeof(int), cudaMemcpyHostToDevice, s));
    if (total > 0) HVO_CUDA(cudaMemcpyAsync(h->d_cand, cand, (size_t)total * sizeof(int), cudaMemcpyHostToDevice, s));
    k_match_candidates<<<div_up(nq * 32, 128), 128, 0, s>>>(reinterpret_cast<const uint4*>(h->d_qdesc), nq, reinterpret_cast<const uint4*>(h->d_desc),
                                                            h->d_off, h->d_cand, h->d_best4);
    HVO_CUDA(cudaGetLastError());
    HVO_CUDA(cudaMemcpyAsync(best4, h->d_best4, (size_t)nq * sizeof(int4), cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaStreamSynchronize(s));
    h->n = 0;  // the frame descriptors were overwritten: hvo_proj_set_frame must be called again before the next search
    h->last_launches = 1;
    return HVO_OK;
}

int hvo_proj_search_candidates(hvo_proj* h, const uint8_t* q, int nq, const uint8_t* t, int nt, const int32_t* offsets, const int32_t* cand,
                               int th_dist, float nnratio, int32_t* match_idx, int32_t* match_dist, int* n_matches) {
    HVO_CHECK_ARG(h && match_idx, "null argument");
    if (n_matches) *n_matches = 0;
    if (nq <= 0) return HVO_OK;
    HVO_CHECK_ARG(q && offsets, "null argument");
    const int total = offsets[nq];
    HVO_CHECK_ARG(total >= 0 && (total == 0 || (cand && t && nt > 0)), "candidate lists without a train set");
    for (int i = 0; i < total; ++i) HVO_CHECK_ARG(cand[i] >= 0 && cand[i] < nt, "candidate index out of range");
    HVO_CUDA(cudaSetDevice(h->device));
    int st = proj_reserve_queries(h, nq);
    if (st == HVO_OK) st = proj_reserve_keys(h, std::max(nt, 1));
    if (st != HVO_OK) return st;
    if (total > h->ccap) {
        if ((st = grow(h->d_cand, (size_t)std::max(total, 4096)))) return st;
        h->ccap = std::max(total, 4096);
    }
    cudaStream_t s = h->stream;
    h->n = 0;  // the frame descriptors are overwritten: hvo_proj_set_frame must be called again before the next windowed search
    HVO_CUDA(cudaMemcpyAsync(h->d_qdesc, q, (size_t)nq * 32, cudaMemcpyHostToDevice, s));
    if (nt > 0) HVO_CUDA(cudaMemcpyAsync(h->d_desc, t, (size_t)nt * 32, cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(h->d_off, offsets, ((size_t)nq + 1) * sizeof(int), cudaMemcpyHostToDevice, s));
    if (total > 0) HVO_CUDA(cudaMemcpyAsync(h->d_cand, cand, (size_t)total * sizeof(int), cudaMemcpyHostToDevice, s));
    const int nk = std::max(nt, 1);
    k_proj_claim_init<<<div_up(nk, 256), 256, 0, s>>>(nullptr, nk, h->d_claim0);
    HVO_CUDA(cudaMemcpyAsync(h->d_claim_a, h->d_claim0, (size_t)nk * sizeof(int), cudaMemcpyDeviceToDevice, s));
    k_proj_fill<<<div_up(nq, 256), 256, 0, s>>>(h->d_choice, nq, -2);
    int launches = 2, rounds = 0;
    int *prev = h->d_claim_a, *next = h->d_claim_b;
    while (true) {
        HVO_CUDA(cudaMemcpyAsync(next, h->d_claim0, (size_t)nk * sizeof(int), cudaMemcpyDeviceToDevice, s));
        HVO_CUDA(cudaMemsetAsync(h->d_flag, 0, sizeof(int), s));
        k_cand_round<<<div_up(nq * 32, 128), 128, 0, s>>>(reinterpret_cast<const uint4*>(h->d_qdesc), nq, reinterpret_cast<const uint4*>(h->d_desc),
                                                          h->d_off, h->d_cand, prev, next, th_dist, nnratio, h->d_choice, h->d_cdist, h->d_flag);
        HVO_CUDA(cudaGetLastError());
        HVO_CUDA(cudaMemcpyAsync(h->h_flag, h->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
        HVO_CUDA(cudaStreamSynchronize(s));
        ++launches; ++rounds;
        if (!h->h_flag[0]) break;
        if (rounds > nq + 1) { set_error("candidate search did not reach its fixed point"); return HVO_ERR_CUDA; }
        std::swap(prev, next);
    }
    h->last_rounds = rounds; h->last_launches = launches;
    HVO_CUDA(cudaMemcpyAsync(match_idx, h->d_choice, (size_t)nq * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (match_dist) HVO_CUDA(cudaMemcpyAsync(match_dist, h->d_cdist, (size_t)nq * sizeof(int), cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaStreamSynchronize(s));
    if (n_matches) { int c = 0; for (int i = 0; i < nq; ++i) c += match_idx[i] >= 0; *n_matches = c; }
    return HVO_OK;
}

int hvo_proj_search_triangulation(hvo_proj* h, const uint8_t* qdesc, const hvo_keypoint* qkeys, const uint8_t* qstereo, int nq, const uint8_t* tdesc,
                                  const hvo_keypoint* tkeys, const uint8_t* tflags, int nt, const int32_t* offsets, const int32_t* cand,
                                  const float* F12, float ex, float ey, const float* scale_factors, const float* level_sigma2, int nlevels,
                                  int only_stereo, int th_low, int32_t* match_idx, int32_t* match_dist, int* n_matches) {
    HVO_CHECK_ARG(h && match_idx, "null argument");
    if (n_matches) *n_matches = 0;
    if (nq <= 0) return HVO_OK;
    HVO_CHECK_ARG(qdesc && qkeys && qstereo && offsets && F12 && scale_factors && level_sigma2, "null argument");
    HVO_CHECK_ARG(nlevels >= 1 && nlevels <= 64, "nlevels out of range (1..64)");
    const int total = offsets[nq];
    HVO_CHECK_ARG(total >= 0 && (total == 0 || (cand && tdesc && tkeys && tflags && nt > 0)), "candidate lists without a train set");
    for (int i = 0; i < total; ++i) HVO_CHECK_ARG(cand[i] >= 0 && cand[i] < nt, "candidate index out of range");
    for (int i = 0; i < nt; ++i) HVO_CHECK_ARG(tkeys[i].octave >= 0 && tkeys[i].octave < nlevels, "train keypoint octave out of range");
    HVO_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    h->n = 0;  // scratch of the windowed search is not touched, but the call owns the stream: keep the contract simple
    uint8_t *d_qd = nullptr, *d_qs = nullptr, *d_td = nullptr, *d_tf = nullptr;
    hvo_keypoint *d_qk = nullptr, *d_tk = nullptr;
    int *d_off = nullptr, *d_cand = nullptr, *d_out = nullptr;
    float* d_tab = nullptr;
    const size_t ntt = (size_t)std::max(nt, 1), tot = (size_t)std::max(total, 1);
    HVO_CUDA(cudaMallocAsync(&d_qd, (size_t)nq * 32, s)); HVO_CUDA(cudaMallocAsync(&d_qk, (size_t)nq * sizeof(hvo_keypoint), s));
    HVO_CUDA(cudaMallocAsync(&d_qs, (size_t)nq, s)); HVO_CUDA(cudaMallocAsync(&d_td, ntt * 32, s));
    HVO_CUDA(cudaMallocAsync(&d_tk, ntt * sizeof(hvo_keypoint), s)); HVO_CUDA(cudaMallocAsync(&d_tf, ntt, s));
    HVO_CUDA(cudaMallocAsync(&d_off, ((size_t)nq + 1) * 4, s)); HVO_CUDA(cudaMallocAsync(&d_cand, tot * 4, s));
    HVO_CUDA(cudaMallocAsync(&d_out, (size_t)nq * 8, s)); HVO_CUDA(cudaMallocAsync(&d_tab, 128 * sizeof(float), s));
    HVO_CUDA(cudaMemcpyAsync(d_qd, qdesc, (size_t)nq * 32, cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(d_qk, qkeys, (size_t)nq * sizeof(hvo_keypoint), cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(d_qs, qstereo, (size_t)nq, cudaMemcpyHostToDevice, s));
    if (nt > 0) {
        HVO_CUDA(cudaMemcpyAsync(d_td, tdesc, (size_t)nt * 32, cudaMemcpyHostToDevice, s));
        HVO_CUDA(cudaMemcpyAsync(d_tk, tkeys, (size_t)nt * sizeof(hvo_keypoint), cudaMemcpyHostToDevice, s));
        HVO_CUDA(cudaMemcpyAsync(d_tf, tflags, (size_t)nt, cudaMemcpyHostToDevice, s));
    }
    HVO_CUDA(cudaMemcpyAsync(d_off, offsets, ((size_t)nq + 1) * 4, cudaMemcpyHostToDevice, s));
    if (total > 0) HVO_CUDA(cudaMemcpyAsync(d_cand, cand, (size_t)total * 4, cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(d_tab, scale_factors, (size_t)nlevels * sizeof(float), cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(d_tab + 64, level_sigma2, (size_t)nlevels * sizeof(float), cudaMemcpyHostToDevice, s));
    TriParams P;
    for (int i = 0; i < 9; ++i) P.F[i] = F12[i];
    P.ex = ex; P.ey = ey; P.only_stereo = only_stereo != 0; P.th_low = th_low;
    k_tri_search<<<div_up(nq * 32, 128), 128, 0, s>>>(reinterpret_cast<const uint4*>(d_qd), d_qk, d_qs, nq, reinterpret_cast<const uint4*>(d_td), d_tk,
                                                      d_tf, d_off, d_cand, P, d_tab, d_tab + 64, d_out, d_out + nq);
    HVO_CUDA(cudaGetLastError());
    HVO_CUDA(cudaMemcpyAsync(match_idx, d_out, (size_t)nq * 4, cudaMemcpyDeviceToHost, s));
    if (match_dist) HVO_CUDA(cudaMemcpyAsync(match_dist, d_out + nq, (size_t)nq * 4, cudaMemcpyDeviceToHost, s));
    void* bufs[] = {d_qd, d_qk, d_qs, d_td, d_tk, d_tf, d_off, d_cand, d_out, d_tab};
    for (void* b : bufs) HVO_CUDA(cudaFreeAsync(b, s));
    HVO_CUDA(cudaStreamSynchronize(s));
    if (n_matches) { int c = 0; for (int i = 0; i < nq; ++i) c += match_idx[i] >= 0; *n_matches = c; }
    h->last_launches = 1; h->last_rounds = 1;
    return HVO_OK;
}

int hvo_proj_timer_start(hvo_proj* h) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[0], h->stream));
    return HVO_OK;
}
int hvo_proj_timer_stop(hvo_proj* h, float* ms_out) {
    HVO_CHECK_ARG(h && ms_out, "null argument");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[1], h->stream));
    HVO_CUDA(cudaEventSynchronize(h->tev[1]));
    HVO_CUDA(cudaEventElapsedTime(ms_out, h->tev[0], h->tev[1]));
    return HVO_OK;
}

}  // extern "C"
