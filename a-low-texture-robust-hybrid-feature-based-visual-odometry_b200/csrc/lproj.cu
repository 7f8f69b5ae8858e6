// Windowed (projection) line matchers for sm_100a.
//
//   Frame::AssignFeaturesToGridForLine      reference src/Frame.cc:849-872 + src/lineIterator.cpp:35-79
//   Frame::GetFeaturesInAreaForLine         src/Frame.cc:1557-1631
//   LSDmatcher::SearchByProjection(F, MapLines, eval_orient, th)   src/LSDmatcher.cpp:709-801   (mode 0)
//   LSDmatcher::SearchByProjection(CurrentFrame, LastFrame, th)    src/LSDmatcher.cpp:561-664   (mode 1)
//
// The reference keeps a std::vector of line indices per grid cell, filled in line order: here a cell is a bit row over the
// frame's lines (bit i = line i crosses the cell), so "the cell's list in push_back order" is "the set bits, ascending".
// A query is one warp: it walks the three sample points, the cells of each window in (ix, iy) order and the words of each
// cell row; the 32 lines of a word are tested in parallel and folded into best / second in ascending order, which is the
// order the reference visits them in.  Lines accepted into the candidate list are remembered in a per-warp bit row (the
// reference's unordered_set).  The greedy "skip lines that already hold a map line" rule is resolved like the point
// matcher's (project.cu): rounds over all queries until no choice changes.  The frame pipeline builds the bit rows of every frame of a call
// (k_lproj_grid, one thread per (frame, line)) and compacts them into mGridForLine's counts and items (k_lproj_grid_compact).
#include <algorithm>
#include <climits>
#include <new>
#include <vector>

#include "hvo_common.cuh"

namespace hvo {

static const int kLGridCols = 64, kLGridRows = 48, kLGridCells = kLGridCols * kLGridRows;
static const int kLMaxWords = 32;  // up to 1024 lines per frame

struct LGridGeom { float min_x, min_y, inv_w, inv_h; };

struct LKey {          // per frame line, everything the per-candidate tests read
    float sx, sy;      // startPoint
    float d2x, d2y;    // (start - end) / |start - end| as GetFeaturesInAreaForLine computes it (float)
    float ocx, ocy;    // ePointInOctave - sPointInOctave (float)
    float length;      // lineLength
    int octave;
};

struct LQuery {  // hvo_lproj_query
    float x1, y1, x2, y2, r, cos_th;
    double dir[3];
    float length;
    int claims;
    int pad[2];
};
static_assert(sizeof(LQuery) == sizeof(hvo_lproj_query), "query layout");

// One thread per (frame, line): ORB_SLAM2::LineIterator over the grid (doubles), one atomicOr per visited cell.  Frame f = blockIdx.x:
// keyline rows [f * stride, + n_f), n_f = counts ? counts[f] : n, bit rows at cells + f * 3072 * W; keys (NULL in the frame pipeline)
// receives the LKey rows.
__global__ void k_lproj_grid(const hvo_keyline* __restrict__ kl, int n, const int32_t* __restrict__ counts, int stride, LGridGeom g, int W,
                             uint32_t* __restrict__ cells, LKey* __restrict__ keys) {
    const int i = blockIdx.y * blockDim.x + threadIdx.x, f = blockIdx.x;
    if (counts) n = min(counts[f], stride);
    if (i >= n) return;
    const hvo_keyline k = kl[(size_t)f * stride + i];
    cells += (size_t)f * kLGridCells * W;
    if (keys) {
        LKey o;
        o.sx = k.startPointX; o.sy = k.startPointY;
        float dx = __fsub_rn(k.startPointX, k.endPointX), dy = __fsub_rn(k.startPointY, k.endPointY);
        const float nrm = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
        o.d2x = __fdiv_rn(dx, nrm); o.d2y = __fdiv_rn(dy, nrm);
        o.ocx = __fsub_rn(k.ePointInOctaveX, k.sPointInOctaveX); o.ocy = __fsub_rn(k.ePointInOctaveY, k.sPointInOctaveY);
        o.length = k.lineLength; o.octave = k.octave;
        keys[i] = o;
    }
    // the reference walks endpoint * inv without the min_x / min_y offset (Frame.cc:849-872)
    double x1 = (double)__fmul_rn(k.startPointX, g.inv_w), y1 = (double)__fmul_rn(k.startPointY, g.inv_h);
    double x2 = (double)__fmul_rn(k.endPointX, g.inv_w), y2 = (double)__fmul_rn(k.endPointY, g.inv_h);
    const bool steep = fabs(y2 - y1) > fabs(x2 - x1);
    if (steep) { double t = x1; x1 = y1; y1 = t; t = x2; x2 = y2; y2 = t; }
    if (x1 > x2) { double t = x1; x1 = x2; x2 = t; t = y1; y1 = y2; y2 = t; }
    const double ddx = x2 - x1, ddy = fabs(y2 - y1);
    double error = ddx / 2.0;
    const int ystep = (y1 < y2) ? 1 : -1;
    int x = (int)x1, y = (int)y1;
    const int maxX = (int)x2;
    for (; x <= maxX; ++x) {
        const int px = steep ? y : x, py = steep ? x : y;
        if (px >= 0 && px < kLGridCols && py >= 0 && py < kLGridRows) atomicOr(&cells[(size_t)(px * kLGridRows + py) * W + (i >> 5)], 1u << (i & 31));
        error -= ddy;
        if (error < 0) { y += ystep; error += ddx; }
    }
}

// One CTA per frame: bit rows -> mGridForLine as counts [f][3072] + items [f][items_stride], a cell's lines ascending (the reference's
// push_back order).  Only the first sum(counts) items are written.
__global__ void __launch_bounds__(1024) k_lproj_grid_compact(const uint32_t* __restrict__ cells, int W, uint16_t* __restrict__ cell_count,
                                                             uint16_t* __restrict__ cell_items, int items_stride) {
    __shared__ int s_part[32];
    const int tid = threadIdx.x, f = blockIdx.x;
    cells += (size_t)f * kLGridCells * W;
    cell_items += (size_t)f * items_stride;
    int v[3], sum = 0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const uint32_t* row = cells + (size_t)(tid * 3 + k) * W;
        int c = 0;
        for (int w = 0; w < W; ++w) c += __popc(row[w]);
        v[k] = c; sum += c;
    }
    int o = block_exclusive_scan3(sum, s_part);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        cell_count[(size_t)f * kLGridCells + tid * 3 + k] = (uint16_t)v[k];
        const uint32_t* row = cells + (size_t)(tid * 3 + k) * W;
        for (int w = 0; w < W; ++w)
            for (uint32_t b = row[w]; b; b &= b - 1) cell_items[o++] = (uint16_t)(32 * w + __ffs(b) - 1);
    }
}

static LGridGeom lgrid_geom(float min_x, float min_y, float max_x, float max_y) {
    LGridGeom g;
    g.min_x = min_x; g.min_y = min_y;
    g.inv_w = (float)kLGridCols / (max_x - min_x);   // Frame.cc:419-420
    g.inv_h = (float)kLGridRows / (max_y - min_y);
    return g;
}

// The frame pipeline's line grids (hvo_frame_grid_outputs): nframes frames of `stride` keyline rows, counts on the device; d_bits =
// scratch of nframes * 3072 * ceil(stride / 32) words.  A line visits at most 64 in-grid cells (LineIterator advances the major axis
// by one cell per step), so 64 * stride items per frame always suffice.
int lproj_grid_frames_launch(cudaStream_t s, const hvo_keyline* d_kl, const int32_t* d_counts, int nframes, int stride, float min_x, float min_y,
                             float max_x, float max_y, uint32_t* d_bits, uint16_t* d_cell_count, uint16_t* d_cell_items) {
    const int W = div_up(stride, 32);
    HVO_CUDA(cudaMemsetAsync(d_bits, 0, (size_t)nframes * kLGridCells * W * sizeof(uint32_t), s));
    k_lproj_grid<<<dim3(nframes, div_up(stride, 128)), 128, 0, s>>>(d_kl, 0, d_counts, stride, lgrid_geom(min_x, min_y, max_x, max_y), W, d_bits, nullptr);
    k_lproj_grid_compact<<<nframes, 1024, 0, s>>>(d_bits, W, d_cell_count, d_cell_items, kLGridCols * stride);
    HVO_CUDA(cudaGetLastError());
    return HVO_OK;
}

// Walks GetFeaturesInAreaForLine for one query (whole warp).  visit(id, pass, sample) is called once per word of candidate
// lines with pass = this lane's line was just accepted into the list; accepted lines of a word are in ascending lane order.
template <class Visit>
__device__ __forceinline__ void lproj_walk(const LGridGeom& g, int W, const uint32_t* __restrict__ cells, const LKey* __restrict__ keys,
                                           const double* __restrict__ func3, float x1, float y1, float x2, float y2, float r, float TH, int lane,
                                           Visit visit) {
    const float xs[3] = {x1, (float)((double)__fadd_rn(x1, x2) / 2.0), x2};
    const float ys[3] = {y1, (float)((double)__fadd_rn(y1, y2) / 2.0), y2};
    float d1x = __fsub_rn(x1, x2), d1y = __fsub_rn(y1, y2);
    const float n1 = __fsqrt_rn(__fadd_rn(__fmul_rn(d1x, d1x), __fmul_rn(d1y, d1y)));
    d1x = __fdiv_rn(d1x, n1); d1y = __fdiv_rn(d1y, n1);
    uint32_t seen = 0;  // lane w: word w of the accepted set
    for (int i = 0; i < 3; ++i) {
        const float x = xs[i], y = ys[i];
        const int cx0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(__fsub_rn(x, g.min_x), r), g.inv_w)));
        if (cx0 >= kLGridCols) continue;
        const int cx1 = min(kLGridCols - 1, (int)ceilf(__fmul_rn(__fadd_rn(__fsub_rn(x, g.min_x), r), g.inv_w)));
        if (cx1 < 0) continue;
        const int cy0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(__fsub_rn(y, g.min_y), r), g.inv_h)));
        if (cy0 >= kLGridRows) continue;
        const int cy1 = min(kLGridRows - 1, (int)ceilf(__fmul_rn(__fadd_rn(__fsub_rn(y, g.min_y), r), g.inv_h)));
        if (cy1 < 0) continue;
        for (int ix = cx0; ix <= cx1; ++ix)
            for (int iy = cy0; iy <= cy1; ++iy) {
                const uint32_t* row = cells + (size_t)(ix * kLGridRows + iy) * W;
                const uint32_t mine = lane < W ? row[lane] & ~seen : 0u;  // lane w: unseen lines of word w in this cell
                unsigned any = __ballot_sync(0xffffffffu, mine != 0u);
                while (any) {
                    const int w = __ffs(any) - 1;
                    any &= any - 1;
                    const uint32_t bits = __shfl_sync(0xffffffffu, mine, w);
                    const int id = 32 * w + lane;
                    bool pass = false;
                    if ((bits >> lane) & 1u) {
                        const LKey k = keys[id];
                        const float cs = fabsf(__fadd_rn(__fmul_rn(d1x, k.d2x), __fmul_rn(d1y, k.d2y)));
                        if (!(cs < TH)) {
                            const double* L = func3 + 3 * (size_t)id;
                            const float dist = (float)__dadd_rn(__dadd_rn(__dmul_rn(L[0], (double)x), __dmul_rn(L[1], (double)y)), L[2]);
                            pass = fabsf(dist) < r;
                        }
                    }
                    const unsigned pm = __ballot_sync(0xffffffffu, pass);
                    if (lane == w) seen |= pm;
                    visit(id, pass, pm);
                }
            }
    }
}

__global__ void __launch_bounds__(32) k_lproj_area(LGridGeom g, int W, const uint32_t* __restrict__ cells, const LKey* __restrict__ keys,
                                                   const double* __restrict__ func3, float x1, float y1, float x2, float y2, float r, float TH,
                                                   int* __restrict__ out, int cap, int* __restrict__ n_out) {
    const int lane = threadIdx.x;
    int cnt = 0;
    lproj_walk(g, W, cells, keys, func3, x1, y1, x2, y2, r, TH, lane, [&](int id, bool pass, unsigned pm) {
        if (pass) { const int o = cnt + __popc(pm & ((1u << lane) - 1u)); if (o < cap) out[o] = id; }
        cnt += __popc(pm);
    });
    if (lane == 0) *n_out = cnt;
}

__global__ void __launch_bounds__(128) k_lproj_round(LGridGeom g, int W, const uint32_t* __restrict__ cells, const LKey* __restrict__ keys,
                                                     const double* __restrict__ func3, const uint4* __restrict__ desc,
                                                     const double* __restrict__ lines3d, const LQuery* __restrict__ qs,
                                                     const uint4* __restrict__ qdesc, int nq, const int* __restrict__ claim_prev,
                                                     int* __restrict__ claim_next, int mode, float nnratio, double th_normal, double cos_th_angle,
                                                     int* __restrict__ choice, int* __restrict__ choice_dist, int* __restrict__ changed) {
    const int k = (blockIdx.x * 128 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (k >= nq) return;
    const LQuery q = qs[k];
    const uint4 qa = qdesc[2 * k], qb = qdesc[2 * k + 1];
    int bestDist = 256, bestLevel = -1, bestDist2 = 256, bestLevel2 = -1, bestIdx = -1;
    lproj_walk(g, W, cells, keys, func3, q.x1, q.y1, q.x2, q.y2, q.r, q.cos_th, lane, [&](int id, bool pass, unsigned pm) {
        int dist = 256, oct = 0;
        bool ok = pass && !(claim_prev[id] < k);
        if (ok) {
            const LKey key = keys[id];
            oct = key.octave;
            if (mode == 0) {   // LSDmatcher.cpp:761-771: float |cos| between the frame line's 3-D direction and the map line's
                const double* P = lines3d + 6 * (size_t)id;
                const double w0 = __dsub_rn(P[0], P[3]), w1 = __dsub_rn(P[1], P[4]), w2 = __dsub_rn(P[2], P[5]);
                // Eigen's unrolled 3-term reduction: x0 + (x1 + x2)
                const float dot = (float)__dadd_rn(__dmul_rn(w0, q.dir[0]), __dadd_rn(__dmul_rn(w1, q.dir[1]), __dmul_rn(w2, q.dir[2])));
                const float mag_f = (float)__dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(w0, w0), __dmul_rn(w1, w1)), __dmul_rn(w2, w2)));
                const float mag_ml = (float)__dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(q.dir[0], q.dir[0]), __dmul_rn(q.dir[1], q.dir[1])), __dmul_rn(q.dir[2], q.dir[2])));
                const float angle = fabsf(__fdiv_rn(dot, __fmul_rn(mag_f, mag_ml)));
                if ((double)angle < th_normal) ok = false;
            } else {           // LSDmatcher.cpp:623-648: 2-D direction (double) and length ratio (float)
                const double cx = (double)key.ocx, cy = (double)key.ocy;
                const double dotp = __dadd_rn(__dmul_rn(cx, q.dir[0]), __dmul_rn(cy, q.dir[1]));
                const double magA = __dsqrt_rn(__dadd_rn(__dmul_rn(cx, cx), __dmul_rn(cy, cy)));
                const double magB = __dsqrt_rn(__dadd_rn(__dmul_rn(q.dir[0], q.dir[0]), __dmul_rn(q.dir[1], q.dir[1])));
                const double angle = fabs(__ddiv_rn(dotp, __dmul_rn(magA, magB)));
                if (angle < cos_th_angle) ok = false;
                const float mx = fmaxf(q.length, key.length), mn = fminf(q.length, key.length);
                if (__fdiv_rn(mn, mx) < 0.75f) ok = false;
            }
            if (ok) {
                const uint4 da = desc[2 * id], db = desc[2 * id + 1];
                dist = __popc(qa.x ^ da.x) + __popc(qa.y ^ da.y) + __popc(qa.z ^ da.z) + __popc(qa.w ^ da.w) + __popc(qb.x ^ db.x) +
                       __popc(qb.y ^ db.y) + __popc(qb.z ^ db.z) + __popc(qb.w ^ db.w);
            }
        }
        unsigned m = __ballot_sync(0xffffffffu, ok);
        while (m) {
            const int j = __ffs(m) - 1;
            m &= m - 1;
            const int d = __shfl_sync(0xffffffffu, dist, j), l = __shfl_sync(0xffffffffu, oct, j), c = __shfl_sync(0xffffffffu, id, j);
            if (d < bestDist) { bestDist2 = bestDist; bestDist = d; bestLevel2 = bestLevel; bestLevel = l; bestIdx = c; }
            else if (mode == 0 && d < bestDist2) { bestLevel2 = l; bestDist2 = d; }
        }
    });
    int pick = -1;
    if (bestDist <= 95 && !(mode == 0 && bestLevel == bestLevel2 && (float)bestDist > __fmul_rn(nnratio, (float)bestDist2))) pick = bestIdx;
    if (lane == 0) {
        if (choice[k] != pick) { choice[k] = pick; *changed = 1; }
        choice_dist[k] = pick >= 0 ? bestDist : 256;
        if (pick >= 0 && q.claims) atomicMin(&claim_next[pick], k);
    }
}

__global__ void k_lproj_claim_init(const uint8_t* __restrict__ claimed, int n, int* __restrict__ a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = (claimed && claimed[i]) ? -1 : INT_MAX;
}
__global__ void k_lproj_fill(int* __restrict__ a, int n, int v) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = v;
}


// ---- Frame::isInFrustum(MapLine*, viewingCosLimit)  (src/Frame.cc:1438-1499) --------------------------------------------------
// One thread per map line; cv::Mat arithmetic as in k_frustum_points (project.cu).  End points and normal are narrowed to float
// first (Mat_<float> << P(0) ...); the mid point is cv::addWeighted(SP, 0.5, EP, 0.5) - mOw; PredictScale is not clamped.
struct LFrustumCam { float R[9], t[3], O[3], fx, fy, cx, cy, min_x, min_y, max_x, max_y; int thr_lo, thr_n; };
struct MapLn { double pos[6], normal[3], dir[3]; float min_dist, max_dist; };   // hvo_map_line
struct TrackLn { float x1, y1, x2, y2; int level; float view_cos; int in_view; };  // hvo_track_line
static_assert(sizeof(MapLn) == sizeof(hvo_map_line) && sizeof(TrackLn) == sizeof(hvo_track_line), "layout");

__device__ __forceinline__ float lgemm_row3(const float* r, float x, float y, float z, float c) {
    const float t = __fadd_rn(__fadd_rn(__fmul_rn(r[0], x), __fmul_rn(r[1], y)), __fmul_rn(r[2], z));
    return (float)((double)t + (double)c);
}
__device__ __forceinline__ TrackLn frustum_line(const LFrustumCam& c, const MapLn& m, float cos_limit, const float* __restrict__ thr) {
    TrackLn o;
    o.x1 = o.y1 = o.x2 = o.y2 = 0.f; o.level = 0; o.view_cos = 0.f; o.in_view = 0;
    const float sx = (float)m.pos[0], sy = (float)m.pos[1], sz = (float)m.pos[2], ex = (float)m.pos[3], ey = (float)m.pos[4], ez = (float)m.pos[5];
    const float SX = lgemm_row3(c.R + 0, sx, sy, sz, c.t[0]), SY = lgemm_row3(c.R + 3, sx, sy, sz, c.t[1]), SZ = lgemm_row3(c.R + 6, sx, sy, sz, c.t[2]);
    const float EX = lgemm_row3(c.R + 0, ex, ey, ez, c.t[0]), EY = lgemm_row3(c.R + 3, ex, ey, ez, c.t[1]), EZ = lgemm_row3(c.R + 6, ex, ey, ez, c.t[2]);
    if (SZ < 0.0f || EZ < 0.0f) return o;
    const float invz1 = __fdiv_rn(1.0f, SZ);
    const float u1 = __fadd_rn(__fmul_rn(__fmul_rn(c.fx, SX), invz1), c.cx), v1 = __fadd_rn(__fmul_rn(__fmul_rn(c.fy, SY), invz1), c.cy);
    if (u1 < c.min_x || u1 > c.max_x) return o;
    if (v1 < c.min_y || v1 > c.max_y) return o;
    const float invz2 = __fdiv_rn(1.0f, EZ);
    const float u2 = __fadd_rn(__fmul_rn(__fmul_rn(c.fx, EX), invz2), c.cx), v2 = __fadd_rn(__fmul_rn(__fmul_rn(c.fy, EY), invz2), c.cy);
    if (u2 < c.min_x || u2 > c.max_x) return o;
    if (v2 < c.min_y || v2 > c.max_y) return o;
    const float mx = __fsub_rn(__fadd_rn(__fmul_rn(sx, 0.5f), __fmul_rn(ex, 0.5f)), c.O[0]);
    const float my = __fsub_rn(__fadd_rn(__fmul_rn(sy, 0.5f), __fmul_rn(ey, 0.5f)), c.O[1]);
    const float mz = __fsub_rn(__fadd_rn(__fmul_rn(sz, 0.5f), __fmul_rn(ez, 0.5f)), c.O[2]);
    const double n2 = __dadd_rn(__dadd_rn(__dmul_rn((double)mx, (double)mx), __dmul_rn((double)my, (double)my)), __dmul_rn((double)mz, (double)mz));
    const float dist = (float)sqrt(n2);
    if (dist < __fmul_rn(0.8f, m.min_dist) || dist > __fmul_rn(1.2f, m.max_dist)) return o;   // Get{Min,Max}DistanceInvariance
    const float nx = (float)m.normal[0], ny = (float)m.normal[1], nz = (float)m.normal[2];
    const double dot = __dadd_rn(__dadd_rn(__dmul_rn((double)mx, (double)nx), __dmul_rn((double)my, (double)ny)), __dmul_rn((double)mz, (double)nz));
    const float view_cos = (float)(dot / (double)dist);
    if (view_cos < cos_limit) return o;
    const float ratio = __fdiv_rn(m.max_dist, dist);
    int level = c.thr_lo;
    for (int k = 0; k < c.thr_n; ++k) level += ratio >= thr[k];
    o.x1 = u1; o.y1 = v1; o.x2 = u2; o.y2 = v2; o.level = level; o.view_cos = view_cos; o.in_view = 1;
    return o;
}
__global__ void __launch_bounds__(128) k_frustum_lines(LFrustumCam c, const MapLn* __restrict__ lines, const uint8_t* __restrict__ skip,
                                                       const uint8_t* __restrict__ claims, int n, float cos_limit, const float* __restrict__ thr,
                                                       float th, TrackLn* __restrict__ track, LQuery* __restrict__ qs, int* __restrict__ n_in_view) {
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= n) return;
    TrackLn o;
    o.x1 = o.y1 = o.x2 = o.y2 = 0.f; o.level = 0; o.view_cos = 0.f; o.in_view = 0;
    if (!(skip && skip[i])) o = frustum_line(c, lines[i], cos_limit, thr);
    if (track) track[i] = o;
    if (qs) {   // LSDmatcher::SearchByProjection(F, vpMapLines, eval_orient, th), LSDmatcher.cpp:727-736
        LQuery q;
        q.length = 0.f; q.pad[0] = q.pad[1] = 0;
        if (o.in_view) {
            float r = ((double)o.view_cos > 0.998) ? 5.0f : 8.0f;      // RadiusByViewingCos, LSDmatcher.cpp:1436-1442
            if (th != 1.0f) r = __fmul_rn(r, th);
            q.x1 = o.x1; q.y1 = o.y1; q.x2 = o.x2; q.y2 = o.y2; q.r = r; q.cos_th = 0.998f;
            q.dir[0] = lines[i].dir[0]; q.dir[1] = lines[i].dir[1]; q.dir[2] = lines[i].dir[2];
            q.claims = claims ? (claims[i] != 0) : 1;
        } else {   // not searched: a window nothing falls into
            q.x1 = q.y1 = q.x2 = q.y2 = -1e30f; q.r = -1.f; q.cos_th = 2.f; q.dir[0] = q.dir[1] = q.dir[2] = 0.0; q.claims = 0;
        }
        qs[i] = q;
    }
    if (n_in_view && o.in_view) atomicAdd(n_in_view, 1);
}

}  // namespace hvo

using namespace hvo;

struct hvo_lproj {
    int device = 0;
    cudaStream_t stream = nullptr;
    int n = 0, W = 1, kcap = 0, qcap = 0;
    bool has3d = false;
    LGridGeom g{0, 0, 0, 0};
    hvo_keyline* d_kl = nullptr;
    LKey* d_keys = nullptr;
    double *d_func = nullptr, *d_l3d = nullptr;
    uint8_t *d_desc = nullptr, *d_claimed = nullptr, *d_qdesc = nullptr;
    uint32_t* d_cells = nullptr;  // [64*48][kLMaxWords]
    int *d_claim0 = nullptr, *d_claim_a = nullptr, *d_claim_b = nullptr, *d_choice = nullptr, *d_cdist = nullptr, *d_flag = nullptr, *d_area = nullptr;
    LQuery* d_q = nullptr;
    int* h_flag = nullptr;
    int last_rounds = 0, last_launches = 0;
    // local-map projection (isInFrustum + search)
    float* d_thr = nullptr; float thr_log = 0.f;
    MapLn* d_lines = nullptr; TrackLn* d_track = nullptr; uint8_t *d_skip = nullptr, *d_claims = nullptr; int* d_count = nullptr;
    int pcap = 0;
};

#define HVO_TRYB(call) do { if ((call) != cudaSuccess) { set_error("%s: %s", #call, cudaGetErrorString(cudaGetLastError())); return HVO_ERR_CUDA; } } while (0)

template <class T>
static int lgrow(T*& p, size_t count) {
    if (p) cudaFree(p);
    p = nullptr;
    HVO_TRYB(cudaMalloc(&p, count * sizeof(T)));
    return HVO_OK;
}

extern "C" {

int hvo_lproj_create(int device, hvo_lproj** out) {
    HVO_CHECK_ARG(out, "null out");
    *out = nullptr;
    int ndev = 0;
    HVO_CUDA(cudaGetDeviceCount(&ndev));
    if (ndev < 1) { set_error("no CUDA device: libhvofront has no CPU fallback"); return HVO_ERR_CUDA; }
    HVO_CHECK_ARG(device >= 0 && device < ndev, "device index out of range");
    hvo_lproj* h = new (std::nothrow) hvo_lproj();
    if (!h) { set_error("out of host memory"); return HVO_ERR_ARG; }
    h->device = device;
    int st = HVO_OK;
    do {
#define HVO_TRY(call) if ((call) != cudaSuccess) { set_error("%s: %s", #call, cudaGetErrorString(cudaGetLastError())); st = HVO_ERR_CUDA; break; }
        HVO_TRY(cudaSetDevice(device));
        HVO_TRY(create_stream(&h->stream));
        const size_t cap = 32 * kLMaxWords;
        HVO_TRY(cudaMalloc(&h->d_cells, (size_t)kLGridCells * kLMaxWords * sizeof(uint32_t)));
        HVO_TRY(cudaMalloc(&h->d_kl, cap * sizeof(hvo_keyline)));
        HVO_TRY(cudaMalloc(&h->d_keys, cap * sizeof(LKey)));
        HVO_TRY(cudaMalloc(&h->d_func, cap * 3 * sizeof(double)));
        HVO_TRY(cudaMalloc(&h->d_l3d, cap * 6 * sizeof(double)));
        HVO_TRY(cudaMalloc(&h->d_desc, cap * 32));
        HVO_TRY(cudaMalloc(&h->d_claimed, cap));
        HVO_TRY(cudaMalloc(&h->d_claim0, cap * sizeof(int)));
        HVO_TRY(cudaMalloc(&h->d_claim_a, cap * sizeof(int)));
        HVO_TRY(cudaMalloc(&h->d_claim_b, cap * sizeof(int)));
        HVO_TRY(cudaMalloc(&h->d_area, cap * sizeof(int)));
        HVO_TRY(cudaMalloc(&h->d_flag, 2 * sizeof(int)));
        HVO_TRY(cudaMallocHost(&h->h_flag, 2 * sizeof(int)));
        h->kcap = (int)cap;
#undef HVO_TRY
    } while (0);
    if (st != HVO_OK) { hvo_lproj_destroy(h); return st; }
    *out = h;
    return HVO_OK;
}

void hvo_lproj_destroy(hvo_lproj* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    void* bufs[] = {h->d_kl, h->d_keys, h->d_func, h->d_l3d, h->d_desc, h->d_claimed, h->d_qdesc, h->d_cells, h->d_claim0, h->d_claim_a,
                    h->d_claim_b, h->d_choice, h->d_cdist, h->d_flag, h->d_area, h->d_q, h->d_thr, h->d_lines, h->d_track, h->d_skip, h->d_claims,
                    h->d_count};
    for (void* b : bufs) if (b) cudaFree(b);
    if (h->h_flag) cudaFreeHost(h->h_flag);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int hvo_lproj_set_frame(hvo_lproj* h, const hvo_keyline* keylines_un, const double* line_functions, const uint8_t* desc, const double* lines3d,
                        int n, float min_x, float min_y, float max_x, float max_y) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CHECK_ARG(n >= 0 && n <= h->kcap, "too many lines (max 1024)");
    HVO_CHECK_ARG(n == 0 || (keylines_un && line_functions && desc), "null keylines / line functions / descriptors");
    HVO_CHECK_ARG(max_x > min_x && max_y > min_y, "empty image bounds");
    HVO_CUDA(cudaSetDevice(h->device));
    h->n = n;
    h->W = std::max(1, div_up(n, 32));
    h->has3d = lines3d != nullptr;
    h->g = lgrid_geom(min_x, min_y, max_x, max_y);
    cudaStream_t s = h->stream;
    HVO_CUDA(cudaMemsetAsync(h->d_cells, 0, (size_t)kLGridCells * h->W * sizeof(uint32_t), s));
    if (n > 0) {
        HVO_CUDA(cudaMemcpyAsync(h->d_kl, keylines_un, (size_t)n * sizeof(hvo_keyline), cudaMemcpyHostToDevice, s));
        HVO_CUDA(cudaMemcpyAsync(h->d_func, line_functions, (size_t)n * 24, cudaMemcpyHostToDevice, s));
        HVO_CUDA(cudaMemcpyAsync(h->d_desc, desc, (size_t)n * 32, cudaMemcpyHostToDevice, s));
        if (lines3d) HVO_CUDA(cudaMemcpyAsync(h->d_l3d, lines3d, (size_t)n * 48, cudaMemcpyHostToDevice, s));
        k_lproj_grid<<<dim3(1, div_up(n, 128)), 128, 0, s>>>(h->d_kl, n, nullptr, 0, h->g, h->W, h->d_cells, h->d_keys);
        HVO_CUDA(cudaGetLastError());
    }
    HVO_CUDA(cudaStreamSynchronize(s));  // the host arrays may be released on return
    h->last_launches = n > 0 ? 1 : 0;
    return HVO_OK;
}

int hvo_lproj_get_grid(hvo_lproj* h, int32_t* cell_count, int32_t* cell_items, int capacity, int* n_items) {
    HVO_CHECK_ARG(h && cell_count && n_items, "null argument");
    HVO_CUDA(cudaSetDevice(h->device));
    std::vector<uint32_t> m((size_t)kLGridCells * h->W);
    HVO_CUDA(cudaMemcpyAsync(m.data(), h->d_cells, m.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    int total = 0;
    for (int c = 0; c < kLGridCells; ++c) {
        int cnt = 0;
        for (int w = 0; w < h->W; ++w) {
            uint32_t b = m[(size_t)c * h->W + w];
            while (b) {
                const int j = __builtin_ctz(b);
                b &= b - 1;
                if (cell_items && total < capacity) cell_items[total] = 32 * w + j;
                ++total; ++cnt;
            }
        }
        cell_count[c] = cnt;
    }
    *n_items = total;
    return HVO_OK;
}

int hvo_lproj_features_in_area(hvo_lproj* h, float x1, float y1, float x2, float y2, float r, float cos_th, int32_t* out, int capacity, int* n_out) {
    HVO_CHECK_ARG(h && out && n_out, "null argument");
    HVO_CHECK_ARG(capacity >= 1, "capacity < 1");
    HVO_CUDA(cudaSetDevice(h->device));
    *n_out = 0;
    if (h->n == 0) return HVO_OK;
    k_lproj_area<<<1, 32, 0, h->stream>>>(h->g, h->W, h->d_cells, h->d_keys, h->d_func, x1, y1, x2, y2, r, cos_th, h->d_area, h->kcap, h->d_flag);
    HVO_CUDA(cudaGetLastError());
    HVO_CUDA(cudaMemcpyAsync(h->h_flag, h->d_flag, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    const int cnt = h->h_flag[0], cp = std::min(cnt, capacity);
    if (cp > 0) HVO_CUDA(cudaMemcpyAsync(out, h->d_area, (size_t)cp * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    *n_out = cnt;
    return HVO_OK;
}

static int lproj_reserve_queries(hvo_lproj* h, int nq) {
    if (nq <= h->qcap) return HVO_OK;
    const int cap = std::max(nq, 1024);
    int st;
    if ((st = lgrow(h->d_q, cap)) || (st = lgrow(h->d_qdesc, (size_t)cap * 32)) || (st = lgrow(h->d_choice, cap)) || (st = lgrow(h->d_cdist, cap))) return st;
    h->qcap = cap;
    return HVO_OK;
}
// the fixed-point rounds over nq device-resident queries (h->d_q, h->d_qdesc)
static int lproj_run_rounds(hvo_lproj* h, int nq, const uint8_t* claimed, int mode, float nnratio, int32_t* match_idx, int32_t* match_dist,
                            int* n_matches, int launches) {
    cudaStream_t s = h->stream;
    if (claimed) HVO_CUDA(cudaMemcpyAsync(h->d_claimed, claimed, (size_t)h->n, cudaMemcpyHostToDevice, s));
    k_lproj_claim_init<<<div_up(h->n, 256), 256, 0, s>>>(claimed ? h->d_claimed : nullptr, h->n, h->d_claim0);
    HVO_CUDA(cudaMemcpyAsync(h->d_claim_a, h->d_claim0, (size_t)h->n * sizeof(int), cudaMemcpyDeviceToDevice, s));
    k_lproj_fill<<<div_up(nq, 256), 256, 0, s>>>(h->d_choice, nq, -2);
    const double th_normal = std::cos(15.0 / 180.0 * M_PI), cos_th_angle = std::cos(10.0 / 180.0 * M_PI);  // LSDmatcher.cpp:713-715, 563-565
    launches += 2;
    int rounds = 0;
    int *prev = h->d_claim_a, *next = h->d_claim_b;
    while (true) {
        HVO_CUDA(cudaMemcpyAsync(next, h->d_claim0, (size_t)h->n * sizeof(int), cudaMemcpyDeviceToDevice, s));
        HVO_CUDA(cudaMemsetAsync(h->d_flag, 0, sizeof(int), s));
        k_lproj_round<<<div_up(nq * 32, 128), 128, 0, s>>>(h->g, h->W, h->d_cells, h->d_keys, h->d_func, reinterpret_cast<const uint4*>(h->d_desc),
                                                           h->d_l3d, h->d_q, reinterpret_cast<const uint4*>(h->d_qdesc), nq, prev, next, mode, nnratio,
                                                           th_normal, cos_th_angle, h->d_choice, h->d_cdist, h->d_flag);
        HVO_CUDA(cudaGetLastError());
        HVO_CUDA(cudaMemcpyAsync(h->h_flag, h->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
        HVO_CUDA(cudaStreamSynchronize(s));
        ++launches; ++rounds;
        if (!h->h_flag[0]) break;  // no choice changed: fixed point == the reference's sequential assignment
        if (rounds > nq + 1) { set_error("line projection search did not reach its fixed point"); return HVO_ERR_CUDA; }
        std::swap(prev, next);
    }
    h->last_rounds = rounds; h->last_launches = launches;
    HVO_CUDA(cudaMemcpyAsync(match_idx, h->d_choice, (size_t)nq * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (match_dist) HVO_CUDA(cudaMemcpyAsync(match_dist, h->d_cdist, (size_t)nq * sizeof(int), cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaStreamSynchronize(s));
    if (n_matches) { int c = 0; for (int i = 0; i < nq; ++i) c += match_idx[i] >= 0; *n_matches = c; }
    return HVO_OK;
}

int hvo_lproj_search(hvo_lproj* h, const hvo_lproj_query* queries, const uint8_t* qdesc, int nq, const uint8_t* claimed, int mode, float nnratio,
                     int32_t* match_idx, int32_t* match_dist, int* n_matches) {
    HVO_CHECK_ARG(h && match_idx, "null argument");
    HVO_CHECK_ARG(mode == 0 || mode == 1, "mode must be 0 (map lines) or 1 (last frame)");
    if (n_matches) *n_matches = 0;
    if (nq <= 0) return HVO_OK;
    HVO_CHECK_ARG(queries && qdesc, "null queries");
    if (h->n == 0) {
        for (int i = 0; i < nq; ++i) { match_idx[i] = -1; if (match_dist) match_dist[i] = 256; }
        return HVO_OK;
    }
    HVO_CHECK_ARG(mode == 1 || h->has3d, "mode 0 needs the frame's 3-D lines (lines3d of hvo_lproj_set_frame)");
    HVO_CUDA(cudaSetDevice(h->device));
    int st = lproj_reserve_queries(h, nq);
    if (st != HVO_OK) return st;
    cudaStream_t s = h->stream;
    HVO_CUDA(cudaMemcpyAsync(h->d_q, queries, (size_t)nq * sizeof(LQuery), cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(h->d_qdesc, qdesc, (size_t)nq * 32, cudaMemcpyHostToDevice, s));
    return lproj_run_rounds(h, nq, claimed, mode, nnratio, match_idx, match_dist, n_matches, 0);
}

// ---- isInFrustum over a batch of map lines, alone or in front of the search ----
static const int kLThrLo = -32, kLThrN = 96;   // MapLine::PredictScale levels representable: [-32, 64]
static int lproj_prepare_frustum(hvo_lproj* h, const hvo_frustum_cam* cam, int n) {
    if (!h->d_thr) { int st; if ((st = lgrow(h->d_thr, kLThrN)) || (st = lgrow(h->d_count, 1))) return st; }
    if (h->thr_log != cam->log_scale_factor) {
        float thr[kLThrN];
        int st = hvo_predict_scale_thresholds(cam->log_scale_factor, kLThrLo, kLThrN, thr);
        if (st != HVO_OK) return st;
        HVO_CUDA(cudaMemcpyAsync(h->d_thr, thr, sizeof(thr), cudaMemcpyHostToDevice, h->stream));
        HVO_CUDA(cudaStreamSynchronize(h->stream));
        h->thr_log = cam->log_scale_factor;
    }
    if (n > h->pcap) {
        const int cap = std::max(n, 2048);
        int st;
        if ((st = lgrow(h->d_lines, cap)) || (st = lgrow(h->d_track, cap)) || (st = lgrow(h->d_skip, cap)) || (st = lgrow(h->d_claims, cap))) return st;
        h->pcap = cap;
    }
    return HVO_OK;
}
static LFrustumCam make_lcam(const hvo_frustum_cam* cam) {
    LFrustumCam c;
    for (int i = 0; i < 9; ++i) c.R[i] = cam->Rcw[i];
    for (int i = 0; i < 3; ++i) { c.t[i] = cam->tcw[i]; c.O[i] = cam->Ow[i]; }
    c.fx = cam->fx; c.fy = cam->fy; c.cx = cam->cx; c.cy = cam->cy;
    c.min_x = cam->min_x; c.min_y = cam->min_y; c.max_x = cam->max_x; c.max_y = cam->max_y; c.thr_lo = kLThrLo; c.thr_n = kLThrN;
    return c;
}

int hvo_lproj_frustum_lines(hvo_lproj* h, const hvo_frustum_cam* cam, const hvo_map_line* lines, int n, float viewing_cos_limit, hvo_track_line* out) {
    HVO_CHECK_ARG(h && cam && out, "null argument");
    if (n <= 0) return HVO_OK;
    HVO_CHECK_ARG(lines, "null map lines");
    HVO_CUDA(cudaSetDevice(h->device));
    int st = lproj_prepare_frustum(h, cam, n);
    if (st != HVO_OK) return st;
    cudaStream_t s = h->stream;
    HVO_CUDA(cudaMemcpyAsync(h->d_lines, lines, (size_t)n * sizeof(MapLn), cudaMemcpyHostToDevice, s));
    k_frustum_lines<<<div_up(n, 128), 128, 0, s>>>(make_lcam(cam), h->d_lines, nullptr, nullptr, n, viewing_cos_limit, h->d_thr, 1.f, h->d_track, nullptr,
                                                   nullptr);
    HVO_CUDA(cudaGetLastError());
    HVO_CUDA(cudaMemcpyAsync(out, h->d_track, (size_t)n * sizeof(TrackLn), cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaStreamSynchronize(s));
    h->last_launches = 1;
    return HVO_OK;
}

int hvo_lproj_search_local_map(hvo_lproj* h, const hvo_frustum_cam* cam, const hvo_map_line* lines, const uint8_t* ldesc, const uint8_t* skip,
                               const uint8_t* claims, int n, float viewing_cos_limit, float th, const uint8_t* claimed, float nnratio,
                               hvo_track_line* track, int32_t* match_idx, int32_t* match_dist, int* n_in_view, int* n_matches) {
    HVO_CHECK_ARG(h && cam && match_idx, "null argument");
    if (n_matches) *n_matches = 0;
    if (n_in_view) *n_in_view = 0;
    if (n <= 0) return HVO_OK;
    HVO_CHECK_ARG(lines && ldesc, "null map lines / descriptors");
    HVO_CHECK_ARG(h->n == 0 || h->has3d, "the search needs the frame's 3-D lines (lines3d of hvo_lproj_set_frame)");
    HVO_CUDA(cudaSetDevice(h->device));
    int st = lproj_prepare_frustum(h, cam, n);
    if (st != HVO_OK || (st = lproj_reserve_queries(h, n)) != HVO_OK) return st;
    cudaStream_t s = h->stream;
    HVO_CUDA(cudaMemcpyAsync(h->d_lines, lines, (size_t)n * sizeof(MapLn), cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemcpyAsync(h->d_qdesc, ldesc, (size_t)n * 32, cudaMemcpyHostToDevice, s));
    if (skip) HVO_CUDA(cudaMemcpyAsync(h->d_skip, skip, (size_t)n, cudaMemcpyHostToDevice, s));
    if (claims) HVO_CUDA(cudaMemcpyAsync(h->d_claims, claims, (size_t)n, cudaMemcpyHostToDevice, s));
    HVO_CUDA(cudaMemsetAsync(h->d_count, 0, sizeof(int), s));
    k_frustum_lines<<<div_up(n, 128), 128, 0, s>>>(make_lcam(cam), h->d_lines, skip ? h->d_skip : nullptr, claims ? h->d_claims : nullptr, n,
                                                   viewing_cos_limit, h->d_thr, th, h->d_track, h->d_q, h->d_count);
    HVO_CUDA(cudaGetLastError());
    if (track) HVO_CUDA(cudaMemcpyAsync(track, h->d_track, (size_t)n * sizeof(TrackLn), cudaMemcpyDeviceToHost, s));
    int count = 0;
    HVO_CUDA(cudaMemcpyAsync(&count, h->d_count, sizeof(int), cudaMemcpyDeviceToHost, s));
    HVO_CUDA(cudaStreamSynchronize(s));
    if (n_in_view) *n_in_view = count;
    if (h->n == 0) {
        for (int i = 0; i < n; ++i) { match_idx[i] = -1; if (match_dist) match_dist[i] = 256; }
        return HVO_OK;
    }
    return lproj_run_rounds(h, n, claimed, 0, nnratio, match_idx, match_dist, n_matches, 1);
}

int hvo_lproj_last_rounds(const hvo_lproj* h) { return h ? h->last_rounds : 0; }
int hvo_lproj_last_launches(const hvo_lproj* h) { return h ? h->last_launches : 0; }

}  // extern "C"
