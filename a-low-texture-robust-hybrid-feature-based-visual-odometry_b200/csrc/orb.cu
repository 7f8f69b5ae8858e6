// ORB extractor kernels for sm_100a (B200).  From-scratch design, batched over frames:
//
//   k_resize_tile x(nlevels-1)  fixed-point bilinear pyramid, bit-exact with cv::resize INTER_LINEAR 8U
//                               (reference ORBextractor.cc:1105-1130); k_resize = the general fallback
//                               (pyramid factors > ~1.3, unaligned level 0)
//   k_fast_strips x1            one CTA per row of reference FAST cells: FAST-9/16 strength, cell-local NMS,
//                               per-cell threshold fallback (ORBextractor.cc:763-826) - no score map in HBM
//   k_octree      x1            one CTA per (frame, level): DistributeOctTree (ORBextractor.cc:537-761)
//                               with parallel key partitioning and the std::list order emulated exactly
//   k_describe    x1            one warp per keypoint: IC_Angle (.cc:75-102), 7x7 Q8 Gaussian of the 37x37
//                               patch in shared memory (.cc:1083-1084), steered rBRIEF-256 (.cc:106-144),
//                               KeyPoint assembly (.cc:835-846,1093-1099), RGB-D depth lookup
//                               (Frame.cc:1940-1961) - no blurred pyramid in HBM
//   k_undistort_kps x1          distorted cameras only: one thread per keypoint, Frame::UndistortKeyPoints
//                               (Frame.cc:1701-1731, cv::undistortPoints in FP64, undistort.cuh) and mvuRight from the
//                               undistorted x.  A kernel of its own: five dependent FP64 iterations on lane 0 of
//                               k_describe would lengthen every describe warp
//
// Float semantics are pinned with explicit round-to-nearest intrinsics (no FMA contraction) so that
// angles, sample coordinates and scaled keypoint positions are bit-identical to the CPU oracle.
#include "orb.cuh"
#include "undistort.cuh"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>

namespace hvo {

// ------------------------------------------------------------------------------------------------------
// constants
// ------------------------------------------------------------------------------------------------------
__device__ __align__(16) const int8_t g_pattern[1024] = {   // read once per CTA, coalesced (lane-varying constant reads serialise)
#include "../../include/hvo_orb_pattern.inc"
};
__constant__ int c_umax[16] = {15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3};
static const int h_umax[16] = {15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3};

static const int kEdge = 19;
static const int kFastMaxZh = 64;    // hCell = ceil(height / floor(height/30)) <= 60
static const int kFastMaxZone = 672; // widest run of cells one strip CTA takes (px)

__device__ __forceinline__ const uint8_t* level_ptr(const OrbGeom& g, const ImgSrc& s, int l, int f, int& pitch) {
    if (l == 0) {
        pitch = s.l0_pitch;
        return s.l0 + (long long)f * s.l0_frame;
    }
    pitch = g.lv[l].pitch;
    return s.pyr + (long long)f * g.pyr_frame_bytes + g.lv[l].img_off;
}

// ------------------------------------------------------------------------------------------------------
// K1: bilinear resize.  One CTA = 128 x 32 destination pixels.  Pass H interpolates every source row the
// tile needs once (thread <-> destination column, coefficients in registers) into shared memory as
// (S0*w0 + S1*w1) >> 4 (15 bits); pass V blends two such rows per destination row and stores 4 px / thread.
// ------------------------------------------------------------------------------------------------------
static const int kRsW = 128, kRsH = 32, kRsMaxSrcRows = 72;

__global__ void __launch_bounds__(256) k_resize(const uint8_t* __restrict__ src, int spitch, long long sframe, int sw,
                                                uint8_t* __restrict__ dst, int dpitch, long long dframe, int dw, int dh,
                                                const int2* __restrict__ xtab, const int4* __restrict__ ytab) {
    __shared__ __align__(8) uint16_t hrow[kRsMaxSrcRows * kRsW];
    const int tid = threadIdx.x, f = blockIdx.z;
    const int tx = blockIdx.x * kRsW, ty = blockIdx.y * kRsH;
    const int ylast = min(ty + kRsH, dh) - 1;
    const int s_base = __ldg(&ytab[ty]).x;
    const int ns = min(__ldg(&ytab[ylast]).y - s_base + 1, kRsMaxSrcRows);
    const uint8_t* S = src + (long long)f * sframe;
    {   // pass H
        const int col = tid & (kRsW - 1), half = tid >> 7;
        const int x = tx + col;
        if (x < dw) {
            const int2 xt = __ldg(&xtab[x]);
            const int sx = xt.x, s1 = min(sx + 1, sw - 1);
            const int w0 = (int)(short)(xt.y & 0xffff), w1 = xt.y >> 16;
            for (int r = half; r < ns; r += 2) {
                const uint8_t* row = S + (long long)(s_base + r) * spitch;
                hrow[r * kRsW + col] = (uint16_t)((__ldg(row + sx) * w0 + __ldg(row + s1) * w1) >> 4);
            }
        }
    }
    __syncthreads();
    {   // pass V
        const int cg = tid & 31, rs = tid >> 5;
        const int x0 = tx + 4 * cg;
        if (x0 < dw) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int y = ty + rs * 4 + j;
                if (y < dh) {
                    const int4 yt = __ldg(&ytab[y]);
                    const uint2 a = *reinterpret_cast<const uint2*>(&hrow[(yt.x - s_base) * kRsW + 4 * cg]);
                    const uint2 b = *reinterpret_cast<const uint2*>(&hrow[(yt.y - s_base) * kRsW + 4 * cg]);
                    const int h0[4] = {(int)(a.x & 0xffff), (int)(a.x >> 16), (int)(a.y & 0xffff), (int)(a.y >> 16)};
                    const int h1[4] = {(int)(b.x & 0xffff), (int)(b.x >> 16), (int)(b.y & 0xffff), (int)(b.y >> 16)};
                    uint32_t packed = 0;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        int v = (((yt.z * h0[i]) >> 16) + ((yt.w * h1[i]) >> 16) + 2) >> 2;
                        v = min(255, max(0, v));
                        packed |= (uint32_t)v << (8 * i);
                    }
                    uint8_t* D = dst + (long long)f * dframe + (long long)y * dpitch + x0;
                    if (x0 + 3 < dw) *reinterpret_cast<uint32_t*>(D) = packed;  // dpitch and x0 are multiples of 4
                    else for (int i = 0; x0 + i < dw; ++i) D[i] = (uint8_t)(packed >> (8 * i));
                }
            }
        }
    }
}

// K1 for the usual pyramid factors (<= ~1.3: the source rows of a tile fit kRtSrcRows x kRtSrcWords words): the source band of the
// tile goes to shared memory first as aligned words (coalesced, every byte read once), pass H reads its two taps per output from
// there (byte offsets in registers, no global latency inside the pass), pass V blends with the row coefficients staged per tile and
// the >> 16 of both products folded into multiply-high.  Same arithmetic as k_resize, bit for bit.
static const int kRtSrcRows = 44, kRtSrcWords = 44;

__global__ void __launch_bounds__(256) k_resize_tile(const uint8_t* __restrict__ src, int spitch, long long sframe, int sw,
                                                     uint8_t* __restrict__ dst, int dpitch, long long dframe, int dw, int dh,
                                                     const int2* __restrict__ xtab, const int4* __restrict__ ytab) {
    __shared__ uint32_t sraw[kRtSrcRows * kRtSrcWords];
    __shared__ __align__(8) uint16_t hrow[kRtSrcRows * kRsW];
    __shared__ int4 syt[kRsH];
    const int tid = threadIdx.x, f = blockIdx.z;
    const int tx = blockIdx.x * kRsW, ty = blockIdx.y * kRsH;
    const int xlast = min(tx + kRsW, dw) - 1, ylast = min(ty + kRsH, dh) - 1;
    const int s_base = __ldg(&ytab[ty]).x;
    const int ns = min(__ldg(&ytab[ylast]).y - s_base + 1, kRtSrcRows);
    const int xs = __ldg(&xtab[tx]).x & ~3;
    const int nwords = min(((min(__ldg(&xtab[xlast]).x + 1, sw - 1) - xs) >> 2) + 1, kRtSrcWords);
    const uint8_t* S = src + (long long)f * sframe + (long long)s_base * spitch + xs;
    if (tid < kRsH) syt[tid] = __ldg(&ytab[min(ty + tid, dh - 1)]);
    {   // source band: 64 threads across the words of a row, 4 rows per sweep
        const int k = tid & 63, r0 = tid >> 6;
        if (k < nwords)
            for (int r = r0; r < ns; r += 4) sraw[r * kRtSrcWords + k] = __ldg(reinterpret_cast<const uint32_t*>(S + (long long)r * spitch) + k);
    }
    __syncthreads();
    {   // pass H
        const int col = tid & (kRsW - 1), half = tid >> 7;
        const int x = tx + col;
        if (x < dw) {
            const int2 xt = __ldg(&xtab[x]);
            const int o0 = xt.x - xs, o1 = min(xt.x + 1, sw - 1) - xs;
            const int w0 = (int)(short)(xt.y & 0xffff), w1 = xt.y >> 16;
            const uint8_t* b = reinterpret_cast<const uint8_t*>(sraw) + half * (kRtSrcWords * 4);
            uint16_t* hr = hrow + half * kRsW + col;
#pragma unroll 4
            for (int r = half; r < ns; r += 2) {
                *hr = (uint16_t)((b[o0] * w0 + b[o1] * w1) >> 4);
                b += 2 * kRtSrcWords * 4;
                hr += 2 * kRsW;
            }
        }
    }
    __syncthreads();
    {   // pass V: 4 columns x 4 rows per thread; ((b0 * h0) >> 16) + ((b1 * h1) >> 16) as multiply-high by the coefficients << 16
        const int cg = tid & 31, rs = tid >> 5;
        const int x0 = tx + 4 * cg;
        if (x0 < dw) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int y = ty + rs * 4 + j;
                if (y < dh) {
                    const int4 yt = syt[rs * 4 + j];
                    const uint2 a = *reinterpret_cast<const uint2*>(&hrow[(yt.x - s_base) * kRsW + 4 * cg]);
                    const uint2 b = *reinterpret_cast<const uint2*>(&hrow[(yt.y - s_base) * kRsW + 4 * cg]);
                    const uint32_t b0 = (uint32_t)yt.z << 16, b1 = (uint32_t)yt.w << 16;
                    const uint32_t v0 = (__umulhi(b0, a.x & 0xffffu) + __umulhi(b1, b.x & 0xffffu) + 2u) >> 2;
                    const uint32_t v1 = (__umulhi(b0, a.x >> 16) + __umulhi(b1, b.x >> 16) + 2u) >> 2;
                    const uint32_t v2 = (__umulhi(b0, a.y & 0xffffu) + __umulhi(b1, b.y & 0xffffu) + 2u) >> 2;
                    const uint32_t v3 = (__umulhi(b0, a.y >> 16) + __umulhi(b1, b.y >> 16) + 2u) >> 2;
                    // b0 + b1 = 2048 and h <= 32640: the sum is at most 255, no saturation needed
                    const uint32_t packed = __byte_perm(__byte_perm(v0, v1, 0x0040), __byte_perm(v2, v3, 0x0040), 0x5410);
                    uint8_t* D = dst + (long long)f * dframe + (long long)y * dpitch + x0;
                    if (x0 + 3 < dw) *reinterpret_cast<uint32_t*>(D) = packed;  // dpitch and x0 are multiples of 4
                    else for (int i = 0; x0 + i < dw; ++i) D[i] = (uint8_t)(packed >> (8 * i));
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// K2: FAST per cell
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool has_run9(uint32_t m16) {
    uint32_t m = m16 | (m16 << 16);
    uint32_t a = m & (m >> 1);
    a &= a >> 2;
    a &= a >> 4;
    a &= m >> 8;
    return (a & 0xffffu) != 0;
}

// Threshold-independent FAST-9/16 strength S = max(A, B) - 1 (see oracle/cvprims.hpp fast_strength):
//   A = max over the 16 arcs of min(v - ring), B = max over arcs of min(ring - v).
__device__ __forceinline__ int fast_strength(const int (&d)[16]) {
    // min / max over every 9-arc as two levels of 3-input min/max (VIMNMX3 on sm_100a)
    int lo3[16], hi3[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        lo3[i] = min(min(d[i], d[(i + 1) & 15]), d[(i + 2) & 15]);
        hi3[i] = max(max(d[i], d[(i + 1) & 15]), d[(i + 2) & 15]);
    }
    int A = -256, B = 256;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        A = max(A, min(min(lo3[i], lo3[(i + 3) & 15]), lo3[(i + 6) & 15]));
        B = min(B, max(max(hi3[i], hi3[(i + 3) & 15]), hi3[(i + 6) & 15]));
    }
    return max(A, -B) - 1;
}

#define HVO_RING(p, st, k)                                                                                   \
    ((k) == 0 ? (p)[3 * (st)] : (k) == 1 ? (p)[3 * (st) + 1] : (k) == 2 ? (p)[2 * (st) + 2] : (k) == 3 ? (p)[(st) + 3] \
     : (k) == 4 ? (p)[3] : (k) == 5 ? (p)[-(st) + 3] : (k) == 6 ? (p)[-2 * (st) + 2] : (k) == 7 ? (p)[-3 * (st) + 1]   \
     : (k) == 8 ? (p)[-3 * (st)] : (k) == 9 ? (p)[-3 * (st) - 1] : (k) == 10 ? (p)[-2 * (st) - 2]                      \
     : (k) == 11 ? (p)[-(st) - 3] : (k) == 12 ? (p)[-3] : (k) == 13 ? (p)[(st) - 3] : (k) == 14 ? (p)[2 * (st) - 2]    \
                                                                                                : (p)[3 * (st) - 1])

// One CTA per STRIP = one row of reference FAST cells of one level of one frame (the zones of a cell row tile the level
// without gaps: cell ROI = zone + 3-px ring, ORBextractor.cc:787-803).  The FAST strength of a pixel depends on the image
// only; what is cell-local is (a) non-max suppression (neighbours outside the cell's zone count as 0) and (b) the
// threshold fallback (ORBextractor.cc:807-814).  So the strip is processed as one image band:
//   fill     the band (zone rows + 3-px ring) goes to shared memory as one bulk copy per row (cp.async.bulk + mbarrier:
//            the copy engine moves the bytes, no LDG/STS issue slots), while the threads clear the score map
//   pass 1   quick reject, 4 pixels per thread on packed bytes; survivors go to a warp-private queue
//   pass 2   exact threshold-independent strength for queued survivors, 32 at a time (dense warps), no CTA barrier
//   pass 3   NMS over the score map (word-wise skip of empty groups), cell-aware; maxima -> list (reuses the band's memory)
//   emit     per-cell ini/min decision, one global atomic per strip
static const int kFastThreads = 256, kFastWarps = kFastThreads / 32;
static const int kFastQueue = 256;   // per-warp survivor queue (entries; >= 31 + 128)
static const int kFastMaxCellsPerStrip = 64;

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Packed 4-pixel FAST ring compare: the 4 ring bytes seen by the 4 pixels of word g at horizontal offset dx (-3..3).
__device__ __forceinline__ uint32_t ring4(const uint32_t* row, int g, int dx) {
    switch (dx) {
        case 0: return row[g];
        case 1: return __byte_perm(row[g], row[g + 1], 0x4321);
        case 2: return __byte_perm(row[g], row[g + 1], 0x5432);
        case 3: return __byte_perm(row[g], row[g + 1], 0x6543);
        case -1: return __byte_perm(row[g - 1], row[g], 0x6543);
        case -2: return __byte_perm(row[g - 1], row[g], 0x5432);
        default: return __byte_perm(row[g - 1], row[g], 0x4321);
    }
}

__global__ void __launch_bounds__(kFastThreads) k_fast_strips(const __grid_constant__ OrbGeom g, ImgSrc src,
                                                              const StripDesc* __restrict__ strips, uint32_t* __restrict__ cand,
                                                              int* __restrict__ ncand, int ini_th, int min_th) {
    extern __shared__ __align__(16) unsigned char fs_smem[];
    __shared__ __align__(8) unsigned long long s_bar;
    __shared__ uint32_t s_queue[kFastWarps][kFastQueue];
    __shared__ int s_nini[kFastMaxCellsPerStrip], s_nmin[kFastMaxCellsPerStrip];
    __shared__ int s_nlist, s_base, s_slot, s_total;

    const StripDesc c = strips[blockIdx.x];
    const int f = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const LevelGeom& L = g.lv[c.level];
    int pitch;
    const uint8_t* img = level_ptr(g, src, c.level, f, pitch);
    const int zh = c.zh, zw = c.zw, th = zh + 6;
    const int low_th = min(ini_th, min_th);

    // band geometry: tile column 0 = image column xal (16-byte aligned), zone starts at tile byte zb0
    const int xal = (c.x0 - 3) & ~15;
    const int zb0 = c.x0 - xal;                       // >= 3
    const int ts = c.tstride;                         // bytes per band row, multiple of 16
    const int tsw = ts >> 2;
    unsigned char* tile_b = fs_smem + 16;             // word -1 of row 0 must be addressable (content unused)
    uint32_t* tile = reinterpret_cast<uint32_t*>(tile_b);
    unsigned char* score = tile_b + c.score_off;      // (zh + 2) rows of ts bytes; row 0 and row zh+1 stay 0
    uint32_t* list = tile;                            // NMS maxima, written after the band is dead

    // ---- fill ----
    const bool bulk = ((pitch & 15) == 0) && ((reinterpret_cast<uintptr_t>(img) & 15) == 0);
    if (tid == 0) {
        s_nlist = 0; s_slot = 0;
        if (bulk) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(&s_bar)));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
    }
    if (tid < kFastMaxCellsPerStrip) { s_nini[tid] = 0; s_nmin[tid] = 0; }
    __syncthreads();
    if (bulk) {
        if (warp == 0) {
            if (lane == 0)
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(&s_bar)), "r"(th * ts) : "memory");
            __syncwarp();
            for (int r = lane; r < th; r += 32) {
                const uint8_t* gp = img + (long long)(c.y0 - 3 + r) * pitch + xal;
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                 smem_addr(tile_b + r * ts)),
                             "l"(gp), "r"(ts), "r"(smem_addr(&s_bar))
                             : "memory");
            }
        }
    } else {
        const int lim = L.w - 1 - xal;
        for (int i = tid; i < th * tsw; i += kFastThreads) {
            const int r = i / tsw, wi = i - r * tsw;
            const uint8_t* p = img + (long long)(c.y0 - 3 + r) * pitch + xal;
            uint32_t w = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) w |= (uint32_t)__ldg(p + min(4 * wi + j, lim)) << (8 * j);
            tile[r * tsw + wi] = w;
        }
    }
    {   // clear the score map while the copy engine works
        uint4* sc4 = reinterpret_cast<uint4*>(score);
        const int n16 = ((zh + 2) * ts) >> 4;
        for (int i = tid; i < n16; i += kFastThreads) sc4[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    if (bulk) {
        uint32_t done = 0;
        while (!done)
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }"
                         : "=r"(done) : "r"(smem_addr(&s_bar)) : "memory");
    }
    __syncthreads();

    // ---- pass 1 + 2 ----
    // A 9-arc always contains ring point 0 or 8 and ring point 4 or 12, so a corner needs |v - ring| > t on one point of each
    // pair.  VABSDIFF4 is native; "byte > t" is the carry trick ((x & 0x7f) + (127 - t)) | x.
    // Survivors (byte flags in bit 7 of `flags`) are compacted into a warp-private queue with four ballots (no shuffles, no loop
    // over the flags) and processed 32 at a time, so the expensive part runs on full warps without a CTA barrier in between.
    const int g0 = zb0 >> 2, g1 = (zb0 + zw - 1) >> 2;
    const bool use_quick = low_th <= 127;
    const uint32_t K = (uint32_t)(127 - min(low_th, 127)) * 0x01010101u;
    uint32_t* q = s_queue[warp];
    int qh = 0, qn = 0;                                  // warp-uniform queue head / tail (monotonic)
    const unsigned lt = (1u << lane) - 1u;
    auto enqueue = [&](uint32_t flags, uint32_t base_pos) -> bool {   // base_pos = zy << 16 | band column of byte 0
        const unsigned m0 = __ballot_sync(0xffffffffu, flags & 0x80u), m1 = __ballot_sync(0xffffffffu, flags & 0x8000u);
        const unsigned m2 = __ballot_sync(0xffffffffu, flags & 0x800000u), m3 = __ballot_sync(0xffffffffu, flags & 0x80000000u);
        const int c0 = __popc(m0), c1 = __popc(m1), c2 = __popc(m2), total = c0 + c1 + c2 + __popc(m3);
        if (total == 0) return false;
        if (flags & 0x80u) q[(qn + __popc(m0 & lt)) & (kFastQueue - 1)] = base_pos;
        if (flags & 0x8000u) q[(qn + c0 + __popc(m1 & lt)) & (kFastQueue - 1)] = base_pos + 1;
        if (flags & 0x800000u) q[(qn + c0 + c1 + __popc(m2 & lt)) & (kFastQueue - 1)] = base_pos + 2;
        if (flags & 0x80000000u) q[(qn + c0 + c1 + c2 + __popc(m3 & lt)) & (kFastQueue - 1)] = base_pos + 3;
        qn += total;
        __syncwarp();
        return true;
    };
    auto strength_at = [&](uint32_t pos) {
        const int py = pos >> 16, px = pos & 0xffff;
        const uint8_t* p = tile_b + (py + 3) * ts + px;
        const int v = *p;
        int d[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) d[k] = v - (int)HVO_RING(p, ts, k);
        const int sc = fast_strength(d);
        if (sc >= low_th) score[(py + 1) * ts + px] = (uint8_t)sc;   // in [low_th, 254]; non-corners stay 0
    };
    for (int zy = warp; zy < zh; zy += kFastWarps) {
        const uint32_t* r0 = tile + (zy + 3) * tsw;
        for (int gb = g0; gb <= g1; gb += 32) {
            const int gi = gb + lane;
            uint32_t maybe = 0;
            if (gi <= g1) {
                const uint32_t v4 = r0[gi];
                const int b0 = 4 * gi;
                maybe = 0x80808080u;
                if (b0 < zb0) maybe &= 0xffffffffu << (8 * (zb0 - b0));
                if (b0 + 3 > zb0 + zw - 1) maybe &= 0xffffffffu >> (8 * (b0 + 3 - (zb0 + zw - 1)));
                if (use_quick) {
                    const uint32_t a0 = __vabsdiffu4(v4, (r0 + 3 * tsw)[gi]), a8 = __vabsdiffu4(v4, (r0 - 3 * tsw)[gi]);
                    const uint32_t a4 = __vabsdiffu4(v4, ring4(r0, gi, 3)), a12 = __vabsdiffu4(v4, ring4(r0, gi, -3));
                    const uint32_t m08 = ((a0 & 0x7f7f7f7fu) + K) | ((a8 & 0x7f7f7f7fu) + K) | a0 | a8;
                    const uint32_t m412 = ((a4 & 0x7f7f7f7fu) + K) | ((a12 & 0x7f7f7f7fu) + K) | a4 | a12;
                    maybe &= m08 & m412;
                }
            }
            if (!enqueue(maybe, ((uint32_t)zy << 16) | (uint32_t)(4 * gi))) continue;
            while (qn - qh >= 32) {
                strength_at(q[(qh + lane) & (kFastQueue - 1)]);
                qh += 32;
            }
            __syncwarp();
        }
    }
    if (lane < qn - qh) strength_at(q[(qh + lane) & (kFastQueue - 1)]);
    __syncthreads();

    // ---- pass 3: cell-local non-max suppression (strict '>' on the 8 neighbours, outside the cell's zone counts as 0).  Same
    //      skeleton: pixels with a score are compacted per warp and tested 32 at a time, branch-free (the guard rows / columns of
    //      the score map are zero, so all 8 neighbours can always be read) ----
    const int wcell = c.wcell;
    const uint32_t cmagic = (1u << 20) / (uint32_t)wcell + 1;   // zx / wcell for zx < 2^12
    const uint32_t* score_w = reinterpret_cast<const uint32_t*>(score);
    qh = qn = 0;
    auto nms_at = [&](uint32_t pos) {
        const int zy = pos >> 16, px = pos & 0xffff, zx = px - zb0;
        int cj = (int)(((uint32_t)zx * cmagic) >> 20);
        if (cj * wcell > zx) --cj;
        const int cx = zx - cj * wcell;
        const uint8_t* sp = score + (zy + 1) * ts + px;
        const int s = sp[0];
        const int up = sp[-ts], dn = sp[ts];
        const int l = max(max((int)sp[-ts - 1], (int)sp[-1]), (int)sp[ts - 1]);
        const int r = max(max((int)sp[-ts + 1], (int)sp[1]), (int)sp[ts + 1]);
        int m = max(up, dn);
        m = max(m, cx > 0 ? l : 0);
        m = max(m, (cx < wcell - 1 && zx < zw - 1) ? r : 0);
        if (s > m) {
            if (s >= ini_th) atomicAdd(&s_nini[cj], 1);
            if (s >= min_th) atomicAdd(&s_nmin[cj], 1);
            list[atomicAdd(&s_nlist, 1)] = (uint32_t)(c.x0 + zx) | ((uint32_t)(c.y0 + zy) << 12) | ((uint32_t)s << 24);
        }
    };
    for (int zy = warp; zy < zh; zy += kFastWarps) {
        const uint32_t* srow = score_w + (zy + 1) * tsw;
        for (int gb = g0; gb <= g1; gb += 32) {
            const int gi = gb + lane;
            uint32_t w = gi <= g1 ? srow[gi] : 0u;
            // byte != 0 -> bit 7 of that byte
            w = (((w & 0x7f7f7f7fu) + 0x7f7f7f7fu) | w) & 0x80808080u;
            if (!enqueue(w, ((uint32_t)zy << 16) | (uint32_t)(4 * gi))) continue;
            while (qn - qh >= 32) {
                nms_at(q[(qh + lane) & (kFastQueue - 1)]);
                qh += 32;
            }
            __syncwarp();
        }
    }
    if (lane < qn - qh) nms_at(q[(qh + lane) & (kFastQueue - 1)]);
    __syncthreads();

    // ---- emit: a cell that has a corner at ini_th keeps those, else the ones at min_th ----
    if (tid == 0) {
        int n = 0;
        for (int j = 0; j < c.ncells; ++j) n += s_nini[j] > 0 ? s_nini[j] : s_nmin[j];
        s_total = n;
        s_base = n > 0 ? atomicAdd(&ncand[f * g.nlevels + c.level], n) : 0;
    }
    __syncthreads();
    if (s_total == 0) return;
    uint32_t* out = cand + (long long)f * g.cand_total + L.cand_off + s_base;
    const int nlist = s_nlist;
    for (int i = tid; i < nlist; i += kFastThreads) {
        const uint32_t e = list[i];
        const int zx = (int)(e & 0xfff) - c.x0, s = (int)(e >> 24);
        int cj = (int)(((uint32_t)zx * cmagic) >> 20);
        if (cj * wcell > zx) --cj;
        const bool keep = s_nini[cj] > 0 ? s >= ini_th : s >= min_th;
        if (keep) {
            const int slot = atomicAdd(&s_slot, 1);
            if (s_base + slot < L.cand_cap) out[slot] = e;
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// K3: quadtree distribution, one CTA per (frame, level)
// ------------------------------------------------------------------------------------------------------
// The reference keeps a std::list of nodes; children are pushed to the FRONT in the order TL,TR,BL,BR and the
// parent is erased.  Here the list is an array in list order (front = index 0).  Per round:
//   * all threads histogram the keys of every splittable node into its 4 quadrants (shared atomics),
//   * thread 0 replays the list bookkeeping (<= quota+3 live nodes) and lays out the next list,
//   * all threads move their keys to the new node positions.
// Phase 2 ("expand the biggest first", ORBextractor.cc:671-735) sorts the splittable nodes by
// (key count, creation order) with a parallel rank sort; ties: later created node first (the oracle's
// documented stand-in for the reference's pointer comparison).
struct OctShared {
    int M, mode, nE, cur;
};
enum { OCT_PHASE1 = 0, OCT_PHASE2 = 1, OCT_DONE = 2 };
enum { NODE_LEAF = 1 };

__device__ __forceinline__ int oct_quadrant(int kx, int ky, const short* r) {
    const int hx = (r[2] - r[0] + 1) >> 1, hy = (r[3] - r[1] + 1) >> 1;  // ceil(w/2), ceil(h/2)
    return (kx < r[0] + hx ? 0 : 1) + (ky < r[1] + hy ? 0 : 2);
}
__device__ __forceinline__ void oct_child_rect(const short* r, int q, short* o) {
    const int hx = (r[2] - r[0] + 1) >> 1, hy = (r[3] - r[1] + 1) >> 1;
    o[0] = (q & 1) ? r[0] + hx : r[0];
    o[2] = (q & 1) ? r[2] : r[0] + hx;
    o[1] = (q & 2) ? r[1] + hy : r[1];
    o[3] = (q & 2) ? r[3] : r[1] + hy;
}

__global__ void __launch_bounds__(256) k_octree(const __grid_constant__ OrbGeom g, const uint32_t* __restrict__ cand_all,
                                                const int* __restrict__ ncand, uint16_t* __restrict__ knode_all,
                                                uint32_t* __restrict__ okp_all, int* __restrict__ on, int cap_nodes,
                                                int* __restrict__ err) {
    extern __shared__ __align__(16) unsigned char oct_smem[];
    const int l = blockIdx.x, f = blockIdx.y, tid = threadIdx.x, nt = blockDim.x;
    const LevelGeom& L = g.lv[l];
    const int N = L.quota;
    int n = ncand[f * g.nlevels + l];
    if (n > L.cand_cap) n = L.cand_cap;
    if (n == 0 || L.nIni < 1 || L.nIni > cap_nodes) {
        if (tid == 0) on[f * g.nlevels + l] = 0;
        return;
    }
    const uint32_t* cand = cand_all + (long long)f * g.cand_total + L.cand_off;
    uint16_t* knode = knode_all + (long long)f * g.cand_total + L.cand_off;
    uint32_t* okp = okp_all + (long long)f * g.kp_total + L.kp_off;

    // shared layout (cap_nodes = quota + 8 entries each)
    const int CN = cap_nodes;
    unsigned long long* best = reinterpret_cast<unsigned long long*>(oct_smem);  // [CN]
    int* cnt4 = reinterpret_cast<int*>(best + CN);                                // [CN][4]
    int* size0 = cnt4 + 4 * CN;                                                   // [2][CN]
    int* e_size = size0 + 2 * CN;                                                 // [CN]
    int* e_pos = e_size + CN;                                                     // [CN]
    int* e_sorted = e_pos + CN;                                                   // [CN]
    short* rect0 = reinterpret_cast<short*>(e_sorted + CN);                       // [2][CN][4]
    short* childpos = rect0 + 2 * CN * 4;                                         // [CN][4]
    short* newpos = childpos + CN * 4;                                            // [CN]
    unsigned char* flags0 = reinterpret_cast<unsigned char*>(newpos + CN);        // [2][CN]
    unsigned char* divided = flags0 + 2 * CN;                                     // [CN]
    __shared__ OctShared S;

    // ---- roots (ORBextractor.cc:541-589) ----
    if (tid == 0) { S.cur = 0; S.M = L.nIni; S.mode = OCT_PHASE1; S.nE = 0; }
    for (int i = tid; i < L.nIni; i += nt) {
        short* r = rect0 + i * 4;
        r[0] = (short)(int)__fmul_rn(L.hX, (float)i);
        r[2] = (short)(int)__fmul_rn(L.hX, (float)(i + 1));
        r[1] = 0;
        r[3] = (short)(L.maxBY - L.minBY);
        size0[i] = 0;
    }
    __syncthreads();
    for (int k = tid; k < n; k += nt) {
        const uint32_t c = cand[k];
        const int kx = (int)(c & 0xfff) - L.minBX;
        int r = (int)__fdiv_rn((float)kx, L.hX);
        r = min(r, L.nIni - 1);
        knode[k] = (uint16_t)r;
        atomicAdd(&size0[r], 1);
    }
    __syncthreads();
    if (tid == 0) {
        int pos = 0;
        for (int r = 0; r < L.nIni; ++r) {
            if (size0[r] == 0) { newpos[r] = -1; continue; }
            newpos[r] = (short)pos;
            for (int j = 0; j < 4; ++j) rect0[(CN + pos) * 4 + j] = rect0[r * 4 + j];
            size0[CN + pos] = size0[r];
            flags0[CN + pos] = size0[r] == 1 ? NODE_LEAF : 0;
            ++pos;
        }
        S.M = pos;
        S.cur = 1;
    }
    __syncthreads();
    for (int k = tid; k < n; k += nt) knode[k] = (uint16_t)newpos[knode[k]];
    __syncthreads();

    // ---- rounds ----
    while (S.mode != OCT_DONE) {
        const int cur = S.cur, M = S.M, mode = S.mode, nE = S.nE;
        short* rect = rect0 + cur * CN * 4;
        short* nrect = rect0 + (cur ^ 1) * CN * 4;
        int* size = size0 + cur * CN;
        int* nsize = size0 + (cur ^ 1) * CN;
        unsigned char* flags = flags0 + cur * CN;
        unsigned char* nflags = flags0 + (cur ^ 1) * CN;

        for (int i = tid; i < 4 * M; i += nt) cnt4[i] = 0;
        for (int i = tid; i < M; i += nt) divided[i] = 0;
        __syncthreads();
        for (int k = tid; k < n; k += nt) {
            const int p = knode[k] & 0x3fff;
            if (!(flags[p] & NODE_LEAF)) {
                const uint32_t c = cand[k];
                const int q = oct_quadrant((int)(c & 0xfff) - L.minBX, (int)((c >> 12) & 0xfff) - L.minBY, rect + p * 4);
                atomicAdd(&cnt4[p * 4 + q], 1);
                knode[k] = (uint16_t)(p | (q << 14));
            }
        }
        if (mode == OCT_PHASE2) {
            // rank sort of the splittable nodes by (size, creation order) ascending
            for (int e = tid; e < nE; e += nt) {
                const int se = e_size[e];
                int rank = 0;
                for (int j = 0; j < nE; ++j) {
                    const int sj = e_size[j];
                    rank += (sj < se || (sj == se && j < e)) ? 1 : 0;
                }
                e_sorted[rank] = e;
            }
        }
        __syncthreads();

        if (tid == 0) {
            int C = 0, newM, nExp = 0, newE = 0;
            if (mode == OCT_PHASE1) {
                // every non-leaf node splits, in list order
                int nLeaf = 0;
                for (int p = 0; p < M; ++p) {
                    if (flags[p] & NODE_LEAF) { newpos[p] = (short)nLeaf++; continue; }
                    divided[p] = 1;
                    for (int q = 0; q < 4; ++q)
                        if (cnt4[p * 4 + q] > 0) childpos[p * 4 + q] = (short)C++;
                }
                newM = C + nLeaf;
                for (int p = 0; p < M; ++p) {
                    if (flags[p] & NODE_LEAF) {
                        const int dst = C + newpos[p];
                        newpos[p] = (short)dst;
                        for (int j = 0; j < 4; ++j) nrect[dst * 4 + j] = rect[p * 4 + j];
                        nsize[dst] = size[p];
                        nflags[dst] = NODE_LEAF;
                    } else {
                        for (int q = 0; q < 4; ++q) {
                            const int cnt = cnt4[p * 4 + q];
                            if (cnt == 0) continue;
                            const int dst = C - 1 - childpos[p * 4 + q];
                            childpos[p * 4 + q] = (short)dst;
                            oct_child_rect(rect + p * 4, q, nrect + dst * 4);
                            nsize[dst] = cnt;
                            nflags[dst] = cnt == 1 ? NODE_LEAF : 0;
                            if (cnt > 1) { ++nExp; e_size[newE] = cnt; e_pos[newE] = dst; ++newE; }
                        }
                    }
                }
                if (newM >= N || newM == M) S.mode = OCT_DONE;
                else if (newM + 3 * nExp > N) S.mode = OCT_PHASE2;
            } else {
                // split the biggest splittable nodes first until the list holds >= N nodes
                int count = M, jstop = nE;  // nodes e_sorted[jstop..nE) get split
                for (int j = nE - 1; j >= 0; --j) {
                    const int p = e_pos[e_sorted[j]];
                    int nchild = 0;
                    for (int q = 0; q < 4; ++q)
                        if (cnt4[p * 4 + q] > 0) { childpos[p * 4 + q] = (short)C++; ++nchild; }
                    divided[p] = 1;
                    count += nchild - 1;
                    jstop = j;
                    if (count >= N) break;
                }
                newM = count;
                int pos = C;
                for (int p = 0; p < M; ++p) {
                    if (divided[p]) continue;
                    newpos[p] = (short)pos;
                    for (int j = 0; j < 4; ++j) nrect[pos * 4 + j] = rect[p * 4 + j];
                    nsize[pos] = size[p];
                    nflags[pos] = flags[p];
                    ++pos;
                }
                for (int j = nE - 1; j >= jstop; --j) {
                    const int p = e_pos[e_sorted[j]];
                    for (int q = 0; q < 4; ++q) {
                        const int cnt = cnt4[p * 4 + q];
                        if (cnt == 0) continue;
                        const int dst = C - 1 - childpos[p * 4 + q];
                        childpos[p * 4 + q] = (short)dst;
                        oct_child_rect(rect + p * 4, q, nrect + dst * 4);
                        nsize[dst] = cnt;
                        nflags[dst] = cnt == 1 ? NODE_LEAF : 0;
                    }
                }
                // new splittable list in creation order (= dst descending from C-1 to 0); e_* are free to overwrite now
                for (int dst = C - 1; dst >= 0; --dst)
                    if (!(nflags[dst] & NODE_LEAF)) { e_size[newE] = nsize[dst]; e_pos[newE] = dst; ++newE; }
                if (newM >= N || newM == M) S.mode = OCT_DONE;
            }
            S.M = newM;
            S.nE = newE;
            S.cur = cur ^ 1;
        }
        __syncthreads();
        for (int k = tid; k < n; k += nt) {
            const int kn = knode[k], p = kn & 0x3fff, q = kn >> 14;
            knode[k] = (uint16_t)(divided[p] ? childpos[p * 4 + q] : newpos[p]);
        }
        __syncthreads();
    }

    // ---- best key per node: max response, ties -> earliest in the reference's candidate order ----
    const int M = S.M;
    for (int i = tid; i < M; i += nt) best[i] = 0ull;
    __syncthreads();
    for (int k = tid; k < n; k += nt) {
        const uint32_t c = cand[k];
        const int x = c & 0xfff, y = (c >> 12) & 0xfff, s = c >> 24;
        const int ci = (y - L.minBY - 3) / L.hCell, cj = (x - L.minBX - 3) / L.wCell;
        const unsigned long long order = ((unsigned long long)(ci * L.nCols + cj) << 24) | ((unsigned long long)y << 12) | (unsigned long long)x;
        const unsigned long long key = ((unsigned long long)s << 48) | (0xffffffffffffull - order);
        atomicMax(&best[knode[k] & 0x3fff], key);
    }
    __syncthreads();
    for (int k = tid; k < n; k += nt) {
        const uint32_t c = cand[k];
        const int x = c & 0xfff, y = (c >> 12) & 0xfff, s = c >> 24;
        const int ci = (y - L.minBY - 3) / L.hCell, cj = (x - L.minBX - 3) / L.wCell;
        const unsigned long long order = ((unsigned long long)(ci * L.nCols + cj) << 24) | ((unsigned long long)y << 12) | (unsigned long long)x;
        const unsigned long long key = ((unsigned long long)s << 48) | (0xffffffffffffull - order);
        const int p = knode[k] & 0x3fff;
        if (best[p] == key && p < L.kp_cap) okp[p] = c;
    }
    if (tid == 0) {
        on[f * g.nlevels + l] = min(M, L.kp_cap);
        if (M > L.kp_cap) atomicExch(err, HVO_ERR_OVERFLOW);
    }
}

// ------------------------------------------------------------------------------------------------------
// K4: orientation + 7x7 sigma-2 Gaussian of the keypoint's patch + steered rBRIEF + output assembly, one warp per keypoint.
//
// The reference blurs every level (ORBextractor.cc:1083-1084) and computeOrbDescriptor (.cc:106-144) then reads 512 samples
// of the blurred level around each keypoint: rotated pattern coordinates reach +-18 (|(-13,-13)| = 18.4), so only the 37x37
// blurred patch matters, i.e. the 43x43 patch of the level itself (BORDER_REFLECT_101 where it leaves the image).  For
// ~1000 keypoints on 950 K pyramid pixels blurring the patches costs less than half the instructions of blurring the levels
// and a third of the DRAM traffic (no blurred pyramid is written or read back), so the blur lives here:
//   load   44 x 12 aligned words of the level (rows cy-21 .. cy+22, the last one only pads the row pairs) -> shared memory
//   angle  IC_Angle (.cc:75-102) on the raw patch: lane <-> column
//   H      cv::GaussianBlur fixed point (Q8 kernel 18,34,48,56,48,34,18): horizontal pass exact in 16 bits, four outputs of two
//          rows per work item with __dp4a on funnel-shifted words; results are stored as vertical PAIRS (row 2r | row 2r+1 << 16)
//   V      vertical pass as four __dp2a per pixel on the row pairs (an output row starting on an odd row uses the pairs one
//          row earlier with the coefficients shifted by one: the extra row gets coefficient 0), rounded (v + 2^15) >> 16;
//          the blurred 37x37 patch overlays the raw one
//   rBRIEF lane i -> descriptor byte i, samples read from shared memory
// ------------------------------------------------------------------------------------------------------
static const int kDescWarps = 4;
static const int kPatRows = 44, kPatWords = 12;   // raw patch: rows cy-21 .. cy+22, 48 bytes from the aligned column at or below cx-21
static const int kPatPairs = kPatRows / 2;
static const int kBlurPitch = 40;                 // columns of the H / blurred patch rows (37 used)

__global__ void __launch_bounds__(kDescWarps * 32) k_describe(const __grid_constant__ OrbGeom g, ImgSrc src,
                                                              const uint32_t* __restrict__ okp_all,
                                                              const int* __restrict__ on, hvo_keypoint* __restrict__ kps,
                                                              uint8_t* __restrict__ desc, int32_t* __restrict__ counts,
                                                              const uint16_t* __restrict__ depth16, float depth_factor,
                                                              float bf, int distorted, float* __restrict__ kp_depth,
                                                              float* __restrict__ kp_uright) {
    __shared__ uint32_t s_pat[256];   // test t of descriptor byte b at word t * 32 + b: (ax, ay, bx, by), conflict-free for lane <-> b
    __shared__ __align__(16) uint32_t s_raw[kDescWarps][kPatRows * kPatWords + 8];
    __shared__ __align__(16) uint32_t s_hp[kDescWarps][kPatPairs * kBlurPitch];
    const int f = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_pat[(i & 7) * 32 + (i >> 3)] = __ldg(reinterpret_cast<const uint32_t*>(g_pattern) + i);
    __syncthreads();

    // locate keypoint gi (level-major) of frame f: lane l holds the count of level l, inclusive scan over the levels
    const int gi = blockIdx.x * kDescWarps + warp;
    const int nl = lane < g.nlevels ? __ldg(&on[f * g.nlevels + lane]) : 0;
    int incl = nl;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    const unsigned below = __ballot_sync(0xffffffffu, incl <= gi);   // levels that end at or before gi: a prefix of the lanes
    const int lvl = __popc(below);
    if (blockIdx.x == 0 && threadIdx.x == 0) counts[f] = min(total, g.out_cap);
    if (gi >= total || gi >= g.out_cap) return;
    const int idx = gi - __shfl_sync(0xffffffffu, incl - nl, lvl);

    const LevelGeom& L = g.lv[lvl];
    const uint32_t c = okp_all[(long long)f * g.kp_total + L.kp_off + idx];
    const int cx = c & 0xfff, cy = (c >> 12) & 0xfff, resp = c >> 24;
    int pitch;
    const uint8_t* img = level_ptr(g, src, lvl, f, pitch);
    uint32_t* raw = s_raw[warp];
    uint32_t* hp = s_hp[warp];

    // ---- load: word k of row r holds level bytes xa + 4k .. + 3 of row reflect101(cy - 21 + r) ----
    const int x0 = cx - 21, xa = x0 & ~3, sh = x0 - xa;   // patch column 0 sits at byte `sh` of a raw row
    const bool aligned = ((pitch & 3) == 0) && ((reinterpret_cast<uintptr_t>(img) & 3) == 0);
    const int lw = L.w, lh = L.h;
    // interior keypoints (the 43 x 43 patch inside the level, every word of it inside the allocation): straight word loads, all in flight
    const bool interior = aligned && xa >= 0 && cx + 21 < lw && cy >= 21 && cy + 21 < lh && (xa + 4 * kPatWords <= pitch || cy + 21 < lh - 1);
    if (interior) {
        const uint8_t* base = img + (long long)(cy - 21) * pitch + xa;
#pragma unroll
        for (int it = 0; it < (kPatRows * kPatWords + 31) / 32; ++it) {
            const int i = lane + 32 * it;
            if (i < kPatRows * kPatWords) {
                const int r = (i * 43691) >> 19, k = i - kPatWords * r;   // i / 12
                raw[i] = __ldg(reinterpret_cast<const uint32_t*>(base + min(r, kPatRows - 2) * pitch + 4 * k));   // row 43 only pads the last pair
            }
        }
    } else {
#pragma unroll 1
        for (int i = lane; i < kPatRows * kPatWords; i += 32) {
            const int r = (i * 43691) >> 19, k = i - kPatWords * r;
            const int y = min(max(reflect101(cy - 21 + r, lh), 0), lh - 1);
            const int x = xa + 4 * k;
            const uint8_t* row = img + (long long)y * pitch;
            uint32_t w = 0;
            if (aligned && x >= 0 && x + 3 < lw) {
                w = __ldg(reinterpret_cast<const uint32_t*>(row + x));
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int xx = min(max(reflect101(x + j, lw), 0), lw - 1);
                    w |= (uint32_t)__ldg(row + xx) << (8 * j);
                }
            }
            raw[i] = w;
        }
    }
    if (lane < 8) raw[kPatRows * kPatWords + lane] = 0u;   // the word behind the last row is read (and multiplied by nothing that is kept)
    __syncwarp();

    // ---- IC_Angle on the unblurred patch: lane <-> column u = lane - 15 ----
    int m10 = 0, m01 = 0;
    if (lane < 31) {
        const int u = lane - 15, au = abs(u);
        const uint8_t* p = reinterpret_cast<const uint8_t*>(raw) + 21 * (kPatWords * 4) + sh + 21 + u;
#pragma unroll
        for (int v = -15; v <= 15; ++v) {
            if (au <= c_umax[v < 0 ? -v : v]) {
                const int val = p[v * (kPatWords * 4)];
                m10 += u * val;
                m01 += v * val;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        m10 += __shfl_xor_sync(0xffffffffu, m10, o);
        m01 += __shfl_xor_sync(0xffffffffu, m01, o);
    }
    const float angle = fast_atan2_deg((float)m01, (float)m10);

    // ---- H pass: item = (row pair, group of 4 columns) ----
    {
        const uint32_t K0123 = 18u | (34u << 8) | (48u << 16) | (56u << 24), K456 = 48u | (34u << 8) | (18u << 16);
        const int fs = 8 * sh;
#pragma unroll 1
        for (int it = 0; it < (kPatPairs * (kBlurPitch / 4) + 31) / 32; ++it) {
            const int item = lane + 32 * it;
            if (item < kPatPairs * (kBlurPitch / 4)) {
                const int rp = (item * 6554) >> 16, cg = item - (kBlurPitch / 4) * rp;   // item / 10
                uint32_t o[2][4];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t* rr = raw + (2 * rp + h) * kPatWords + cg;
                    const uint32_t w0 = rr[0], w1 = rr[1], w2 = rr[2], w3 = rr[3];
                    const uint32_t A = __funnelshift_r(w0, w1, fs), B = __funnelshift_r(w1, w2, fs), C = __funnelshift_r(w2, w3, fs);
                    o[h][0] = __dp4a(A, K0123, __dp4a(B, K456, 0u));
                    o[h][1] = __dp4a(__byte_perm(A, B, 0x4321), K0123, __dp4a(__byte_perm(B, C, 0x4321), K456, 0u));
                    o[h][2] = __dp4a(__byte_perm(A, B, 0x5432), K0123, __dp4a(__byte_perm(B, C, 0x5432), K456, 0u));
                    o[h][3] = __dp4a(__byte_perm(A, B, 0x6543), K0123, __dp4a(__byte_perm(B, C, 0x6543), K456, 0u));
                }
                *reinterpret_cast<uint4*>(&hp[rp * kBlurPitch + 4 * cg]) =
                    make_uint4(__byte_perm(o[0][0], o[1][0], 0x5410), __byte_perm(o[0][1], o[1][1], 0x5410), __byte_perm(o[0][2], o[1][2], 0x5410),
                               __byte_perm(o[0][3], o[1][3], 0x5410));
            }
        }
    }
    __syncwarp();

    // ---- V pass: lane = (band of 14 output rows, group of 4 columns); the blurred patch overlays the raw one ----
    if (lane < 30) {
        const int band = lane / 10, cg = lane - 10 * band;
        const int y0 = 14 * band;   // even: every iteration makes the even row y and the odd row y + 1 from the same four row pairs
        // row pairs {2p, 2p+1}: the even output row y uses pairs y/2 .. y/2+3 with (k0,k1)(k2,k3)(k4,k5)(k6,0), the odd row y+1 the same
        // pairs with (0,k0)(k1,k2)(k3,k4)(k5,k6)
        const uint32_t E0 = 18u | (34u << 8), E1 = 48u | (56u << 8), E2 = 48u | (34u << 8), E3 = 18u;
        const uint32_t O0 = 18u << 8, O1 = 34u | (48u << 8), O2 = 56u | (48u << 8), O3 = 34u | (18u << 8);
        const uint4* hp4 = reinterpret_cast<const uint4*>(hp) + cg;
        const int p0 = y0 >> 1;
        uint4 P0 = hp4[p0 * (kBlurPitch / 4)], P1 = hp4[(p0 + 1) * (kBlurPitch / 4)], P2 = hp4[(p0 + 2) * (kBlurPitch / 4)];
        uint32_t* bl = raw + y0 * (kBlurPitch / 4) + cg;
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            const uint4 P3 = hp4[min(p0 + j + 3, kPatPairs - 1) * (kBlurPitch / 4)];   // rows past 36 (last band) are computed and dropped
            {
                const uint32_t a0 = __dp2a_lo(P0.x, E0, __dp2a_lo(P1.x, E1, __dp2a_lo(P2.x, E2, __dp2a_lo(P3.x, E3, 32768u))));
                const uint32_t a1 = __dp2a_lo(P0.y, E0, __dp2a_lo(P1.y, E1, __dp2a_lo(P2.y, E2, __dp2a_lo(P3.y, E3, 32768u))));
                const uint32_t a2 = __dp2a_lo(P0.z, E0, __dp2a_lo(P1.z, E1, __dp2a_lo(P2.z, E2, __dp2a_lo(P3.z, E3, 32768u))));
                const uint32_t a3 = __dp2a_lo(P0.w, E0, __dp2a_lo(P1.w, E1, __dp2a_lo(P2.w, E2, __dp2a_lo(P3.w, E3, 32768u))));
                if (y0 + 2 * j < 37) bl[(2 * j) * (kBlurPitch / 4)] = __byte_perm(__byte_perm(a0, a1, 0x0062), __byte_perm(a2, a3, 0x0062), 0x5410);
            }
            {
                const uint32_t a0 = __dp2a_lo(P0.x, O0, __dp2a_lo(P1.x, O1, __dp2a_lo(P2.x, O2, __dp2a_lo(P3.x, O3, 32768u))));
                const uint32_t a1 = __dp2a_lo(P0.y, O0, __dp2a_lo(P1.y, O1, __dp2a_lo(P2.y, O2, __dp2a_lo(P3.y, O3, 32768u))));
                const uint32_t a2 = __dp2a_lo(P0.z, O0, __dp2a_lo(P1.z, O1, __dp2a_lo(P2.z, O2, __dp2a_lo(P3.z, O3, 32768u))));
                const uint32_t a3 = __dp2a_lo(P0.w, O0, __dp2a_lo(P1.w, O1, __dp2a_lo(P2.w, O2, __dp2a_lo(P3.w, O3, 32768u))));
                if (y0 + 2 * j + 1 < 37) bl[(2 * j + 1) * (kBlurPitch / 4)] = __byte_perm(__byte_perm(a0, a1, 0x0062), __byte_perm(a2, a3, 0x0062), 0x5410);
            }
            P0 = P1; P1 = P2; P2 = P3;
        }
    }
    __syncwarp();

    // ---- steered rBRIEF on the blurred patch: lane i -> descriptor byte i ----
    const float factorPI = 0.017453292519943295769236907684886f;  // (float)(CV_PI / 180.f)
    const float ang = __fmul_rn(angle, factorPI);
    const float a = (float)cos((double)ang), b = (float)sin((double)ang);
    const uint8_t* ctr = reinterpret_cast<const uint8_t*>(raw) + 18 * kBlurPitch + 18;
    int val = 0;
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const uint32_t pw = s_pat[t * 32 + lane];
        const float ax = (float)(int8_t)(pw & 0xff), ay = (float)(int8_t)((pw >> 8) & 0xff), bx = (float)(int8_t)((pw >> 16) & 0xff), by = (float)(int8_t)(pw >> 24);
        const int r0 = __float2int_rn(__fadd_rn(__fmul_rn(ax, b), __fmul_rn(ay, a)));
        const int c0 = __float2int_rn(__fsub_rn(__fmul_rn(ax, a), __fmul_rn(ay, b)));
        const int r1 = __float2int_rn(__fadd_rn(__fmul_rn(bx, b), __fmul_rn(by, a)));
        const int c1 = __float2int_rn(__fsub_rn(__fmul_rn(bx, a), __fmul_rn(by, b)));
        const int t0 = ctr[r0 * kBlurPitch + c0], t1 = ctr[r1 * kBlurPitch + c1];
        val |= (t0 < t1 ? 1 : 0) << t;
    }
    const long long o = (long long)f * g.out_cap + gi;
    desc[o * 32 + lane] = (uint8_t)val;

    if (lane == 0) {
        float x = (float)cx, y = (float)cy;
        if (lvl != 0) { x = __fmul_rn(x, L.scale); y = __fmul_rn(y, L.scale); }
        hvo_keypoint k;
        k.x = x; k.y = y; k.size = L.kp_size; k.angle = angle; k.response = (float)resp; k.octave = lvl; k.class_id = -1;
        kps[o] = k;
        if (depth16 != nullptr) {
            const int u = min((int)x, g.width - 1), v = min((int)y, g.height - 1);
            const float d = __fmul_rn((float)depth16[((long long)f * g.height + v) * g.width + u], depth_factor);
            const bool ok = d > 0.f && d < 7.0f;
            kp_depth[o] = ok ? d : -1.f;
            // mvuRight = kpU.pt.x - bf / d needs the UNDISTORTED x (Frame.cc:1944, 1957): only formed here when mvKeysUn == mvKeys
            kp_uright[o] = (ok && !distorted) ? __fsub_rn(x, __fdiv_rn(bf, d)) : -1.f;
        }
    }
}

// Frame::UndistortKeyPoints (Frame.cc:1701-1731) and the mvuRight of ComputeStereoFromRGBD (:1953-1958) on the keypoints k_describe
// wrote: row i of frame blockIdx.y, rows at or past counts[f] untouched.  kp_depth > 0 exactly where k_describe found 0 < d < 7.
__global__ void __launch_bounds__(128) k_undistort_kps(const hvo_camera cam, int cap, const hvo_keypoint* __restrict__ kps,
                                                       const int32_t* __restrict__ counts, const float* __restrict__ kp_depth, float bf,
                                                       hvo_keypoint* __restrict__ kps_un, float* __restrict__ kp_uright) {
    const int f = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= min(counts[f], cap)) return;
    const long long o = (long long)f * cap + i;
    hvo_keypoint k = kps[o];
    if (cam.k1 != 0.f) undistort_point(cam, k.x, k.y, &k.x, &k.y);   // the reference tests k1 only (Frame.cc:1703)
    if (kps_un) kps_un[o] = k;
    if (kp_uright) {
        const float d = kp_depth[o];
        kp_uright[o] = d > 0.f ? __fsub_rn(k.x, __fdiv_rn(bf, d)) : -1.f;
    }
}

// ------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------
static inline int cv_round_f(float v) { return (int)lrintf(v); }

static short sat_short_round(float v) {
    int i = (int)lrintf(v);
    return (short)std::min(32767, std::max(-32768, i));
}

}  // namespace hvo

using namespace hvo;

int hvo_orb::init() {
    const int n = p.nlevels;
    // ---- scale tables and per-level quotas (ORBextractor.cc:408-444) ----
    const double sfd = (double)p.scale_factor;
    sf.assign(n, 1.f); isf.assign(n, 1.f); sigma2.assign(n, 1.f); isigma2.assign(n, 1.f);
    for (int i = 1; i < n; ++i) {
        sf[i] = (float)((double)sf[i - 1] * sfd);
        sigma2[i] = sf[i] * sf[i];
    }
    for (int i = 0; i < n; ++i) { isf[i] = 1.0f / sf[i]; isigma2[i] = 1.0f / sigma2[i]; }
    nfeat.assign(n, 0);
    {
        const float factor = (float)(1.0 / sfd);
        float want = (float)p.nfeatures * (1.f - factor) / (1.f - (float)std::pow((double)factor, (double)n));
        int sum = 0;
        for (int l = 0; l < n - 1; ++l) {
            nfeat[l] = cv_round_f(want);
            sum += nfeat[l];
            want *= factor;
        }
        nfeat[n - 1] = std::max(p.nfeatures - sum, 0);
    }
    umax.assign(h_umax, h_umax + 16);

    // ---- level geometry ----
    std::memset(&g, 0, sizeof(g));
    g.nlevels = n; g.width = width; g.height = height;
    long long off = 0;
    int cand_off = 0, kp_off = 0;
    std::vector<StripDesc> strips;
    fast_smem = 0;
    max_quota = 0;
    for (int l = 0; l < n; ++l) {
        LevelGeom& L = g.lv[l];
        L.w = cv_round_f((float)width * isf[l]);
        L.h = cv_round_f((float)height * isf[l]);
        if (L.w > 4095 || L.h > 4095) { set_error("image too large (max 4095 px per side)"); return HVO_ERR_ARG; }
        if (l == 0) { L.pitch = width; L.img_off = 0; }
        else { L.pitch = (int)align_up((size_t)L.w, 128); L.img_off = off; off += (long long)L.pitch * L.h; }
        L.minBX = kEdge - 3; L.minBY = kEdge - 3; L.maxBX = L.w - kEdge + 3; L.maxBY = L.h - kEdge + 3;
        L.quota = nfeat[l];
        L.scale = sf[l];
        L.kp_size = (float)(int)(31 * sf[l]);
        const float fw = (float)(L.maxBX - L.minBX), fh = (float)(L.maxBY - L.minBY);
        L.nCols = (int)(fw / 30.f); L.nRows = (int)(fh / 30.f);
        L.cand_off = cand_off; L.cand_cap = 0;
        L.kp_off = kp_off; L.kp_cap = L.quota + 4;
        kp_off += L.kp_cap;
        max_quota = std::max(max_quota, L.quota);
        if (L.nCols < 1 || L.nRows < 1 || L.maxBX <= L.minBX || L.maxBY <= L.minBY) {
            // level too small for a single 30-px cell: the reference divides by zero here; produce no keypoints
            L.nCols = L.nRows = 0; L.wCell = L.hCell = 1; L.nIni = 0; L.hX = 1.f;
            continue;
        }
        L.wCell = (int)std::ceil(fw / L.nCols); L.hCell = (int)std::ceil(fh / L.nRows);
        L.nIni = (int)std::round((float)(L.maxBX - L.minBX) / (L.maxBY - L.minBY));
        L.hX = L.nIni > 0 ? (float)(L.maxBX - L.minBX) / L.nIni : 1.f;
        const int max_seg_cells = std::max(1, kFastMaxZone / L.wCell);   // a strip = a run of cells of one cell row
        for (int i = 0; i < L.nRows; ++i) {
            const float iniY = (float)(L.minBY + i * L.hCell);
            float maxY = iniY + L.hCell + 6;
            if (iniY >= L.maxBY - 3) continue;
            if (maxY > L.maxBY) maxY = (float)L.maxBY;
            const int zh = (int)maxY - (int)iniY - 6;
            if (zh <= 0) continue;
            if (zh > kFastMaxZh) { set_error("internal: FAST cell higher than %d", kFastMaxZh); return HVO_ERR_ARG; }
            StripDesc st;
            std::memset(&st, 0, sizeof(st));
            int listcap = 0;
            auto flush = [&]() {
                if (st.ncells == 0) return;
                const int xal = (st.x0 - 3) & ~15, zb0 = st.x0 - xal;
                st.tstride = (short)align_up((size_t)(zb0 + st.zw + 8), 16);
                st.score_off = (int)align_up(std::max<size_t>((size_t)(zh + 6) * st.tstride, (size_t)listcap * 4), 16);
                fast_smem = std::max(fast_smem, (size_t)16 + st.score_off + (size_t)(zh + 2) * st.tstride);
                strips.push_back(st);
                std::memset(&st, 0, sizeof(st));
                listcap = 0;
            };
            for (int j = 0; j < L.nCols; ++j) {
                const float iniX = (float)(L.minBX + j * L.wCell);
                float maxX = iniX + L.wCell + 6;
                if (iniX >= L.maxBX - 6) continue;
                if (maxX > L.maxBX) maxX = (float)L.maxBX;
                const int zw = (int)maxX - (int)iniX - 6;
                if (zw <= 0) continue;
                if (st.ncells == 0) {
                    st.level = (short)l; st.x0 = (short)((int)iniX + 3); st.y0 = (short)((int)iniY + 3); st.zh = (short)zh;
                    st.wcell = (short)L.wCell;
                }
                st.zw += (short)zw; st.ncells += 1;
                const int nms_cap = ((zw + 1) / 2) * ((zh + 1) / 2);  // NMS survivors are never 8-adjacent
                L.cand_cap += nms_cap; listcap += nms_cap;
                if (st.ncells == max_seg_cells) flush();
            }
            flush();
        }
        cand_off += L.cand_cap;
    }
    if (max_quota + 8 > 16383) { set_error("nfeatures too large"); return HVO_ERR_ARG; }
    g.pyr_frame_bytes = (long long)align_up((size_t)off, 256);
    g.cand_total = std::max(cand_off, 1);
    g.kp_total = kp_off;
    g.out_cap = kp_off;
    nstrips = (int)strips.size();

    // ---- CUDA resources ----
    HVO_CUDA(cudaSetDevice(device));
    pin_carveout(k_resize); pin_carveout(k_resize_tile); pin_carveout(k_fast_strips); pin_carveout(k_octree); pin_carveout(k_describe);
    HVO_CUDA(create_stream(&stream));
    for (auto& e : ev) HVO_CUDA(cudaEventCreate(&e));
    for (auto& e : tev) HVO_CUDA(cudaEventCreate(&e));
    const size_t B = (size_t)max_batch;
    HVO_CUDA(cudaMalloc(&d_pyr, std::max<size_t>(B * (size_t)g.pyr_frame_bytes, 256)));
    HVO_CUDA(cudaMalloc(&d_cand, B * g.cand_total * sizeof(uint32_t)));
    HVO_CUDA(cudaMalloc(&d_knode, B * g.cand_total * sizeof(uint16_t)));
    HVO_CUDA(cudaMalloc(&d_ncand, B * n * sizeof(int)));
    HVO_CUDA(cudaMalloc(&d_okp, B * g.kp_total * sizeof(uint32_t)));
    HVO_CUDA(cudaMalloc(&d_on, B * n * sizeof(int)));
    HVO_CUDA(cudaMalloc(&d_err, sizeof(int)));
    HVO_CUDA(cudaMemset(d_err, 0, sizeof(int)));
    HVO_CUDA(cudaMalloc(&d_strips, std::max<size_t>(strips.size(), 1) * sizeof(StripDesc)));
    if (!strips.empty()) HVO_CUDA(cudaMemcpy(d_strips, strips.data(), strips.size() * sizeof(StripDesc), cudaMemcpyHostToDevice));
    if (fast_smem > 200 * 1024) { set_error("internal: FAST strip needs %zu bytes of shared memory", fast_smem); return HVO_ERR_ARG; }
    {   // the attribute is per function (shared by all handles on the device): only ever raise it
        static size_t s_fast_smem_max[64] = {0};
        if (device < 64 && fast_smem > s_fast_smem_max[device]) {
            HVO_CUDA(cudaFuncSetAttribute(k_fast_strips, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fast_smem));
            s_fast_smem_max[device] = fast_smem;
        }
    }

    // ---- resize tables (cv::resize INTER_LINEAR 8U coefficient generation, oracle/cvprims.hpp) ----
    std::vector<int2> xt;
    std::vector<int4> yt;
    xtab_off.assign(n, 0); ytab_off.assign(n, 0);
    for (int l = 1; l < n; ++l) {
        const LevelGeom& S = g.lv[l - 1];
        const LevelGeom& D = g.lv[l];
        xtab_off[l] = (int)xt.size(); ytab_off[l] = (int)yt.size();
        const double scale_x = 1.0 / ((double)D.w / S.w), scale_y = 1.0 / ((double)D.h / S.h);
        for (int dx = 0; dx < D.w; ++dx) {
            float fx = (float)((dx + 0.5) * scale_x - 0.5);
            int sx = (int)std::floor(fx);
            fx -= sx;
            if (sx < 0) { fx = 0; sx = 0; }
            if (sx >= S.w - 1) { fx = 0; sx = S.w - 1; }
            const short w0 = sat_short_round((1.f - fx) * 2048.f), w1 = sat_short_round(fx * 2048.f);
            xt.push_back(make_int2(sx, (int)(unsigned short)w0 | ((int)w1 << 16)));
        }
        for (int dy = 0; dy < D.h; ++dy) {
            float fy = (float)((dy + 0.5) * scale_y - 0.5);
            int sy = (int)std::floor(fy);
            fy -= sy;
            const short b0 = sat_short_round((1.f - fy) * 2048.f), b1 = sat_short_round(fy * 2048.f);
            const int sy0 = std::min(std::max(sy, 0), S.h - 1), sy1 = std::min(std::max(sy + 1, 0), S.h - 1);
            yt.push_back(make_int4(sy0, sy1, b0, b1));
        }
    }
    resize_tile_ok.assign(n, 0);
    for (int l = 1; l < n; ++l) {   // does every 128 x 32 destination tile read at most kRtSrcRows x kRtSrcWords source words?
        const LevelGeom& S = g.lv[l - 1];
        const LevelGeom& D = g.lv[l];
        bool ok = true;
        for (int ty = 0; ty < D.h && ok; ty += kRsH) {
            const int yl = std::min(ty + kRsH, D.h) - 1;
            ok = yt[ytab_off[l] + yl].y - yt[ytab_off[l] + ty].x + 1 <= kRtSrcRows;
        }
        for (int tx = 0; tx < D.w && ok; tx += kRsW) {
            const int xl = std::min(tx + kRsW, D.w) - 1;
            const int xs = xt[xtab_off[l] + tx].x & ~3;
            ok = ((std::min(xt[xtab_off[l] + xl].x + 1, S.w - 1) - xs) >> 2) + 1 <= kRtSrcWords;
        }
        resize_tile_ok[l] = ok ? 1 : 0;
    }
    HVO_CUDA(cudaMalloc(&d_xtab, std::max<size_t>(xt.size(), 1) * sizeof(int2)));
    HVO_CUDA(cudaMalloc(&d_ytab, std::max<size_t>(yt.size(), 1) * sizeof(int4)));
    if (!xt.empty()) HVO_CUDA(cudaMemcpy(d_xtab, xt.data(), xt.size() * sizeof(int2), cudaMemcpyHostToDevice));
    if (!yt.empty()) HVO_CUDA(cudaMemcpy(d_ytab, yt.data(), yt.size() * sizeof(int4), cudaMemcpyHostToDevice));

    // quadtree shared memory: see the layout in k_octree
    const size_t CN = (size_t)max_quota + 8;
    oct_smem = CN * (8 + 16 + 8 + 4 + 4 + 4 + 16 + 8 + 2 + 2 + 1) + 64;
    if (oct_smem > 200 * 1024) { set_error("nfeatures too large for the quadtree kernel"); return HVO_ERR_ARG; }
    // the attribute is per function (shared by all handles on the device): only ever raise it
    static size_t s_oct_smem_max[64] = {0};
    const size_t want = std::max<size_t>(oct_smem, 48 * 1024);
    if (device < 64 && want > s_oct_smem_max[device]) {
        HVO_CUDA(cudaFuncSetAttribute(k_octree, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)want));
        s_oct_smem_max[device] = want;
    }
    return HVO_OK;
}

void hvo_orb::release() {
    cudaSetDevice(device);
    if (stream) cudaStreamSynchronize(stream);
    void* bufs[] = {d_l0, d_depth, d_pyr, d_xtab, d_ytab, d_strips, d_cand, d_ncand, d_knode, d_okp, d_on, d_err,
                    d_kps, d_desc, d_counts, d_kpdepth, d_kpuright};
    for (void* b : bufs) if (b) cudaFree(b);
    for (auto& e : ev) if (e) cudaEventDestroy(e);
    for (auto& e : tev) if (e) cudaEventDestroy(e);
    if (stream) cudaStreamDestroy(stream);
}

int hvo_orb::run(const uint8_t* d_gray, int nframes, hvo_keypoint* d_kps_out, uint8_t* d_desc_out, int32_t* d_counts_out,
                 const uint16_t* d_depth16, const hvo_rgbd_params* rgbd, float* d_kp_depth, float* d_kp_uright) {
    const int n = p.nlevels, B = nframes;
    int launches = 0;
    ImgSrc src;
    src.l0 = d_gray; src.l0_frame = (long long)width * height; src.l0_pitch = width; src.pyr = d_pyr;
    last_l0 = d_gray;
    last_nframes = nframes;
    if (profiling) HVO_CUDA(cudaEventRecord(ev[0], stream));
    HVO_CUDA(cudaMemsetAsync(d_ncand, 0, (size_t)B * n * sizeof(int), stream));
    // K1: pyramid, level l from level l-1
    for (int l = 1; l < n; ++l) {
        const LevelGeom& S = g.lv[l - 1];
        const LevelGeom& D = g.lv[l];
        const uint8_t* sp = l == 1 ? d_gray : d_pyr + S.img_off;
        const long long sframe = l == 1 ? src.l0_frame : g.pyr_frame_bytes;
        dim3 grd(div_up(D.w, kRsW), div_up(D.h, kRsH), B);
        timeline_mark(stream, "k_resize");
        // the shared-memory band kernel needs aligned source words (level 0 is the caller's buffer) and a tile's source rows to fit
        const bool tile_ok = resize_tile_ok[l] && (S.pitch & 3) == 0 && (reinterpret_cast<uintptr_t>(sp) & 3) == 0 && (sframe & 3) == 0;
        if (tile_ok)
            k_resize_tile<<<grd, 256, 0, stream>>>(sp, S.pitch, sframe, S.w, d_pyr + D.img_off, D.pitch, g.pyr_frame_bytes, D.w, D.h,
                                                   d_xtab + xtab_off[l], d_ytab + ytab_off[l]);
        else
            k_resize<<<grd, 256, 0, stream>>>(sp, S.pitch, sframe, S.w, d_pyr + D.img_off, D.pitch, g.pyr_frame_bytes, D.w, D.h,
                                              d_xtab + xtab_off[l], d_ytab + ytab_off[l]);
        ++launches;
    }
    if (profiling) HVO_CUDA(cudaEventRecord(ev[1], stream));
    // K2: FAST cells
    if (nstrips > 0) {
        timeline_mark(stream, "k_fast_strips");
        k_fast_strips<<<dim3(nstrips, B), kFastThreads, fast_smem, stream>>>(g, src, d_strips, d_cand, d_ncand, p.ini_th_fast, p.min_th_fast);
        ++launches;
    }
    if (profiling) HVO_CUDA(cudaEventRecord(ev[2], stream));
    // K3: quadtree
    timeline_mark(stream, "k_octree");
    k_octree<<<dim3(n, B), 256, oct_smem, stream>>>(g, d_cand, d_ncand, d_knode, d_okp, d_on, max_quota + 8, d_err);
    ++launches;
    if (profiling) HVO_CUDA(cudaEventRecord(ev[3], stream));
    // K4: describe (the 7x7 blur of the reference's pyramid is computed per keypoint patch inside; stage 'blur' stays in the
    // stage-time record as an empty interval)
    if (profiling) HVO_CUDA(cudaEventRecord(ev[4], stream));
    const bool rgbd_on = d_depth16 != nullptr && rgbd != nullptr && d_kp_depth != nullptr && d_kp_uright != nullptr;
    timeline_mark(stream, "k_describe");
    k_describe<<<dim3(div_up(g.out_cap, kDescWarps), B), kDescWarps * 32, 0, stream>>>(
        g, src, d_okp, d_on, d_kps_out, d_desc_out, d_counts_out, rgbd_on ? d_depth16 : nullptr,
        rgbd_on ? rgbd->depth_factor : 0.f, rgbd_on ? rgbd->bf : 0.f, rgbd_on ? rgbd->distorted : 0, d_kp_depth, d_kp_uright);
    ++launches;
    if (profiling) { HVO_CUDA(cudaEventRecord(ev[5], stream)); have_stage_times = true; }
    HVO_CUDA(cudaGetLastError());
    last_launches = launches;
    return HVO_OK;
}

int hvo_orb::undistort(const hvo_camera& cam, const hvo_keypoint* d_kps, const int32_t* d_counts, int nframes, const float* d_kp_depth,
                       float bf, hvo_keypoint* d_kps_un, float* d_kp_uright) {
    timeline_mark(stream, "k_undistort_kps");
    k_undistort_kps<<<dim3(div_up(g.out_cap, 128), nframes), 128, 0, stream>>>(cam, g.out_cap, d_kps, d_counts, d_kp_depth, bf, d_kps_un,
                                                                              d_kp_uright);
    HVO_CUDA(cudaGetLastError());
    return HVO_OK;
}
