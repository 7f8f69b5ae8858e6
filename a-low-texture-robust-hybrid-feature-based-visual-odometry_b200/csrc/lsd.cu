// Line extractor for sm_100a.  Replaces ORB_SLAM2::LINEextractor::operator() (reference src/LineExtractor.cpp:329-380):
//   line_descriptor::LSDDetector::detect (Thirdparty/line_descriptor/src/LSDDetector_custom.cpp:105-215), which runs
//   cv::createLineSegmentDetector()->detect() (OpenCV imgproc LSD, default parameters) on octave 0 and fills KeyLines,
//   the response sort + truncation to nLSDFeature (:351-360), LBD (lbd.cu) and the 2-D line functions (:365-377).
//
//   k_lsd_prep      fused cv::GaussianBlur(7x7, sigma 0.75; Q8 taps 0,4,56,136,56,4,0) + cv::resize(0.8, INTER_LINEAR_EXACT,
//                   8.8 fixed point) + LSD ll_angle: 2x2 gradient, level-line angle (cv::fastAtan2), cosf/sinf of the angle;
//                   one shared-memory tile per CTA; 16 B per scaled pixel go to HBM {angle, cos, sin, gx|gy}
//   k_lsd_order     one CTA per frame: stable counting sort of the defined pixels into 1024 gradient-magnitude bins,
//                   descending (warp-private histograms in shared memory, match_any ranks) = LSD's seed order
//   k_lsd_grow      one warp per frame: the ordered, inherently sequential part (region growing with a running mean
//                   angle, rectangle fit, density refinement).  Lanes hold the 8 neighbours of three consecutive region
//                   points; the `used` map is a bitmap in global memory (no shared memory: 32 frames per SM, and the
//                   kernel co-resides with the other pipelines); sums over a region are warp reductions.
//                   Frames are independent, so a batch fills the machine with one warp per frame.
//   k_line_keylines one CTA per frame: KeyLine fields, rank by response (ties: libstdc++'s std::sort order), keep nLSDFeature,
//                   2-D line functions
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <new>
#include <vector>

#include "std_sort.cuh"
#include "hvo_common.cuh"

struct hvo_lbd;
namespace hvo {
int lbd_compute_on_stream(hvo_lbd* h, cudaStream_t stream, const uint8_t* d_gray, int nframes, const hvo_keyline* d_keylines,
                          const int32_t* d_counts, uint8_t* d_desc);

static const double kLsdPi = 3.1415926535897932384626433832795;
#define LSD_NOTDEF (-1024.0f)
#define LSD_DEG2RAD (3.1415926535897932384626433832795 / 180)
#define LSD_2PI (2 * 3.1415926535897932384626433832795)
#define LSD_32PI ((3 * 3.1415926535897932384626433832795) / 2)
#define LSD_PI 3.1415926535897932384626433832795
static const unsigned kFull = 0xffffffffu;

struct __align__(16) LsdPix {
    float ang;  // level-line angle in degrees (cv::fastAtan2), LSD_NOTDEF where the gradient is below threshold
    float c, s; // cosf / sinf of float(angle in radians)
    int gxgy;   // gx (low 16) | gy (high 16): modgrad = sqrt((gx^2 + gy^2) / 4.0)
};

struct LinCoef { int ofs; uint16_t c1; uint16_t mode; };  // INTER_LINEAR_EXACT: mode 0 interior, 1 low border, 2 high border

static const int kPW = 64, kPH = 16;                 // scaled-pixel tile of k_lsd_prep
static const int kSrcW = 96, kSrcH = 28;             // raw tile capacity (scale 0.8: 1.25 * (tile + 1) + 2 + 4 halo, + 3 bytes of word alignment)

// i / d and i % d for 0 <= i < 4096, 1 <= d <= 128 without an integer division (magic = ceil(65536 / d))
struct FastDiv { uint32_t magic; int d; };
__device__ __forceinline__ FastDiv fastdiv_make(int d) { return FastDiv{(65536u + (uint32_t)d - 1u) / (uint32_t)d, d}; }
__device__ __forceinline__ void fastdiv(const FastDiv& f, int i, int& q, int& r) {
    q = (int)(((uint32_t)i * f.magic) >> 16);
    if (q * f.d > i) --q;
    r = i - q * f.d;
}

// --------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_lsd_prep(const uint8_t* __restrict__ gray, int W, int H, long long frame_px, int sw, int sh,
                                                  const LinCoef* __restrict__ cx, const LinCoef* __restrict__ cy,
                                                  const float2* __restrict__ cstab, int sq_low_max, LsdPix* __restrict__ pix,
                                                  uint8_t* __restrict__ scaled_out, int* __restrict__ maxsq, uint32_t* __restrict__ sqkey) {
    __shared__ __align__(4) uint8_t raw[kSrcH][kSrcW];
    __shared__ uint16_t hb[kSrcH][kSrcW];
    __shared__ uint8_t bl[kSrcH][kSrcW];
    __shared__ uint16_t hr[kSrcH][kPW + 2];
    __shared__ uint8_t sc[kPH + 1][kPW + 4];
    __shared__ int s_max;
    const int x0 = blockIdx.x * kPW, y0 = blockIdx.y * kPH, f = blockIdx.z, tid = threadIdx.x;
    const uint8_t* img = gray + (long long)f * frame_px;
    const int x1 = min(x0 + kPW, sw - 1), y1 = min(y0 + kPH, sh - 1);  // last scaled col / row needed (incl. +1 halo)
    const int nx = x1 - x0 + 1, ny = y1 - y0 + 1;
    // blurred source window needed by the resize taps
    const int bx0 = cx[x0].ofs, bx1 = min(cx[x1].ofs + 1, W - 1), by0 = cy[y0].ofs, by1 = min(cy[y1].ofs + 1, H - 1);
    const int bw = bx1 - bx0 + 1, bh = by1 - by0 + 1;  // <= kSrcW - 4, kSrcH - 4
    const int rw = bw + 4, rh = bh + 4;
    if (tid == 0) s_max = 0;
    // raw tile: columns bx0 - 2 .. bx1 + 2, rows by0 - 2 .. by1 + 2.  Interior tiles (no border reflection, 4-byte aligned rows)
    // are fetched as aligned 32-bit words; `shb` = bytes between the aligned origin and the first column the tile needs.
    const int rx0 = bx0 - 2, ry0 = by0 - 2;
    const bool interior = rx0 >= 0 && ry0 >= 0 && rx0 + rw <= W && ry0 + rh <= H && (W & 3) == 0 && (frame_px & 3) == 0 &&
                          (reinterpret_cast<uintptr_t>(gray) & 3) == 0;
    const int shb = interior ? (rx0 & 3) : 0;
    if (interior) {
        const int nwr = (shb + rw + 3) >> 2;  // words per row, <= kSrcW / 4 (the last word may reach past the tile, not past the row)
        const FastDiv dw = fastdiv_make(nwr);
        const uint8_t* base = img + (long long)ry0 * W + (rx0 - shb);
        for (int i = tid; i < nwr * rh; i += 256) {
            int r, c;
            fastdiv(dw, i, r, c);
            reinterpret_cast<uint32_t*>(&raw[r][0])[c] = __ldg(reinterpret_cast<const uint32_t*>(base + (long long)r * W) + c);
        }
    } else {
        const FastDiv dr = fastdiv_make(rw);
        for (int i = tid; i < rw * rh; i += 256) {
            int r, c;
            fastdiv(dr, i, r, c);
            const int y = reflect101(ry0 + r, H), x = reflect101(rx0 + c, W);
            raw[r][c] = __ldg(img + (long long)y * W + x);
        }
    }
    __syncthreads();
    const FastDiv db = fastdiv_make(bw), dn = fastdiv_make(nx);
    for (int i = tid; i < bw * rh; i += 256) {  // horizontal taps 4,56,136,56,4 (the 7-tap kernel's outer taps are 0)
        int r, c;
        fastdiv(db, i, r, c);
        const uint8_t* p = &raw[r][c + shb];
        hb[r][c] = (uint16_t)(4 * (p[0] + p[4]) + 56 * (p[1] + p[3]) + 136 * p[2]);
    }
    __syncthreads();
    for (int i = tid; i < bw * bh; i += 256) {
        int r, c;
        fastdiv(db, i, r, c);
        const uint32_t acc = 4u * (hb[r][c] + hb[r + 4][c]) + 56u * (hb[r + 1][c] + hb[r + 3][c]) + 136u * hb[r + 2][c];
        bl[r][c] = (uint8_t)((acc + 32768u) >> 16);
    }
    __syncthreads();
    for (int i = tid; i < nx * bh; i += 256) {  // horizontal resize, 8.8 fixed point
        int r, c;
        fastdiv(dn, i, r, c);
        const LinCoef k = cx[x0 + c];
        uint16_t v;
        if (k.mode == 0) v = (uint16_t)(bl[r][k.ofs - bx0] * (256 - k.c1) + bl[r][k.ofs - bx0 + 1] * k.c1);
        else v = (uint16_t)(bl[r][k.ofs - bx0] << 8);  // ofs = 0 (low border) or W-1 (high border)
        hr[r][c] = v;
    }
    __syncthreads();
    for (int i = tid; i < nx * ny; i += 256) {  // vertical resize
        int r, c;
        fastdiv(dn, i, r, c);
        const LinCoef k = cy[y0 + r];
        uint8_t v;
        if (k.mode == 0) v = (uint8_t)((hr[k.ofs - by0][c] * (256u - k.c1) + hr[k.ofs - by0 + 1][c] * (uint32_t)k.c1 + 32768u) >> 16);
        else v = (uint8_t)((hr[k.ofs - by0][c] + 128) >> 8);
        sc[r][c] = v;
    }
    __syncthreads();
    int lmax = 0;
    for (int i = tid; i < kPW * kPH; i += 256) {
        const int r = i / kPW, c = i - r * kPW;
        const int x = x0 + c, y = y0 + r;
        if (x >= sw || y >= sh) continue;
        LsdPix p;
        p.ang = LSD_NOTDEF; p.c = 0.f; p.s = 0.f; p.gxgy = 0;
        uint32_t key = 0u;   // gx^2 + gy^2 of a defined pixel, 0 otherwise: all k_lsd_order needs (4 instead of 16 bytes per pixel)
        if (x < sw - 1 && y < sh - 1) {
            const int DA = sc[r + 1][c + 1] - sc[r][c], BC = sc[r][c + 1] - sc[r + 1][c];
            const int gx = DA + BC, gy = DA - BC;
            const int sq = gx * gx + gy * gy;
            p.gxgy = (gx & 0xffff) | (gy << 16);
            // modgrad = sqrt(sq / 4.0) <= rho  <=>  sq <= sq_low_max (the largest integer for which the reference's double test holds)
            if (sq > sq_low_max) {
                p.ang = fast_atan2_deg((float)gx, (float)-gy);
                const float2 cs = __ldg(&cstab[(gx + 510) * 1021 + (gy + 510)]);
                p.c = cs.x; p.s = cs.y;
                lmax = max(lmax, sq);
                key = (uint32_t)sq;
            }
        }
        const long long o = (long long)f * sw * sh + (long long)y * sw + x;
        pix[o] = p;
        sqkey[o] = key;
        if (scaled_out) scaled_out[o] = sc[r][c];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lmax = max(lmax, __shfl_xor_sync(kFull, lmax, o));
    if ((tid & 31) == 0 && lmax > 0) atomicMax(&s_max, lmax);
    __syncthreads();
    if (tid == 0 && s_max > 0) atomicMax(&maxsq[f], s_max);
}

// --------------------------------------------------------------------------------------------------------------------
// Seed order = cv::LineSegmentDetector's ordered_points restricted to the defined pixels: bin = int(modgrad * 1023 /
// max_grad), descending; scan order inside a bin.  (Undefined pixels are skipped by the seed loop, so they are not listed.)
static const int kOrdWarps = 32, kBins = 1024;

// `key` (written by k_lsd_prep; the region buffer of k_lsd_grow, unused until then): gx^2 + gy^2 per defined pixel, 0 otherwise.  The
// counting pass replaces it in place by bin + 1, which the scatter pass reads back: the 16-byte pixel records are not touched and the
// double-precision square root runs once per pixel.
__device__ __forceinline__ int lsd_bin(uint32_t sq, double bin_coef) {
    return (int)(sqrt((double)(int)sq / 4.0) * bin_coef);
}

__global__ void __launch_bounds__(1024) k_lsd_order(uint32_t* __restrict__ key, int npix, const int* __restrict__ maxsq,
                                                     uint32_t* __restrict__ order, int* __restrict__ norder) {
    extern __shared__ uint32_t hist[];  // [kOrdWarps][kBins]
    __shared__ uint32_t s_warp[32];
    const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    uint32_t* K = key + (long long)f * npix;
    uint32_t* out = order + (long long)f * npix;
    const int mq = maxsq[f];
    if (mq <= 0) { if (tid == 0) norder[f] = 0; return; }
    const double bin_coef = (double)(kBins - 1) / sqrt((double)mq / 4.0);
    for (int i = tid; i < kOrdWarps * kBins; i += 1024) hist[i] = 0;
    __syncthreads();
    const int seg = (npix + kOrdWarps - 1) / kOrdWarps, s0 = wid * seg, s1 = min(npix, s0 + seg);
    uint32_t* myh = hist + wid * kBins;
    // four loads in flight per lane: with one CTA per SM the passes are bound by memory-level parallelism, not by bandwidth
    for (int i = s0 + lane; i < s1; i += 128) {
        uint32_t q[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) q[u] = (i + 32 * u < s1) ? K[i + 32 * u] : 0u;
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (q[u]) { const int bin = lsd_bin(q[u], bin_coef); atomicAdd(&myh[bin], 1u); K[i + 32 * u] = (uint32_t)bin + 1u; }
    }
    __syncthreads();
    {   // thread t owns bin (kBins-1-t): descending bins <-> ascending t
        const int b = kBins - 1 - tid;
        uint32_t run = 0;
        for (int w = 0; w < kOrdWarps; ++w) { const uint32_t c = hist[w * kBins + b]; hist[w * kBins + b] = run; run += c; }
        // exclusive scan of the bin totals over tid
        uint32_t v = run;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t n = __shfl_up_sync(kFull, v, o); if (lane >= o) v += n; }
        if (lane == 31) s_warp[wid] = v;
        __syncthreads();
        if (wid == 0) {
            uint32_t wv = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const uint32_t n = __shfl_up_sync(kFull, wv, o); if (lane >= o) wv += n; }
            s_warp[lane] = wv;
        }
        __syncthreads();
        const uint32_t base = v - run + (wid ? s_warp[wid - 1] : 0);
        if (tid == 1023) norder[f] = (int)(base + run);
        for (int w = 0; w < kOrdWarps; ++w) hist[w * kBins + b] += base;
    }
    __syncthreads();
    for (int i0 = s0; i0 < s1; i0 += 128) {
        int bins[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { const int i = i0 + 32 * u + lane; bins[u] = (i < s1) ? (int)K[i] - 1 : -1; }
#pragma unroll
        for (int u = 0; u < 4; ++u) {   // scan order inside a bin: the four groups of 32 pixels go in order
            const int bin = bins[u];
            if (!__any_sync(kFull, bin >= 0)) continue;
            const unsigned peers = __match_any_sync(kFull, bin);
            uint32_t pos = 0;
            if (bin >= 0) pos = myh[bin] + __popc(peers & ((1u << lane) - 1u));
            __syncwarp();
            if (bin >= 0) {
                out[pos] = (uint32_t)(i0 + 32 * u + lane);
                if ((int)(__ffs(peers) - 1) == lane) myh[bin] += __popc(peers);
            }
            __syncwarp();
        }
    }
}

// --------------------------------------------------------------------------------------------------------------------
struct LsdRect { double x1, y1, x2, y2, width; };

__device__ __forceinline__ bool lsd_aligned(double theta, double a, double prec) {
    double n = theta - a;
    if (n < 0) n = -n;
    if (n > LSD_32PI) { n -= LSD_2PI; if (n < 0) n = -n; }
    return n <= prec;
}
__device__ __forceinline__ double lsd_angle_diff_signed(double a, double b) {
    double d = a - b;
    while (d <= -LSD_PI) d += LSD_2PI;
    while (d > LSD_PI) d -= LSD_2PI;
    return d;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(kFull, v, o));
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(kFull, v, o));
    return v;
}
__device__ __forceinline__ bool used_get(const uint32_t* used, int i) { return (used[i >> 5] >> (i & 31)) & 1u; }
__device__ __forceinline__ double lsd_modgrad(int gxgy) {
    const int gx = (int)(short)(gxgy & 0xffff), gy = gxgy >> 16;
    return sqrt((double)(gx * gx + gy * gy) / 4.0);
}

// LineSegmentDetectorImpl::region_grow.  Warp-collective; returns the region size, reg[] holds x | y << 16.
static const int kRing = 256;  // most recent region points, kept in shared memory (the frontier is read from here)

__device__ __forceinline__ void lsd_prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
// a pixel joined the region: it will be a centre a few steps from now; pull the records of its 3x3 neighbourhood into L1
__device__ __forceinline__ void lsd_prefetch_nbhd(const LsdPix* __restrict__ pix, int w, int h, int xx, int yy) {
    const int x0 = max(xx - 1, 0), x1 = min(xx + 1, w - 1);
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy) {
        const int y = yy + dy;
        if (y < 0 || y >= h) continue;
        lsd_prefetch_l1(pix + y * w + x0);
        lsd_prefetch_l1(pix + y * w + x1);
    }
}

__device__ int lsd_region_grow(const LsdPix* __restrict__ pix, volatile uint32_t* reg, volatile uint32_t* ring, uint32_t* used, int w,
                               int h, uint32_t seed_xy, double prec, double& reg_angle_out, int lane) {
    const int si = (int)(seed_xy >> 16) * w + (int)(seed_xy & 0xffff);
    const LsdPix sp = pix[si];
    double reg_angle = (double)sp.ang * LSD_DEG2RAD;
    float sumdx = (float)cos(reg_angle), sumdy = (float)sin(reg_angle);
    if (lane == 0) { reg[0] = seed_xy; ring[0] = seed_xy; used[si >> 5] |= 1u << (si & 31); }
    __syncwarp();
    int n = 1, i = 0;
    const int cidx = lane / 9, k = lane - cidx * 9;
    const int ddy = k / 3 - 1, ddx = k - (k / 3) * 3 - 1;
    while (i < n) {
        const int nb = min(3, n - i);
        bool def = false, isused = true;
        int xx = 0, yy = 0, ni = -1;
        LsdPix p;
        p.ang = LSD_NOTDEF; p.c = 0.f; p.s = 0.f;
        if (cidx < nb && k != 4) {
            const int ci = i + cidx;
            const uint32_t c = (n - ci <= kRing) ? ring[ci & (kRing - 1)] : reg[ci];
            xx = (int)(c & 0xffff) + ddx; yy = (int)(c >> 16) + ddy;
            if (xx >= 0 && yy >= 0 && xx < w && yy < h) {
                ni = yy * w + xx;
                // record and `used` bit are requested together; pixels accepted later in this step are tracked in `isused` below,
                // so the bitmap is not read again after the record has arrived
                isused = used_get(used, ni);
                p = pix[ni];
                def = p.ang != LSD_NOTDEF;
            }
        }
        const double a = (double)p.ang * LSD_DEG2RAD;
        for (int c = 0; c < nb; ++c) {
            const bool cand = def && cidx == c && !isused;
            unsigned pending = __ballot_sync(kFull, cand);
            while (pending) {
                const bool al = cand && lsd_aligned(reg_angle, a, prec);
                const unsigned m = __ballot_sync(kFull, al) & pending;
                if (!m) break;
                const int j = __ffs(m) - 1;
                if (lane == j) {
                    const uint32_t packed = (uint32_t)xx | ((uint32_t)yy << 16);
                    used[ni >> 5] |= 1u << (ni & 31);
                    reg[n] = packed;
                    ring[n & (kRing - 1)] = packed;
                    lsd_prefetch_nbhd(pix, w, h, xx, yy);
                }
                if (ni == __shfl_sync(kFull, ni, j)) isused = true;  // the same pixel seen from a later centre of this step
                const float cs = __shfl_sync(kFull, p.c, j), sn = __shfl_sync(kFull, p.s, j);
                sumdx = __fadd_rn(sumdx, cs);
                sumdy = __fadd_rn(sumdy, sn);
                reg_angle = (double)fast_atan2_deg(sumdy, sumdx) * LSD_DEG2RAD;
                ++n;
                pending &= ~((2u << j) - 1u);
            }
            __syncwarp();
        }
        i += nb;
    }
    reg_angle_out = reg_angle;
    return n;
}

// region2rect + get_theta.  Sums are warp reductions (summation order differs from the sequential reference by
// rounding only; every decision downstream is made on the same formulas).
__device__ void lsd_region2rect(const LsdPix* __restrict__ pix, const volatile uint32_t* reg, int n, int w, double reg_angle, double prec,
                                LsdRect& rec, int lane) {
    double x = 0, y = 0, sum = 0;
    for (int i = lane; i < n; i += 32) {
        const uint32_t c = reg[i];
        const int px = c & 0xffff, py = c >> 16;
        const double wt = lsd_modgrad(pix[py * w + px].gxgy);
        x += (double)px * wt; y += (double)py * wt; sum += wt;
    }
    x = warp_sum(x); y = warp_sum(y); sum = warp_sum(sum);
    x /= sum; y /= sum;
    double Ixx = 0, Iyy = 0, Ixy = 0;
    for (int i = lane; i < n; i += 32) {
        const uint32_t c = reg[i];
        const int px = c & 0xffff, py = c >> 16;
        const double wt = lsd_modgrad(pix[py * w + px].gxgy);
        const double dx = (double)px - x, dy = (double)py - y;
        Ixx += dy * dy * wt; Iyy += dx * dx * wt; Ixy -= dx * dy * wt;
    }
    Ixx = warp_sum(Ixx); Iyy = warp_sum(Iyy); Ixy = warp_sum(Ixy);
    const double lambda = 0.5 * (Ixx + Iyy - sqrt((Ixx - Iyy) * (Ixx - Iyy) + 4.0 * Ixy * Ixy));
    double theta = (fabs(Ixx) > fabs(Iyy)) ? (double)fast_atan2_deg((float)(lambda - Ixx), (float)Ixy)
                                           : (double)fast_atan2_deg((float)Ixy, (float)(lambda - Iyy));
    theta *= LSD_DEG2RAD;
    if (fabs(lsd_angle_diff_signed(theta, reg_angle)) > prec) theta += LSD_PI;
    const double dx = cos(theta), dy = sin(theta);
    double l_min = 0, l_max = 0, w_min = 0, w_max = 0;
    for (int i = lane; i < n; i += 32) {
        const uint32_t c = reg[i];
        const double rx = (double)(int)(c & 0xffff) - x, ry = (double)(int)(c >> 16) - y;
        const double l = rx * dx + ry * dy, ww = -rx * dy + ry * dx;
        l_max = fmax(l_max, l); l_min = fmin(l_min, l);
        w_max = fmax(w_max, ww); w_min = fmin(w_min, ww);
    }
    l_max = warp_max(l_max); l_min = warp_min(l_min); w_max = warp_max(w_max); w_min = warp_min(w_min);
    rec.x1 = x + l_min * dx; rec.y1 = y + l_min * dy; rec.x2 = x + l_max * dx; rec.y2 = y + l_max * dy;
    rec.width = w_max - w_min;
    if (rec.width < 1.0) rec.width = 1.0;
}

__device__ __forceinline__ double lsd_density(int n, const LsdRect& r) {
    const double dx = r.x2 - r.x1, dy = r.y2 - r.y1;
    return (double)n / (sqrt(dx * dx + dy * dy) * r.width);
}

#ifndef HVO_GROW_MINBLOCKS
#define HVO_GROW_MINBLOCKS 32  /* 64 registers, no spills: 32 resident warps per SM instead of 24 */
#endif
__global__ void __launch_bounds__(32, HVO_GROW_MINBLOCKS) k_lsd_grow(const LsdPix* __restrict__ pix, int w, int h, const uint32_t* __restrict__ order,
                                                 const int* __restrict__ norder, uint32_t* __restrict__ regbuf, int min_reg_size,
                                                 double prec, double density_th, double inv_scale_div, float* __restrict__ seg,
                                                 int seg_cap, int* __restrict__ nseg, uint32_t* __restrict__ usedbuf) {
    __shared__ uint32_t ring[kRing];
    const int f = blockIdx.x, lane = threadIdx.x;
    const int npix = w * h;
    // `used` map: one bit per pixel in global memory (L1/L2 resident, touched only around the growing region).  Keeping it
    // out of shared memory lets 32 frames share an SM and lets this latency-bound kernel co-reside with the other pipelines.
    uint32_t* used = usedbuf + (size_t)f * ((npix + 31) >> 5);
    const LsdPix* P = pix + (long long)f * npix;
    const uint32_t* ord = order + (long long)f * npix;
    volatile uint32_t* reg = regbuf + (long long)f * npix;
    float* out = seg + (long long)f * seg_cap * 4;
    const int nwords = (npix + 31) >> 5;
    for (int i = lane; i < nwords; i += 32) used[i] = 0;
    __syncwarp();
    const int no = norder[f];
    int ns = 0;
    for (int base = 0; base < no; base += 32) {
        const bool valid = base + lane < no;
        const uint32_t idx = valid ? ord[base + lane] : 0u;
        unsigned remaining = kFull;
        while (true) {
            const unsigned m = __ballot_sync(kFull, valid && !used_get(used, (int)idx)) & remaining;
            if (!m) break;
            const int j = __ffs(m) - 1;
            remaining &= ~((2u << j) - 1u);
            const uint32_t sidx = __shfl_sync(kFull, idx, j);
            const uint32_t seed = (sidx % (uint32_t)w) | ((sidx / (uint32_t)w) << 16);
            double reg_angle;
            int n = lsd_region_grow(P, reg, ring, used, w, h, seed, prec, reg_angle, lane);
            if (n < min_reg_size) continue;
            LsdRect rec;
            lsd_region2rect(P, reg, n, w, reg_angle, prec, rec, lane);
            bool ok = true;
            if (lsd_density(n, rec) < density_th) {
                // ---- refine: try a tighter angle tolerance around the seed ----
                const double xc = (double)(seed & 0xffff), yc = (double)(seed >> 16);
                const double ang_c = (double)P[sidx].ang * LSD_DEG2RAD;
                double sum = 0, s_sum = 0;
                int cnt = 0;
                for (int i = lane; i < n; i += 32) {
                    const uint32_t c = reg[i];
                    const int px = c & 0xffff, py = c >> 16, pi = py * w + px;
                    atomicAnd(&used[pi >> 5], ~(1u << (pi & 31)));
                    const double ddx = (double)px - xc, ddy = (double)py - yc;
                    if (sqrt(ddx * ddx + ddy * ddy) < rec.width) {
                        const double d = lsd_angle_diff_signed((double)P[pi].ang * LSD_DEG2RAD, ang_c);
                        sum += d; s_sum += d * d; ++cnt;
                    }
                }
                sum = warp_sum(sum); s_sum = warp_sum(s_sum);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(kFull, cnt, o);
                __syncwarp();
                const double mean_angle = sum / (double)cnt;
                const double tau = 2.0 * sqrt((s_sum - 2.0 * mean_angle * sum) / (double)cnt + mean_angle * mean_angle);
                n = lsd_region_grow(P, reg, ring, used, w, h, seed, tau, reg_angle, lane);
                if (n < 2) ok = false;
                if (ok) {
                    lsd_region2rect(P, reg, n, w, reg_angle, prec, rec, lane);
                    double density = lsd_density(n, rec);
                    if (density < density_th) {
                        // ---- reduce_region_radius ----
                        const double d1x = rec.x1 - xc, d1y = rec.y1 - yc, d2x = rec.x2 - xc, d2y = rec.y2 - yc;
                        const double r1 = d1x * d1x + d1y * d1y, r2 = d2x * d2x + d2y * d2y;
                        double rad_sq = r1 > r2 ? r1 : r2;
                        while (density < density_th) {
                            rad_sq *= 0.75 * 0.75;
                            int kept = 0;
                            for (int i0 = 0; i0 < n; i0 += 32) {
                                const int i = i0 + lane;
                                uint32_t c = 0;
                                bool keep = false;
                                if (i < n) {
                                    c = reg[i];
                                    const int px = c & 0xffff, py = c >> 16;
                                    const double ddx = (double)px - xc, ddy = (double)py - yc;
                                    keep = !(ddx * ddx + ddy * ddy > rad_sq);
                                    if (!keep) { const int pi = py * w + px; atomicAnd(&used[pi >> 5], ~(1u << (pi & 31))); }
                                }
                                const unsigned km = __ballot_sync(kFull, keep);
                                __syncwarp();
                                if (keep) reg[kept + __popc(km & ((1u << lane) - 1u))] = c;
                                kept += __popc(km);
                                __syncwarp();
                            }
                            n = kept;
                            if (n < 2) { ok = false; break; }
                            lsd_region2rect(P, reg, n, w, reg_angle, prec, rec, lane);
                            density = lsd_density(n, rec);
                        }
                    }
                }
            }
            if (!ok) continue;
            if (lane == 0 && ns < seg_cap) {
                out[4 * ns + 0] = (float)((rec.x1 + 0.5) / inv_scale_div);
                out[4 * ns + 1] = (float)((rec.y1 + 0.5) / inv_scale_div);
                out[4 * ns + 2] = (float)((rec.x2 + 0.5) / inv_scale_div);
                out[4 * ns + 3] = (float)((rec.y2 + 0.5) / inv_scale_div);
            }
            ++ns;
        }
    }
    if (lane == 0) nseg[f] = ns;
}

// --------------------------------------------------------------------------------------------------------------------
struct KeyLineOut {  // cv::line_descriptor::KeyLine POD, 68 bytes (hvo_keyline)
    float angle;
    int class_id, octave;
    float pt_x, pt_y, response, size;
    float startPointX, startPointY, endPointX, endPointY;
    float sPointInOctaveX, sPointInOctaveY, ePointInOctaveX, ePointInOctaveY;
    float lineLength;
    int numOfPixels;
};

__device__ __forceinline__ void lsd_clamp_extremes(float e[4], int W, int H) {  // checkLineExtremes, LSDDetector_custom.cpp:76-103
    if (e[0] < 0) e[0] = 0;
    if (e[0] >= W) e[0] = (float)W - 1.0f;
    if (e[2] < 0) e[2] = 0;
    if (e[2] >= W) e[2] = (float)W - 1.0f;
    if (e[1] < 0) e[1] = 0;
    if (e[1] >= H) e[1] = (float)H - 1.0f;
    if (e[3] < 0) e[3] = 0;
    if (e[3] >= H) e[3] = (float)H - 1.0f;
}
__device__ __forceinline__ float lsd_length(const float e[4]) {
    const double a = (double)__fsub_rn(e[0], e[2]), b = (double)__fsub_rn(e[1], e[3]);
    return (float)sqrt(a * a + b * b);
}

// Idx = uint16_t: the sorted index list and the ranks live in shared memory (seg_cap <= 65535, 4 bytes per possible segment).
// Idx = uint32_t: they live in `scratch` ([B][2 seg_cap] in global memory), for images whose segment bound exceeds either limit.
template <class Idx>
__global__ void __launch_bounds__(256) k_line_keylines(const float* __restrict__ seg, int seg_cap, const int* __restrict__ nseg, int W, int H,
                                                       int nfeat, int max_lines, float* __restrict__ resp, KeyLineOut* __restrict__ kls,
                                                       double* __restrict__ linevec, int32_t* __restrict__ counts, uint32_t* __restrict__ scratch) {
    const int f = blockIdx.x, tid = threadIdx.x;
    const int n = min(nseg[f], seg_cap);
    const float* S = seg + (long long)f * seg_cap * 4;
    float* R = resp + (long long)f * seg_cap;
    const bool select = n > nfeat;
    const float inv_max = (float)max(W, H);
    if (select) {
        for (int i = tid; i < n; i += 256) {
            float e[4] = {S[4 * i], S[4 * i + 1], S[4 * i + 2], S[4 * i + 3]};
            lsd_clamp_extremes(e, W, H);
            R[i] = __fdiv_rn(lsd_length(e), inv_max);
        }
        __syncthreads();
    }
    const int nout = select ? nfeat : n;
    if (tid == 0) counts[f] = min(nout, max_lines);
    // sort_lines_by_response (LineExtractor.cpp:351-360) is an unstable std::sort.  Without equal responses the result is the
    // plain descending rank (computed in parallel); with ties the order is libstdc++'s, replayed by one thread (std_sort.cuh).
    extern __shared__ uint16_t kl_sm[];   // [seg_cap] sorted index list, then [seg_cap] rank of every input line
    Idx* sidx;
    if constexpr (sizeof(Idx) == 2) sidx = kl_sm;
    else sidx = scratch + (long long)f * seg_cap * 2;
    Idx* srank = sidx + seg_cap;
    if (select) {
        int tie = 0;
        for (int i = tid; i < n; i += 256) {
            const float r = R[i];
            int rank = 0;
            for (int j = 0; j < n; ++j) { const float q = R[j]; rank += (q > r || (q == r && j < i)) ? 1 : 0; tie |= (q == r && j != i) ? 1 : 0; }
            srank[i] = (Idx)rank;
            sidx[i] = (Idx)i;
        }
        if (__syncthreads_or(tie)) {
            if (tid == 0) stdsort::sort(sidx, n, [R](Idx a, Idx b) { return R[a] > R[b]; });
            __syncthreads();
            for (int k = tid; k < n; k += 256) srank[sidx[k]] = (Idx)k;
            __syncthreads();
        }
    }
    for (int i = tid; i < n; i += 256) {
        int rank = i;
        if (select) {
            rank = srank[i];
            if (rank >= nfeat) continue;
        }
        if (rank >= max_lines) continue;
        float e[4] = {S[4 * i], S[4 * i + 1], S[4 * i + 2], S[4 * i + 3]};
        lsd_clamp_extremes(e, W, H);
        KeyLineOut kl;
        kl.startPointX = e[0]; kl.startPointY = e[1]; kl.endPointX = e[2]; kl.endPointY = e[3];  // octaveScale = pow(scale, 0) = 1
        kl.sPointInOctaveX = e[0]; kl.sPointInOctaveY = e[1]; kl.ePointInOctaveX = e[2]; kl.ePointInOctaveY = e[3];
        kl.lineLength = lsd_length(e);
        const int xa = __float2int_rn(e[0]), ya = __float2int_rn(e[1]), xb = __float2int_rn(e[2]), yb = __float2int_rn(e[3]);
        kl.numOfPixels = max(abs(xb - xa), abs(yb - ya)) + 1;  // cv::LineIterator(...).count, 8-connected, endpoints inside the image
        kl.angle = (float)atan2((double)__fsub_rn(e[3], e[1]), (double)__fsub_rn(e[2], e[0]));
        kl.class_id = rank;
        kl.octave = 0;
        kl.size = __fmul_rn(__fsub_rn(e[2], e[0]), __fsub_rn(e[3], e[1]));
        kl.response = __fdiv_rn(kl.lineLength, inv_max);
        kl.pt_x = __fdiv_rn(__fadd_rn(e[2], e[0]), 2.f);
        kl.pt_y = __fdiv_rn(__fadd_rn(e[3], e[1]), 2.f);
        kls[(long long)f * max_lines + rank] = kl;
        // lineVec2d (LineExtractor.cpp:365-377): (sp x ep) / sqrt(l0^2 + l1^2), doubles
        const double sx = e[0], sy = e[1], ex = e[2], ey = e[3];
        const double l0 = sy - ey, l1 = ex - sx, l2 = sx * ey - sy * ex;
        const double nn = sqrt(l0 * l0 + l1 * l1);
        double* lv = linevec + ((long long)f * max_lines + rank) * 3;
        lv[0] = l0 / nn; lv[1] = l1 / nn; lv[2] = l2 / nn;
    }
}


// --------------------------------------------------------------------------------------------------------------------
// Frame::cullingLine (reference src/Frame.cc:952-1116): merge near-collinear KeyLines, rebuild the KeyLines, sort by
// response.  One warp per frame.  Pair tests of one leader i run 32 candidates j at a time (a candidate's outcome depends
// only on tags set by earlier leaders); the per-line terms of PointLineDistance (:1117-1126) and TwoLineAngle
// (:1127-1140) are computed once per line with the reference's own operation order.  Each group is then folded with
// MergeTwoLines (:1141-1203) by one lane.  The LBD pass on the new KeyLines (:1094-1096) follows on the same stream.
struct CullLine {  // per input line: 72 bytes
    double A, B, C, den;   // (y2 - y1), (x1 - x2), (x2 y1 - x1 y2), sqrt((y2 - y1)^2 + (x1 - x2)^2)
    double a0, a1, nrm;    // line function after the two divisions by its third component; its norm
    float m12x, m12y, m21x, m21y;  // (start + end) / 2 and (end + start) / 2 + start (sic, :975)
};

__device__ __forceinline__ void cull_merge_two(const float l1[4], const float l2[4], float out[4]) {  // MergeTwoLines
    const float ax = l1[0], ay = l1[1], bx = l1[2], by = l1[3];
    const float cx = l2[0], cy = l2[1], dx = l2[2], dy = l2[3];
    const float dlix = __fsub_rn(bx, ax), dliy = __fsub_rn(by, ay), dljx = __fsub_rn(dx, cx), dljy = __fsub_rn(dy, cy);
    const double li = sqrt((double)__fmul_rn(dlix, dlix) + (double)__fmul_rn(dliy, dliy));
    const double lj = sqrt((double)__fmul_rn(dljx, dljx) + (double)__fmul_rn(dljy, dljy));
    const double xg = (li * (double)__fadd_rn(ax, bx) + lj * (double)__fadd_rn(cx, dx)) / (2.0 * (li + lj));
    const double yg = (li * (double)__fadd_rn(ay, by) + lj * (double)__fadd_rn(cy, dy)) / (2.0 * (li + lj));
    const double kPi = 3.1415926535897932384626433832795;
    double thi, thj, thr;
    if (dlix == 0.0f) thi = kPi / 2.0;
    // the reference's atan(float) binds to the float overload (Frame.cc:33 'using namespace std'): a float-precision angle.
    // Here: the correctly rounded float (libm's atanf is within 1 ulp of it, not pinned by the reference).
    else thi = (double)(float)atan((double)__fdiv_rn(dliy, dlix));
    if (dljx == 0.0f) thj = kPi / 2.0;
    else thj = (double)(float)atan((double)__fdiv_rn(dljy, dljx));
    if (fabs(thi - thj) <= kPi / 2.0) {
        thr = (li * thi + lj * thj) / (li + lj);
    } else {
        const double tmp = thj - kPi * (thj / fabs(thj));
        thr = li * thi + lj * tmp;
        thr /= (li + lj);
    }
    const double s = sin(thr), c = cos(thr);
    const double axg = ((double)ay - yg) * s + ((double)ax - xg) * c;
    const double bxg = ((double)by - yg) * s + ((double)bx - xg) * c;
    const double cxg = ((double)cy - yg) * s + ((double)cx - xg) * c;
    const double dxg = ((double)dy - yg) * s + ((double)dx - xg) * c;
    const double d1 = fmin(axg, fmin(bxg, fmin(cxg, dxg)));
    const double d2 = fmax(axg, fmax(bxg, fmax(cxg, dxg)));
    out[0] = (float)(d1 * c + xg);
    out[1] = (float)(d1 * s + yg);
    out[2] = (float)(d2 * c + xg);
    out[3] = (float)(d2 * s + yg);
}

// cv::clipLine on 64-bit points (OpenCV imgproc drawing.cpp, un-vendored; the oracle's restatement is pinned to cv2)
__device__ bool cull_clip_line(long long width, long long height, long long& x1, long long& y1, long long& x2, long long& y2) {
    const long long right = width - 1, bottom = height - 1;
    int c1 = (x1 < 0) + (x1 > right) * 2 + (y1 < 0) * 4 + (y1 > bottom) * 8;
    int c2 = (x2 < 0) + (x2 > right) * 2 + (y2 < 0) * 4 + (y2 > bottom) * 8;
    if ((c1 & c2) == 0 && (c1 | c2) != 0) {
        long long a;
        if (c1 & 12) {
            a = c1 < 8 ? 0 : bottom;
            x1 += (long long)((double)(a - y1) * (double)(x2 - x1) / (double)(y2 - y1));
            y1 = a;
            c1 = (x1 < 0) + (x1 > right) * 2;
        }
        if (c2 & 12) {
            a = c2 < 8 ? 0 : bottom;
            x2 += (long long)((double)(a - y2) * (double)(x2 - x1) / (double)(y2 - y1));
            y2 = a;
            c2 = (x2 < 0) + (x2 > right) * 2;
        }
        if ((c1 & c2) == 0 && (c1 | c2) != 0) {
            if (c1) {
                a = c1 == 1 ? 0 : right;
                y1 += (long long)((double)(a - x1) * (double)(y2 - y1) / (double)(x2 - x1));
                x1 = a;
                c1 = 0;
            }
            if (c2) {
                a = c2 == 1 ? 0 : right;
                y2 += (long long)((double)(a - x2) * (double)(y2 - y1) / (double)(x2 - x1));
                x2 = a;
                c2 = 0;
            }
        }
    }
    return (c1 | c2) == 0;
}
__device__ int cull_line_count(int W, int H, const float e[4]) {  // cv::LineIterator(img, Point(p1), Point(p2)).count, 8-connected
    long long x1 = __float2int_rn(e[0]), y1 = __float2int_rn(e[1]), x2 = __float2int_rn(e[2]), y2 = __float2int_rn(e[3]);
    if ((unsigned long long)x1 >= (unsigned long long)W || (unsigned long long)x2 >= (unsigned long long)W ||
        (unsigned long long)y1 >= (unsigned long long)H || (unsigned long long)y2 >= (unsigned long long)H) {
        if (!cull_clip_line(W, H, x1, y1, x2, y2)) return 0;
    }
    const long long dx = x2 > x1 ? x2 - x1 : x1 - x2, dy = y2 > y1 ? y2 - y1 : y1 - y2;
    return (int)(dx > dy ? dx : dy) + 1;
}

__global__ void __launch_bounds__(32) k_line_cull(KeyLineOut* __restrict__ kls, double* __restrict__ linevec, int32_t* __restrict__ counts,
                                                 int max_lines, int W, int H, double dis, double cos_th, double endpoint_dis,
                                                 CullLine* __restrict__ scratch, float* __restrict__ newline) {
    extern __shared__ int16_t cull_sm[];  // grp[max_lines] (leader of a merged line, -1 none), then tag bytes
    int16_t* grp = cull_sm;
    uint8_t* tag = (uint8_t*)(cull_sm + 2 * max_lines);
    const int f = blockIdx.x, lane = threadIdx.x;
    const int n = min(counts[f], max_lines);
    KeyLineOut* K = kls + (long long)f * max_lines;
    double* LV = linevec + (long long)f * max_lines * 3;
    CullLine* S = scratch + (long long)f * max_lines;
    float* NL = newline + (long long)f * max_lines * 5;  // x1 y1 x2 y2 response
    for (int i = lane; i < n; i += 32) {
        const KeyLineOut k = K[i];
        CullLine c;
        const double x1 = k.startPointX, y1 = k.startPointY, x2 = k.endPointX, y2 = k.endPointY;
        c.A = y2 - y1; c.B = x1 - x2; c.C = (x2 * y1) - (x1 * y2);
        c.den = sqrt((y2 - y1) * (y2 - y1) + (x1 - x2) * (x1 - x2));
        double v0 = LV[3 * i], v1 = LV[3 * i + 1];
        const double v2 = LV[3 * i + 2];
        v0 /= v2; v1 /= v2;
        c.a0 = v0 / v2; c.a1 = v1 / v2;
        c.nrm = sqrt(c.a0 * c.a0 + c.a1 * c.a1);
        c.m12x = __fmul_rn(__fadd_rn(k.startPointX, k.endPointX), 0.5f);
        c.m12y = __fmul_rn(__fadd_rn(k.startPointY, k.endPointY), 0.5f);
        c.m21x = __fadd_rn(__fmul_rn(__fadd_rn(k.endPointX, k.startPointX), 0.5f), k.startPointX);
        c.m21y = __fadd_rn(__fmul_rn(__fadd_rn(k.endPointY, k.startPointY), 0.5f), k.startPointY);
        S[i] = c;
        grp[i] = -1; tag[i] = 0;
    }
    __syncwarp();
    // ---- step 1: pair tests ----
    for (int i = 0; i < n; ++i) {
        if (tag[i]) continue;  // warp-uniform (shared memory)
        const CullLine ci = S[i];
        const KeyLineOut ki = K[i];
        bool any = false;
        for (int base = i + 1; base < n; base += 32) {
            const int j = base + lane;
            bool hit = false;
            if (j < n && !tag[j]) {
                const CullLine cj = S[j];
                const double dis12 = fabs(cj.A * (double)ci.m12x + cj.B * (double)ci.m12y + cj.C) / cj.den;
                const double dis21 = fabs(ci.A * (double)cj.m21x + ci.B * (double)cj.m21y + ci.C) / ci.den;
                if (dis12 < dis || dis21 < dis) {
                    const double a = ci.a0 * cj.a0 + ci.a1 * cj.a1;
                    const double ang = fabs(a / (ci.nrm * cj.nrm));
                    if (fabs(ang) > cos_th) {
                        const KeyLineOut kj = K[j];
                        const double x11 = ki.startPointX, x12 = ki.endPointX, y11 = ki.startPointY, y12 = ki.endPointY;
                        const double x21 = kj.startPointX, x22 = kj.endPointX, y21 = kj.startPointY, y22 = kj.endPointY;
                        // sorted extents: [min, second, third, max] of the four x (y) coordinates
                        const double xlo1 = fmin(x11, x12), xhi1 = fmax(x11, x12), xlo2 = fmin(x21, x22), xhi2 = fmax(x21, x22);
                        const double ylo1 = fmin(y11, y12), yhi1 = fmax(y11, y12), ylo2 = fmin(y21, y22), yhi2 = fmax(y21, y22);
                        const double bx0 = fmin(xlo1, xlo2), bx3 = fmax(xhi1, xhi2), bx1 = fmin(fmax(xlo1, xlo2), fmin(xhi1, xhi2)),
                                     bx2 = fmax(fmax(xlo1, xlo2), fmin(xhi1, xhi2));
                        const double by0 = fmin(ylo1, ylo2), by3 = fmax(yhi1, yhi2), by1 = fmin(fmax(ylo1, ylo2), fmin(yhi1, yhi2)),
                                     by2 = fmax(fmax(ylo1, ylo2), fmin(yhi1, yhi2));
                        hit = true;
                        if (bx3 - bx0 > fabs(x11 - x12) + fabs(x21 - x22) && bx2 - bx1 > endpoint_dis) hit = false;
                        if (hit && by3 - by0 > fabs(y11 - y12) + fabs(y21 - y22) && by2 - by1 > endpoint_dis) hit = false;
                    }
                }
            }
            if (hit) { grp[j] = (int16_t)i; tag[j] = 1; }
            any |= __any_sync(kFull, hit);
        }
        if (any && lane == 0) { tag[i] = 1; grp[i] = (int16_t)i; }
        __syncwarp();
    }
    // ---- step 2: fold every group (one lane per leader), keep the untouched lines; output order = index order ----
    int nout = 0;
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        bool keep = false;
        float cur[4] = {0.f, 0.f, 0.f, 0.f};
        if (i < n) {
            const KeyLineOut k = K[i];
            cur[0] = k.startPointX; cur[1] = k.startPointY; cur[2] = k.endPointX; cur[3] = k.endPointY;
            if (grp[i] == i) {
                keep = true;
                for (int j = i + 1; j < n; ++j) {
                    if (grp[j] != i) continue;
                    const KeyLineOut kj = K[j];
                    const float y1[4] = {kj.startPointX, kj.startPointY, kj.endPointX, kj.endPointY};
                    float m[4];
                    cull_merge_two(cur, y1, m);
                    cur[0] = m[0]; cur[1] = m[1]; cur[2] = m[2]; cur[3] = m[3];
                }
            } else if (!tag[i]) {
                keep = true;
            }
        }
        const unsigned km = __ballot_sync(kFull, keep);
        if (keep) {
            const int o = nout + __popc(km & ((1u << lane) - 1u));
            const double a = (double)__fsub_rn(cur[0], cur[2]), b = (double)__fsub_rn(cur[1], cur[3]);
            const float len = (float)sqrt(a * a + b * b);
            NL[5 * o] = cur[0]; NL[5 * o + 1] = cur[1]; NL[5 * o + 2] = cur[2]; NL[5 * o + 3] = cur[3];
            NL[5 * o + 4] = __fdiv_rn(len, (float)max(W, H));
        }
        nout += __popc(km);
    }
    __syncwarp();
    // ---- step 3: KeyLines of the new segments at their response rank.  std::sort (Frame.cc:1087) is unstable: without equal
    //      responses the order is the plain descending rank; with ties it is libstdc++'s, replayed by one lane (std_sort.cuh) ----
    uint16_t* sidx = (uint16_t*)grp;                       // the group leaders are dead here: [max_lines] sorted index list
    uint16_t* srank = sidx + max_lines;                    // [max_lines] rank of every new line
    {
        int tie = 0;
        for (int i = lane; i < nout; i += 32) {
            const float r = NL[5 * i + 4];
            int rank = 0;
            for (int j = 0; j < nout; ++j) { const float q = NL[5 * j + 4]; rank += (q > r || (q == r && j < i)) ? 1 : 0; tie |= (q == r && j != i) ? 1 : 0; }
            srank[i] = (uint16_t)rank;
            sidx[i] = (uint16_t)i;
        }
        __syncwarp();
        if (__any_sync(0xffffffffu, tie)) {
            if (lane == 0) stdsort::sort(sidx, nout, [NL](uint16_t a, uint16_t b) { return NL[5 * a + 4] > NL[5 * b + 4]; });
            __syncwarp();
            for (int k = lane; k < nout; k += 32) srank[sidx[k]] = (uint16_t)k;
            __syncwarp();
        }
    }
    for (int i = lane; i < nout; i += 32) {
        const float e[4] = {NL[5 * i], NL[5 * i + 1], NL[5 * i + 2], NL[5 * i + 3]};
        const float r = NL[5 * i + 4];
        const int rank = srank[i];
        KeyLineOut kl;
        kl.startPointX = e[0]; kl.startPointY = e[1]; kl.endPointX = e[2]; kl.endPointY = e[3];
        kl.sPointInOctaveX = e[0]; kl.sPointInOctaveY = e[1]; kl.ePointInOctaveX = e[2]; kl.ePointInOctaveY = e[3];
        kl.lineLength = lsd_length(e);
        kl.octave = 0;
        kl.angle = (float)atan2((double)__fsub_rn(e[3], e[1]), (double)__fsub_rn(e[2], e[0]));  // reference: atan2f
        kl.size = __fmul_rn(__fsub_rn(e[2], e[0]), __fsub_rn(e[3], e[1]));
        kl.pt_x = __fdiv_rn(__fadd_rn(e[2], e[0]), 2.f);
        kl.pt_y = __fdiv_rn(__fadd_rn(e[3], e[1]), 2.f);
        kl.numOfPixels = cull_line_count(W, H, e);
        kl.response = r;
        kl.class_id = rank;
        K[rank] = kl;
        const double sx = e[0], sy = e[1], ex = e[2], ey = e[3];
        const double l0 = sy - ey, l1 = ex - sx, l2 = sx * ey - sy * ex;
        const double nn = sqrt(l0 * l0 + l1 * l1);
        LV[3 * rank] = l0 / nn; LV[3 * rank + 1] = l1 / nn; LV[3 * rank + 2] = l2 / nn;
    }
    if (lane == 0) counts[f] = nout;
}

}  // namespace hvo

using namespace hvo;

extern "C" {
int hvo_lbd_create(int width, int height, int max_batch, int max_lines, int device, hvo_lbd** out);
void hvo_lbd_destroy(hvo_lbd* h);
}

struct hvo_line {
    int device = 0, width = 0, height = 0, max_batch = 0, nfeat = 0;
    int sw = 0, sh = 0, seg_cap = 0, min_reg_size = 0;
    double rho = 0, prec = 0;
    int sq_low_max = 0;  // gradient threshold of LSD as an integer bound on gx^2 + gy^2
    cudaStream_t stream = nullptr;
    cudaEvent_t tev[2] = {nullptr, nullptr};
    cudaEvent_t sev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    bool profiling = false;
    float stage_ms[4] = {0, 0, 0, 0};
    hvo_lbd* lbd = nullptr;
    uint8_t* d_gray = nullptr;
    LinCoef *d_cx = nullptr, *d_cy = nullptr;
    float2* d_cstab = nullptr;
    LsdPix* d_pix = nullptr;
    uint8_t* d_scaled = nullptr;
    int* d_maxsq = nullptr;
    uint32_t *d_order = nullptr, *d_reg = nullptr, *d_used = nullptr;
    int *d_norder = nullptr, *d_nseg = nullptr;
    float *d_seg = nullptr, *d_resp = nullptr;
    KeyLineOut* d_kl = nullptr;
    double* d_linevec = nullptr;
    int32_t* d_counts = nullptr;
    uint8_t* d_desc = nullptr;
    bool cull = false;               // run Frame::cullingLine after the extractor (hvo_line_set_culling)
    CullLine* d_cull = nullptr;      // [B][nfeat]
    float* d_newline = nullptr;      // [B][nfeat][5]
    uint32_t* d_klscratch = nullptr; // [B][2 seg_cap]: k_line_keylines<uint32_t>'s index and rank lists (null: the uint16_t kernel)
    int last_launches = 0;
};

// cv::fastAtan2 on the host (this file is compiled with -ffp-contract=off: every operation individually rounded)
static float host_fast_atan2_deg(float y, float x) {
    const float scale = (float)(180.0 / kLsdPi);
    const float p1 = 0.9997878412794807f * scale, p3 = -0.3258083974640975f * scale, p5 = 0.1555786518463281f * scale,
                p7 = -0.04432655554792128f * scale;
    const float ax = std::fabs(x), ay = std::fabs(y);
    float a, c, c2;
    if (ax >= ay) { c = ay / (ax + (float)DBL_EPSILON); c2 = c * c; a = (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c; }
    else { c = ax / (ay + (float)DBL_EPSILON); c2 = c * c; a = 90.f - (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c; }
    if (x < 0) a = 180.f - a;
    if (y < 0) a = 360.f - a;
    return a;
}

static void lsd_exact_coeffs(int src, int dst, double inv_scale, std::vector<LinCoef>& out) {
    // cv::resize INTER_LINEAR_EXACT coefficient rule (8.8 fixed point): see oracle/lsd_oracle.cpp for the cv2 pin
    const double scale = 1.0 / inv_scale;
    out.resize(dst);
    for (int v = 0; v < dst; ++v) {
        const double f = scale * ((double)v + 0.5) - 0.5;
        const int i = (int)std::floor(f);
        LinCoef c{0, 0, 1};
        if (i >= 0 && src > 1) {
            if (i < src - 1) { c.ofs = i; c.c1 = (uint16_t)std::lrint((f - (double)i) * 256.0); c.mode = 0; }
            else { c.ofs = src - 1; c.mode = 2; }
        }
        out[v] = c;
    }
}

static int line_detect_device(hvo_line* h, const uint8_t* d_gray, int nframes) {
    const int npix = h->sw * h->sh;
    cudaStream_t s = h->stream;
    if (h->profiling) cudaEventRecord(h->sev[0], s);
    HVO_CUDA(cudaMemsetAsync(h->d_maxsq, 0, (size_t)nframes * sizeof(int), s));
    timeline_mark(s, "k_lsd_prep");
    k_lsd_prep<<<dim3(div_up(h->sw, kPW), div_up(h->sh, kPH), nframes), 256, 0, s>>>(
        d_gray, h->width, h->height, (long long)h->width * h->height, h->sw, h->sh, h->d_cx, h->d_cy, h->d_cstab, h->sq_low_max, h->d_pix,
        h->d_scaled, h->d_maxsq, h->d_reg);
    if (h->profiling) cudaEventRecord(h->sev[1], s);
    timeline_mark(s, "k_lsd_order");
    k_lsd_order<<<nframes, 1024, kOrdWarps * kBins * sizeof(uint32_t), s>>>(h->d_reg, npix, h->d_maxsq, h->d_order, h->d_norder);
    if (h->profiling) cudaEventRecord(h->sev[2], s);
    timeline_mark(s, "k_lsd_grow");
    k_lsd_grow<<<nframes, 32, 0, s>>>(h->d_pix, h->sw, h->sh, h->d_order, h->d_norder, h->d_reg, h->min_reg_size, h->prec, 0.7, 0.8,
                                      h->d_seg, h->seg_cap, h->d_nseg, h->d_used);
    if (h->profiling) cudaEventRecord(h->sev[3], s);
    h->last_launches = 3;
    HVO_CUDA(cudaGetLastError());
    return HVO_OK;
}

// Frame::cullingLine(im, 5, 2.5, 15, 30) (src/Frame.cc:939) on device-resident KeyLines, in place, then LBD on the result
static int line_cull_device(hvo_line* h, const uint8_t* d_gray, int nframes, KeyLineOut* d_kl, uint8_t* d_desc, double* d_linevec,
                            int32_t* d_counts) {
    const size_t sm = (size_t)h->nfeat * 5 + 16;   // grp int16 (reused as the sorted index list), rank u16, tag bytes
    timeline_mark(h->stream, "k_line_cull");
    k_line_cull<<<nframes, 32, sm, h->stream>>>(d_kl, d_linevec, d_counts, h->nfeat, h->width, h->height, 5.0, std::cos(2.5 * 0.0174533),
                                                15.0, h->d_cull, h->d_newline);
    HVO_CUDA(cudaGetLastError());
    return lbd_compute_on_stream(h->lbd, h->stream, d_gray, nframes, reinterpret_cast<const hvo_keyline*>(d_kl), d_counts, d_desc);
}

static int line_extract_device(hvo_line* h, const uint8_t* d_gray, int nframes, KeyLineOut* d_kl, uint8_t* d_desc, double* d_linevec,
                               int32_t* d_counts) {
    int st = line_detect_device(h, d_gray, nframes);
    if (st != HVO_OK) return st;
    if (h->d_klscratch) {
        timeline_mark(h->stream, "k_line_keylines<uint32_t>");
        k_line_keylines<uint32_t><<<nframes, 256, 0, h->stream>>>(h->d_seg, h->seg_cap, h->d_nseg, h->width, h->height, h->nfeat, h->nfeat, h->d_resp,
                                                                d_kl, d_linevec, d_counts, h->d_klscratch);
    } else {
        timeline_mark(h->stream, "k_line_keylines");
        k_line_keylines<uint16_t><<<nframes, 256, (size_t)h->seg_cap * 4, h->stream>>>(h->d_seg, h->seg_cap, h->d_nseg, h->width, h->height, h->nfeat, h->nfeat,
                                                                                h->d_resp, d_kl, d_linevec, d_counts, nullptr);
    }
    HVO_CUDA(cudaGetLastError());
    if (h->cull) {
        // the reference computes LBD twice (LineExtractor.cpp:361-363, Frame.cc:1094-1096) and discards the first result;
        // only the descriptors of the culled KeyLines survive, so only those are computed
        st = line_cull_device(h, d_gray, nframes, d_kl, d_desc, d_linevec, d_counts);
        h->last_launches = 8;
    } else {
        st = lbd_compute_on_stream(h->lbd, h->stream, d_gray, nframes, reinterpret_cast<const hvo_keyline*>(d_kl), d_counts, d_desc);
        h->last_launches = 7;
    }
    if (h->profiling) cudaEventRecord(h->sev[4], h->stream);
    return st;
}

namespace hvo {
cudaStream_t line_stream(hvo_line* h) { return h->stream; }  // internal: frame.cu chains the stages on events
const int* line_segment_counts(hvo_line* h) { return h->d_nseg; }  // internal: > line_segment_cap means the segment buffer overflowed
int line_segment_cap(hvo_line* h) { return h->seg_cap; }
}

extern "C" {

int hvo_line_create(const hvo_line_params* p, int width, int height, int max_batch, int device, hvo_line** out) {
    HVO_CHECK_ARG(out, "null out");
    *out = nullptr;
    HVO_CHECK_ARG(p, "null params");
    HVO_CHECK_ARG(width >= 16 && height >= 16 && width <= 8192 && height <= 8192, "image size out of range");
    HVO_CHECK_ARG(max_batch >= 1, "max_batch < 1");
    HVO_CHECK_ARG(p->n_features >= 1 && p->n_features <= 4096, "n_features out of range");
    HVO_CHECK_ARG(p->n_octaves == 1, "only LINE.nLevels = 1 is supported (every shipped YAML; see DESIGN.md)");
    int ndev = 0;
    HVO_CUDA(cudaGetDeviceCount(&ndev));
    if (ndev < 1) { set_error("no CUDA device: libhvofront has no CPU fallback"); return HVO_ERR_CUDA; }
    HVO_CHECK_ARG(device >= 0 && device < ndev, "device index out of range");
    hvo_line* h = new (std::nothrow) hvo_line();
    if (!h) { set_error("out of host memory"); return HVO_ERR_ARG; }
    h->device = device; h->width = width; h->height = height; h->max_batch = max_batch; h->nfeat = p->n_features;
    h->sw = (int)std::lrint((double)width * 0.8);
    h->sh = (int)std::lrint((double)height * 0.8);
    h->prec = kLsdPi * 22.5 / 180;
    h->rho = 2.0 / std::sin(h->prec);
    h->sq_low_max = -1;
    for (int sq = 0; sq <= 2 * 510 * 510 && std::sqrt((double)sq / 4.0) <= h->rho; ++sq) h->sq_low_max = sq;
    const double log_nt = 5 * (std::log10((double)h->sw) + std::log10((double)h->sh)) / 2 + std::log10(11.0);
    h->min_reg_size = (int)(size_t)(-log_nt / std::log10(22.5 / 180));
    h->seg_cap = ((h->sw - 1) * (h->sh - 1)) / (h->min_reg_size > 0 ? h->min_reg_size : 1) + 1;  // every segment owns >= min_reg_size pixels
    // test aid: a smaller segment buffer, to provoke HVO_ERR_OVERFLOW (the bound above cannot be exceeded by construction)
    if (const char* e = getenv("HVO_DEBUG_LINE_SEGCAP")) h->seg_cap = std::max(1, std::min(h->seg_cap, atoi(e)));
    std::vector<LinCoef> cx, cy;
    lsd_exact_coeffs(width, h->sw, 0.8, cx);
    lsd_exact_coeffs(height, h->sh, 0.8, cy);
    // cosf/sinf of float(angle) for every possible gradient (gx, gy in [-510, 510]): region_grow accumulates them in
    // float, and libm's cosf/sinf are not correctly rounded, so the table is built by the same libm the CPU path calls.
    std::vector<float2> tab((size_t)1021 * 1021);
    for (int gx = -510; gx <= 510; ++gx)
        for (int gy = -510; gy <= 510; ++gy) {
            const float fa = (float)((double)host_fast_atan2_deg((float)gx, (float)-gy) * (kLsdPi / 180));
            tab[(size_t)(gx + 510) * 1021 + (gy + 510)] = make_float2(cosf(fa), sinf(fa));
        }
    // the shared-memory tiles of k_lsd_prep are sized for the 0.8 scale; verify the source window of every tile fits
    for (int x0 = 0; x0 < h->sw; x0 += kPW) {
        const int x1 = std::min(x0 + kPW, h->sw - 1);
        if (std::min(cx[x1].ofs + 1, width - 1) - cx[x0].ofs + 1 + 4 > kSrcW) { set_error("internal: prep tile too wide"); delete h; return HVO_ERR_ARG; }
    }
    for (int y0 = 0; y0 < h->sh; y0 += kPH) {
        const int y1 = std::min(y0 + kPH, h->sh - 1);
        if (std::min(cy[y1].ofs + 1, height - 1) - cy[y0].ofs + 1 + 4 > kSrcH) { set_error("internal: prep tile too tall"); delete h; return HVO_ERR_ARG; }
    }
    int st = HVO_OK;
    do {
#define HVO_TRY(call) if ((call) != cudaSuccess) { set_error("%s: %s", #call, cudaGetErrorString(cudaGetLastError())); st = HVO_ERR_CUDA; break; }
        HVO_TRY(cudaSetDevice(device));
        pin_carveout(k_lsd_prep); pin_carveout(k_lsd_order); pin_carveout(k_lsd_grow); pin_carveout(k_line_keylines<uint16_t>); pin_carveout(k_line_keylines<uint32_t>);
        pin_carveout(k_line_cull);
        HVO_TRY(create_stream(&h->stream));
        for (auto& e : h->tev) HVO_TRY(cudaEventCreate(&e));
        if (st != HVO_OK) break;
        for (auto& e : h->sev) HVO_TRY(cudaEventCreate(&e));
        if (st != HVO_OK) break;
        const size_t B = (size_t)max_batch, px = (size_t)width * height, spx = (size_t)h->sw * h->sh, ml = (size_t)h->nfeat;
        HVO_TRY(cudaMalloc(&h->d_gray, B * px));
        HVO_TRY(cudaMalloc(&h->d_cx, cx.size() * sizeof(LinCoef)));
        HVO_TRY(cudaMalloc(&h->d_cy, cy.size() * sizeof(LinCoef)));
        HVO_TRY(cudaMalloc(&h->d_cstab, tab.size() * sizeof(float2)));
        HVO_TRY(cudaMalloc(&h->d_pix, B * spx * sizeof(LsdPix)));
        HVO_TRY(cudaMalloc(&h->d_scaled, B * spx));
        HVO_TRY(cudaMalloc(&h->d_maxsq, B * sizeof(int)));
        HVO_TRY(cudaMalloc(&h->d_order, B * spx * sizeof(uint32_t)));
        HVO_TRY(cudaMalloc(&h->d_reg, B * spx * sizeof(uint32_t)));
        HVO_TRY(cudaMalloc(&h->d_used, B * ((spx + 31) / 32) * sizeof(uint32_t)));
        HVO_TRY(cudaMalloc(&h->d_norder, B * sizeof(int)));
        HVO_TRY(cudaMalloc(&h->d_nseg, B * sizeof(int)));
        HVO_TRY(cudaMalloc(&h->d_seg, B * (size_t)h->seg_cap * 4 * sizeof(float)));
        HVO_TRY(cudaMalloc(&h->d_resp, B * (size_t)h->seg_cap * sizeof(float)));
        HVO_TRY(cudaMalloc(&h->d_kl, B * ml * sizeof(KeyLineOut)));
        HVO_TRY(cudaMalloc(&h->d_linevec, B * ml * 3 * sizeof(double)));
        HVO_TRY(cudaMalloc(&h->d_counts, B * sizeof(int32_t)));
        HVO_TRY(cudaMalloc(&h->d_desc, B * ml * 32));
        HVO_TRY(cudaMalloc(&h->d_cull, B * ml * sizeof(CullLine)));
        HVO_TRY(cudaMalloc(&h->d_newline, B * ml * 5 * sizeof(float)));
        HVO_TRY(cudaMemcpy(h->d_cx, cx.data(), cx.size() * sizeof(LinCoef), cudaMemcpyHostToDevice));
        HVO_TRY(cudaMemcpy(h->d_cy, cy.data(), cy.size() * sizeof(LinCoef), cudaMemcpyHostToDevice));
        HVO_TRY(cudaMemcpy(h->d_cstab, tab.data(), tab.size() * sizeof(float2), cudaMemcpyHostToDevice));
        HVO_TRY(cudaFuncSetAttribute(k_lsd_order, cudaFuncAttributeMaxDynamicSharedMemorySize, kOrdWarps * kBins * (int)sizeof(uint32_t)));
        {   // k_line_keylines<uint16_t> keeps two u16 per possible segment in shared memory; the attribute is per function: only ever
            // raise it.  Beyond 65535 segments or 200 KB, k_line_keylines<uint32_t> keeps two u32 per possible segment in global memory.
            static size_t s_kl_smem_max[64] = {0};
            const size_t want = std::max<size_t>((size_t)h->seg_cap * 4, 48 * 1024);
            if (want > 200 * 1024 || h->seg_cap > 65535) {
                HVO_TRY(cudaMalloc(&h->d_klscratch, B * (size_t)h->seg_cap * 2 * sizeof(uint32_t)));
            } else if (device < 64 && want > s_kl_smem_max[device]) {
                HVO_TRY(cudaFuncSetAttribute(k_line_keylines<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)want));
                s_kl_smem_max[device] = want;
            }
        }
#undef HVO_TRY
    } while (0);
    if (st == HVO_OK) st = hvo_lbd_create(width, height, max_batch, h->nfeat, device, &h->lbd);
    if (st != HVO_OK) { hvo_line_destroy(h); return st; }
    *out = h;
    return HVO_OK;
}

void hvo_line_destroy(hvo_line* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->lbd) hvo_lbd_destroy(h->lbd);
    void* bufs[] = {h->d_gray, h->d_cx, h->d_cy, h->d_cstab, h->d_pix, h->d_scaled, h->d_maxsq, h->d_order, h->d_reg, h->d_used, h->d_norder,
                    h->d_nseg, h->d_seg, h->d_resp, h->d_kl, h->d_linevec, h->d_counts, h->d_desc, h->d_cull, h->d_newline, h->d_klscratch};
    for (void* b : bufs) if (b) cudaFree(b);
    for (auto& e : h->tev) if (e) cudaEventDestroy(e);
    for (auto& e : h->sev) if (e) cudaEventDestroy(e);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int hvo_line_set_culling(hvo_line* h, int enable) {
    HVO_CHECK_ARG(h, "null handle");
    h->cull = enable != 0;
    return HVO_OK;
}

int hvo_line_cull_batch_device(hvo_line* h, const uint8_t* d_gray, int nframes, hvo_keyline* d_keylines, uint8_t* d_desc, double* d_linevec3,
                               int32_t* d_counts) {
    HVO_CHECK_ARG(h && d_gray && d_keylines && d_desc && d_linevec3 && d_counts, "null argument");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch, "nframes out of range for this handle");
    HVO_CUDA(cudaSetDevice(h->device));
    return line_cull_device(h, d_gray, nframes, reinterpret_cast<KeyLineOut*>(d_keylines), d_desc, d_linevec3, d_counts);
}

int hvo_line_cull(hvo_line* h, const uint8_t* gray, size_t stride, hvo_keyline* keylines, double* linevec3, int n, uint8_t* desc,
                  int* n_out) {
    HVO_CHECK_ARG(h && n_out, "null argument");
    *n_out = 0;
    if (!gray || n <= 0) return HVO_OK;
    HVO_CHECK_ARG(keylines && linevec3 && desc, "null argument");
    HVO_CHECK_ARG(stride >= (size_t)h->width, "stride smaller than width");
    HVO_CHECK_ARG(n <= h->nfeat, "more KeyLines than hvo_line_max_lines()");
    HVO_CUDA(cudaSetDevice(h->device));
    const int32_t cnt_in = n;
    HVO_CUDA(cudaMemcpy2DAsync(h->d_gray, h->width, gray, stride, h->width, h->height, cudaMemcpyHostToDevice, h->stream));
    HVO_CUDA(cudaMemcpyAsync(h->d_kl, keylines, (size_t)n * sizeof(KeyLineOut), cudaMemcpyHostToDevice, h->stream));
    HVO_CUDA(cudaMemcpyAsync(h->d_linevec, linevec3, (size_t)n * 3 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    HVO_CUDA(cudaMemcpyAsync(h->d_counts, &cnt_in, sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    int st = line_cull_device(h, h->d_gray, 1, h->d_kl, h->d_desc, h->d_linevec, h->d_counts);
    if (st != HVO_OK) return st;
    int32_t cnt = 0, nseg = 0;
    HVO_CUDA(cudaMemcpyAsync(&cnt, h->d_counts, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaMemcpyAsync(&nseg, h->d_nseg, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    if (nseg > h->seg_cap) { set_error("LSD segment buffer overflow (%d segments, capacity %d)", nseg, h->seg_cap); return HVO_ERR_OVERFLOW; }
    if (cnt > 0) {
        HVO_CUDA(cudaMemcpyAsync(keylines, h->d_kl, (size_t)cnt * sizeof(KeyLineOut), cudaMemcpyDeviceToHost, h->stream));
        HVO_CUDA(cudaMemcpyAsync(desc, h->d_desc, (size_t)cnt * 32, cudaMemcpyDeviceToHost, h->stream));
        HVO_CUDA(cudaMemcpyAsync(linevec3, h->d_linevec, (size_t)cnt * 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        HVO_CUDA(cudaStreamSynchronize(h->stream));
    }
    *n_out = cnt;
    return HVO_OK;
}

int hvo_line_max_lines(const hvo_line* h) { return h ? h->nfeat : 0; }
int hvo_line_segment_capacity(const hvo_line* h) { return h ? h->seg_cap : 0; }
int hvo_line_scaled_size(const hvo_line* h, int* sw, int* sh) {
    HVO_CHECK_ARG(h && sw && sh, "null argument");
    *sw = h->sw; *sh = h->sh;
    return HVO_OK;
}

int hvo_line_detect_batch(hvo_line* h, const uint8_t* gray, int nframes, float* segments4, int seg_capacity, int32_t* counts) {
    HVO_CHECK_ARG(h && gray && segments4 && counts, "null argument");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch, "nframes out of range for this handle");
    HVO_CHECK_ARG(seg_capacity >= 1, "seg_capacity < 1");
    HVO_CUDA(cudaSetDevice(h->device));
    const size_t px = (size_t)h->width * h->height;
    HVO_CUDA(cudaMemcpyAsync(h->d_gray, gray, (size_t)nframes * px, cudaMemcpyHostToDevice, h->stream));
    int st = line_detect_device(h, h->d_gray, nframes);
    if (st != HVO_OK) return st;
    HVO_CUDA(cudaMemcpyAsync(counts, h->d_nseg, (size_t)nframes * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    const int cpy = seg_capacity < h->seg_cap ? seg_capacity : h->seg_cap;
    HVO_CUDA(cudaMemcpy2DAsync(segments4, (size_t)seg_capacity * 16, h->d_seg, (size_t)h->seg_cap * 16, (size_t)cpy * 16, nframes,
                               cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return HVO_OK;
}

int hvo_line_extract_batch(hvo_line* h, const uint8_t* gray, int nframes, hvo_keyline* keylines, uint8_t* desc, double* linevec3,
                           int32_t* counts) {
    HVO_CHECK_ARG(h && gray && keylines && desc && counts, "null argument");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch, "nframes out of range for this handle");
    HVO_CUDA(cudaSetDevice(h->device));
    const size_t px = (size_t)h->width * h->height, n = (size_t)nframes, ml = (size_t)h->nfeat;
    HVO_CUDA(cudaMemcpyAsync(h->d_gray, gray, n * px, cudaMemcpyHostToDevice, h->stream));
    int st = line_extract_device(h, h->d_gray, nframes, h->d_kl, h->d_desc, h->d_linevec, h->d_counts);
    if (st != HVO_OK) return st;
    HVO_CUDA(cudaMemcpyAsync(counts, h->d_counts, n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaMemcpyAsync(keylines, h->d_kl, n * ml * sizeof(KeyLineOut), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaMemcpyAsync(desc, h->d_desc, n * ml * 32, cudaMemcpyDeviceToHost, h->stream));
    if (linevec3) HVO_CUDA(cudaMemcpyAsync(linevec3, h->d_linevec, n * ml * 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    std::vector<int32_t> nseg(n);
    HVO_CUDA(cudaMemcpyAsync(nseg.data(), h->d_nseg, n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    for (int f = 0; f < nframes; ++f)
        if (nseg[f] > h->seg_cap) { set_error("LSD segment buffer overflow in frame %d (%d segments, capacity %d)", f, nseg[f], h->seg_cap); return HVO_ERR_OVERFLOW; }
    return HVO_OK;
}

int hvo_line_extract(hvo_line* h, const uint8_t* gray, size_t stride, hvo_keyline* keylines, uint8_t* desc, double* linevec3, int capacity,
                     int* n_out) {
    HVO_CHECK_ARG(h && n_out, "null argument");
    *n_out = 0;
    if (!gray) return HVO_OK;  // empty image: the reference returns silently (LineExtractor.cpp:331-332)
    HVO_CHECK_ARG(keylines && desc, "null argument");
    HVO_CHECK_ARG(stride >= (size_t)h->width, "stride smaller than width");
    HVO_CHECK_ARG(capacity >= h->nfeat, "capacity smaller than hvo_line_max_lines()");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaMemcpy2DAsync(h->d_gray, h->width, gray, stride, h->width, h->height, cudaMemcpyHostToDevice, h->stream));
    int st = line_extract_device(h, h->d_gray, 1, h->d_kl, h->d_desc, h->d_linevec, h->d_counts);
    if (st != HVO_OK) return st;
    int32_t cnt = 0, nseg = 0;
    HVO_CUDA(cudaMemcpyAsync(&cnt, h->d_counts, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaMemcpyAsync(&nseg, h->d_nseg, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    if (nseg > h->seg_cap) { set_error("LSD segment buffer overflow (%d segments, capacity %d)", nseg, h->seg_cap); return HVO_ERR_OVERFLOW; }
    if (cnt > 0) {
        HVO_CUDA(cudaMemcpyAsync(keylines, h->d_kl, (size_t)cnt * sizeof(KeyLineOut), cudaMemcpyDeviceToHost, h->stream));
        HVO_CUDA(cudaMemcpyAsync(desc, h->d_desc, (size_t)cnt * 32, cudaMemcpyDeviceToHost, h->stream));
        if (linevec3) HVO_CUDA(cudaMemcpyAsync(linevec3, h->d_linevec, (size_t)cnt * 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        HVO_CUDA(cudaStreamSynchronize(h->stream));
    }
    *n_out = cnt;
    return HVO_OK;
}

int hvo_line_extract_batch_device(hvo_line* h, const uint8_t* d_gray, int nframes, hvo_keyline* d_keylines, uint8_t* d_desc,
                                  double* d_linevec3, int32_t* d_counts) {
    HVO_CHECK_ARG(h && d_gray && d_keylines && d_desc && d_linevec3 && d_counts, "null argument");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch, "nframes out of range for this handle");
    HVO_CUDA(cudaSetDevice(h->device));
    return line_extract_device(h, d_gray, nframes, reinterpret_cast<KeyLineOut*>(d_keylines), d_desc, d_linevec3, d_counts);
}

int hvo_line_get_scaled(hvo_line* h, int frame, uint8_t* out) {
    HVO_CHECK_ARG(h && out, "null argument");
    HVO_CHECK_ARG(frame >= 0 && frame < h->max_batch, "frame out of range");
    HVO_CUDA(cudaSetDevice(h->device));
    const size_t spx = (size_t)h->sw * h->sh;
    HVO_CUDA(cudaMemcpyAsync(out, h->d_scaled + frame * spx, spx, cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return HVO_OK;
}

int hvo_line_get_seed_order(hvo_line* h, int frame, uint32_t* out, int cap, int* n_out) {
    HVO_CHECK_ARG(h && out && n_out, "null argument");
    HVO_CHECK_ARG(frame >= 0 && frame < h->max_batch, "frame out of range");
    HVO_CUDA(cudaSetDevice(h->device));
    int n = 0;
    HVO_CUDA(cudaMemcpyAsync(&n, h->d_norder + frame, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    *n_out = n;
    const int m = n < cap ? n : cap;
    if (m > 0) {
        HVO_CUDA(cudaMemcpyAsync(out, h->d_order + (size_t)frame * h->sw * h->sh, (size_t)m * 4, cudaMemcpyDeviceToHost, h->stream));
        HVO_CUDA(cudaStreamSynchronize(h->stream));
    }
    return HVO_OK;
}

int hvo_line_set_profiling(hvo_line* h, int enable) {
    HVO_CHECK_ARG(h, "null handle");
    h->profiling = enable != 0;
    return HVO_OK;
}
int hvo_line_stage_times(hvo_line* h, float* ms4) {
    HVO_CHECK_ARG(h && ms4, "null argument");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventSynchronize(h->sev[4]));
    for (int i = 0; i < 4; ++i) HVO_CUDA(cudaEventElapsedTime(&ms4[i], h->sev[i], h->sev[i + 1]));
    return HVO_OK;
}
int hvo_line_last_launches(const hvo_line* h) { return h ? h->last_launches : 0; }
int hvo_line_sync(hvo_line* h) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return HVO_OK;
}
int hvo_line_timer_start(hvo_line* h) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[0], h->stream));
    return HVO_OK;
}
int hvo_line_timer_stop(hvo_line* h, float* ms_out) {
    HVO_CHECK_ARG(h && ms_out, "null argument");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[1], h->stream));
    HVO_CUDA(cudaEventSynchronize(h->tev[1]));
    HVO_CUDA(cudaEventElapsedTime(ms_out, h->tev[0], h->tev[1]));
    return HVO_OK;
}

}  // extern "C"
