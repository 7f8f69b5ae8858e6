// Manhattan::computeNormalsLPVO for sm_100a (reference src/Manhattan.cpp:237-393; called from Frame::ExtractMainImgPtNormals
// until the Manhattan axes are initialised, src/Frame.cc:218-228).
//
// The reference builds a vertex map, six tangent maps and a mask, takes seven full cv::integral images (CV_32F -> CV_64F)
// and then reads them at a 15-px lattice only.  Here nothing is materialised per pixel: a thread walks one image row with
// seven running double sums (cv::integral's own row order) and keeps them at the lattice columns (84 at 640 px); a second
// kernel adds the rows up per column (cv::integral's column order) and keeps the lattice rows; a third takes the box means, the
// cross product and cv::normalize, and compacts the valid samples in the reference's push_back order.  The additions
// happen in cv::integral's order, so the sums are the same doubles.
//
// Reference bug, not reproduced: the live caller passes the raw CV_16U depth Mat and the function reads it as float
// (SURVEY section 8, row D6).  This implements the intended float-depth behaviour: z = (float)raw * depth_factor.
#include <algorithm>
#include <new>

#include "lpvo.cuh"

namespace hvo {

static const int kCell = 10, kDensity = 15;

__device__ __forceinline__ bool lpvo_bad(float z) { return z < 0.2f || z > 7.0f; }
__device__ __forceinline__ float3 lpvo_vertex(const LpvoGeom& g, int u, int v, float z) {
    if (!(z > 0.2f && z < 7.0f)) return make_float3(0.f, 0.f, 0.f);  // vertexMap stays zero (Manhattan.cpp:250)
    return make_float3(__fmul_rn(__fmul_rn((float)u - g.cx, z), g.inv_fx), __fmul_rn(__fmul_rn((float)v - g.cy, z), g.inv_fy), z);
}

// rowsum[f][k][v][c]: running sum of map k along row v up to and including lattice column c (c even: u = 15 j, c odd: u = 15 j + 10)
__global__ void __launch_bounds__(64) k_lpvo_rows(const uint16_t* __restrict__ depth, LpvoGeom g, double* __restrict__ rowsum) {
    const int v = blockIdx.x * 64 + threadIdx.x, f = blockIdx.y;
    if (v >= g.H) return;
    const int W = g.W, H = g.H, ncs = 2 * g.nsu;
    const uint16_t* D = depth + (size_t)f * W * H;
    double* out = rowsum + (size_t)f * 7 * H * ncs + (size_t)v * ncs;
    const size_t kstride = (size_t)H * ncs;
    double s[7] = {0, 0, 0, 0, 0, 0, 0};
    const bool inner = v >= 1 && v < H - 1;
    const uint16_t* r0 = D + (size_t)v * W;
    const uint16_t* rm = D + (size_t)(inner ? v - 1 : v) * W;
    const uint16_t* rp = D + (size_t)(inner ? v + 1 : v) * W;
    float zl = 0.f, zc = __fmul_rn((float)r0[0], g.factor), zr = W > 1 ? __fmul_rn((float)r0[1], g.factor) : 0.f;
    int next15 = 0;  // u of the next lattice column pair: 15 j and 15 j + 10
    for (int u = 0; u < W; ++u) {
        if (inner && u >= 1 && u < W - 1) {
            const float zu = __fmul_rn((float)rm[u], g.factor), zd = __fmul_rn((float)rp[u], g.factor);
            if (!(lpvo_bad(zc) || lpvo_bad(zl) || lpvo_bad(zr) || lpvo_bad(zu) || lpvo_bad(zd))) {
                const float3 a = lpvo_vertex(g, u + 1, v, zr), b = lpvo_vertex(g, u - 1, v, zl);
                const float3 c = lpvo_vertex(g, u, v + 1, zd), d = lpvo_vertex(g, u, v - 1, zu);
                s[0] += (double)__fsub_rn(a.x, b.x); s[1] += (double)__fsub_rn(a.y, b.y); s[2] += (double)__fsub_rn(a.z, b.z);
                s[3] += (double)__fsub_rn(c.x, d.x); s[4] += (double)__fsub_rn(c.y, d.y); s[5] += (double)__fsub_rn(c.z, d.z);
                s[6] += 1.0;
            }
        }
        const int du = u - next15;
        if (du == 0 || du == kCell) {
            const int c = 2 * (next15 / kDensity) + (du ? 1 : 0);
            if (c < ncs) {
#pragma unroll
                for (int k = 0; k < 7; ++k) out[k * kstride + c] = s[k];
            }
            if (du) next15 += kDensity;
        }
        zl = zc; zc = zr;
        zr = (u + 2 < W) ? __fmul_rn((float)r0[u + 2], g.factor) : 0.f;
    }
}

// integ[f][k][r][c]: integral image at lattice row r (r even: v = 15 i, r odd: v = 15 i + 10) and lattice column c.
// One thread per lattice column, as many CTAs across as the width needs (170 columns at 1280 px).
static const int kColsBlock = 96;
__global__ void __launch_bounds__(kColsBlock) k_lpvo_cols(LpvoGeom g, const double* __restrict__ rowsum, double* __restrict__ integ) {
    const int c = blockIdx.x * kColsBlock + threadIdx.x, k = blockIdx.y, f = blockIdx.z;
    const int ncs = 2 * g.nsu, nrs = 2 * g.nsv, H = g.H;
    if (c >= ncs) return;
    const double* in = rowsum + ((size_t)f * 7 + k) * H * ncs + c;
    double* out = integ + ((size_t)f * 7 + k) * nrs * ncs + c;
    double acc = 0;
    int next15 = 0;
    for (int v = 0; v < H; ++v) {
        acc += in[(size_t)v * ncs];
        const int dv = v - next15;
        if (dv == 0 || dv == kCell) {
            const int r = 2 * (next15 / kDensity) + (dv ? 1 : 0);
            if (r < nrs) out[(size_t)r * ncs] = acc;
            if (dv) next15 += kDensity;
        }
    }
}

// one CTA per frame: box means, normal, cv::normalize; valid samples compacted in (v, u) scan order
__global__ void __launch_bounds__(256) k_lpvo_normals(const uint16_t* __restrict__ depth, LpvoGeom g, const double* __restrict__ integ,
                                                       double* __restrict__ normals3, float* __restrict__ zout, int32_t* __restrict__ pix2,
                                                       int32_t* __restrict__ counts) {
    __shared__ int s_warp[8], s_base;
    const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int W = g.W, H = g.H, ncs = 2 * g.nsu, nrs = 2 * g.nsv, cap = g.nsu * g.nsv;
    const uint16_t* D = depth + (size_t)f * W * H;
    const double* I = integ + (size_t)f * 7 * nrs * ncs;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int base = 0; base < cap; base += 256) {
        const int idx = base + tid;
        bool valid = false;
        double nrm[3] = {0, 0, 0};
        float zc = 0.f;
        int u = 0, v = 0;
        if (idx < cap) {
            const int i = idx / g.nsu, j = idx - i * g.nsu;
            u = kCell + kDensity * j; v = kCell + kDensity * i;
            auto Z = [&](int vv, int uu) { return __fmul_rn((float)D[(size_t)vv * W + uu], g.factor); };
            zc = Z(v, u);
            valid = !(lpvo_bad(zc) || lpvo_bad(Z(v, u - 1)) || lpvo_bad(Z(v, u + 1)) || lpvo_bad(Z(v - 1, u)) || lpvo_bad(Z(v + 1, u)));
            if (valid) {
                const int r1 = 2 * i + 1, r0 = 2 * i, c1 = 2 * j + 1, c0 = 2 * j;  // (v, u), (v - 10, u - 10)
                double m[7];
#pragma unroll
                for (int k = 0; k < 7; ++k) {
                    const double* J = I + (size_t)k * nrs * ncs;
                    m[k] = __dadd_rn(__dsub_rn(__dsub_rn(J[r1 * ncs + c1], J[r0 * ncs + c1]), J[r1 * ncs + c0]), J[r0 * ncs + c0]);
                }
                const double num = (double)(int)m[6];
                double uv[3], vv[3];
#pragma unroll
                for (int k = 0; k < 3; ++k) { uv[k] = __ddiv_rn(m[k], num); vv[k] = __ddiv_rn(m[3 + k], num); }
                const double n0 = __dsub_rn(__dmul_rn(vv[1], uv[2]), __dmul_rn(vv[2], uv[1]));
                const double n1 = __dsub_rn(__dmul_rn(vv[2], uv[0]), __dmul_rn(vv[0], uv[2]));
                const double n2 = __dsub_rn(__dmul_rn(vv[0], uv[1]), __dmul_rn(vv[1], uv[0]));
                // cv::normalize as cv2 4.13.0 computes it: norm from fused multiply-adds in element order, scale = 1 / norm
                const double ss = __fma_rn(n2, n2, __fma_rn(n1, n1, __dmul_rn(n0, n0)));
                const double norm = __dsqrt_rn(ss), scale = norm > DBL_EPSILON ? __ddiv_rn(1.0, norm) : 0.0;
                nrm[0] = __dmul_rn(n0, scale); nrm[1] = __dmul_rn(n1, scale); nrm[2] = __dmul_rn(n2, scale);
                if (!(zc > 0.2f && zc < 7.0f)) zc = 0.f;  // depth_normals takes vertexMap z (zero at exactly 0.2 / 7.0)
            }
        }
        const unsigned bal = __ballot_sync(0xffffffffu, valid);
        if (lane == 0) s_warp[wid] = __popc(bal);
        __syncthreads();
        int off = s_base;
        for (int w = 0; w < wid; ++w) off += s_warp[w];
        if (valid) {
            const size_t o = (size_t)f * cap + off + __popc(bal & ((1u << lane) - 1));
            normals3[o * 3 + 0] = nrm[0]; normals3[o * 3 + 1] = nrm[1]; normals3[o * 3 + 2] = nrm[2];
            zout[o] = zc;
            pix2[o * 2] = u; pix2[o * 2 + 1] = v;
        }
        __syncthreads();
        if (tid == 0) { int t = 0; for (int w = 0; w < 8; ++w) t += s_warp[w]; s_base += t; }
        __syncthreads();
    }
    if (tid == 0) counts[f] = s_base;
}

LpvoGeom lpvo_geom(const hvo_plane_params& cam, int width, int height) {
    LpvoGeom g;
    g.W = width; g.H = height;
    g.nsu = (width - 1 - kCell + kDensity - 1) / kDensity;   // u = 10; u < W - 1; u += 15
    g.nsv = (height - 1 - kCell + kDensity - 1) / kDensity;
    g.cx = cam.cx; g.cy = cam.cy; g.inv_fx = 1.0f / cam.fx; g.inv_fy = 1.0f / cam.fy; g.factor = cam.depth_factor;
    return g;
}

static size_t lpvo_rowsum_bytes(const LpvoGeom& g, int frames) { return (size_t)frames * 7 * g.H * 2 * g.nsu * sizeof(double); }
static size_t lpvo_integ_bytes(const LpvoGeom& g, int frames) { return (size_t)frames * 7 * 2 * g.nsv * 2 * g.nsu * sizeof(double); }

int lpvo_scratch_alloc(const LpvoGeom& g, int frames, LpvoScratch* s) {
    HVO_CUDA(cudaMalloc(&s->rowsum, lpvo_rowsum_bytes(g, frames)));
    HVO_CUDA(cudaMalloc(&s->integ, lpvo_integ_bytes(g, frames)));
    s->frames = frames;
    return HVO_OK;
}

void lpvo_scratch_free(LpvoScratch* s) {
    if (s->rowsum) cudaFree(s->rowsum);
    if (s->integ) cudaFree(s->integ);
    *s = LpvoScratch{};
}

int lpvo_launch(cudaStream_t s, const LpvoGeom& g, const LpvoScratch& sc, const uint16_t* d_depth, int n, double* d_normals3, float* d_z,
                int32_t* d_pix2, int32_t* d_counts, int* launches) {
    const size_t px = (size_t)g.W * g.H, cap = (size_t)lpvo_capacity(g);
    for (int off = 0; off < n; off += sc.frames) {   // sub-batches: the scratch holds sc.frames frames
        const int m = std::min(sc.frames, n - off);
        const uint16_t* D = d_depth + off * px;
        k_lpvo_rows<<<dim3(div_up(g.H, 64), m), 64, 0, s>>>(D, g, sc.rowsum);
        k_lpvo_cols<<<dim3(div_up(2 * g.nsu, kColsBlock), 7, m), kColsBlock, 0, s>>>(g, sc.rowsum, sc.integ);
        k_lpvo_normals<<<m, 256, 0, s>>>(D, g, sc.integ, d_normals3 + off * cap * 3, d_z + off * cap, d_pix2 + off * cap * 2, d_counts + off);
        HVO_CUDA(cudaGetLastError());
        *launches += 3;
    }
    return HVO_OK;
}

}  // namespace hvo

using namespace hvo;

struct hvo_lpvo {
    int device = 0, max_batch = 0, cap = 0;
    LpvoGeom g;
    LpvoScratch scratch;   // max_batch frames: one pass of the chain per call
    cudaStream_t stream = nullptr;
    cudaEvent_t tev[2] = {nullptr, nullptr};
    uint16_t* d_depth = nullptr;
    double* d_normals = nullptr;
    float* d_z = nullptr;
    int32_t *d_pix = nullptr, *d_counts = nullptr;
};

static int lpvo_run(hvo_lpvo* h, const uint16_t* d_depth, int n, double* d_normals3, float* d_z, int32_t* d_pix2, int32_t* d_counts) {
    int launches = 0;
    return lpvo_launch(h->stream, h->g, h->scratch, d_depth, n, d_normals3, d_z, d_pix2, d_counts, &launches);
}

extern "C" {

int hvo_lpvo_create(const hvo_plane_params* cam, int width, int height, int max_batch, int device, hvo_lpvo** out) {
    HVO_CHECK_ARG(out, "null out");
    *out = nullptr;
    HVO_CHECK_ARG(cam, "null params");
    HVO_CHECK_ARG(width >= 32 && height >= 32 && width <= 8192 && height <= 8192, "image size out of range");
    HVO_CHECK_ARG(max_batch >= 1, "max_batch < 1");
    int ndev = 0;
    HVO_CUDA(cudaGetDeviceCount(&ndev));
    if (ndev < 1) { set_error("no CUDA device: libhvofront has no CPU fallback"); return HVO_ERR_CUDA; }
    HVO_CHECK_ARG(device >= 0 && device < ndev, "device index out of range");
    hvo_lpvo* h = new (std::nothrow) hvo_lpvo();
    if (!h) { set_error("out of host memory"); return HVO_ERR_ARG; }
    h->device = device; h->max_batch = max_batch;
    h->g = lpvo_geom(*cam, width, height);
    h->cap = lpvo_capacity(h->g);
    int st = HVO_OK;
    do {
#define HVO_TRY(call) if ((call) != cudaSuccess) { set_error("%s: %s", #call, cudaGetErrorString(cudaGetLastError())); st = HVO_ERR_CUDA; break; }
        HVO_TRY(cudaSetDevice(device));
        HVO_TRY(create_stream(&h->stream));
        HVO_TRY(cudaEventCreate(&h->tev[0]));
        HVO_TRY(cudaEventCreate(&h->tev[1]));
        const size_t B = (size_t)max_batch, px = (size_t)width * height;
        HVO_TRY(cudaMalloc(&h->d_depth, B * px * 2));
        if ((st = lpvo_scratch_alloc(h->g, max_batch, &h->scratch)) != HVO_OK) break;
        HVO_TRY(cudaMalloc(&h->d_normals, B * h->cap * 3 * sizeof(double)));
        HVO_TRY(cudaMalloc(&h->d_z, B * h->cap * sizeof(float)));
        HVO_TRY(cudaMalloc(&h->d_pix, B * h->cap * 2 * sizeof(int32_t)));
        HVO_TRY(cudaMalloc(&h->d_counts, B * sizeof(int32_t)));
#undef HVO_TRY
    } while (0);
    if (st != HVO_OK) { hvo_lpvo_destroy(h); return st; }
    *out = h;
    return HVO_OK;
}

void hvo_lpvo_destroy(hvo_lpvo* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    void* bufs[] = {h->d_depth, h->d_normals, h->d_z, h->d_pix, h->d_counts};
    for (void* b : bufs) if (b) cudaFree(b);
    lpvo_scratch_free(&h->scratch);
    for (auto& e : h->tev) if (e) cudaEventDestroy(e);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int hvo_lpvo_capacity(const hvo_lpvo* h) { return h ? h->cap : 0; }

int hvo_lpvo_compute_batch_device(hvo_lpvo* h, const uint16_t* d_depth16, int nframes, double* d_normals3, float* d_depth, int32_t* d_pix2,
                                  int32_t* d_counts) {
    HVO_CHECK_ARG(h && d_depth16 && d_normals3 && d_depth && d_pix2 && d_counts, "null argument");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch, "nframes out of range for this handle");
    HVO_CUDA(cudaSetDevice(h->device));
    return lpvo_run(h, d_depth16, nframes, d_normals3, d_depth, d_pix2, d_counts);
}

int hvo_lpvo_compute_batch(hvo_lpvo* h, const uint16_t* depth16, int nframes, double* normals3, float* depth, int32_t* pix2, int32_t* counts) {
    HVO_CHECK_ARG(h && depth16 && normals3 && depth && pix2 && counts, "null argument");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch, "nframes out of range for this handle");
    HVO_CUDA(cudaSetDevice(h->device));
    const size_t n = (size_t)nframes, px = (size_t)h->g.W * h->g.H, c = (size_t)h->cap;
    HVO_CUDA(cudaMemcpyAsync(h->d_depth, depth16, n * px * 2, cudaMemcpyHostToDevice, h->stream));
    int st = lpvo_run(h, h->d_depth, nframes, h->d_normals, h->d_z, h->d_pix, h->d_counts);
    if (st != HVO_OK) return st;
    HVO_CUDA(cudaMemcpyAsync(normals3, h->d_normals, n * c * 24, cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaMemcpyAsync(depth, h->d_z, n * c * 4, cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaMemcpyAsync(pix2, h->d_pix, n * c * 8, cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaMemcpyAsync(counts, h->d_counts, n * 4, cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return HVO_OK;
}

int hvo_lpvo_sync(hvo_lpvo* h) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return HVO_OK;
}
int hvo_lpvo_timer_start(hvo_lpvo* h) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[0], h->stream));
    return HVO_OK;
}
int hvo_lpvo_timer_stop(hvo_lpvo* h, float* ms_out) {
    HVO_CHECK_ARG(h && ms_out, "null argument");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[1], h->stream));
    HVO_CUDA(cudaEventSynchronize(h->tev[1]));
    HVO_CUDA(cudaEventElapsedTime(ms_out, h->tev[0], h->tev[1]));
    return HVO_OK;
}

}  // extern "C"
