// Surface normals of Frame::ComputePlanes (reference src/Frame.cc:2155-2212) for sm_100a: 3x-subsampled organised
// cloud + PCL-style IntegralImageNormalEstimation (AVERAGE_3D_GRADIENT, max depth change factor 0.05, smoothing 10,
// BORDER_POLICY_IGNORE), normals kept at odd (row, col) of the cloud.  PCL is un-vendored; the algorithm follows the
// oracle's restatement (oracle/normals_oracle.cpp).
//
//   k_sn_cloud    back-projection of every 3rd pixel (float, reference operation order) + depth-change mask as a
//                 gather (the reference scatters zeros to the right / lower neighbour)
//   k_sn_rowscan  3-D central differences + per-row prefix sums in double (thread <-> cloud row)
//   k_sn_colscan  column prefix sums -> summed-area tables (thread <-> column x 6 channels, coalesced)
//   k_sn_chamfer  two-pass 3-4 chamfer distance map: one warp per frame, lanes do the three upper (lower) taps,
//                 the left (right) dependency is replayed serially in float so every value matches the sequential scan
//   k_sn_normals  window = min(distance, smoothing), box sums, n = gy x gx, normalise (double), flip to the viewpoint
#include <cmath>
#include <new>

#include "hvo_common.cuh"

namespace hvo {

struct SnGeom {
    int W, H, cw, ch;
    float factor, fx, fy, cx, cy, max_change, smoothing;
};

__global__ void k_sn_cloud(const uint16_t* __restrict__ depth, SnGeom g, float* __restrict__ pts, float* __restrict__ dist) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y, f = blockIdx.z;
    if (c >= g.cw) return;
    const uint16_t* D = depth + (long long)f * g.W * g.H;
    auto z_at = [&](int rr, int cc) { return (float)D[(long long)(3 * rr) * g.W + 3 * cc] * g.factor; };
    const float z = z_at(r, c);
    const int n = 3 * c, m = 3 * r;
    float* p = pts + ((long long)f * g.ch * g.cw + (long long)r * g.cw + c) * 3;
    p[2] = z;
    p[0] = ((float)n - g.cx) * z / g.fx;
    p[1] = ((float)m - g.cy) * z / g.fy;
    bool zero = false;
    auto th = [&](float d) { return g.max_change * (fabsf(d) + 1.0f) * 2.0f; };
    if (r < g.ch - 1 && c < g.cw - 1) {
        const float t = th(z);
        zero = fabsf(z - z_at(r, c + 1)) > t || fabsf(z - z_at(r + 1, c)) > t;
    }
    if (!zero && c >= 1 && r < g.ch - 1) { const float zl = z_at(r, c - 1); zero = fabsf(zl - z) > th(zl); }
    if (!zero && r >= 1 && c < g.cw - 1) { const float zu = z_at(r - 1, c); zero = fabsf(zu - z) > th(zu); }
    dist[(long long)f * g.ch * g.cw + (long long)r * g.cw + c] = zero ? 0.f : (float)(g.cw + g.ch);
}

// SAT layout: [f][ch+1][cw+1][6] doubles (dx.xyz, dy.xyz)
// The table adds the terms (float differences widened to double) in another order than PCL's recurrence (up + left - up-left
// + term).  A double sum of floats is exact only while the bits of all its terms fit in 53 places; terms of very different
// exponents (a difference of 1e-9 next to one of 10) round, and then the order can change the last bit of a window sum.  Depth
// images keep the terms within that range: tests/test_normals_reference.py requires the oracle's bits on every scene, shape
// and parameter set it runs.
// One warp per SAT row: 32 cloud columns at a time, lane <-> column.  Every lane forms its six central differences, the
// warp adds them up with a shuffle scan and each lane stores its six doubles next to its neighbours' (48 B per lane,
// 1.5 KB contiguous per warp).  Round 1 had one thread per row writing 48-byte records 10 KB apart (2.4 ms per 1184 frames).
__global__ void __launch_bounds__(128) k_sn_rowscan(const float* __restrict__ pts, SnGeom g, double* __restrict__ sat) {
    const int r = blockIdx.x * 4 + (threadIdx.x >> 5), f = blockIdx.y, lane = threadIdx.x & 31;
    if (r > g.ch) return;
    const int iw = g.cw + 1;
    double* row = sat + ((long long)f * (g.ch + 1) + r) * iw * 6;
    if (r == 0) {
        for (int i = lane; i < iw * 6; i += 32) row[i] = 0.0;
        return;
    }
    if (lane < 6) row[lane] = 0.0;
    const int rr = r - 1;  // cloud row
    const bool inner_row = rr >= 1 && rr < g.ch - 1;
    const float* P = pts + (long long)f * g.ch * g.cw * 3;
    double carry[6] = {0, 0, 0, 0, 0, 0};
    for (int c0 = 0; c0 < g.cw; c0 += 32) {
        const int c = c0 + lane;
        double v[6] = {0, 0, 0, 0, 0, 0};
        if (inner_row && c >= 1 && c < g.cw - 1) {
            const float* L = P + ((long long)rr * g.cw + c - 1) * 3;
            const float* R = P + ((long long)rr * g.cw + c + 1) * 3;
            const float* U = P + ((long long)(rr - 1) * g.cw + c) * 3;
            const float* Dn = P + ((long long)(rr + 1) * g.cw + c) * 3;
            v[0] = (double)(R[0] - L[0]); v[1] = (double)(R[1] - L[1]); v[2] = (double)(R[2] - L[2]);
            v[3] = (double)(Dn[0] - U[0]); v[4] = (double)(Dn[1] - U[1]); v[5] = (double)(Dn[2] - U[2]);
        }
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                const double t = __shfl_up_sync(0xffffffffu, v[k], o);
                if (lane >= o) v[k] += t;
            }
#pragma unroll
        for (int k = 0; k < 6; ++k) v[k] += carry[k];
        if (c < g.cw) {
            double2* o2 = reinterpret_cast<double2*>(row + (long long)(c + 1) * 6);   // (c + 1) * 48 B: 16-byte aligned
            o2[0] = make_double2(v[0], v[1]); o2[1] = make_double2(v[2], v[3]); o2[2] = make_double2(v[4], v[5]);
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) carry[k] = __shfl_sync(0xffffffffu, v[k], 31);
    }
}

__global__ void k_sn_colscan(SnGeom g, double* __restrict__ sat) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, f = blockIdx.y;  // i over (cw+1)*6
    const int iw6 = (g.cw + 1) * 6;
    if (i >= iw6) return;
    double* S = sat + (long long)f * (g.ch + 1) * iw6;
    double acc = 0.0;
    for (int r = 1; r <= g.ch; ++r) {
        acc += S[(long long)r * iw6 + i];
        S[(long long)r * iw6 + i] = acc;
    }
}

// kChamferFrames frames per CTA, one warp each.  The three upper (lower) taps of a row are lane-parallel per frame; the left (right)
// dependency is a float chain that has to be replayed in order, so it is done for all the CTA's frames at once by the first lanes of
// warp 0 (lane j <-> frame j): the serial part costs kChamferFrames times fewer instructions than with one active lane per warp.
static const int kChamferFrames = 8;
__global__ void __launch_bounds__(32 * kChamferFrames) k_sn_chamfer(SnGeom g, float* __restrict__ dist_all, int nf) {
    extern __shared__ float sm[];  // per frame 3 rows of cw floats: prev (or next), cur, m
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31, cw = g.cw, ch = g.ch;
    const int f = blockIdx.x * kChamferFrames + wid;
    const bool live = f < nf;
    float* dist = dist_all + (long long)(live ? f : 0) * ch * cw;
    float* base = sm + (size_t)wid * 3 * cw;
    int ia = 0, ib = 1;                       // row roles rotate identically in every warp
    float* m = base + 2 * cw;
    auto serial_fwd = [&]() {
        if (wid == 0 && lane < kChamferFrames && blockIdx.x * kChamferFrames + lane < nf) {
            float* bb = sm + (size_t)lane * 3 * cw + ib * cw;
            const float* mm = sm + (size_t)lane * 3 * cw + 2 * cw;
            float left = bb[0];
            int c = 1;
            for (; c + 3 < cw; c += 4) {   // loads first: only add / min / select are on the dependent chain
                const float m0 = mm[c], m1 = mm[c + 1], m2 = mm[c + 2], m3 = mm[c + 3];
                const float b0 = bb[c], b1 = bb[c + 1], b2 = bb[c + 2], b3 = bb[c + 3];
                float v = fminf(m0, left + 1.0f); const float r0 = v < b0 ? v : b0;
                v = fminf(m1, r0 + 1.0f); const float r1 = v < b1 ? v : b1;
                v = fminf(m2, r1 + 1.0f); const float r2 = v < b2 ? v : b2;
                v = fminf(m3, r2 + 1.0f); const float r3 = v < b3 ? v : b3;
                bb[c] = r0; bb[c + 1] = r1; bb[c + 2] = r2; bb[c + 3] = r3;
                left = r3;
            }
            for (; c < cw; ++c) {
                const float v = fminf(mm[c], left + 1.0f);
                float cur = bb[c];
                if (v < cur) { cur = v; bb[c] = v; }
                left = cur;
            }
        }
    };
    auto serial_bwd = [&]() {
        if (wid == 0 && lane < kChamferFrames && blockIdx.x * kChamferFrames + lane < nf) {
            float* bb = sm + (size_t)lane * 3 * cw + ib * cw;
            const float* mm = sm + (size_t)lane * 3 * cw + 2 * cw;
            float right = bb[cw - 1];
            int c = cw - 2;
            for (; c - 3 >= 0; c -= 4) {
                const float m0 = mm[c], m1 = mm[c - 1], m2 = mm[c - 2], m3 = mm[c - 3];
                const float b0 = bb[c], b1 = bb[c - 1], b2 = bb[c - 2], b3 = bb[c - 3];
                float v = fminf(m0, right + 1.0f); const float r0 = v < b0 ? v : b0;
                v = fminf(m1, r0 + 1.0f); const float r1 = v < b1 ? v : b1;
                v = fminf(m2, r1 + 1.0f); const float r2 = v < b2 ? v : b2;
                v = fminf(m3, r2 + 1.0f); const float r3 = v < b3 ? v : b3;
                bb[c] = r0; bb[c - 1] = r1; bb[c - 2] = r2; bb[c - 3] = r3;
                right = r3;
            }
            for (; c >= 0; --c) {
                const float v = fminf(mm[c], right + 1.0f);
                float cur = bb[c];
                if (v < cur) { cur = v; bb[c] = v; }
                right = cur;
            }
        }
    };
    // forward pass
    if (live) for (int c = lane; c < cw; c += 32) base[ia * cw + c] = dist[c];
    __syncthreads();
    for (int r = 1; r < ch; ++r) {
        float *a = base + ia * cw, *b = base + ib * cw;
        if (live) {
            for (int c = lane; c < cw; c += 32) b[c] = dist[(long long)r * cw + c];
            __syncwarp();
            for (int c = 1 + lane; c < cw; c += 32) {
                const float ur = (c + 1 < cw) ? a[c + 1] : b[0];  // PCL reads one element past the previous row
                m[c] = fminf(fminf(a[c - 1] + 1.4f, a[c] + 1.0f), ur + 1.4f);
            }
        }
        __syncthreads();
        serial_fwd();
        __syncthreads();
        if (live) for (int c = lane; c < cw; c += 32) dist[(long long)r * cw + c] = b[c];
        const int t = ia; ia = ib; ib = t;
    }
    // backward pass: row `ia` holds the last row
    for (int r = ch - 2; r >= 0; --r) {
        float *a = base + ia * cw, *b = base + ib * cw;
        if (live) {
            for (int c = lane; c < cw; c += 32) b[c] = dist[(long long)r * cw + c];
            __syncwarp();
            for (int c = lane; c <= cw - 2; c += 32) {
                const float ll = (c >= 1) ? a[c - 1] : b[cw - 1];  // PCL reads one element before the next row
                m[c] = fminf(fminf(ll + 1.4f, a[c] + 1.0f), a[c + 1] + 1.4f);
            }
        }
        __syncthreads();
        serial_bwd();
        __syncthreads();
        if (live) for (int c = lane; c < cw; c += 32) dist[(long long)r * cw + c] = b[c];
        const int t = ia; ia = ib; ib = t;
    }
}

__global__ void k_sn_normals(SnGeom g, const float* __restrict__ pts, const float* __restrict__ dist, const double* __restrict__ sat,
                             float* __restrict__ out8) {
    const int ow = g.cw / 2, oh = g.ch / 2;
    const int i = blockIdx.x * blockDim.x + threadIdx.x, f = blockIdx.y;
    if (i >= ow * oh) return;
    const int m = 2 * (i / ow) + 1, n = 2 * (i % ow) + 1;
    const long long idx = (long long)f * g.ch * g.cw + (long long)m * g.cw + n;
    const float* p = pts + idx * 3;
    const float nanv = __int_as_float(0x7fc00000);
    float nx = nanv, ny = nanv, nz = nanv;
    const int border = (int)g.smoothing;
    if (m >= border && m < g.ch - border && n >= border && n < g.cw - border) {
        const float smoothing = fminf(dist[idx], g.smoothing);
        if (smoothing > 2.0f) {
            const int rw = (int)smoothing, sx = n - rw / 2, sy = m - rw / 2, iw = g.cw + 1;
            const double* S = sat + (long long)f * (g.ch + 1) * iw * 6;
            const double* ul = S + ((long long)sy * iw + sx) * 6;
            const double* ur = ul + rw * 6;
            const double* ll = S + ((long long)(sy + rw) * iw + sx) * 6;
            const double* lr = ll + rw * 6;
            double gx[3], gy[3];
            for (int k = 0; k < 3; ++k) {
                gx[k] = lr[k] + ul[k] - ur[k] - ll[k];
                gy[k] = lr[3 + k] + ul[3 + k] - ur[3 + k] - ll[3 + k];
            }
            const double v0 = gy[1] * gx[2] - gy[2] * gx[1], v1 = gy[2] * gx[0] - gy[0] * gx[2], v2 = gy[0] * gx[1] - gy[1] * gx[0];
            const double len2 = v0 * v0 + v1 * v1 + v2 * v2;
            if (len2 != 0.0) {
                const double l = sqrt(len2);
                nx = (float)(v0 / l); ny = (float)(v1 / l); nz = (float)(v2 / l);
                const float cos_theta = (0.f - p[0]) * nx + (0.f - p[1]) * ny + (0.f - p[2]) * nz;
                if (cos_theta < 0) { nx = -nx; ny = -ny; nz = -nz; }
            }
        }
    }
    float* o = out8 + ((long long)f * ow * oh + i) * 8;
    o[0] = nx; o[1] = ny; o[2] = nz; o[3] = p[0]; o[4] = p[1]; o[5] = p[2]; o[6] = (float)(n * 3); o[7] = (float)(m * 3);
}

}  // namespace hvo

using namespace hvo;

struct hvo_normals {
    int device = 0, max_batch = 0;
    SnGeom g;
    cudaStream_t stream = nullptr;
    cudaEvent_t tev[2] = {nullptr, nullptr};
    uint16_t* d_depth = nullptr;
    float *d_pts = nullptr, *d_dist = nullptr, *d_out = nullptr;
    double* d_sat = nullptr;
    int n_out = 0;
};

static int sn_run(hvo_normals* h, const uint16_t* d_depth, int nf, float* d_out) {
    const SnGeom& g = h->g;
    timeline_mark(h->stream, "k_sn_cloud");
    k_sn_cloud<<<dim3(div_up(g.cw, 128), g.ch, nf), 128, 0, h->stream>>>(d_depth, g, h->d_pts, h->d_dist);
    timeline_mark(h->stream, "k_sn_rowscan");
    k_sn_rowscan<<<dim3(div_up(g.ch + 1, 4), nf), 128, 0, h->stream>>>(h->d_pts, g, h->d_sat);
    timeline_mark(h->stream, "k_sn_colscan");
    k_sn_colscan<<<dim3(div_up((g.cw + 1) * 6, 128), nf), 128, 0, h->stream>>>(g, h->d_sat);
    timeline_mark(h->stream, "k_sn_chamfer");
    k_sn_chamfer<<<div_up(nf, kChamferFrames), 32 * kChamferFrames, (size_t)kChamferFrames * 3 * g.cw * sizeof(float), h->stream>>>(g, h->d_dist, nf);
    timeline_mark(h->stream, "k_sn_normals");
    k_sn_normals<<<dim3(div_up(h->n_out, 128), nf), 128, 0, h->stream>>>(g, h->d_pts, h->d_dist, h->d_sat, d_out);
    HVO_CUDA(cudaGetLastError());
    return HVO_OK;
}

namespace hvo {
cudaStream_t normals_stream(hvo_normals* h) { return h->stream; }  // internal: frame.cu chains the stages on events
}

extern "C" {

int hvo_normals_create(const hvo_normals_params* p, int width, int height, int max_batch, int device, hvo_normals** out) {
    HVO_CHECK_ARG(p && out, "null argument");
    *out = nullptr;
    HVO_CHECK_ARG(width >= 64 && height >= 64 && max_batch >= 1, "size out of range");
    HVO_CHECK_ARG(max_batch <= 65535, "max_batch > 65535 (the frame index is a grid y / z coordinate)");
    HVO_CHECK_ARG(p->fx != 0.f && p->fy != 0.f, "focal length is zero");
    int ndev = 0;
    HVO_CUDA(cudaGetDeviceCount(&ndev));
    if (ndev < 1) { set_error("no CUDA device: libhvofront has no CPU fallback"); return HVO_ERR_CUDA; }
    HVO_CHECK_ARG(device >= 0 && device < ndev, "device index out of range");
    // k_sn_chamfer keeps 3 cloud rows of each of its kChamferFrames frames in shared memory: 96 * ceil(width / 3) bytes
    const int cw = (int)std::ceil(width / 3.0);
    const size_t chamfer_smem = (size_t)kChamferFrames * 3 * cw * sizeof(float);
    int smem_optin = 0;
    HVO_CUDA(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    if (chamfer_smem > (size_t)smem_optin) {
        set_error("bad argument: width %d needs %zu B of shared memory per chamfer block, the device allows %d B (width <= %d)", width,
                  chamfer_smem, smem_optin, 3 * (smem_optin / (int)(kChamferFrames * 3 * sizeof(float))));
        return HVO_ERR_ARG;
    }
    hvo_normals* h = new (std::nothrow) hvo_normals();
    if (!h) { set_error("out of host memory"); return HVO_ERR_ARG; }
    h->device = device; h->max_batch = max_batch;
    SnGeom& g = h->g;
    g.W = width; g.H = height; g.cw = (int)std::ceil(width / 3.0); g.ch = (int)std::ceil(height / 3.0);
    g.factor = p->depth_factor; g.fx = p->fx; g.fy = p->fy; g.cx = p->cx; g.cy = p->cy;
    g.max_change = p->max_depth_change_factor; g.smoothing = p->normal_smoothing_size;
    h->n_out = (g.cw / 2) * (g.ch / 2);
    const size_t B = (size_t)max_batch, np = (size_t)g.cw * g.ch;
    cudaError_t e = cudaSetDevice(device);
    pin_carveout(k_sn_cloud); pin_carveout(k_sn_rowscan); pin_carveout(k_sn_colscan); pin_carveout(k_sn_chamfer); pin_carveout(k_sn_normals);
    // widths over 1536 need more than the default 48 KB; the limit is the device's (one value for every handle, so handles of
    // different widths cannot lower it for each other), each launch asks for what its width needs
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_sn_chamfer, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
    if (e == cudaSuccess) e = create_stream(&h->stream);
    if (e == cudaSuccess) e = cudaEventCreate(&h->tev[0]);
    if (e == cudaSuccess) e = cudaEventCreate(&h->tev[1]);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_depth, B * width * height * 2);
    if (e == cudaSuccess) e = cudaMalloc(&h->d_pts, B * np * 3 * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&h->d_dist, B * np * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&h->d_sat, B * (size_t)(g.cw + 1) * (g.ch + 1) * 6 * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&h->d_out, B * h->n_out * 8 * sizeof(float));
    if (e != cudaSuccess) { set_error("hvo_normals_create: %s", cudaGetErrorString(e)); hvo_normals_destroy(h); return HVO_ERR_CUDA; }
    *out = h;
    return HVO_OK;
}

void hvo_normals_destroy(hvo_normals* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    void* bufs[] = {h->d_depth, h->d_pts, h->d_dist, h->d_sat, h->d_out};
    for (void* b : bufs) if (b) cudaFree(b);
    for (auto& e : h->tev) if (e) cudaEventDestroy(e);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int hvo_normals_count(const hvo_normals* h) { return h ? h->n_out : 0; }

int hvo_normals_compute_batch(hvo_normals* h, const uint16_t* depth16, int nframes, float* out8) {
    HVO_CHECK_ARG(h && depth16 && out8, "null argument");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch, "nframes out of range for this handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaMemcpyAsync(h->d_depth, depth16, (size_t)nframes * h->g.W * h->g.H * 2, cudaMemcpyHostToDevice, h->stream));
    int st = sn_run(h, h->d_depth, nframes, h->d_out);
    if (st != HVO_OK) return st;
    HVO_CUDA(cudaMemcpyAsync(out8, h->d_out, (size_t)nframes * h->n_out * 8 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return HVO_OK;
}

int hvo_normals_compute_batch_device(hvo_normals* h, const uint16_t* d_depth16, int nframes, float* d_out8) {
    HVO_CHECK_ARG(h && d_depth16 && d_out8, "null argument");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch, "nframes out of range for this handle");
    HVO_CUDA(cudaSetDevice(h->device));
    return sn_run(h, d_depth16, nframes, d_out8);
}

int hvo_normals_get_distance_map(hvo_normals* h, int frame, float* out) {
    HVO_CHECK_ARG(h && out, "null argument");
    HVO_CHECK_ARG(frame >= 0 && frame < h->max_batch, "frame out of range");
    HVO_CUDA(cudaSetDevice(h->device));
    const size_t np = (size_t)h->g.cw * h->g.ch;
    HVO_CUDA(cudaMemcpyAsync(out, h->d_dist + frame * np, np * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return HVO_OK;
}

int hvo_normals_sync(hvo_normals* h) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return HVO_OK;
}
int hvo_normals_timer_start(hvo_normals* h) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[0], h->stream));
    return HVO_OK;
}
int hvo_normals_timer_stop(hvo_normals* h, float* ms_out) {
    HVO_CHECK_ARG(h && ms_out, "null argument");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[1], h->stream));
    HVO_CUDA(cudaEventSynchronize(h->tev[1]));
    HVO_CUDA(cudaEventElapsedTime(ms_out, h->tev[0], h->tev[1]));
    return HVO_OK;
}

}  // extern "C"
