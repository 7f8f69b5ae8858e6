// Shared host/device helpers for libhvofront (sm_100a only).
#pragma once
#include <cuda_runtime.h>

#include <cfloat>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>

#include "../../include/hvo_capi.h"

namespace hvo {

void set_error(const char* fmt, ...);

#define HVO_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) {                                                                \
            ::hvo::set_error("%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            return HVO_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

#define HVO_CHECK_ARG(cond, msg)                            \
    do {                                                    \
        if (!(cond)) {                                      \
            ::hvo::set_error("bad argument: %s", msg);      \
            return HVO_ERR_ARG;                             \
        }                                                   \
    } while (0)

// Kernels of different pipelines only share an SM when they ask for the same L1/shared-memory split, so every
// long-running kernel is pinned to one carveout (percent of the 256 KB unified array given to shared memory).
int smem_carveout_percent();
template <class K>
static inline void pin_carveout(K kernel) {
    const int pc = smem_carveout_percent();
    if (pc >= 0) cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pc);
}

// Every handle owns one non-blocking stream.  hvo_frame gives the pipelines whose kernels are latency-bound (lines,
// planes) a higher stream priority than the streaming pipelines (ORB, normals), so the long ordered kernels are placed
// first and the streaming kernels fill the remaining warp slots: set_next_stream_priority applies to the calling
// thread's next create_stream calls (0 = default).
void set_next_stream_priority(int priority);
cudaError_t create_stream(cudaStream_t* s);

// Profiling aid (hvo_timeline_*): when enabled, every kernel launch site records a timed event on its stream first, so the
// start of each kernel and the overlap between the pipelines' streams can be read back as one timeline.  Off by default.
void timeline_mark(cudaStream_t s, const char* name);

static inline int div_up(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t a, size_t b) { return (a + b - 1) / b * b; }

// Exclusive scan over a 1024-thread CTA of 3 consecutive values per thread (the 64 x 48 = 3072 cells of a frame grid): returns the
// prefix of thread tid's first value.  s_part: 32 ints of shared memory; ends with a __syncthreads, so s_part may be reused.
__device__ __forceinline__ int block_exclusive_scan3(int sum, int* s_part) {
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    int pre = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, pre, o); if (lane >= o) pre += t; }
    if (lane == 31) s_part[wid] = pre;
    __syncthreads();
    if (wid == 0) {
        int w = s_part[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += t; }
        s_part[lane] = w;
    }
    __syncthreads();
    const int base = pre - sum + (wid > 0 ? s_part[wid - 1] : 0);
    __syncthreads();
    return base;
}

__device__ __forceinline__ int reflect101(int p, int n) {
    // single reflection is enough for |overshoot| < n (halo radii here are <= 21 px)
    if (p < 0) p = -p;
    if (p >= n) p = 2 * (n - 1) - p;
    return p;
}

// cv::fastAtan2 (degrees): float32 polynomial, every operation individually rounded (no FMA).
__device__ __forceinline__ float fast_atan2_deg(float y, float x) {
    const float scale = 57.295779513082320876798154814105f;  // (float)(180 / CV_PI)
    const float p1 = __fmul_rn(0.9997878412794807f, scale), p3 = __fmul_rn(-0.3258083974640975f, scale),
                p5 = __fmul_rn(0.1555786518463281f, scale), p7 = __fmul_rn(-0.04432655554792128f, scale);
    const float ax = fabsf(x), ay = fabsf(y);
    const float eps = (float)DBL_EPSILON;
    float a, c, c2;
    if (ax >= ay) {
        c = __fdiv_rn(ay, __fadd_rn(ax, eps));
        c2 = __fmul_rn(c, c);
        a = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c);
    } else {
        c = __fdiv_rn(ax, __fadd_rn(ay, eps));
        c2 = __fmul_rn(c, c);
        a = __fsub_rn(90.f, __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c));
    }
    if (x < 0) a = __fsub_rn(180.f, a);
    if (y < 0) a = __fsub_rn(360.f, a);
    return a;
}

}  // namespace hvo
