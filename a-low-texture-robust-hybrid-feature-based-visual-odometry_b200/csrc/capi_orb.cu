// C ABI for the ORB extractor (include/hvo_capi.h).  No torch types, no exceptions across the boundary.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <vector>

#include "orb.cuh"
#include "undistort.cuh"

namespace hvo {
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
static thread_local int g_stream_priority = 0;
void set_next_stream_priority(int priority) { g_stream_priority = priority; }
cudaError_t create_stream(cudaStream_t* s) { return cudaStreamCreateWithPriority(s, cudaStreamNonBlocking, g_stream_priority); }
struct TimelineEntry { cudaEvent_t ev; const char* name; cudaStream_t stream; };
static std::mutex g_tl_mutex;
static std::vector<TimelineEntry> g_tl;
static bool g_tl_on = false;
void timeline_mark(cudaStream_t s, const char* name) {
    // A TIMED event record in front of every kernel (one reused event per host thread and device; nobody reads it).  Measured on B200
    // with the pipelines side by side (1024-frame calls): in a process that also holds a multi-rank NCCL communicator the step takes
    // 79 ms without it and 65 ms with it (untimed records do not help; a single process without NCCL runs 65 ms either way).  The
    // timestamp makes the stream drain completely before its next kernel is handed to the work distributor, so a pipeline's pending
    // kernels do not sit in front of the other pipelines' ready ones.  HVO_FRAME_MARKS=0 switches it off (tuning aid).
    static const bool marks = [] { const char* e = getenv("HVO_FRAME_MARKS"); return !(e && e[0] == '0'); }();
    if (marks && !g_tl_on) {
        static thread_local cudaEvent_t ev[64] = {nullptr};
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return; }
        if (!ev[dev] && cudaEventCreate(&ev[dev]) != cudaSuccess) { cudaGetLastError(); ev[dev] = nullptr; return; }
        if (cudaEventRecord(ev[dev], s) != cudaSuccess) cudaGetLastError();
        return;
    }
    if (!g_tl_on) return;
    std::lock_guard<std::mutex> lk(g_tl_mutex);
    if (g_tl.size() >= 4096) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, s);
    g_tl.push_back({e, name, s});
}
int smem_carveout_percent() {
    // HVO_CARVEOUT (percent, -1 = leave the driver default) is a tuning aid; the default is chosen in DESIGN.md section 4
    static const int pc = [] { const char* e = getenv("HVO_CARVEOUT"); return e ? atoi(e) : -1; }();
    return pc;
}
}  // namespace hvo

using namespace hvo;

namespace hvo {
cudaStream_t orb_stream(hvo_orb* h) { return h->stream; }  // internal: frame.cu chains the stages on events
int* orb_error_flag(hvo_orb* h) { return h->d_err; }         // internal: frame.cu folds the device error flags into its own status
}

extern "C" {

const char* hvo_last_error(void) { return g_err; }
int hvo_timeline_enable(int on) {
    std::lock_guard<std::mutex> lk(g_tl_mutex);
    for (auto& t : g_tl) cudaEventDestroy(t.ev);
    g_tl.clear();
    g_tl_on = on != 0;
    return HVO_OK;
}
/* After the work has been synchronised: one line per mark, "ms-since-first-mark stream-id name". */
int hvo_timeline_dump(char* buf, int capacity) {
    HVO_CHECK_ARG(buf && capacity > 0, "null buffer");
    std::lock_guard<std::mutex> lk(g_tl_mutex);
    int off = 0;
    buf[0] = 0;
    std::vector<cudaStream_t> streams;
    for (auto& t : g_tl) {
        float ms = 0.f;
        if (cudaEventSynchronize(t.ev) != cudaSuccess || cudaEventElapsedTime(&ms, g_tl[0].ev, t.ev) != cudaSuccess) { cudaGetLastError(); continue; }
        int sid = -1;
        for (size_t i = 0; i < streams.size(); ++i) if (streams[i] == t.stream) sid = (int)i;
        if (sid < 0) { sid = (int)streams.size(); streams.push_back(t.stream); }
        const int n = snprintf(buf + off, (size_t)(capacity - off), "%.3f %d %s\n", ms, sid, t.name);
        if (n < 0 || off + n >= capacity) break;
        off += n;
    }
    return HVO_OK;
}

const char* hvo_version(void) { return "hvofront sm_100a " __DATE__; }

int hvo_device_count(int* n_out) {
    HVO_CHECK_ARG(n_out, "n_out is null");
    *n_out = 0;
    HVO_CUDA(cudaGetDeviceCount(n_out));
    return HVO_OK;
}

int hvo_orb_create(const hvo_orb_params* params, int width, int height, int max_batch, int device, hvo_orb** out) {
    HVO_CHECK_ARG(params && out, "null params/out");
    *out = nullptr;
    HVO_CHECK_ARG(params->nlevels >= 1 && params->nlevels <= HVO_MAX_LEVELS, "nlevels out of range");
    HVO_CHECK_ARG(params->nfeatures >= 1, "nfeatures < 1");
    HVO_CHECK_ARG(params->scale_factor > 1.0f && params->scale_factor <= 2.0f, "scale_factor must be in (1, 2]");
    HVO_CHECK_ARG(params->ini_th_fast >= 1 && params->min_th_fast >= 1 && params->ini_th_fast <= 254 &&
                      params->min_th_fast <= 254, "FAST thresholds must be in [1,254]");
    HVO_CHECK_ARG(width >= 64 && height >= 64, "image smaller than 64x64");
    HVO_CHECK_ARG(max_batch >= 1, "max_batch < 1");
    int ndev = 0;
    HVO_CUDA(cudaGetDeviceCount(&ndev));
    if (ndev < 1) { set_error("no CUDA device: libhvofront has no CPU fallback"); return HVO_ERR_CUDA; }
    HVO_CHECK_ARG(device >= 0 && device < ndev, "device index out of range");
    hvo_orb* h = new (std::nothrow) hvo_orb();
    if (!h) { set_error("out of host memory"); return HVO_ERR_ARG; }
    h->p = *params; h->width = width; h->height = height; h->max_batch = max_batch; h->device = device;
    int st = h->init();
    if (st != HVO_OK) { h->release(); delete h; return st; }
    *out = h;
    return HVO_OK;
}

void hvo_orb_destroy(hvo_orb* h) {
    if (!h) return;
    h->release();
    delete h;
}

int hvo_orb_capacity(const hvo_orb* h) { return h ? h->g.out_cap : 0; }

int hvo_orb_get_tables(const hvo_orb* h, float* sf, float* isf, float* s2, float* is2, int32_t* nfeat) {
    HVO_CHECK_ARG(h, "null handle");
    for (int i = 0; i < h->p.nlevels; ++i) {
        if (sf) sf[i] = h->sf[i];
        if (isf) isf[i] = h->isf[i];
        if (s2) s2[i] = h->sigma2[i];
        if (is2) is2[i] = h->isigma2[i];
        if (nfeat) nfeat[i] = h->nfeat[i];
    }
    return HVO_OK;
}

static int ensure_host_staging(hvo_orb* h, bool depth) {
    const size_t B = (size_t)h->max_batch, cap = (size_t)h->g.out_cap;
    if (!h->d_l0) {
        HVO_CUDA(cudaMalloc(&h->d_l0, B * h->width * h->height));
        HVO_CUDA(cudaMalloc(&h->d_kps, B * cap * sizeof(hvo_keypoint)));
        HVO_CUDA(cudaMalloc(&h->d_desc, B * cap * 32));
        HVO_CUDA(cudaMalloc(&h->d_counts, B * sizeof(int32_t)));
    }
    if (depth && !h->d_depth) {
        HVO_CUDA(cudaMalloc(&h->d_depth, B * h->width * h->height * sizeof(uint16_t)));
        HVO_CUDA(cudaMalloc(&h->d_kpdepth, B * cap * sizeof(float)));
        HVO_CUDA(cudaMalloc(&h->d_kpuright, B * cap * sizeof(float)));
    }
    return HVO_OK;
}

static int check_device_error(hvo_orb* h) {
    int e = 0;
    HVO_CUDA(cudaMemcpyAsync(&e, h->d_err, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    if (e != 0) {
        cudaMemsetAsync(h->d_err, 0, sizeof(int), h->stream);
        set_error("device-side capacity overflow (code %d)", e);
        return HVO_ERR_OVERFLOW;
    }
    return HVO_OK;
}

int hvo_orb_extract_batch_device(hvo_orb* h, const uint8_t* d_gray, int nframes, hvo_keypoint* d_kps, uint8_t* d_desc,
                                 int32_t* d_counts, const uint16_t* d_depth16, const hvo_rgbd_params* rgbd,
                                 float* d_kp_depth, float* d_kp_uright) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CHECK_ARG(d_gray && d_kps && d_desc && d_counts, "null device buffer");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch, "nframes out of range for this handle");
    HVO_CUDA(cudaSetDevice(h->device));
    return h->run(d_gray, nframes, d_kps, d_desc, d_counts, d_depth16, rgbd, d_kp_depth, d_kp_uright);
}

int hvo_orb_sync(hvo_orb* h) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return check_device_error(h);
}

int hvo_orb_extract_batch(hvo_orb* h, const uint8_t* gray, int nframes, hvo_keypoint* kps, uint8_t* desc, int32_t* counts,
                          const uint16_t* depth16, const hvo_rgbd_params* rgbd, float* kp_depth, float* kp_uright) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CHECK_ARG(gray && kps && desc && counts, "null host buffer");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch, "nframes out of range for this handle");
    const bool use_depth = depth16 != nullptr;
    if (use_depth) HVO_CHECK_ARG(rgbd && kp_depth && kp_uright, "depth given without rgbd params / outputs");
    HVO_CUDA(cudaSetDevice(h->device));
    int st = ensure_host_staging(h, use_depth);
    if (st != HVO_OK) return st;
    const size_t fb = (size_t)h->width * h->height, cap = (size_t)h->g.out_cap, n = (size_t)nframes;
    HVO_CUDA(cudaMemcpyAsync(h->d_l0, gray, n * fb, cudaMemcpyHostToDevice, h->stream));
    if (use_depth) HVO_CUDA(cudaMemcpyAsync(h->d_depth, depth16, n * fb * 2, cudaMemcpyHostToDevice, h->stream));
    st = h->run(h->d_l0, nframes, h->d_kps, h->d_desc, h->d_counts, use_depth ? h->d_depth : nullptr, rgbd, h->d_kpdepth,
                h->d_kpuright);
    if (st != HVO_OK) return st;
    HVO_CUDA(cudaMemcpyAsync(kps, h->d_kps, n * cap * sizeof(hvo_keypoint), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaMemcpyAsync(desc, h->d_desc, n * cap * 32, cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaMemcpyAsync(counts, h->d_counts, n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (use_depth) {
        HVO_CUDA(cudaMemcpyAsync(kp_depth, h->d_kpdepth, n * cap * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
        HVO_CUDA(cudaMemcpyAsync(kp_uright, h->d_kpuright, n * cap * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    }
    return check_device_error(h);  // synchronises the stream
}

int hvo_orb_extract(hvo_orb* h, const uint8_t* gray, size_t stride, hvo_keypoint* kps, uint8_t* desc, int capacity,
                    int* n_out) {
    HVO_CHECK_ARG(h && n_out, "null handle / n_out");
    *n_out = 0;
    if (gray == nullptr) return HVO_OK;  // empty image: silent return, as ORBextractor.cc:1044-1045
    HVO_CHECK_ARG(kps && desc, "null output buffer");
    HVO_CHECK_ARG(stride >= (size_t)h->width, "stride smaller than width");
    HVO_CUDA(cudaSetDevice(h->device));
    int st = ensure_host_staging(h, false);
    if (st != HVO_OK) return st;
    const size_t cap = (size_t)h->g.out_cap;
    HVO_CUDA(cudaMemcpy2DAsync(h->d_l0, h->width, gray, stride, h->width, h->height, cudaMemcpyHostToDevice, h->stream));
    st = h->run(h->d_l0, 1, h->d_kps, h->d_desc, h->d_counts, nullptr, nullptr, nullptr, nullptr);
    if (st != HVO_OK) return st;
    int32_t n = 0;
    HVO_CUDA(cudaMemcpyAsync(&n, h->d_counts, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    if (n > capacity) { set_error("capacity %d too small for %d keypoints (use hvo_orb_capacity)", capacity, n); return HVO_ERR_ARG; }
    if (n > 0) {
        HVO_CUDA(cudaMemcpyAsync(kps, h->d_kps, (size_t)n * sizeof(hvo_keypoint), cudaMemcpyDeviceToHost, h->stream));
        HVO_CUDA(cudaMemcpyAsync(desc, h->d_desc, (size_t)n * 32, cudaMemcpyDeviceToHost, h->stream));
    }
    (void)cap;
    st = check_device_error(h);
    if (st != HVO_OK) return st;
    *n_out = n;
    return HVO_OK;
}

int hvo_orb_timer_start(hvo_orb* h) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[0], h->stream));
    return HVO_OK;
}
int hvo_orb_timer_stop(hvo_orb* h, float* ms_out) {
    HVO_CHECK_ARG(h && ms_out, "null handle / ms_out");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[1], h->stream));
    HVO_CUDA(cudaEventSynchronize(h->tev[1]));
    HVO_CUDA(cudaEventElapsedTime(ms_out, h->tev[0], h->tev[1]));
    return HVO_OK;
}
int hvo_orb_set_profiling(hvo_orb* h, int enable) {
    HVO_CHECK_ARG(h, "null handle");
    h->profiling = enable != 0;
    h->have_stage_times = false;
    return HVO_OK;
}
int hvo_orb_stage_times(hvo_orb* h, float* ms5) {
    HVO_CHECK_ARG(h && ms5, "null handle / ms5");
    if (!h->have_stage_times) { set_error("no profiled call recorded"); return HVO_ERR_STATE; }
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventSynchronize(h->ev[5]));
    for (int i = 0; i < 5; ++i) HVO_CUDA(cudaEventElapsedTime(&ms5[i], h->ev[i], h->ev[i + 1]));
    return HVO_OK;
}
int hvo_stereo_uright_from_depth(const hvo_keypoint* keys_un, const float* kp_depth, int n, float bf, float* uright) {
    HVO_CHECK_ARG(n >= 0 && (n == 0 || (keys_un && kp_depth && uright)), "null argument");
    for (int i = 0; i < n; ++i) {
        const float d = kp_depth[i];
        uright[i] = d > 0.f ? keys_un[i].x - bf / d : -1.f;   // host code is built with -ffp-contract=off
    }
    return HVO_OK;
}

static bool camera_ok(const hvo_camera* c) {
    return c && c->fx != 0.f && c->fy != 0.f && std::isfinite(c->fx) && std::isfinite(c->fy) && std::isfinite(c->cx) && std::isfinite(c->cy);
}

int hvo_undistort_points(const hvo_camera* cam, const float* xy, int n, float* xy_un) {
    HVO_CHECK_ARG(camera_ok(cam), "camera missing or fx / fy zero or not finite");
    HVO_CHECK_ARG(n >= 0 && (n == 0 || (xy && xy_un)), "null argument");
    for (int i = 0; i < n; ++i) undistort_point(*cam, xy[2 * i], xy[2 * i + 1], &xy_un[2 * i], &xy_un[2 * i + 1]);
    return HVO_OK;
}

int hvo_image_bounds(const hvo_camera* cam, int width, int height, float* min_x, float* max_x, float* min_y, float* max_y) {
    HVO_CHECK_ARG(camera_ok(cam), "camera missing or fx / fy zero or not finite");
    HVO_CHECK_ARG(min_x && max_x && min_y && max_y && width > 0 && height > 0, "bad argument");
    if (cam->k1 == 0.f) {   // the reference tests mDistCoef.at<float>(0) only
        *min_x = 0.f; *max_x = (float)width; *min_y = 0.f; *max_y = (float)height;
        return HVO_OK;
    }
    const float c[8] = {0.f, 0.f, (float)width, 0.f, 0.f, (float)height, (float)width, (float)height};
    float u[8];
    for (int i = 0; i < 4; ++i) undistort_point(*cam, c[2 * i], c[2 * i + 1], &u[2 * i], &u[2 * i + 1]);
    *min_x = std::min(u[0], u[4]); *max_x = std::max(u[2], u[6]);
    *min_y = std::min(u[1], u[3]); *max_y = std::max(u[5], u[7]);
    return HVO_OK;
}

int hvo_orb_undistort_batch_device(hvo_orb* h, const hvo_camera* cam, const hvo_keypoint* d_kps, const int32_t* d_counts, int nframes,
                                   const float* d_kp_depth, float bf, hvo_keypoint* d_kps_un, float* d_kp_uright) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CHECK_ARG(camera_ok(cam), "camera missing or fx / fy zero or not finite");
    HVO_CHECK_ARG(d_kps && d_counts, "null device buffer");
    HVO_CHECK_ARG(!d_kp_uright || d_kp_depth, "kp_uright needs kp_depth");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= 65535, "nframes out of range (1..65535)");
    HVO_CUDA(cudaSetDevice(h->device));
    return h->undistort(*cam, d_kps, d_counts, nframes, d_kp_depth, bf, d_kps_un, d_kp_uright);
}

int hvo_orb_last_launches(const hvo_orb* h) { return h ? h->last_launches : 0; }

int hvo_orb_level_size(const hvo_orb* h, int level, int* w, int* h_out) {
    HVO_CHECK_ARG(h && w && h_out, "null argument");
    HVO_CHECK_ARG(level >= 0 && level < h->p.nlevels, "level out of range");
    *w = h->g.lv[level].w;
    *h_out = h->g.lv[level].h;
    return HVO_OK;
}

int hvo_orb_get_pyramid_level(hvo_orb* h, int frame, int level, uint8_t* out, size_t out_stride) {
    HVO_CHECK_ARG(h && out, "null argument");
    HVO_CHECK_ARG(level >= 0 && level < h->p.nlevels, "level out of range");
    HVO_CHECK_ARG(frame >= 0 && frame < h->last_nframes, "frame out of range of the last call");
    const hvo::LevelGeom& L = h->g.lv[level];
    HVO_CHECK_ARG(out_stride >= (size_t)L.w, "out_stride smaller than the level width");
    HVO_CUDA(cudaSetDevice(h->device));
    const uint8_t* srcp = level == 0 ? h->last_l0 + (size_t)frame * h->width * h->height
                                     : h->d_pyr + (size_t)frame * h->g.pyr_frame_bytes + L.img_off;
    HVO_CUDA(cudaMemcpy2DAsync(out, out_stride, srcp, L.pitch, L.w, L.h, cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return HVO_OK;
}

int hvo_orb_get_candidates(hvo_orb* h, int frame, int level, int32_t* xys, int cap, int* n_out) {
    HVO_CHECK_ARG(h && xys && n_out, "null argument");
    HVO_CHECK_ARG(level >= 0 && level < h->p.nlevels, "level out of range");
    HVO_CHECK_ARG(frame >= 0 && frame < h->last_nframes, "frame out of range of the last call");
    HVO_CUDA(cudaSetDevice(h->device));
    const hvo::LevelGeom& L = h->g.lv[level];
    int n = 0;
    HVO_CUDA(cudaMemcpyAsync(&n, h->d_ncand + (size_t)frame * h->p.nlevels + level, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    n = n < L.cand_cap ? n : L.cand_cap;
    *n_out = n;
    const int m = n < cap ? n : cap;
    if (m > 0) {
        uint32_t* tmp = new (std::nothrow) uint32_t[m];
        if (!tmp) { set_error("out of host memory"); return HVO_ERR_ARG; }
        cudaError_t e = cudaMemcpyAsync(tmp, h->d_cand + (size_t)frame * h->g.cand_total + L.cand_off, (size_t)m * 4,
                                        cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
        if (e != cudaSuccess) { delete[] tmp; set_error("cudaMemcpy: %s", cudaGetErrorString(e)); return HVO_ERR_CUDA; }
        for (int i = 0; i < m; ++i) {
            xys[3 * i] = tmp[i] & 0xfff;
            xys[3 * i + 1] = (tmp[i] >> 12) & 0xfff;
            xys[3 * i + 2] = tmp[i] >> 24;
        }
        delete[] tmp;
    }
    return HVO_OK;
}

}  // extern "C"
