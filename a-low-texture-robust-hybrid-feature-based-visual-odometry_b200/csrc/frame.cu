// Frame-level front-end for sm_100a: the extraction part of Frame::Frame(imGray, imDepth, ...) of the reference
// (src/Frame.cc:188-233), where std::threads run ExtractORBNDepth (ORB + ComputeStereoFromRGBD, :874-884),
// ExtractLSD (LINEextractor::operator(), :895-903) and ComputePlanes (PlaneDetection + surface normals, :2104-2212)
// on the same frame, plus ExtractMainImgPtNormals (Manhattan::computeNormalsLPVO, :218-228, :1324-1328) while the
// Manhattan axes are not initialised.  Here the frame (gray + raw 16-bit depth) is uploaded once and the pipelines run on
// CUDA streams chained by events to a master stream, so a batch of frames is one call and one device-timed region.
#include <algorithm>
#include <cstdlib>
#include <new>

#include "hvo_common.cuh"
#include "lpvo.cuh"

struct hvo_orb;
struct hvo_line;
struct hvo_plane;
struct hvo_normals;
namespace hvo {
cudaStream_t orb_stream(hvo_orb* h);
cudaStream_t line_stream(hvo_line* h);
cudaStream_t plane_stream(hvo_plane* h);
cudaStream_t normals_stream(hvo_normals* h);
int* orb_error_flag(hvo_orb* h);
const int* line_segment_counts(hvo_line* h);
int line_segment_cap(hvo_line* h);
const int32_t* plane_status(hvo_plane* h);
int bow_frame_launch(hvo_bow* h, cudaStream_t s, const uint8_t* d_desc, const int32_t* d_counts, int nframes, int stride, int levelsup,
                     double* d_weight, const hvo_frame_bow_outputs* o);
int bow_max_features();
int proj_grid_frames_launch(cudaStream_t s, const hvo_keypoint* d_kps, const int32_t* d_counts, int nframes, int stride, float min_x, float min_y,
                            float max_x, float max_y, uint16_t* d_cell_count, uint16_t* d_cell_items);
int lproj_grid_frames_launch(cudaStream_t s, const hvo_keyline* d_kl, const int32_t* d_counts, int nframes, int stride, float min_x, float min_y,
                             float max_x, float max_y, uint32_t* d_bits, uint16_t* d_cell_count, uint16_t* d_cell_items);
}  // namespace hvo
using namespace hvo;

enum { ST_ORB = 1, ST_LINE = 2, ST_PLANE = 4, ST_NORMALS = 8 };
static const int kMaxLanes = 8;
static const int kGridCells = 64 * 48;   // FRAME_GRID_COLS x FRAME_GRID_ROWS
// frames per pass of the LPVO chain (rows -> cols -> normals): its scratch is 2.6 MB / frame at 640x480 and 7.8 MB at 1280x720, so a
// chunk-sized copy would take 10.5 GB at 4096 frames.  Measured on B200 (DESIGN section 4): 16 passes of 256 frames take 34.9 ms per
// 4096 frames, one pass of 4096 (hvo_lpvo) 29.0 ms; 0.66 GB of scratch is worth the 6 ms on a stage only the first frames ask for.
static const int kLpvoFrames = 256;

// Device-side capacity faults of the pipelines (ORB quadtree arena, LSD segment buffer, plane refinement queue) are folded,
// on the pipeline's own stream right after its kernels, into one sticky record per frame handle: fault[0] = lowest frame index
// (within its call) that overflowed, fault[1] = OR of the pipeline codes.  hvo_frame_sync / hvo_frame_timer_stop /
// hvo_frame_extract_batch read it back and return HVO_ERR_OVERFLOW ("reported, never silent", hvo_capi.h).
enum { FAULT_ORB = 1, FAULT_LINE = 2, FAULT_PLANE = 4 };
__global__ void k_frame_fold_status(const int* __restrict__ flags, int n, int stride_is_zero, int threshold, int base, int code, int* __restrict__ fault) {
    for (int f = blockIdx.x * blockDim.x + threadIdx.x; f < n; f += gridDim.x * blockDim.x) {
        if (flags[stride_is_zero ? 0 : f] > threshold) {
            atomicMin(&fault[0], base + f);
            atomicOr(&fault[1], code);
        }
    }
}

// Compact host outputs: 4-bit plane labels and normal-only surface normals, packed on the device before the download.
__global__ void k_pack_membership4(const uint8_t* __restrict__ m8, uint8_t* __restrict__ m4, long long npairs8) {
    // 16 labels in, 8 bytes out per thread
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npairs8; i += (long long)gridDim.x * blockDim.x) {
        const uint4 v = reinterpret_cast<const uint4*>(m8)[i];
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
        uint32_t o[2] = {0u, 0u};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            // bytes b0 b1 b2 b3 (255 -> 15) -> two output bytes (b0 | b1 << 4), (b2 | b3 << 4)
            const uint32_t n = w[k] & 0x0f0f0f0fu;                      // 255 & 15 = 15 = none; labels are < 15
            const uint32_t packed = (n & 0xfu) | ((n >> 4) & 0xf0u) | ((n >> 8) & 0xf00u) | ((n >> 12) & 0xf000u);
            o[k >> 1] |= packed << (16 * (k & 1));
        }
        reinterpret_cast<uint2*>(m4)[i] = make_uint2(o[0], o[1]);
    }
}
__global__ void k_pack_normals3(const float* __restrict__ n8, float* __restrict__ n3, long long rows) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < rows; i += (long long)gridDim.x * blockDim.x) {
        const float4 v = reinterpret_cast<const float4*>(n8)[2 * i];
        n3[3 * i] = v.x; n3[3 * i + 1] = v.y; n3[3 * i + 2] = v.z;
    }
}

// One lane = the staging of one chunk of `cap` frames in flight: input buffers, output buffers, an upload stream and one download
// stream per pipeline.  The pipeline handles (kernels' scratch and streams) belong to lane 0 and are shared by every lane: the
// kernels of consecutive chunks run one after the other anyway (see lane_launch), so a second copy of the 15 MB / frame of scratch
// would buy nothing, while sharing it lets a chunk be as large as the ordered kernels want (4096+ frames) inside 180 GB.
struct FrameLane {
    int cap = 0;
    bool owns = false;          // lane 0 owns the pipeline handles
    cudaStream_t down[4] = {nullptr, nullptr, nullptr, nullptr};  // host API: downloads of pipeline i (ORB, lines, planes, normals)
    cudaEvent_t fork_depth = nullptr;  // host API: the chunk's depth has arrived (the plane pipeline starts on it; gray follows)
    hvo_orb* orb = nullptr;
    hvo_line* line = nullptr;
    hvo_plane* plane = nullptr;
    hvo_normals* normals = nullptr;
    cudaStream_t up = nullptr;  // host API: uploads of this lane's chunks
    cudaEvent_t fork = nullptr, join[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t cdone[4] = {nullptr, nullptr, nullptr, nullptr};  // kernels of a pipeline done (recorded before its downloads)
    uint8_t* d_gray = nullptr;
    uint16_t* d_depth = nullptr;
    hvo_frame_outputs d_out;  // device staging of every output (host API)
    hvo_frame_bow_outputs d_bow{};  // device staging of the BoW outputs (host API; allocated while a vocabulary is attached)
    hvo_frame_grid_outputs d_grid{};  // device staging of the grid outputs (host API; allocated by the first call that asks for grids)
    hvo_frame_lpvo_outputs d_lpvo{};  // device staging of the LPVO outputs (host API; allocated by the first call that asks for them)
};

struct hvo_frame {
    hvo_frame_params p;
    int device = 0, width = 0, height = 0, max_batch = 0, nlanes = 0;
    FrameLane lane[kMaxLanes];
    cudaStream_t stream = nullptr;  // master: fork/join of the device API, timing
    cudaEvent_t fork = nullptr, tev[2] = {nullptr, nullptr};
    int orb_cap = 0, max_lines = 0, normals_count = 0, last_launches = 0;
    int last_lane = -1;  // lane of the most recent chunk: the next chunk's kernels start after its kernels
    int next_lane = 0;   // host API: lane of the next chunk (round-robin across calls)
    int* d_fault = nullptr;   // {first faulty frame, pipeline codes}, sticky until read
    int* h_fault = nullptr;   // pinned copy
    bool undistort = false;   // distorted camera with coefficients: mvKeysUn / mvuRight are formed on the device
    hvo_camera cam{};
    hvo_bow* bow = nullptr;   // attached vocabulary (hvo_frame_set_vocabulary)
    int levelsup = 4;
    double* d_bow_weight = nullptr;   // per-row leaf weights of one chunk: shared by the lanes, whose ORB kernels run in order on one stream
    float min_x = 0.f, max_x = 0.f, min_y = 0.f, max_y = 0.f;   // mnMinX .. mnMaxY (Frame::ComputeImageBounds), the grids' bounds
    uint32_t* d_lgrid_bits = nullptr;   // line grid bit rows of one chunk: shared by the lanes, whose line kernels run in order on one stream
    LpvoGeom lpvo_g{};                  // Manhattan::computeNormalsLPVO's lattice for the handle's camera and image size
    LpvoScratch lpvo_scratch;           // min(kLpvoFrames, chunk) frames: shared by the lanes, whose normals kernels run in order on one stream
};

static const int kNoFault = 0x7fffffff;

// rows [off, off + n) of every output array
static hvo_frame_outputs outputs_at(const hvo_frame* h, const hvo_frame_outputs& o, size_t off) {
    const size_t c = (size_t)h->orb_cap, l = (size_t)h->max_lines, px = (size_t)h->width * h->height;
    hvo_frame_outputs r = o;
    if (o.kps) r.kps = o.kps + off * c;
    if (o.desc) r.desc = o.desc + off * c * 32;
    if (o.kp_counts) r.kp_counts = o.kp_counts + off;
    if (o.kp_depth) r.kp_depth = o.kp_depth + off * c;
    if (o.kp_uright) r.kp_uright = o.kp_uright + off * c;
    if (o.keylines) r.keylines = o.keylines + off * l;
    if (o.line_desc) r.line_desc = o.line_desc + off * l * 32;
    if (o.linevec3) r.linevec3 = o.linevec3 + off * l * 3;
    if (o.line_counts) r.line_counts = o.line_counts + off;
    if (o.n_planes) r.n_planes = o.n_planes + off;
    if (o.planes7) r.planes7 = o.planes7 + off * (size_t)h->p.max_planes * 7;
    if (o.membership) r.membership = o.membership + off * px;
    if (o.membership8) r.membership8 = o.membership8 + off * px;
    if (o.membership4) r.membership4 = o.membership4 + off * (px / 2);
    if (o.normals8) r.normals8 = o.normals8 + off * (size_t)h->normals_count * 8;
    if (o.normals3) r.normals3 = o.normals3 + off * (size_t)h->normals_count * 3;
    if (o.kps_un) r.kps_un = o.kps_un + off * c;
    return r;
}
static hvo_frame_bow_outputs outputs_at(const hvo_frame* h, const hvo_frame_bow_outputs& o, size_t off) {
    const size_t c = (size_t)h->orb_cap;
    hvo_frame_bow_outputs r = o;
    if (o.bow_counts) r.bow_counts = o.bow_counts + off;
    if (o.bow_words) r.bow_words = o.bow_words + off * c;
    if (o.bow_values) r.bow_values = o.bow_values + off * c;
    if (o.fv_order) r.fv_order = o.fv_order + off * c;
    if (o.fv_counts) r.fv_counts = o.fv_counts + off;
    if (o.node_of) r.node_of = o.node_of + off * c;
    if (o.word_of) r.word_of = o.word_of + off * c;
    return r;
}
static hvo_frame_lpvo_outputs outputs_at(const hvo_frame* h, const hvo_frame_lpvo_outputs& o, size_t off) {
    const size_t c = (size_t)lpvo_capacity(h->lpvo_g);
    hvo_frame_lpvo_outputs r = o;
    if (o.normals3) r.normals3 = o.normals3 + off * c * 3;
    if (o.depth) r.depth = o.depth + off * c;
    if (o.pix2) r.pix2 = o.pix2 + off * c * 2;
    if (o.counts) r.counts = o.counts + off;
    return r;
}
static hvo_frame_grid_outputs outputs_at(const hvo_frame* h, const hvo_frame_grid_outputs& o, size_t off) {
    hvo_frame_grid_outputs r = o;
    if (o.grid_counts) r.grid_counts = o.grid_counts + off * kGridCells;
    if (o.grid_items) r.grid_items = o.grid_items + off * (size_t)h->orb_cap;
    if (o.lgrid_counts) r.lgrid_counts = o.lgrid_counts + off * kGridCells;
    if (o.lgrid_items) r.lgrid_items = o.lgrid_items + off * 64 * (size_t)h->max_lines;
    return r;
}

// The pipelines of one lane on n frames: wait for `start`, run, optionally copy each stage's results back on its own
// stream, record the lane's join events.  Launch order = placement order: the ordered (latency-bound) pipelines first.
// `after`: lane whose kernels must have finished first (host API: chunks compute one after the other, so the ordered kernels
// of two chunks never slow each other down, while the copies of the neighbouring chunks run beside the kernels).
//
// Two schedules (measured on B200, whole front-end, device-resident): SIDE BY SIDE (every pipeline starts at once on its own stream)
// is what a small batch wants - a single frame takes max(planes, lines) instead of their sum - but each of the ordered kernels fills
// the register file with one warp / CTA per frame by itself, and from about 2000 frames on running them beside each other only makes
// them slower (4736 frames: 16.2 K frames/s side by side, 18.2 K one after the other; ORB / normals beside the ordered kernels:
// 16.5-17.3 K).  So a chunk of >= kSerialFrames frames runs its pipelines ONE AFTER THE OTHER (planes, lines, ORB, normals), each at
// its saturating batch, and the download of a pipeline's results runs beside the kernels of the next one.
// bo (device, NULL = no BoW) / host_bo (host, NULL = nothing to download): the BoW kernels follow the ORB kernels on the ORB stream; their
// downloads are the first of phase 2.  go / host_go likewise for the grids (a NULL pair = no such grid): the point grid follows the
// undistortion on the ORB stream, the line grid the line kernels on the line stream; each is downloaded with its pipeline's results.
// lo / host_lo likewise for the LPVO normals: their chain follows the surface normals on the normals stream (so it sits beside the ordered
// pipelines side by side, and runs last in the serial schedule) and is downloaded with them.
// HVO_FRAME_SERIAL=0 / 1 forces one schedule (tuning aid).  Also measured for 1024-frame chunks and rejected: planes || lines first and
// ORB || normals afterwards (87 instead of 65-79 ms), a third priority level that puts planes above lines (no change).
static const int kSerialFrames = 2048;
static int lane_launch(hvo_frame* h, FrameLane& L, cudaEvent_t start, cudaEvent_t start_depth, const uint8_t* d_gray, const uint16_t* d_depth, int n,
                       int base, const hvo_frame_outputs& o, const hvo_frame_outputs* host, const hvo_frame_bow_outputs* bo,
                       const hvo_frame_bow_outputs* host_bo, const hvo_frame_grid_outputs* go, const hvo_frame_grid_outputs* host_go,
                       const hvo_frame_lpvo_outputs* lo, const hvo_frame_lpvo_outputs* host_lo, int* launches, FrameLane* after = nullptr) {
    const size_t N = (size_t)n, px = (size_t)h->width * h->height;
    static const int serial_env = [] { const char* e = getenv("HVO_FRAME_SERIAL"); return e ? atoi(e) : -1; }();
    const bool serial = serial_env >= 0 ? serial_env == 1 : n >= kSerialFrames;
    // side by side on one lane: every pipeline stream is already in order behind its own previous chunk
    if (after == &L && !serial) after = nullptr;
    cudaEvent_t prev_done = nullptr;   // serial schedule: the pipeline launched before this one
    auto wait_start = [&](cudaStream_t s, bool depth_only) -> int {
        HVO_CUDA(cudaStreamWaitEvent(s, (depth_only && start_depth) ? start_depth : start, 0));
        if (serial && prev_done) {
            HVO_CUDA(cudaStreamWaitEvent(s, prev_done, 0));
        } else if (after) {   // (serial: only the first pipeline waits for the previous chunk, the others follow it)
            for (int i = 0; i < 4; ++i)
                if (h->p.stages & (i == 0 ? ST_ORB : i == 1 ? ST_LINE : i == 2 ? ST_PLANE : ST_NORMALS)) HVO_CUDA(cudaStreamWaitEvent(s, after->cdone[i], 0));
        }
        return HVO_OK;
    };
    // ---- phase 1: the kernels of every pipeline are queued before any copy.  (A device-to-host copy into pageable memory
    // blocks the calling thread until the stream gets there; queued behind the plane kernels it would keep the other
    // pipelines from even starting.) ----
    if (h->p.stages & ST_PLANE) {
        cudaStream_t s = plane_stream(L.plane);
        if (int ws = wait_start(s, true)) return ws;
        int st = o.membership8 ? hvo_plane_detect_batch_device_u8(L.plane, d_depth, n, o.n_planes, o.planes7, h->p.max_planes, o.membership, o.membership8)
                               : hvo_plane_detect_batch_device(L.plane, d_depth, n, o.n_planes, o.planes7, h->p.max_planes, o.membership);
        if (st != HVO_OK) return st;
        *launches += hvo_plane_last_launches(L.plane) + 1;
        if (o.membership4 && o.membership8) {
            const long long n16 = (long long)(N * px / 16);
            k_pack_membership4<<<(int)std::min<long long>((n16 + 255) / 256, 148 * 16), 256, 0, s>>>(o.membership8, o.membership4, n16);
            ++*launches;
        }
        k_frame_fold_status<<<(n + 255) / 256, 256, 0, s>>>(plane_status(L.plane), n, 0, 0, base, FAULT_PLANE, h->d_fault);
        HVO_CUDA(cudaEventRecord(L.cdone[2], s));
        prev_done = L.cdone[2];
    }
    if (h->p.stages & ST_LINE) {
        cudaStream_t s = line_stream(L.line);
        if (int ws = wait_start(s, false)) return ws;
        int st = hvo_line_extract_batch_device(L.line, d_gray, n, o.keylines, o.line_desc, o.linevec3, o.line_counts);
        if (st != HVO_OK) return st;
        *launches += hvo_line_last_launches(L.line) + 1;
        if (go && go->lgrid_counts) {   // on the keylines returned (after cullingLine when line_cull is set), as Frame::Frame
            st = lproj_grid_frames_launch(s, o.keylines, o.line_counts, n, h->max_lines, h->min_x, h->min_y, h->max_x, h->max_y, h->d_lgrid_bits,
                                          go->lgrid_counts, go->lgrid_items);
            if (st != HVO_OK) return st;
            *launches += 2;
        }
        k_frame_fold_status<<<(n + 255) / 256, 256, 0, s>>>(line_segment_counts(L.line), n, 0, line_segment_cap(L.line), base, FAULT_LINE, h->d_fault);
        HVO_CUDA(cudaEventRecord(L.cdone[1], s));
        prev_done = L.cdone[1];
    }
    if (h->p.stages & ST_ORB) {
        cudaStream_t s = orb_stream(L.orb);
        if (int ws = wait_start(s, false)) return ws;
        hvo_rgbd_params rg{h->p.depth_factor, h->p.bf, h->p.distorted};
        int st = hvo_orb_extract_batch_device(L.orb, d_gray, n, o.kps, o.desc, o.kp_counts, d_depth, &rg, o.kp_depth, o.kp_uright);
        if (st != HVO_OK) return st;
        *launches += hvo_orb_last_launches(L.orb) + 1;
        if (h->undistort) {
            st = hvo_orb_undistort_batch_device(L.orb, &h->cam, o.kps, o.kp_counts, n, o.kp_depth, h->p.bf, o.kps_un, o.kp_uright);
            if (st != HVO_OK) return st;
            ++*launches;
        }
        if (go && go->grid_counts) {    // on mvKeysUn
            st = proj_grid_frames_launch(s, h->undistort ? o.kps_un : o.kps, o.kp_counts, n, h->orb_cap, h->min_x, h->min_y, h->max_x, h->max_y,
                                         go->grid_counts, go->grid_items);
            if (st != HVO_OK) return st;
            ++*launches;
        }
        if (bo) {
            st = bow_frame_launch(h->bow, s, o.desc, o.kp_counts, n, h->orb_cap, h->levelsup, h->d_bow_weight, bo);
            if (st != HVO_OK) return st;
            *launches += 2;
        }
        k_frame_fold_status<<<1, 32, 0, s>>>(orb_error_flag(L.orb), 1, 1, 0, base, FAULT_ORB, h->d_fault);   // one flag per chunk
        HVO_CUDA(cudaMemsetAsync(orb_error_flag(L.orb), 0, sizeof(int), s));
        HVO_CUDA(cudaEventRecord(L.cdone[0], s));
        prev_done = L.cdone[0];
    }
    if (h->p.stages & ST_NORMALS) {
        cudaStream_t s = normals_stream(L.normals);
        if (int ws = wait_start(s, false)) return ws;
        int st = hvo_normals_compute_batch_device(L.normals, d_depth, n, o.normals8);
        if (st != HVO_OK) return st;
        *launches += 5;
        if (o.normals3) {
            const long long rows = (long long)(N * (size_t)h->normals_count);
            k_pack_normals3<<<(int)std::min<long long>((rows + 255) / 256, 148 * 16), 256, 0, s>>>(o.normals8, o.normals3, rows);
            ++*launches;
        }
        if (lo) {
            st = lpvo_launch(s, h->lpvo_g, h->lpvo_scratch, d_depth, n, lo->normals3, lo->depth, lo->pix2, lo->counts, launches);
            if (st != HVO_OK) return st;
        }
        HVO_CUDA(cudaEventRecord(L.cdone[3], s));
        prev_done = L.cdone[3];
    }
    // ---- phase 2: results back to the host on the lane's download streams (one per pipeline, each behind its pipeline's kernels:
    // the shared pipeline streams stay free for the next chunk), then the join events ----
    auto down_stream = [&](int i, cudaStream_t pipe, cudaStream_t* out) -> int {
        *out = pipe;
        if (host) { HVO_CUDA(cudaStreamWaitEvent(L.down[i], L.cdone[i], 0)); *out = L.down[i]; }
        return HVO_OK;
    };
    // the BoW rows first, on the ORB download stream: side by side they are ready long before the planes, so a download into pageable
    // memory (which holds the calling thread until it is done) runs while the ordered pipelines still compute instead of after them
    if (host && host_bo) {
        cudaStream_t s;
        if (int ds = down_stream(0, orb_stream(L.orb), &s)) return ds;
        const size_t c = (size_t)h->orb_cap;
        HVO_CUDA(cudaMemcpyAsync(host_bo->bow_counts, bo->bow_counts, N * 4, cudaMemcpyDeviceToHost, s));
        HVO_CUDA(cudaMemcpyAsync(host_bo->bow_words, bo->bow_words, N * c * 4, cudaMemcpyDeviceToHost, s));
        HVO_CUDA(cudaMemcpyAsync(host_bo->bow_values, bo->bow_values, N * c * 8, cudaMemcpyDeviceToHost, s));
        if (host_bo->fv_order) HVO_CUDA(cudaMemcpyAsync(host_bo->fv_order, bo->fv_order, N * c * 4, cudaMemcpyDeviceToHost, s));
        if (host_bo->fv_counts) HVO_CUDA(cudaMemcpyAsync(host_bo->fv_counts, bo->fv_counts, N * 4, cudaMemcpyDeviceToHost, s));
        if (host_bo->node_of) HVO_CUDA(cudaMemcpyAsync(host_bo->node_of, bo->node_of, N * c * 4, cudaMemcpyDeviceToHost, s));
        if (host_bo->word_of) HVO_CUDA(cudaMemcpyAsync(host_bo->word_of, bo->word_of, N * c * 4, cudaMemcpyDeviceToHost, s));
    }
    if (h->p.stages & ST_PLANE) {
        cudaStream_t s;
        if (int ds = down_stream(2, plane_stream(L.plane), &s)) return ds;
        if (host) {
            HVO_CUDA(cudaMemcpyAsync(host->n_planes, o.n_planes, N * 4, cudaMemcpyDeviceToHost, s));
            HVO_CUDA(cudaMemcpyAsync(host->planes7, o.planes7, N * (size_t)h->p.max_planes * 56, cudaMemcpyDeviceToHost, s));
            if (host->membership) HVO_CUDA(cudaMemcpyAsync(host->membership, o.membership, N * px * 4, cudaMemcpyDeviceToHost, s));
            if (host->membership8) HVO_CUDA(cudaMemcpyAsync(host->membership8, o.membership8, N * px, cudaMemcpyDeviceToHost, s));
            if (host->membership4) HVO_CUDA(cudaMemcpyAsync(host->membership4, o.membership4, N * (px / 2), cudaMemcpyDeviceToHost, s));
        }
        timeline_mark(s, "end_planes");
        HVO_CUDA(cudaEventRecord(L.join[2], s));
    }
    if (h->p.stages & ST_LINE) {
        cudaStream_t s;
        if (int ds = down_stream(1, line_stream(L.line), &s)) return ds;
        if (host) {
            const size_t c = (size_t)h->max_lines;
            HVO_CUDA(cudaMemcpyAsync(host->line_counts, o.line_counts, N * 4, cudaMemcpyDeviceToHost, s));
            HVO_CUDA(cudaMemcpyAsync(host->keylines, o.keylines, N * c * sizeof(hvo_keyline), cudaMemcpyDeviceToHost, s));
            HVO_CUDA(cudaMemcpyAsync(host->line_desc, o.line_desc, N * c * 32, cudaMemcpyDeviceToHost, s));
            if (host->linevec3) HVO_CUDA(cudaMemcpyAsync(host->linevec3, o.linevec3, N * c * 24, cudaMemcpyDeviceToHost, s));
            if (host_go && host_go->lgrid_counts) {
                HVO_CUDA(cudaMemcpyAsync(host_go->lgrid_counts, go->lgrid_counts, N * kGridCells * 2, cudaMemcpyDeviceToHost, s));
                HVO_CUDA(cudaMemcpyAsync(host_go->lgrid_items, go->lgrid_items, N * 64 * c * 2, cudaMemcpyDeviceToHost, s));
            }
        }
        timeline_mark(s, "end_lines");
        HVO_CUDA(cudaEventRecord(L.join[1], s));
    }
    if (h->p.stages & ST_ORB) {
        cudaStream_t s;
        if (int ds = down_stream(0, orb_stream(L.orb), &s)) return ds;
        if (host) {
            const size_t c = (size_t)h->orb_cap;
            HVO_CUDA(cudaMemcpyAsync(host->kp_counts, o.kp_counts, N * 4, cudaMemcpyDeviceToHost, s));
            HVO_CUDA(cudaMemcpyAsync(host->kps, o.kps, N * c * sizeof(hvo_keypoint), cudaMemcpyDeviceToHost, s));
            HVO_CUDA(cudaMemcpyAsync(host->desc, o.desc, N * c * 32, cudaMemcpyDeviceToHost, s));
            if (host->kp_depth) HVO_CUDA(cudaMemcpyAsync(host->kp_depth, o.kp_depth, N * c * 4, cudaMemcpyDeviceToHost, s));
            if (host->kp_uright) HVO_CUDA(cudaMemcpyAsync(host->kp_uright, o.kp_uright, N * c * 4, cudaMemcpyDeviceToHost, s));
            if (host->kps_un) HVO_CUDA(cudaMemcpyAsync(host->kps_un, o.kps_un, N * c * sizeof(hvo_keypoint), cudaMemcpyDeviceToHost, s));
            if (host_go && host_go->grid_counts) {
                HVO_CUDA(cudaMemcpyAsync(host_go->grid_counts, go->grid_counts, N * kGridCells * 2, cudaMemcpyDeviceToHost, s));
                HVO_CUDA(cudaMemcpyAsync(host_go->grid_items, go->grid_items, N * c * 2, cudaMemcpyDeviceToHost, s));
            }
        }
        timeline_mark(s, "end_orb");
        HVO_CUDA(cudaEventRecord(L.join[0], s));
    }
    if (h->p.stages & ST_NORMALS) {
        cudaStream_t s;
        if (int ds = down_stream(3, normals_stream(L.normals), &s)) return ds;
        if (host && host->normals8) HVO_CUDA(cudaMemcpyAsync(host->normals8, o.normals8, N * (size_t)h->normals_count * 32, cudaMemcpyDeviceToHost, s));
        if (host && host->normals3) HVO_CUDA(cudaMemcpyAsync(host->normals3, o.normals3, N * (size_t)h->normals_count * 12, cudaMemcpyDeviceToHost, s));
        if (host && host_lo) {
            const size_t c = (size_t)lpvo_capacity(h->lpvo_g);
            HVO_CUDA(cudaMemcpyAsync(host_lo->counts, lo->counts, N * 4, cudaMemcpyDeviceToHost, s));
            HVO_CUDA(cudaMemcpyAsync(host_lo->normals3, lo->normals3, N * c * 24, cudaMemcpyDeviceToHost, s));
            HVO_CUDA(cudaMemcpyAsync(host_lo->depth, lo->depth, N * c * 4, cudaMemcpyDeviceToHost, s));
            if (host_lo->pix2) HVO_CUDA(cudaMemcpyAsync(host_lo->pix2, lo->pix2, N * c * 8, cudaMemcpyDeviceToHost, s));
        }
        timeline_mark(s, "end_normals");
        HVO_CUDA(cudaEventRecord(L.join[3], s));
    }
    return HVO_OK;
}

static int wait_joins(hvo_frame* h, cudaStream_t s, FrameLane& L) {
    for (int i = 0; i < 4; ++i)
        if (h->p.stages & (i == 0 ? ST_ORB : i == 1 ? ST_LINE : i == 2 ? ST_PLANE : ST_NORMALS)) HVO_CUDA(cudaStreamWaitEvent(s, L.join[i], 0));
    return HVO_OK;
}

// After the master stream has been synchronised: read the sticky fault record, reset it, report.
static int frame_check_fault(hvo_frame* h) {
    HVO_CUDA(cudaMemcpyAsync(h->h_fault, h->d_fault, 2 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    if (h->h_fault[1] == 0) return HVO_OK;
    const int frame = h->h_fault[0], code = h->h_fault[1];
    h->h_fault[0] = kNoFault; h->h_fault[1] = 0;
    HVO_CUDA(cudaMemcpyAsync(h->d_fault, h->h_fault, 2 * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    set_error("device-side capacity overflow in frame %d of its call:%s%s%s (the outputs of that frame are truncated)", frame,
              (code & FAULT_ORB) ? " ORB quadtree arena" : "", (code & FAULT_LINE) ? " LSD segment buffer" : "",
              (code & FAULT_PLANE) ? " plane refinement queue" : "");
    return HVO_ERR_OVERFLOW;
}

extern "C" {

int hvo_membership4_expand(const uint8_t* labels4, int npixels, int32_t* labels) {
    HVO_CHECK_ARG(labels4 && labels && npixels >= 0 && (npixels & 1) == 0, "bad argument");
    for (int i = 0; i < npixels / 2; ++i) {
        const int a = labels4[i] & 15, b = labels4[i] >> 4;
        labels[2 * i] = a == 15 ? -1 : a;
        labels[2 * i + 1] = b == 15 ? -1 : b;
    }
    return HVO_OK;
}

int hvo_normals3_expand(const float* normals3, const uint16_t* depth16, int width, int height, float fx, float fy, float cx, float cy,
                        float depth_factor, float* normals8) {
    HVO_CHECK_ARG(normals3 && depth16 && normals8 && width > 0 && height > 0, "bad argument");
    const int cw = (width + 2) / 3, ch = (height + 2) / 3, ow = cw / 2, oh = ch / 2;
    for (int i = 0; i < ow * oh; ++i) {
        const int m = 2 * (i / ow) + 1, n = 2 * (i % ow) + 1;
        // the subsampled cloud of Frame::ComputePlanes (Frame.cc:2158-2171), float arithmetic as on the device (no FMA)
        const float z = (float)depth16[(size_t)(3 * m) * width + 3 * n] * depth_factor;
        float* o = normals8 + (size_t)i * 8;
        o[0] = normals3[3 * i]; o[1] = normals3[3 * i + 1]; o[2] = normals3[3 * i + 2];
        o[3] = ((float)(3 * n) - cx) * z / fx;
        o[4] = ((float)(3 * m) - cy) * z / fy;
        o[5] = z;
        o[6] = (float)(n * 3); o[7] = (float)(m * 3);
    }
    return HVO_OK;
}

int hvo_frame_create(const hvo_frame_params* p, int width, int height, int max_batch, int device, hvo_frame** out) {
    HVO_CHECK_ARG(out, "null out");
    *out = nullptr;
    HVO_CHECK_ARG(p, "null params");
    HVO_CHECK_ARG((p->stages & 15) != 0, "no stage selected");
    HVO_CHECK_ARG(max_batch >= 1 && p->max_planes >= 1, "max_batch / max_planes < 1");
    HVO_CHECK_ARG(p->lanes >= 0 && p->lanes <= kMaxLanes, "lanes out of range (0..8)");
    int ndev = 0;
    HVO_CUDA(cudaGetDeviceCount(&ndev));
    if (ndev < 1) { set_error("no CUDA device: libhvofront has no CPU fallback"); return HVO_ERR_CUDA; }
    HVO_CHECK_ARG(device >= 0 && device < ndev, "device index out of range");
    hvo_frame* h = new (std::nothrow) hvo_frame();
    if (!h) { set_error("out of host memory"); return HVO_ERR_ARG; }
    h->p = *p; h->device = device; h->width = width; h->height = height; h->max_batch = max_batch;
    h->undistort = p->distorted != 0 && (p->k1 != 0.f || p->k2 != 0.f || p->p1 != 0.f || p->p2 != 0.f || p->k3 != 0.f);
    h->cam = hvo_camera{p->fx, p->fy, p->cx, p->cy, p->k1, p->k2, p->p1, p->p2, p->k3};
    // default: two lanes once a chunk still holds >= 1024 frames (measured on B200: the ordered kernels, one warp / CTA per
    // frame, need about that many frames per launch; 4 x 256 is 25 % slower than 1 x 1024)
    int nl = p->lanes > 0 ? p->lanes : (max_batch >= 2048 ? 2 : 1);
    if (const char* e = getenv("HVO_FRAME_LANES")) nl = std::min(kMaxLanes, std::max(1, atoi(e)));  // tuning aid
    nl = std::min(nl, max_batch);
    h->nlanes = nl;
    const int cap = (max_batch + nl - 1) / nl;
    int st = HVO_OK;
    // lines and planes are chains of long latency-bound kernels (one warp / CTA per frame): they get the high-priority
    // streams so they are resident from the start; ORB and normals (streaming kernels with large grids) fill in around them
    int prio_lo = 0, prio_hi = 0;
    HVO_CUDA(cudaSetDevice(device));
    HVO_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    const char* env_prio = getenv("HVO_FRAME_PRIORITIES");  // tuning aid: "0" = all streams at the default priority
    if (env_prio && env_prio[0] == '0') prio_lo = prio_hi = 0;
    for (int li = 0; li < nl && st == HVO_OK; ++li) {
        FrameLane& L = h->lane[li];
        L.cap = cap;
        L.d_out = hvo_frame_outputs{};
        if (li > 0) {   // the pipelines (scratch + streams) are lane 0's
            L.orb = h->lane[0].orb; L.line = h->lane[0].line; L.plane = h->lane[0].plane; L.normals = h->lane[0].normals;
            continue;
        }
        L.owns = true;
        set_next_stream_priority(prio_lo);
        if (st == HVO_OK && (p->stages & ST_ORB)) st = hvo_orb_create(&p->orb, width, height, cap, device, &L.orb);
        set_next_stream_priority(prio_hi);
        if (st == HVO_OK && (p->stages & ST_LINE)) st = hvo_line_create(&p->line, width, height, cap, device, &L.line);
        if (st == HVO_OK && L.line) st = hvo_line_set_culling(L.line, p->line_cull);
        if (st == HVO_OK && (p->stages & ST_PLANE)) {
            hvo_plane_params pp{p->fx, p->fy, p->cx, p->cy, p->depth_factor};
            st = hvo_plane_create(&pp, width, height, cap, device, &L.plane);
        }
        set_next_stream_priority(prio_lo);
        if (st == HVO_OK && (p->stages & ST_NORMALS)) {
            hvo_normals_params np{p->fx, p->fy, p->cx, p->cy, p->depth_factor, 0.05f, 10.0f};  // Frame.cc:2179-2180
            st = hvo_normals_create(&np, width, height, cap, device, &L.normals);
        }
    }
    set_next_stream_priority(0);
    if (st != HVO_OK) { hvo_frame_destroy(h); return st; }
    const FrameLane& L0 = h->lane[0];
    h->orb_cap = L0.orb ? hvo_orb_capacity(L0.orb) : 0;
    h->max_lines = L0.line ? hvo_line_max_lines(L0.line) : 0;
    h->normals_count = L0.normals ? hvo_normals_count(L0.normals) : 0;
    h->lpvo_g = lpvo_geom(hvo_plane_params{p->fx, p->fy, p->cx, p->cy, p->depth_factor}, width, height);
    // Frame::ComputeImageBounds; a handle that does not undistort has the reference's k1 == 0 bounds
    h->max_x = (float)width; h->max_y = (float)height;
    if (h->undistort) st = hvo_image_bounds(&h->cam, width, height, &h->min_x, &h->max_x, &h->min_y, &h->max_y);
    if (st != HVO_OK) { hvo_frame_destroy(h); return st; }
    do {
#define HVO_TRY(call) if ((call) != cudaSuccess) { set_error("%s: %s", #call, cudaGetErrorString(cudaGetLastError())); st = HVO_ERR_CUDA; break; }
        HVO_TRY(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        HVO_TRY(cudaEventCreateWithFlags(&h->fork, cudaEventDisableTiming));
        for (auto& e : h->tev) HVO_TRY(cudaEventCreate(&e));
        if (st != HVO_OK) break;
        HVO_TRY(cudaMalloc(&h->d_fault, 2 * sizeof(int)));
        HVO_TRY(cudaHostAlloc(&h->h_fault, 2 * sizeof(int), cudaHostAllocDefault));
        h->h_fault[0] = kNoFault; h->h_fault[1] = 0;
        HVO_TRY(cudaMemcpy(h->d_fault, h->h_fault, 2 * sizeof(int), cudaMemcpyHostToDevice));
        const size_t B = (size_t)cap, px = (size_t)width * height;
        for (int li = 0; li < nl && st == HVO_OK; ++li) {
            FrameLane& L = h->lane[li];
            HVO_TRY(cudaStreamCreateWithFlags(&L.up, cudaStreamNonBlocking));
            HVO_TRY(cudaEventCreateWithFlags(&L.fork, cudaEventDisableTiming));
            HVO_TRY(cudaEventCreateWithFlags(&L.fork_depth, cudaEventDisableTiming));
            for (auto& d : L.down) HVO_TRY(cudaStreamCreateWithFlags(&d, cudaStreamNonBlocking));
            if (st != HVO_OK) break;
            for (auto& e : L.join) HVO_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            if (st != HVO_OK) break;
            for (auto& e : L.cdone) HVO_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            if (st != HVO_OK) break;
            HVO_TRY(cudaMalloc(&L.d_gray, B * px));
            HVO_TRY(cudaMalloc(&L.d_depth, B * px * 2));
            hvo_frame_outputs& o = L.d_out;
            if (L.orb) {
                const size_t c = (size_t)h->orb_cap;
                HVO_TRY(cudaMalloc(&o.kps, B * c * sizeof(hvo_keypoint)));
                HVO_TRY(cudaMalloc(&o.desc, B * c * 32));
                HVO_TRY(cudaMalloc(&o.kp_counts, B * 4));
                HVO_TRY(cudaMalloc(&o.kp_depth, B * c * 4));
                HVO_TRY(cudaMalloc(&o.kp_uright, B * c * 4));
                if (h->undistort) HVO_TRY(cudaMalloc(&o.kps_un, B * c * sizeof(hvo_keypoint)));
            }
            if (L.line) {
                const size_t c = (size_t)h->max_lines;
                HVO_TRY(cudaMalloc(&o.keylines, B * c * sizeof(hvo_keyline)));
                HVO_TRY(cudaMalloc(&o.line_desc, B * c * 32));
                HVO_TRY(cudaMalloc(&o.linevec3, B * c * 24));
                HVO_TRY(cudaMalloc(&o.line_counts, B * 4));
            }
            if (L.plane) {
                HVO_TRY(cudaMalloc(&o.n_planes, B * 4));
                HVO_TRY(cudaMalloc(&o.planes7, B * (size_t)p->max_planes * 56));
                HVO_TRY(cudaMalloc(&o.membership, B * px * 4));
                HVO_TRY(cudaMalloc(&o.membership8, B * px));
                HVO_TRY(cudaMalloc(&o.membership4, B * (px / 2) + 16));
            }
            if (L.normals) {
                HVO_TRY(cudaMalloc(&o.normals8, B * (size_t)h->normals_count * 32));
                HVO_TRY(cudaMalloc(&o.normals3, B * (size_t)h->normals_count * 12));
            }
        }
#undef HVO_TRY
    } while (0);
    if (st != HVO_OK) { hvo_frame_destroy(h); return st; }
    *out = h;
    return HVO_OK;
}

static void frame_detach_vocabulary(hvo_frame* h) {
    for (FrameLane& L : h->lane) {
        hvo_frame_bow_outputs& o = L.d_bow;
        void* bufs[] = {o.bow_counts, o.bow_words, o.bow_values, o.fv_order, o.fv_counts, o.node_of, o.word_of};
        for (void* b : bufs) if (b) cudaFree(b);
        o = hvo_frame_bow_outputs{};
    }
    if (h->d_bow_weight) cudaFree(h->d_bow_weight);
    h->d_bow_weight = nullptr;
    hvo_bow_destroy(h->bow);
    h->bow = nullptr;
}

void hvo_frame_destroy(hvo_frame* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    frame_detach_vocabulary(h);
    for (int li = 0; li < kMaxLanes; ++li) {
        FrameLane& L = h->lane[li];
        if (L.owns) {
            if (L.orb) hvo_orb_destroy(L.orb);
            if (L.line) hvo_line_destroy(L.line);
            if (L.plane) hvo_plane_destroy(L.plane);
            if (L.normals) hvo_normals_destroy(L.normals);
        }
        for (auto& d : L.down) if (d) cudaStreamDestroy(d);
        if (L.fork_depth) cudaEventDestroy(L.fork_depth);
        hvo_frame_outputs& o = L.d_out;
        void* bufs[] = {L.d_gray, L.d_depth, o.kps, o.desc, o.kp_counts, o.kp_depth, o.kp_uright, o.keylines, o.line_desc, o.linevec3,
                        o.line_counts, o.n_planes, o.planes7, o.membership, o.membership8, o.normals8, o.membership4, o.normals3, o.kps_un};
        for (void* b : bufs) if (b) cudaFree(b);
        void* gbufs[] = {L.d_grid.grid_counts, L.d_grid.grid_items, L.d_grid.lgrid_counts, L.d_grid.lgrid_items,
                         L.d_lpvo.normals3, L.d_lpvo.depth, L.d_lpvo.pix2, L.d_lpvo.counts};
        for (void* b : gbufs) if (b) cudaFree(b);
        if (L.fork) cudaEventDestroy(L.fork);
        for (auto& e : L.join) if (e) cudaEventDestroy(e);
        for (auto& e : L.cdone) if (e) cudaEventDestroy(e);
        if (L.up) cudaStreamDestroy(L.up);
    }
    if (h->d_fault) cudaFree(h->d_fault);
    if (h->d_lgrid_bits) cudaFree(h->d_lgrid_bits);
    lpvo_scratch_free(&h->lpvo_scratch);
    if (h->h_fault) cudaFreeHost(h->h_fault);
    if (h->fork) cudaEventDestroy(h->fork);
    for (auto& e : h->tev) if (e) cudaEventDestroy(e);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int hvo_frame_capacities(const hvo_frame* h, int* orb_capacity, int* max_lines, int* normals_count) {
    HVO_CHECK_ARG(h, "null handle");
    if (orb_capacity) *orb_capacity = h->orb_cap;
    if (max_lines) *max_lines = h->max_lines;
    if (normals_count) *normals_count = h->normals_count;
    return HVO_OK;
}

int hvo_frame_lanes(const hvo_frame* h, int* lanes, int* chunk) {
    HVO_CHECK_ARG(h, "null handle");
    if (lanes) *lanes = h->nlanes;
    if (chunk) *chunk = h->lane[0].cap;
    return HVO_OK;
}

static int frame_check_outputs(const hvo_frame* h, const hvo_frame_outputs* o, bool device) {
    HVO_CHECK_ARG(o, "null outputs");
    if (h->p.stages & ST_ORB) HVO_CHECK_ARG(o->kps && o->desc && o->kp_counts, "ORB outputs missing");
    if (h->p.stages & ST_LINE) HVO_CHECK_ARG(o->keylines && o->line_desc && o->line_counts, "line outputs missing");
    if (h->p.stages & ST_PLANE) HVO_CHECK_ARG(o->n_planes && o->planes7 && (o->membership || (!device && (o->membership8 || o->membership4))), "plane outputs missing");
    if (h->p.stages & ST_NORMALS) HVO_CHECK_ARG(o->normals8 || (!device && o->normals3), "normals output missing");
    if (o->kps_un) HVO_CHECK_ARG(h->undistort && (h->p.stages & ST_ORB), "kps_un needs the ORB stage and a distorted camera with coefficients");
    if (o->membership4) {
        HVO_CHECK_ARG(h->p.max_planes <= 15, "membership4 needs max_planes <= 15");
        HVO_CHECK_ARG(((size_t)h->width * h->height) % 16 == 0, "membership4 needs width * height divisible by 16");
        if (device) HVO_CHECK_ARG(o->membership8, "membership4 on the device needs membership8 as well");
    }
    return HVO_OK;
}

static int frame_check_bow_outputs(const hvo_frame* h, const hvo_frame_bow_outputs* b, bool device) {
    if (!b) return HVO_OK;
    HVO_CHECK_ARG(h->bow, "BoW outputs need a vocabulary (hvo_frame_set_vocabulary)");
    HVO_CHECK_ARG(b->bow_counts && b->bow_words && b->bow_values, "bow_counts / bow_words / bow_values missing");
    HVO_CHECK_ARG(!b->fv_order || b->node_of, "fv_order needs node_of");
    if (device) HVO_CHECK_ARG(b->fv_order && b->fv_counts && b->node_of && b->word_of, "device BoW outputs: every array is required");
    return HVO_OK;
}

static int frame_check_grid_outputs(const hvo_frame* h, const hvo_frame_grid_outputs* g, const hvo_frame_outputs* o, bool device) {
    if (!g) return HVO_OK;
    HVO_CHECK_ARG(!g->grid_counts == !g->grid_items && !g->lgrid_counts == !g->lgrid_items, "grid_counts / grid_items and lgrid_counts / lgrid_items go in pairs");
    if (g->grid_counts) {
        HVO_CHECK_ARG(h->p.stages & ST_ORB, "point grid outputs need the ORB stage");
        HVO_CHECK_ARG(h->orb_cap <= 65535, "point grid outputs need orb_capacity <= 65535 (uint16 items)");
        if (device && h->undistort) HVO_CHECK_ARG(o->kps_un, "point grids of an undistorting handle are built on kps_un: the device call needs it");
    }
    if (g->lgrid_counts) {
        HVO_CHECK_ARG(h->p.stages & ST_LINE, "line grid outputs need the line stage");
        HVO_CHECK_ARG(h->max_lines <= 65535, "line grid outputs need max_lines <= 65535 (uint16 items)");
    }
    return HVO_OK;
}

static int frame_check_lpvo_outputs(const hvo_frame* h, const hvo_frame_lpvo_outputs* l, bool device) {
    if (!l) return HVO_OK;
    HVO_CHECK_ARG(h->p.stages & ST_NORMALS, "LPVO outputs need the normals stage");
    HVO_CHECK_ARG(l->normals3 && l->depth && l->counts, "LPVO normals3 / depth / counts missing");
    if (device) HVO_CHECK_ARG(l->pix2, "device LPVO outputs: every array is required");
    return HVO_OK;
}

// Allocated by the first call that asks for LPVO outputs, kept until destroy: the chain's scratch (kLpvoFrames frames, shared by the
// lanes) and, for the host calls, every lane's device staging of the four arrays.
static int frame_reserve_lpvo(hvo_frame* h, bool host) {
    if (!h->lpvo_scratch.frames) {
        const int st = lpvo_scratch_alloc(h->lpvo_g, std::min(kLpvoFrames, h->lane[0].cap), &h->lpvo_scratch);
        if (st != HVO_OK) { lpvo_scratch_free(&h->lpvo_scratch); return st; }
    }
    const size_t B = (size_t)h->lane[0].cap, c = (size_t)lpvo_capacity(h->lpvo_g);
    for (int li = 0; host && li < h->nlanes; ++li) {
        hvo_frame_lpvo_outputs& o = h->lane[li].d_lpvo;
        if (!o.normals3) HVO_CUDA(cudaMalloc(&o.normals3, B * c * 24));
        if (!o.depth) HVO_CUDA(cudaMalloc(&o.depth, B * c * 4));
        if (!o.pix2) HVO_CUDA(cudaMalloc(&o.pix2, B * c * 8));
        if (!o.counts) HVO_CUDA(cudaMalloc(&o.counts, B * 4));
    }
    return HVO_OK;
}

// Allocated by the first call that asks for a grid, kept until destroy: the line grid's bit rows (one chunk, shared by the lanes) and, for
// the host calls, every lane's device staging of the requested grids.
static int frame_reserve_grids(hvo_frame* h, const hvo_frame_grid_outputs* g, bool host) {
    const size_t B = (size_t)h->lane[0].cap;
    if (g->lgrid_counts && !h->d_lgrid_bits) HVO_CUDA(cudaMalloc(&h->d_lgrid_bits, B * kGridCells * div_up(h->max_lines, 32) * sizeof(uint32_t)));
    for (int li = 0; host && li < h->nlanes; ++li) {
        hvo_frame_grid_outputs& o = h->lane[li].d_grid;
        if (g->grid_counts) {
            if (!o.grid_counts) HVO_CUDA(cudaMalloc(&o.grid_counts, B * kGridCells * 2));
            if (!o.grid_items) HVO_CUDA(cudaMalloc(&o.grid_items, B * h->orb_cap * 2));
        }
        if (g->lgrid_counts) {
            if (!o.lgrid_counts) HVO_CUDA(cudaMalloc(&o.lgrid_counts, B * kGridCells * 2));
            if (!o.lgrid_items) HVO_CUDA(cudaMalloc(&o.lgrid_items, B * 64 * h->max_lines * 2));
        }
    }
    return HVO_OK;
}

int hvo_frame_set_vocabulary(hvo_frame* h, int n_nodes, const int32_t* child_start, const int32_t* child_ids, const uint8_t* node_desc,
                             const double* node_weight, const int32_t* node_word, int depth_levels, int levelsup) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CHECK_ARG(n_nodes >= 0, "n_nodes < 0");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaStreamSynchronize(h->stream));   // queued calls may still use the BoW buffers
    frame_detach_vocabulary(h);
    if (n_nodes == 0) return HVO_OK;
    HVO_CHECK_ARG(h->p.stages & ST_ORB, "a vocabulary needs the ORB stage");
    HVO_CHECK_ARG(h->orb_cap <= bow_max_features(), "orb_capacity > 4096: too many features per frame for the BoW sort");
    int st = hvo_bow_create(h->device, &h->bow);   // (also makes h->device current)
    if (st == HVO_OK) st = hvo_bow_set_vocabulary(h->bow, n_nodes, child_start, child_ids, node_desc, node_weight, node_word, depth_levels);
    const size_t c = (size_t)h->orb_cap;
    do {
#define HVO_TRY(call) if ((call) != cudaSuccess) { set_error("%s: %s", #call, cudaGetErrorString(cudaGetLastError())); st = HVO_ERR_CUDA; break; }
        if (st != HVO_OK) break;
        HVO_TRY(cudaMalloc(&h->d_bow_weight, (size_t)h->lane[0].cap * c * 8));
        for (int li = 0; li < h->nlanes && st == HVO_OK; ++li) {
            const size_t B = (size_t)h->lane[li].cap;
            hvo_frame_bow_outputs& o = h->lane[li].d_bow;
            HVO_TRY(cudaMalloc(&o.bow_counts, B * 4));
            HVO_TRY(cudaMalloc(&o.bow_words, B * c * 4));
            HVO_TRY(cudaMalloc(&o.bow_values, B * c * 8));
            HVO_TRY(cudaMalloc(&o.fv_order, B * c * 4));
            HVO_TRY(cudaMalloc(&o.fv_counts, B * 4));
            HVO_TRY(cudaMalloc(&o.node_of, B * c * 4));
            HVO_TRY(cudaMalloc(&o.word_of, B * c * 4));
        }
#undef HVO_TRY
    } while (0);
    if (st != HVO_OK) { frame_detach_vocabulary(h); return st; }
    h->levelsup = levelsup;
    return HVO_OK;
}

int hvo_frame_extract_batch_device_lpvo(hvo_frame* h, const uint8_t* d_gray, const uint16_t* d_depth16, int nframes, const hvo_frame_outputs* d_out,
                                        const hvo_frame_bow_outputs* d_bow, const hvo_frame_grid_outputs* d_grid, const hvo_frame_lpvo_outputs* d_lpvo) {
    HVO_CHECK_ARG(h && d_gray && d_depth16, "null argument");
    HVO_CHECK_ARG(nframes >= 1 && nframes <= h->max_batch, "nframes out of range for this handle");
    int st = frame_check_outputs(h, d_out, true);
    if (st == HVO_OK) st = frame_check_bow_outputs(h, d_bow, true);
    if (st == HVO_OK) st = frame_check_grid_outputs(h, d_grid, d_out, true);
    if (st == HVO_OK) st = frame_check_lpvo_outputs(h, d_lpvo, true);
    if (st != HVO_OK) return st;
    if (h->p.stages & ST_ORB) HVO_CHECK_ARG(d_out->kp_depth && d_out->kp_uright, "kp_depth / kp_uright missing");
    if (h->p.stages & ST_LINE) HVO_CHECK_ARG(d_out->linevec3, "linevec3 missing");
    HVO_CUDA(cudaSetDevice(h->device));
    if (d_grid && (st = frame_reserve_grids(h, d_grid, false)) != HVO_OK) return st;
    if (d_lpvo && (st = frame_reserve_lpvo(h, false)) != HVO_OK) return st;
    const size_t px = (size_t)h->width * h->height;
    HVO_CUDA(cudaEventRecord(h->fork, h->stream));
    int launches = 0, used = 0;
    // the batch is spread evenly over the lanes; the chunks compute one after the other (measured: two chunks whose ordered
    // kernels overlap are slower than the same chunks back to back)
    // as few chunks as the lane capacity allows, of equal size (the ordered kernels are latency-bound: one warp / CTA per frame, so
    // a chunk of 1024 is faster than two of 512)
    const int nchunks = (nframes + h->lane[0].cap - 1) / h->lane[0].cap;
    const int per = (nframes + nchunks - 1) / nchunks;
    for (int off = 0; off < nframes; off += per, ++used) {
        FrameLane& L = h->lane[used];
        const int n = std::min(per, nframes - off);
        const hvo_frame_bow_outputs bo = d_bow ? outputs_at(h, *d_bow, (size_t)off) : hvo_frame_bow_outputs{};
        const hvo_frame_grid_outputs go = d_grid ? outputs_at(h, *d_grid, (size_t)off) : hvo_frame_grid_outputs{};
        const hvo_frame_lpvo_outputs lo = d_lpvo ? outputs_at(h, *d_lpvo, (size_t)off) : hvo_frame_lpvo_outputs{};
        st = lane_launch(h, L, h->fork, nullptr, d_gray + (size_t)off * px, d_depth16 + (size_t)off * px, n, off, outputs_at(h, *d_out, (size_t)off), nullptr,
                         d_bow ? &bo : nullptr, nullptr, d_grid ? &go : nullptr, nullptr, d_lpvo ? &lo : nullptr, nullptr, &launches,
                         h->last_lane >= 0 ? &h->lane[h->last_lane] : nullptr);
        if (st != HVO_OK) return st;
        h->last_lane = used;
    }
    for (int li = 0; li < used; ++li) {
        st = wait_joins(h, h->stream, h->lane[li]);
        if (st != HVO_OK) return st;
    }
    h->last_launches = launches;
    return HVO_OK;
}

int hvo_frame_extract_batch_device_grid(hvo_frame* h, const uint8_t* d_gray, const uint16_t* d_depth16, int nframes, const hvo_frame_outputs* d_out,
                                        const hvo_frame_bow_outputs* d_bow, const hvo_frame_grid_outputs* d_grid) {
    return hvo_frame_extract_batch_device_lpvo(h, d_gray, d_depth16, nframes, d_out, d_bow, d_grid, nullptr);
}

int hvo_frame_extract_batch_device_bow(hvo_frame* h, const uint8_t* d_gray, const uint16_t* d_depth16, int nframes, const hvo_frame_outputs* d_out,
                                       const hvo_frame_bow_outputs* d_bow) {
    return hvo_frame_extract_batch_device_grid(h, d_gray, d_depth16, nframes, d_out, d_bow, nullptr);
}

int hvo_frame_extract_batch_device(hvo_frame* h, const uint8_t* d_gray, const uint16_t* d_depth16, int nframes, const hvo_frame_outputs* d_out) {
    return hvo_frame_extract_batch_device_grid(h, d_gray, d_depth16, nframes, d_out, nullptr, nullptr);
}

int hvo_frame_extract_batch_async_lpvo(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                                       const hvo_frame_bow_outputs* bow, const hvo_frame_grid_outputs* grid, const hvo_frame_lpvo_outputs* lpvo) {
    HVO_CHECK_ARG(h && gray && depth16, "null argument");
    HVO_CHECK_ARG(nframes >= 1, "nframes < 1");
    int st = frame_check_outputs(h, out, false);
    if (st == HVO_OK) st = frame_check_bow_outputs(h, bow, false);
    if (st == HVO_OK) st = frame_check_grid_outputs(h, grid, out, false);
    if (st == HVO_OK) st = frame_check_lpvo_outputs(h, lpvo, false);
    if (st != HVO_OK) return st;
    HVO_CUDA(cudaSetDevice(h->device));
    if (grid && (st = frame_reserve_grids(h, grid, true)) != HVO_OK) return st;
    if (lpvo && (st = frame_reserve_lpvo(h, true)) != HVO_OK) return st;
    const size_t px = (size_t)h->width * h->height;
    // chunks: as few as the lane capacity allows, of equal size.  Chunks go round-robin through the lanes ACROSS calls
    // (next_lane), so that the upload of a one-chunk call overlaps the kernels of the previous call on the other lane.
    const int cap = h->lane[0].cap;
    const int nchunks = (nframes + cap - 1) / cap;
    const int per = (nframes + nchunks - 1) / nchunks;
    int launches = 0, k = 0;
    bool lane_used[kMaxLanes] = {false};
    for (int off = 0; off < nframes; off += per, ++k) {
        const int li = h->next_lane;
        h->next_lane = (h->next_lane + 1) % h->nlanes;
        lane_used[li] = true;
        FrameLane& L = h->lane[li];
        const int n = std::min(per, nframes - off);
        st = wait_joins(h, L.up, L);  // the lane's previous chunk (of this or an earlier call) must be done with the staging buffers
        if (st != HVO_OK) return st;
        // depth first: the plane pipeline (first in the serial schedule) needs nothing else, the gray upload runs beside its kernels
        HVO_CUDA(cudaMemcpyAsync(L.d_depth, depth16 + (size_t)off * px, (size_t)n * px * 2, cudaMemcpyHostToDevice, L.up));
        HVO_CUDA(cudaEventRecord(L.fork_depth, L.up));
        HVO_CUDA(cudaMemcpyAsync(L.d_gray, gray + (size_t)off * px, (size_t)n * px, cudaMemcpyHostToDevice, L.up));
        HVO_CUDA(cudaEventRecord(L.fork, L.up));
        hvo_frame_outputs d = L.d_out;
        if (!out->membership8 && !out->membership4) d.membership8 = nullptr;
        if (!out->membership4) d.membership4 = nullptr;
        if (!out->normals3) d.normals3 = nullptr;
        if (!out->kps_un && !(grid && grid->grid_counts)) d.kps_un = nullptr;   // (the point grid is built on kps_un)
        hvo_frame_grid_outputs dg{};   // the requested pairs of the lane's grid staging
        if (grid && grid->grid_counts) { dg.grid_counts = L.d_grid.grid_counts; dg.grid_items = L.d_grid.grid_items; }
        if (grid && grid->lgrid_counts) { dg.lgrid_counts = L.d_grid.lgrid_counts; dg.lgrid_items = L.d_grid.lgrid_items; }
        const hvo_frame_outputs hostk = outputs_at(h, *out, (size_t)off);
        const hvo_frame_bow_outputs hostb = bow ? outputs_at(h, *bow, (size_t)off) : hvo_frame_bow_outputs{};
        const hvo_frame_grid_outputs hostg = grid ? outputs_at(h, *grid, (size_t)off) : hvo_frame_grid_outputs{};
        const hvo_frame_lpvo_outputs hostl = lpvo ? outputs_at(h, *lpvo, (size_t)off) : hvo_frame_lpvo_outputs{};
        st = lane_launch(h, L, L.fork, L.fork_depth, L.d_gray, L.d_depth, n, off, d, &hostk, bow ? &L.d_bow : nullptr, bow ? &hostb : nullptr,
                         grid ? &dg : nullptr, grid ? &hostg : nullptr, lpvo ? &L.d_lpvo : nullptr, lpvo ? &hostl : nullptr, &launches,
                         h->last_lane >= 0 ? &h->lane[h->last_lane] : nullptr);
        if (st != HVO_OK) return st;
        h->last_lane = li;
    }
    for (int li = 0; li < h->nlanes; ++li) {
        if (!lane_used[li]) continue;
        st = wait_joins(h, h->stream, h->lane[li]);
        if (st != HVO_OK) return st;
    }
    h->last_launches = launches;
    return HVO_OK;
}

int hvo_frame_extract_batch_async_grid(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                                       const hvo_frame_bow_outputs* bow, const hvo_frame_grid_outputs* grid) {
    return hvo_frame_extract_batch_async_lpvo(h, gray, depth16, nframes, out, bow, grid, nullptr);
}

int hvo_frame_extract_batch_async_bow(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                                      const hvo_frame_bow_outputs* bow) {
    return hvo_frame_extract_batch_async_grid(h, gray, depth16, nframes, out, bow, nullptr);
}

int hvo_frame_extract_batch_async(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out) {
    return hvo_frame_extract_batch_async_grid(h, gray, depth16, nframes, out, nullptr, nullptr);
}

int hvo_frame_extract_batch_lpvo(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                                 const hvo_frame_bow_outputs* bow, const hvo_frame_grid_outputs* grid, const hvo_frame_lpvo_outputs* lpvo) {
    const int st = hvo_frame_extract_batch_async_lpvo(h, gray, depth16, nframes, out, bow, grid, lpvo);
    if (st != HVO_OK) return st;
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return frame_check_fault(h);
}

int hvo_frame_extract_batch_grid(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                                 const hvo_frame_bow_outputs* bow, const hvo_frame_grid_outputs* grid) {
    return hvo_frame_extract_batch_lpvo(h, gray, depth16, nframes, out, bow, grid, nullptr);
}

int hvo_frame_extract_batch_bow(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                                const hvo_frame_bow_outputs* bow) {
    return hvo_frame_extract_batch_grid(h, gray, depth16, nframes, out, bow, nullptr);
}

int hvo_frame_extract_batch(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out) {
    return hvo_frame_extract_batch_grid(h, gray, depth16, nframes, out, nullptr, nullptr);
}

int hvo_frame_image_bounds(const hvo_frame* h, float* min_x, float* max_x, float* min_y, float* max_y) {
    HVO_CHECK_ARG(h && min_x && max_x && min_y && max_y, "null argument");
    *min_x = h->min_x; *max_x = h->max_x; *min_y = h->min_y; *max_y = h->max_y;
    return HVO_OK;
}

int hvo_frame_line_grid_capacity(const hvo_frame* h) { return h ? 64 * h->max_lines : 0; }

int hvo_frame_lpvo_capacity(const hvo_frame* h) { return h && (h->p.stages & ST_NORMALS) ? lpvo_capacity(h->lpvo_g) : 0; }

int hvo_frame_last_launches(const hvo_frame* h) { return h ? h->last_launches : 0; }
int hvo_frame_sync(hvo_frame* h) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaStreamSynchronize(h->stream));
    return frame_check_fault(h);
}
int hvo_frame_timer_start(hvo_frame* h) {
    HVO_CHECK_ARG(h, "null handle");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[0], h->stream));
    return HVO_OK;
}
int hvo_frame_timer_stop(hvo_frame* h, float* ms_out) {
    HVO_CHECK_ARG(h && ms_out, "null argument");
    HVO_CUDA(cudaSetDevice(h->device));
    HVO_CUDA(cudaEventRecord(h->tev[1], h->stream));
    HVO_CUDA(cudaEventSynchronize(h->tev[1]));
    HVO_CUDA(cudaEventElapsedTime(ms_out, h->tev[0], h->tev[1]));
    return frame_check_fault(h);
}

}  // extern "C"
