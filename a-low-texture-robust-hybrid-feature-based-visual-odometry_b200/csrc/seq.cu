// Offline sequences on several GPUs of one box, in ONE process: frames are partitioned across the devices (contiguous ranges, so the
// host gather is "every device writes its own rows of the caller's arrays"), one host thread + one hvo_frame handle (its streams)
// per device, no NCCL, no collective.  This is config 5 of BASELINE.json as the reference would use it: extraction has no
// cross-frame state (SURVEY.md section 8e), so Frame construction of different frames is independent work.
#include <algorithm>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "hvo_common.cuh"

using namespace hvo;

struct hvo_seq {
    std::vector<int> devices;
    std::vector<hvo_frame*> handles;
    int width = 0, height = 0, call_frames = 0;
    hvo_frame_params p;
    int orb_cap = 0, max_lines = 0, normals_count = 0, lpvo_cap = 0;
    float last_ms = 0.f;                 // slowest device of the last call (CUDA events on its master stream)
    std::vector<float> dev_ms;
};

static hvo_frame_outputs seq_outputs_at(const hvo_seq* s, const hvo_frame_outputs& o, size_t off) {
    const size_t c = (size_t)s->orb_cap, l = (size_t)s->max_lines, px = (size_t)s->width * s->height, nc = (size_t)s->normals_count;
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
    if (o.planes7) r.planes7 = o.planes7 + off * (size_t)s->p.max_planes * 7;
    if (o.membership) r.membership = o.membership + off * px;
    if (o.membership8) r.membership8 = o.membership8 + off * px;
    if (o.membership4) r.membership4 = o.membership4 + off * (px / 2);
    if (o.normals8) r.normals8 = o.normals8 + off * nc * 8;
    if (o.normals3) r.normals3 = o.normals3 + off * nc * 3;
    if (o.kps_un) r.kps_un = o.kps_un + off * c;
    return r;
}
static hvo_frame_bow_outputs seq_outputs_at(const hvo_seq* s, const hvo_frame_bow_outputs& o, size_t off) {
    const size_t c = (size_t)s->orb_cap;
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

static hvo_frame_grid_outputs seq_outputs_at(const hvo_seq* s, const hvo_frame_grid_outputs& o, size_t off) {
    hvo_frame_grid_outputs r = o;
    if (o.grid_counts) r.grid_counts = o.grid_counts + off * 3072;
    if (o.grid_items) r.grid_items = o.grid_items + off * (size_t)s->orb_cap;
    if (o.lgrid_counts) r.lgrid_counts = o.lgrid_counts + off * 3072;
    if (o.lgrid_items) r.lgrid_items = o.lgrid_items + off * 64 * (size_t)s->max_lines;
    return r;
}

static hvo_frame_lpvo_outputs seq_outputs_at(const hvo_seq* s, const hvo_frame_lpvo_outputs& o, size_t off) {
    const size_t c = (size_t)s->lpvo_cap;
    hvo_frame_lpvo_outputs r = o;
    if (o.normals3) r.normals3 = o.normals3 + off * c * 3;
    if (o.depth) r.depth = o.depth + off * c;
    if (o.pix2) r.pix2 = o.pix2 + off * c * 2;
    if (o.counts) r.counts = o.counts + off;
    return r;
}

extern "C" {

int hvo_seq_create(const hvo_frame_params* p, int width, int height, const int* devices, int ndevices, int frames_per_call, hvo_seq** out) {
    HVO_CHECK_ARG(out, "null out");
    *out = nullptr;
    HVO_CHECK_ARG(p && devices && ndevices >= 1 && ndevices <= 64 && frames_per_call >= 1, "bad argument");
    hvo_seq* s = new (std::nothrow) hvo_seq();
    if (!s) { set_error("out of host memory"); return HVO_ERR_ARG; }
    s->p = *p; s->width = width; s->height = height; s->call_frames = frames_per_call;
    s->devices.assign(devices, devices + ndevices);
    s->handles.assign(ndevices, nullptr);
    s->dev_ms.assign(ndevices, 0.f);
    for (int i = 0; i < ndevices; ++i) {
        const int st = hvo_frame_create(p, width, height, frames_per_call, devices[i], &s->handles[i]);
        if (st != HVO_OK) { hvo_seq_destroy(s); return st; }
    }
    hvo_frame_capacities(s->handles[0], &s->orb_cap, &s->max_lines, &s->normals_count);
    s->lpvo_cap = hvo_frame_lpvo_capacity(s->handles[0]);
    *out = s;
    return HVO_OK;
}

void hvo_seq_destroy(hvo_seq* s) {
    if (!s) return;
    for (hvo_frame* h : s->handles) if (h) hvo_frame_destroy(h);
    delete s;
}

int hvo_seq_devices(const hvo_seq* s) { return s ? (int)s->devices.size() : 0; }

int hvo_seq_capacities(const hvo_seq* s, int* orb_capacity, int* max_lines, int* normals_count) {
    HVO_CHECK_ARG(s, "null handle");
    if (orb_capacity) *orb_capacity = s->orb_cap;
    if (max_lines) *max_lines = s->max_lines;
    if (normals_count) *normals_count = s->normals_count;
    return HVO_OK;
}

// frames [first, first + count) of device d out of n: contiguous, sizes differ by at most one
void hvo_seq_shard(int nframes, int ndevices, int d, int* first, int* count) {
    const int base = nframes / ndevices, rem = nframes % ndevices;
    *first = d * base + std::min(d, rem);
    *count = base + (d < rem ? 1 : 0);
}

int hvo_seq_set_vocabulary(hvo_seq* s, int n_nodes, const int32_t* child_start, const int32_t* child_ids, const uint8_t* node_desc,
                           const double* node_weight, const int32_t* node_word, int depth_levels, int levelsup) {
    HVO_CHECK_ARG(s, "null handle");
    for (size_t d = 0; d < s->handles.size(); ++d) {
        const int st = hvo_frame_set_vocabulary(s->handles[d], n_nodes, child_start, child_ids, node_desc, node_weight, node_word, depth_levels, levelsup);
        if (st != HVO_OK) return st;
    }
    return HVO_OK;
}

int hvo_seq_extract_lpvo(hvo_seq* s, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                         const hvo_frame_bow_outputs* bow, const hvo_frame_grid_outputs* grid, const hvo_frame_lpvo_outputs* lpvo) {
    HVO_CHECK_ARG(s && gray && depth16 && out && nframes >= 1, "bad argument");
    const int nd = (int)s->devices.size();
    const size_t px = (size_t)s->width * s->height;
    std::vector<int> status(nd, HVO_OK);
    std::vector<std::string> errors(nd);
    std::vector<std::thread> workers;
    for (int d = 0; d < nd; ++d) {
        workers.emplace_back([&, d]() {
            int first = 0, count = 0;
            hvo_seq_shard(nframes, nd, d, &first, &count);
            if (count == 0) return;
            hvo_frame* h = s->handles[d];
            int st = hvo_frame_timer_start(h);
            // queued calls of at most call_frames frames: the upload of call k+1 overlaps the kernels of call k
            for (int off = 0; st == HVO_OK && off < count; off += s->call_frames) {
                const int n = std::min(s->call_frames, count - off);
                const hvo_frame_outputs o = seq_outputs_at(s, *out, (size_t)(first + off));
                const hvo_frame_bow_outputs b = bow ? seq_outputs_at(s, *bow, (size_t)(first + off)) : hvo_frame_bow_outputs{};
                const hvo_frame_grid_outputs g = grid ? seq_outputs_at(s, *grid, (size_t)(first + off)) : hvo_frame_grid_outputs{};
                const hvo_frame_lpvo_outputs l = lpvo ? seq_outputs_at(s, *lpvo, (size_t)(first + off)) : hvo_frame_lpvo_outputs{};
                st = hvo_frame_extract_batch_async_lpvo(h, gray + (size_t)(first + off) * px, depth16 + (size_t)(first + off) * px, n, &o, bow ? &b : nullptr,
                                                        grid ? &g : nullptr, lpvo ? &l : nullptr);
            }
            float ms = 0.f;
            const int st2 = hvo_frame_timer_stop(h, &ms);   // waits for every download of this device; reports device-side faults
            s->dev_ms[d] = ms;
            status[d] = st != HVO_OK ? st : st2;
            if (status[d] != HVO_OK) errors[d] = hvo_last_error();   // the error string is per thread
        });
    }
    for (auto& w : workers) w.join();
    s->last_ms = *std::max_element(s->dev_ms.begin(), s->dev_ms.end());
    for (int d = 0; d < nd; ++d)
        if (status[d] != HVO_OK) { set_error("device %d: %s", s->devices[d], errors[d].c_str()); return status[d]; }
    return HVO_OK;
}

int hvo_seq_extract_grid(hvo_seq* s, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                         const hvo_frame_bow_outputs* bow, const hvo_frame_grid_outputs* grid) {
    return hvo_seq_extract_lpvo(s, gray, depth16, nframes, out, bow, grid, nullptr);
}

int hvo_seq_extract_bow(hvo_seq* s, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                        const hvo_frame_bow_outputs* bow) {
    return hvo_seq_extract_grid(s, gray, depth16, nframes, out, bow, nullptr);
}

int hvo_seq_extract(hvo_seq* s, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out) {
    return hvo_seq_extract_grid(s, gray, depth16, nframes, out, nullptr, nullptr);
}

int hvo_seq_image_bounds(const hvo_seq* s, float* min_x, float* max_x, float* min_y, float* max_y) {
    HVO_CHECK_ARG(s, "null handle");
    return hvo_frame_image_bounds(s->handles[0], min_x, max_x, min_y, max_y);
}

int hvo_seq_line_grid_capacity(const hvo_seq* s) { return s ? hvo_frame_line_grid_capacity(s->handles[0]) : 0; }

int hvo_seq_lpvo_capacity(const hvo_seq* s) { return s ? s->lpvo_cap : 0; }

float hvo_seq_last_ms(const hvo_seq* s) { return s ? s->last_ms : 0.f; }

}  // extern "C"
