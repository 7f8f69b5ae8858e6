// ORB extractor, B200-native.  Device-visible geometry + host-side handle.
// Replaces ORB_SLAM2::ORBextractor (reference include/ORBextractor.h:46-110, src/ORBextractor.cc).
#pragma once
#include <vector>

#include "hvo_common.cuh"

namespace hvo {

struct LevelGeom {
    int w, h, pitch;          // level image size; pitch in bytes (levels >= 1: 128-byte aligned)
    long long img_off;        // byte offset of the level inside one frame's pyramid block (levels >= 1)
    int minBX, minBY, maxBX, maxBY;  // FAST search window (ORBextractor.cc:771-774)
    int nCols, nRows, wCell, hCell;  // cell grid (ORBextractor.cc:779-785)
    int quota;                // mnFeaturesPerLevel[l]
    int cand_off, cand_cap;   // slice of the per-frame candidate arena
    int kp_off, kp_cap;       // slice of the per-frame quadtree output arena
    int nIni;                 // quadtree roots (ORBextractor.cc:541)
    float hX;                 // root width
    float scale;              // mvScaleFactor[l]
    float kp_size;            // (float)(int)(31 * scale)
};

struct OrbGeom {
    int nlevels, width, height;
    int cand_total, kp_total;  // per-frame arena sizes (entries)
    int out_cap;               // rows per frame in the caller's kps/desc buffers
    long long pyr_frame_bytes; // bytes per frame of levels >= 1
    LevelGeom lv[HVO_MAX_LEVELS];
};

struct ImgSrc {  // where the pyramid of frame f lives
    const uint8_t* l0;  // level 0 = the caller's frames
    long long l0_frame; // bytes per frame
    int l0_pitch;
    uint8_t* pyr;       // levels >= 1
};

struct StripDesc {  // one FAST strip = the detection zones of a run of cells of one reference cell row (zone = ROI minus the 3-px ring)
    short level, x0, y0, zw, zh;  // zone origin (level coords) and size: zw = sum of the cells' zone widths
    short wcell, ncells;          // cell pitch in x (the last cell of a row may be narrower), cells in the run
    short tstride;                // bytes per row of the band in shared memory (multiple of 16)
    int score_off;                // byte offset of the score map behind the band
};

}  // namespace hvo

struct hvo_orb {
    hvo_orb_params p;
    int width = 0, height = 0, max_batch = 0, device = 0;
    hvo::OrbGeom g;
    std::vector<float> sf, isf, sigma2, isigma2;
    std::vector<int> nfeat, umax;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t tev[2] = {nullptr, nullptr};
    bool profiling = false, have_stage_times = false;
    int last_launches = 0, last_nframes = 0;
    int nstrips = 0, max_quota = 0;
    size_t oct_smem = 0, fast_smem = 0;
    // device buffers
    uint8_t* d_l0 = nullptr;        // staging for host frames [B][h][w]
    uint16_t* d_depth = nullptr;    // staging for host depth [B][h][w]
    uint8_t* d_pyr = nullptr;       // [B][pyr_frame_bytes]
    int2* d_xtab = nullptr;         // per level: {sx, w0 | w1 << 16}
    int4* d_ytab = nullptr;         // per level: {sy0, sy1, b0, b1}
    std::vector<int> xtab_off, ytab_off;
    std::vector<char> resize_tile_ok;  // per level: the shared-memory band kernel applies (pyramid factor small enough)
    hvo::StripDesc* d_strips = nullptr;
    uint32_t* d_cand = nullptr;     // [B][cand_total] packed x | y << 12 | score << 24
    int* d_ncand = nullptr;         // [B][nlevels]
    uint16_t* d_knode = nullptr;    // [B][cand_total] quadtree scratch
    uint32_t* d_okp = nullptr;      // [B][kp_total] quadtree output, list order
    int* d_on = nullptr;            // [B][nlevels]
    int* d_err = nullptr;           // device error flag
    hvo_keypoint* d_kps = nullptr;  // [B][out_cap]   (host-path staging)
    uint8_t* d_desc = nullptr;      // [B][out_cap][32]
    int32_t* d_counts = nullptr;    // [B]
    float* d_kpdepth = nullptr;     // [B][out_cap]
    float* d_kpuright = nullptr;    // [B][out_cap]
    const uint8_t* last_l0 = nullptr;  // level-0 source of the last call (for inspection)

    int init();
    void release();
    int run(const uint8_t* d_gray, int nframes, hvo_keypoint* d_kps_out, uint8_t* d_desc_out, int32_t* d_counts_out,
            const uint16_t* d_depth16, const hvo_rgbd_params* rgbd, float* d_kp_depth, float* d_kp_uright);
    int undistort(const hvo_camera& cam, const hvo_keypoint* d_kps, const int32_t* d_counts, int nframes, const float* d_kp_depth, float bf,
                  hvo_keypoint* d_kps_un, float* d_kp_uright);
};
