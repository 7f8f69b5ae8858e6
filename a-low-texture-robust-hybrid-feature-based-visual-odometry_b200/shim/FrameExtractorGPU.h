// Drop-in for the extraction block of Frame::Frame(imGray, imDepth, timeStamp, extractors, ...) (reference src/Frame.cc:188-233 and
// the grid threads at :304-307): one frame call (hvo_frame_extract_batch_lpvo, max_batch = 1, the pipelines side by side) fills every
// member that threads A-C and the two grid threads fill, and, on request, returns the rows thread D's Manhattan::computeNormalsLPVO
// pushes back.  INTEGRATION.md §5 shows the patch:
//
//     hvo_shim::FrameExtractorGPU fx(w, h, nFeatures, fScaleFactor, nLevels, fIniThFAST, fMinThFAST,   // Tracking, once
//                                    1, 1.2f, nLSDFeature, 0.125, mK, mDistCoef, mbf, mDepthMapFactor);
//     fx.setVocabulary(*mpORBvocabulary);                                                           // optional: mBowVec / mFeatVec
//     fx.extract(imGray, imDepth, *this, !bManhInit, &ptNormals, &depthNormals);                    // Frame::Frame, instead of the threads
//
// Filled: N, mvKeys, mvKeysUn, mDescriptors (N x 32 CV_8U), mvDepth, mvuRight; NL, mvKeylinesUn, mLdesc, mvKeyLineFunctions (after
// cullingLine); planeDetector (plane_num_, plane_vertices_, cloud.vertices of member pixels, plane_filter.extractedPlanes);
// vSurfaceNormal; mGrid, mGridForLine; mBowVec / mFeatVec with a vocabulary attached.  The first successful call also sets the static
// mnMinX .. mnMaxY and mfGridElementWidthInv / mfGridElementHeightInv from the handle's bounds (hvo_frame_image_bounds), which is what
// the reference's first Frame computes in ComputeImageBounds.  The scale tables stay with the reference's ORBextractor (Frame.cc:162-168).
//
// Errors (no device, an image that is not CV_8UC1, a depth that is not CV_16UC1, a size other than the handle's, any C-ABI failure)
// print the reason and leave every output empty, as the per-class shims do: the tracker then sees a textureless frame.  One object per
// Tracking, used by one thread at a time, like the reference's extractors.
#ifndef HVO_SHIM_FRAMEEXTRACTORGPU_H
#define HVO_SHIM_FRAMEEXTRACTORGPU_H

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include <opencv2/core/core.hpp>

#include "hvo_capi.h"
#include "FrameGridGPU.h"
#include "ORBVocabularyGPU.h"
#include "PlaneExtractor.h"
#include "UndistortGPU.h"

namespace hvo_shim {

// One row of hvo_normals_compute_batch / normals8 (normal.xyz, cameraPosition.xyz, FramePosition.x, .y) into the reference's
// SurfaceNormal, each field converted to its own member type.
template <class SurfaceNormalT>
inline void setSurfaceNormal(SurfaceNormalT& s, const float* e) {
    s.normal.x = (decltype(s.normal.x))e[0];
    s.normal.y = (decltype(s.normal.y))e[1];
    s.normal.z = (decltype(s.normal.z))e[2];
    s.cameraPosition.x = (decltype(s.cameraPosition.x))e[3];
    s.cameraPosition.y = (decltype(s.cameraPosition.y))e[4];
    s.cameraPosition.z = (decltype(s.cameraPosition.z))e[5];
    s.FramePosition.x = (decltype(s.FramePosition.x))e[6];
    s.FramePosition.y = (decltype(s.FramePosition.y))e[7];
}

class FrameExtractorGPU {
public:
    // The values Tracking reads from the settings file: ORBextractor.* (as passed to ORBextractor), the LINEextractor arguments, mK and
    // mDistCoef (CV_32F, 4 or 5 coefficients), mbf and mDepthMapFactor (metres per raw depth unit, 1 / DepthMapFactor), plus the image
    // size.  maxPlanes bounds the planes kept per frame (the PlaneDetection shim keeps 64).
    FrameExtractorGPU(int width, int height, int nFeatures, float scaleFactor, int nLevels, int iniThFAST, int minThFAST, int lsdOctaves,
                      float lsdScale, unsigned int nLSDFeature, double minLineLength, const cv::Mat& K, const cv::Mat& distCoef, float bf,
                      float depthMapFactor, int maxPlanes = 64, int device = 0)
        : w_(width), h_(height) {
        const hvo_camera c = cameraOf(K, distCoef);
        hvo_frame_params p;
        std::memset(&p, 0, sizeof(p));
        p.orb.nfeatures = nFeatures; p.orb.scale_factor = scaleFactor; p.orb.nlevels = nLevels;
        p.orb.ini_th_fast = iniThFAST; p.orb.min_th_fast = minThFAST;
        p.line.n_octaves = lsdOctaves; p.line.scale = lsdScale; p.line.n_features = (int)nLSDFeature; p.line.min_line_length = minLineLength;
        p.fx = c.fx; p.fy = c.fy; p.cx = c.cx; p.cy = c.cy;
        p.depth_factor = depthMapFactor; p.bf = bf;
        p.k1 = c.k1; p.k2 = c.k2; p.p1 = c.p1; p.p2 = c.p2; p.k3 = c.k3;
        undistorts_ = c.k1 != 0.f || c.k2 != 0.f || c.p1 != 0.f || c.p2 != 0.f || c.k3 != 0.f;
        p.distorted = undistorts_ ? 1 : 0;
        p.stages = HVO_STAGE_ALL; p.max_planes = maxPlanes; p.line_cull = 1;  // Frame::ExtractLSD runs cullingLine (Frame.cc:939)
        plane_cam_.fx = c.fx; plane_cam_.fy = c.fy; plane_cam_.cx = c.cx; plane_cam_.cy = c.cy; plane_cam_.depth_factor = depthMapFactor;
        max_planes_ = maxPlanes;
        labels8_ = maxPlanes <= 254;  // one byte per pixel, 255 = no plane
        if (hvo_frame_create(&p, width, height, 1, device, &fh_) != HVO_OK ||
            hvo_frame_capacities(fh_, &orb_cap_, &max_lines_, &normals_count_) != HVO_OK ||
            hvo_frame_image_bounds(fh_, &min_x_, &max_x_, &min_y_, &max_y_) != HVO_OK) {
            error_ = hvo_last_error();
            hvo_frame_destroy(fh_);
            fh_ = nullptr;
            return;
        }
        lgrid_cap_ = hvo_frame_line_grid_capacity(fh_);
        lpvo_cap_ = hvo_frame_lpvo_capacity(fh_);
        const size_t px = (size_t)width * height;
        kps_.resize(orb_cap_); kps_un_.resize(undistorts_ ? orb_cap_ : 0); desc_.resize((size_t)orb_cap_ * 32);
        kp_depth_.resize(orb_cap_); kp_uright_.resize(orb_cap_);
        keylines_.resize(max_lines_); line_desc_.resize((size_t)max_lines_ * 32); linevec3_.resize((size_t)max_lines_ * 3);
        planes7_.resize((size_t)maxPlanes * 7);
        if (labels8_) labels8v_.resize(px); else labels32v_.resize(px);
        normals3_.resize((size_t)normals_count_ * 3); normals8_.resize((size_t)normals_count_ * 8);
        grid_counts_.resize(3072); grid_items_.resize(orb_cap_); lgrid_counts_.resize(3072); lgrid_items_.resize(lgrid_cap_);
        lpvo_normals3_.resize((size_t)lpvo_cap_ * 3); lpvo_depth_.resize(lpvo_cap_);
    }
    ~FrameExtractorGPU() { hvo_frame_destroy(fh_); }
    FrameExtractorGPU(const FrameExtractorGPU&) = delete;
    FrameExtractorGPU& operator=(const FrameExtractorGPU&) = delete;

    // Attach the reference's vocabulary (read once through VocabularyArrays): every later extract also fills mBowVec / mFeatVec as
    // Frame::ComputeBoW would, transform(mDescriptors rows, mBowVec, mFeatVec, levelsup).
    template <class TVoc>
    bool setVocabulary(const TVoc& voc, int levelsup = 4) {
        bow_ = false;
        if (!fh_) { std::fprintf(stderr, "FrameExtractorGPU: %s\n", error_.c_str()); return false; }
        const VocabularyArrays<TVoc> a(voc);
        if (hvo_frame_set_vocabulary(fh_, a.n_nodes(), a.child_start.data(), a.child_ids.empty() ? nullptr : a.child_ids.data(), a.desc.data(),
                                     a.weight.data(), a.word.data(), a.levels, levelsup) != HVO_OK) {
            std::fprintf(stderr, "FrameExtractorGPU: %s\n", hvo_last_error());
            return false;
        }
        bow_counts_.resize(1); fv_counts_.resize(1);
        bow_words_.resize(orb_cap_); bow_values_.resize(orb_cap_); fv_order_.resize(orb_cap_); node_of_.resize(orb_cap_);
        bow_ = true;
        return true;
    }

    // imGray CV_8UC1 and imDepth16 CV_16UC1 (the raw depth, before Tracking's convertTo) of the handle's size.  wantLpvo: the tracker
    // would start thread D (!bManhInit); ptNormals / depthNormals (may be null) then receive computeNormalsLPVO's pt_normals (3x1 CV_64F)
    // and depth_normals in its push_back order.  Returns false, with every output empty, on any error.
    template <class FrameT>
    bool extract(const cv::Mat& imGray, const cv::Mat& imDepth16, FrameT& F, bool wantLpvo, std::vector<cv::Mat>* ptNormals,
                 std::vector<float>* depthNormals) {
        clear(F, ptNormals, depthNormals);
        fill_seconds_ = 0.0;
        if (!fh_) return fail(error_.c_str());
        if (imGray.type() != CV_8UC1 || imDepth16.type() != CV_16UC1) return fail("the image must be CV_8UC1 and the depth CV_16UC1");
        if (imGray.cols != w_ || imGray.rows != h_ || imDepth16.cols != w_ || imDepth16.rows != h_) return fail("the image size differs from the handle's");
        const uint8_t* gray = continuous(imGray, 1, gray_);
        const uint16_t* depth = reinterpret_cast<const uint16_t*>(continuous(imDepth16, 2, depth_));
        int32_t nkp = 0, nl = 0, np = 0, lcount = 0;
        hvo_frame_outputs o;
        std::memset(&o, 0, sizeof(o));
        o.kps = kps_.data(); o.desc = desc_.data(); o.kp_counts = &nkp; o.kp_depth = kp_depth_.data(); o.kp_uright = kp_uright_.data();
        o.kps_un = undistorts_ ? kps_un_.data() : nullptr;
        o.keylines = reinterpret_cast<hvo_keyline*>(keylines_.data()); o.line_desc = line_desc_.data(); o.linevec3 = linevec3_.data(); o.line_counts = &nl;
        o.n_planes = &np; o.planes7 = planes7_.data();
        if (labels8_) o.membership8 = labels8v_.data(); else o.membership = labels32v_.data();
        o.normals3 = normals3_.data();
        hvo_frame_bow_outputs b = {bow_counts_.data(), bow_words_.data(), bow_values_.data(), fv_order_.data(), fv_counts_.data(), node_of_.data(), nullptr};
        hvo_frame_grid_outputs g = {grid_counts_.data(), grid_items_.data(), lgrid_counts_.data(), lgrid_items_.data()};
        hvo_frame_lpvo_outputs lp = {lpvo_normals3_.data(), lpvo_depth_.data(), nullptr, &lcount};
        if (hvo_frame_extract_batch_lpvo(fh_, gray, depth, 1, &o, bow_ ? &b : nullptr, &g, wantLpvo ? &lp : nullptr) != HVO_OK) return fail(hvo_last_error());
        const auto t0 = std::chrono::steady_clock::now();
        if (hvo_normals3_expand(normals3_.data(), depth, w_, h_, plane_cam_.fx, plane_cam_.fy, plane_cam_.cx, plane_cam_.cy, plane_cam_.depth_factor,
                                normals8_.data()) != HVO_OK)
            return fail(hvo_last_error());

        // thread A: ExtractORBNDepth (Frame.cc:874-884), UndistortKeyPoints, ComputeStereoFromRGBD
        static_assert(sizeof(F.mvKeys[0]) == sizeof(hvo_keypoint), "cv::KeyPoint layout");
        F.N = nkp;
        F.mvKeys.resize(nkp);
        std::memcpy((void*)F.mvKeys.data(), kps_.data(), (size_t)nkp * sizeof(hvo_keypoint));
        if (undistorts_) {
            F.mvKeysUn.resize(nkp);
            std::memcpy((void*)F.mvKeysUn.data(), kps_un_.data(), (size_t)nkp * sizeof(hvo_keypoint));
        } else {
            F.mvKeysUn = F.mvKeys;
        }
        rows32(desc_.data(), nkp, F.mDescriptors);
        F.mvDepth.assign(kp_depth_.begin(), kp_depth_.begin() + nkp);
        F.mvuRight.assign(kp_uright_.begin(), kp_uright_.begin() + nkp);

        // thread B: ExtractLSD with cullingLine (Frame.cc:895-950)
        static_assert(sizeof(F.mvKeylinesUn[0]) == sizeof(hvo_keyline), "KeyLine layout");
        F.NL = nl;
        F.mvKeylinesUn.resize(nl);
        std::memcpy((void*)F.mvKeylinesUn.data(), keylines_.data(), (size_t)nl * sizeof(hvo_keyline));
        rows32(line_desc_.data(), nl, F.mLdesc);
        F.mvKeyLineFunctions.resize(nl);
        for (int i = 0; i < nl; ++i)
            for (int k = 0; k < 3; ++k) F.mvKeyLineFunctions[i][k] = linevec3_[(size_t)i * 3 + k];

        // thread C: ComputePlanes (Frame.cc:2104-2212): the planes and the surface normals
        const int n = std::min(np, max_planes_);
        if (labels8_) F.planeDetector.assignPlanes(n, planes7_.data(), labels8v_.data(), depth, w_, h_, plane_cam_);
        else F.planeDetector.assignPlanes(n, planes7_.data(), labels32v_.data(), depth, w_, h_, plane_cam_);
        F.vSurfaceNormal.resize(normals_count_);
        for (int i = 0; i < normals_count_; ++i) setSurfaceNormal(F.vSurfaceNormal[i], &normals8_[(size_t)i * 8]);

        // the grid threads (Frame.cc:304-307) and Frame::ComputeBoW (:1692-1699)
        fillGrid(grid_counts_.data(), grid_items_.data(), F.mGrid);
        fillGrid(lgrid_counts_.data(), lgrid_items_.data(), F.mGridForLine);
        if (bow_) fill(bow_words_.data(), bow_values_.data(), bow_counts_[0], fv_order_.data(), fv_counts_[0], node_of_.data(), F.mBowVec, F.mFeatVec);

        // thread D: ExtractMainImgPtNormals -> Manhattan::computeNormalsLPVO (Frame.cc:218-228)
        if (wantLpvo) {
            for (int i = 0; i < lcount; ++i) {
                const double* v = &lpvo_normals3_[(size_t)i * 3];
                if (ptNormals) ptNormals->push_back((cv::Mat_<double>(3, 1) << v[0], v[1], v[2]));
                if (depthNormals) depthNormals->push_back(lpvo_depth_[i]);
            }
        }

        if (!bounds_set_) {  // the reference's first Frame (mbInitialComputations): ComputeImageBounds and the grid cell inverses
            F.mnMinX = min_x_; F.mnMaxX = max_x_; F.mnMinY = min_y_; F.mnMaxY = max_y_;
            F.mfGridElementWidthInv = static_cast<float>(64) / static_cast<float>(F.mnMaxX - F.mnMinX);
            F.mfGridElementHeightInv = static_cast<float>(48) / static_cast<float>(F.mnMaxY - F.mnMinY);
            bounds_set_ = true;
        }
        fill_seconds_ = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        return true;
    }

    // Host time of the last successful extract spent filling the Frame from the call's rows (everything after the frame call returned).
    double lastFillSeconds() const { return fill_seconds_; }
    // The frame handle underneath (null when creation failed), for callers that also want the raw C-ABI rows.
    hvo_frame* handle() const { return fh_; }

private:
    template <class FrameT>
    static void clear(FrameT& F, std::vector<cv::Mat>* ptNormals, std::vector<float>* depthNormals) {
        F.N = 0; F.mvKeys.clear(); F.mvKeysUn.clear(); F.mDescriptors.release(); F.mvDepth.clear(); F.mvuRight.clear();
        F.NL = 0; F.mvKeylinesUn.clear(); F.mLdesc.release(); F.mvKeyLineFunctions.clear();
        F.planeDetector.plane_num_ = 0; F.planeDetector.plane_vertices_.clear(); F.planeDetector.cloud.vertices.clear();
        F.planeDetector.plane_filter.extractedPlanes.clear();
        F.vSurfaceNormal.clear();
        for (int ix = 0; ix < 64; ++ix)
            for (int iy = 0; iy < 48; ++iy) { F.mGrid[ix][iy].clear(); F.mGridForLine[ix][iy].clear(); }
        F.mBowVec.clear(); F.mFeatVec.clear();
        if (ptNormals) ptNormals->clear();
        if (depthNormals) depthNormals->clear();
    }
    static bool fail(const char* why) {
        std::fprintf(stderr, "FrameExtractorGPU: %s\n", why);
        return false;
    }
    // n rows of 32 bytes into an n x 32 CV_8U matrix (released when n == 0, as the reference's extractors leave it)
    static void rows32(const uint8_t* src, int n, cv::Mat& m) {
        if (n == 0) { m.release(); return; }
        m.create(n, 32, CV_8U);
        for (int i = 0; i < n; ++i) std::memcpy(m.ptr(i), src + (size_t)i * 32, 32);
    }
    // the image's rows back to back (the frame call takes packed rows); no copy for a continuous image
    static const uint8_t* continuous(const cv::Mat& m, int elem, std::vector<uint8_t>& buf) {
        const size_t row = (size_t)m.cols * elem;
        if (m.isContinuous()) return m.ptr(0);
        buf.resize(row * m.rows);
        for (int y = 0; y < m.rows; ++y) std::memcpy(&buf[(size_t)y * row], m.ptr(y), row);
        return buf.data();
    }

    hvo_frame* fh_ = nullptr;
    std::string error_;
    int w_, h_, max_planes_ = 0;
    int orb_cap_ = 0, max_lines_ = 0, normals_count_ = 0, lgrid_cap_ = 0, lpvo_cap_ = 0;
    bool undistorts_ = false, labels8_ = true, bow_ = false, bounds_set_ = false;
    float min_x_ = 0.f, max_x_ = 0.f, min_y_ = 0.f, max_y_ = 0.f;
    hvo_plane_params plane_cam_;
    double fill_seconds_ = 0.0;
    std::vector<uint8_t> gray_, depth_;
    std::vector<hvo_keypoint> kps_, kps_un_;
    std::vector<uint8_t> desc_, line_desc_, labels8v_;
    std::vector<float> kp_depth_, kp_uright_, normals3_, normals8_, lpvo_depth_;
    std::vector<hvo_keyline> keylines_;
    std::vector<double> linevec3_, planes7_, bow_values_, lpvo_normals3_;
    std::vector<int32_t> labels32v_, bow_counts_, bow_words_, fv_order_, fv_counts_, node_of_;
    std::vector<uint16_t> grid_counts_, grid_items_, lgrid_counts_, lgrid_items_;
};

}  // namespace hvo_shim

#endif
