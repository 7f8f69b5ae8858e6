// Drop-in replacement for the reference's include/PlaneExtractor.h (class PlaneDetection, :36-56) forwarding to the C ABI
// of libhvofront.so.  Frame::ComputePlanes (src/Frame.cc:2104-2130) compiles against it unchanged:
//
//   planeDetector.readColorImage(imRGB);
//   planeDetector.readDepthImage(Depth, K, depthMapFactor);
//   planeDetector.runPlaneDetection(imDepth.rows, imDepth.cols);
//   for (i < planeDetector.plane_num_) { planeDetector.plane_vertices_[i]; planeDetector.cloud.vertices[j][0..2];
//                                         planeDetector.plane_filter.extractedPlanes[i]->normal / ->center; }
//
// VertexT is Eigen::Vector3d in the reference (typedef VertexType); any type with operator[] works.  The point cloud
// (7.4 MB per frame in the reference) is not produced on the device: cloud.vertices is filled on the host only for the
// pixels that belong to a plane, which are the only ones Frame::ComputePlanes reads.
#ifndef HVO_SHIM_PLANEEXTRACTOR_H
#define HVO_SHIM_PLANEEXTRACTOR_H

#include <cstdio>
#include <memory>
#include <vector>

#include <opencv2/core/core.hpp>

#include "hvo_capi.h"

#ifndef HVO_SHIM_VERTEX_TYPE
#include <Eigen/Core>
typedef Eigen::Vector3d VertexType;
#else
typedef HVO_SHIM_VERTEX_TYPE VertexType;
#endif

struct ImagePointCloud {
    std::vector<VertexType> vertices;  // filled for plane members only (see above)
    int w = 0, h = 0;
    inline int width() const { return w; }
    inline int height() const { return h; }
};

namespace hvo_shim {
struct PlaneSegLite { double normal[3]; double center[3]; int N; };  // the members of ahc::PlaneSeg that Frame.cc reads
struct PlaneFilterLite { std::vector<std::shared_ptr<PlaneSegLite>> extractedPlanes; };
}  // namespace hvo_shim

class PlaneDetection {
public:
    ImagePointCloud cloud;
    hvo_shim::PlaneFilterLite plane_filter;
    std::vector<std::vector<int>> plane_vertices_;  // vertex indices each plane contains
    cv::Mat seg_img_;
    cv::Mat color_img_;
    int plane_num_ = 0;

    PlaneDetection() {}
    ~PlaneDetection() { hvo_plane_destroy(h_); }
    PlaneDetection(const PlaneDetection& o) : cloud(o.cloud), plane_filter(o.plane_filter), plane_vertices_(o.plane_vertices_),
                                             seg_img_(o.seg_img_), color_img_(o.color_img_), plane_num_(o.plane_num_) {}  // Frame is copied by value
    PlaneDetection& operator=(const PlaneDetection& o) {
        cloud = o.cloud; plane_filter = o.plane_filter; plane_vertices_ = o.plane_vertices_; seg_img_ = o.seg_img_;
        color_img_ = o.color_img_; plane_num_ = o.plane_num_;
        return *this;
    }

    bool readColorImage(cv::Mat RGBImg) { color_img_ = RGBImg; return true; }  // only used for debug drawing in the reference

    bool readDepthImage(cv::Mat depthImg, cv::Mat& K, float kScaleFactor) {
        if (depthImg.empty() || depthImg.type() != CV_16U) {  // PlaneExtractor.cpp:34-38
            std::printf("WARNING: cannot read depth image. No such a file, or the image format is not 16UC1\n");
            return false;
        }
        hvo_plane_params p;
        p.fx = K.at<float>(0, 0); p.fy = K.at<float>(1, 1); p.cx = K.at<float>(0, 2); p.cy = K.at<float>(1, 2);
        p.depth_factor = kScaleFactor;
        if (!h_ || depthImg.cols != w_ || depthImg.rows != hgt_ || p.fx != p_.fx || p.fy != p_.fy || p.cx != p_.cx || p.cy != p_.cy ||
            p.depth_factor != p_.depth_factor) {
            hvo_plane_destroy(h_);
            h_ = nullptr;
            if (hvo_plane_create(&p, depthImg.cols, depthImg.rows, 1, 0, &h_) != HVO_OK) {
                std::fprintf(stderr, "PlaneDetection: %s\n", hvo_last_error());
                return false;
            }
            p_ = p; w_ = depthImg.cols; hgt_ = depthImg.rows;
        }
        depth_.resize((size_t)w_ * hgt_);
        for (int y = 0; y < hgt_; ++y) std::memcpy(&depth_[(size_t)y * w_], depthImg.ptr<unsigned short>(y), (size_t)w_ * 2);
        cloud.w = w_; cloud.h = hgt_;
        return true;
    }

    void runPlaneDetection(int /*kDepthHeight*/, int /*kDepthWidth*/) {
        plane_num_ = 0;
        plane_vertices_.clear();
        plane_filter.extractedPlanes.clear();
        if (!h_ || depth_.empty()) return;
        const int maxp = 64;
        std::vector<double> planes((size_t)maxp * 7);
        membership_.resize(depth_.size());
        int32_t n = 0;
        if (hvo_plane_detect(h_, depth_.data(), &n, planes.data(), maxp, membership_.data()) != HVO_OK) {
            std::fprintf(stderr, "PlaneDetection: %s\n", hvo_last_error());
            return;
        }
        if (n > maxp) n = maxp;
        assignPlanes(n, planes.data(), membership_.data(), depth_.data(), w_, hgt_, p_);
    }

    // Fills plane_num_, plane_vertices_, cloud and plane_filter from one frame's plane outputs of the C ABI: planes7 [n][7], the
    // labels [w*h] (plane id; any value outside [0, n), such as -1 or 255, is no plane), the raw depth and the camera the planes were
    // detected with.  runPlaneDetection and hvo_shim::FrameExtractorGPU (the frame call's int32 or one-byte labels) both fill through it.
    template <class LabelT>
    void assignPlanes(int n, const double* planes7, const LabelT* labels, const uint16_t* depth, int w, int h, const hvo_plane_params& cam) {
        const int npx = w * h;
        plane_num_ = n;
        plane_vertices_.assign(n, std::vector<int>());
        plane_filter.extractedPlanes.clear();
        cloud.w = w; cloud.h = h;
        cloud.vertices.resize(npx);
        const double f = (double)cam.depth_factor, fx = (double)cam.fx, fy = (double)cam.fy, cx = (double)cam.cx, cy = (double)cam.cy;
        for (int i = 0; i < npx; ++i) {
            const int m = labels[i];
            if (m < 0 || m >= n) continue;
            plane_vertices_[m].push_back(i);
            const int row = i / w, col = i - row * w;
            const double z = (double)depth[i] * f;  // PlaneExtractor.cpp:44-53
            cloud.vertices[i][0] = ((double)col - cx) * z / fx;
            cloud.vertices[i][1] = ((double)row - cy) * z / fy;
            cloud.vertices[i][2] = z;
        }
        for (int i = 0; i < n; ++i) {
            auto s = std::make_shared<hvo_shim::PlaneSegLite>();
            for (int k = 0; k < 3; ++k) { s->normal[k] = planes7[7 * i + k]; s->center[k] = planes7[7 * i + 3 + k]; }
            s->N = (int)planes7[7 * i + 6];
            plane_filter.extractedPlanes.push_back(s);
        }
    }

    const std::vector<int32_t>& membership() const { return membership_; }

private:
    hvo_plane* h_ = nullptr;
    hvo_plane_params p_{};
    int w_ = 0, hgt_ = 0;
    std::vector<uint16_t> depth_;
    std::vector<int32_t> membership_;
};

#endif
