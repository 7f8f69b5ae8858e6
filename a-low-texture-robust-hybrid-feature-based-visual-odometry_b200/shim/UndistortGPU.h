// Bodies of Frame::UndistortKeyPoints and Frame::ComputeImageBounds (reference src/Frame.cc:1701-1760) over the C ABI of
// libhvofront.so (hvo_undistort_points / hvo_image_bounds: cv::undistortPoints of OpenCV 4.13, bit for bit, without calib3d).
// For callers of the per-class extractors; the frame handle (hvo_frame_*) undistorts on the device by itself.  The two-body patch:
//
//   void Frame::UndistortKeyPoints() { hvo_shim::undistortKeyPoints(mvKeys, mK, mDistCoef, mvKeysUn); }
//   void Frame::ComputeImageBounds(const cv::Mat& imLeft) {
//       hvo_shim::computeImageBounds(mK, mDistCoef, imLeft.cols, imLeft.rows, mnMinX, mnMaxX, mnMinY, mnMaxY);
//   }
#ifndef HVO_SHIM_UNDISTORT_GPU_H
#define HVO_SHIM_UNDISTORT_GPU_H

#include <cstdio>
#include <vector>

#include <opencv2/core/core.hpp>

#include "hvo_capi.h"

namespace hvo_shim {

// mK (3x3 CV_32F) and mDistCoef (4 or 5 x 1 CV_32F, k3 only when Camera.k3 != 0)
inline hvo_camera cameraOf(const cv::Mat& K, const cv::Mat& distCoef) {
    hvo_camera c;
    c.fx = K.at<float>(0, 0); c.fy = K.at<float>(1, 1); c.cx = K.at<float>(0, 2); c.cy = K.at<float>(1, 2);
    const int nd = distCoef.rows * distCoef.cols;
    c.k1 = distCoef.at<float>(0); c.k2 = distCoef.at<float>(1); c.p1 = distCoef.at<float>(2); c.p2 = distCoef.at<float>(3);
    c.k3 = nd > 4 ? distCoef.at<float>(4) : 0.f;
    return c;
}

// mvKeysUn = mvKeys with pt undistorted; unchanged when k1 == 0, as the reference (which tests k1 only)
inline void undistortKeyPoints(const std::vector<cv::KeyPoint>& keys, const cv::Mat& K, const cv::Mat& distCoef, std::vector<cv::KeyPoint>& keysUn) {
    keysUn = keys;
    if (distCoef.at<float>(0) == 0.f || keys.empty()) return;
    const hvo_camera cam = cameraOf(K, distCoef);
    std::vector<float> xy(2 * keys.size());
    for (size_t i = 0; i < keys.size(); ++i) { xy[2 * i] = keys[i].pt.x; xy[2 * i + 1] = keys[i].pt.y; }
    if (hvo_undistort_points(&cam, xy.data(), (int)keys.size(), xy.data()) != HVO_OK) {
        std::fprintf(stderr, "undistortKeyPoints: %s\n", hvo_last_error());
        return;
    }
    for (size_t i = 0; i < keys.size(); ++i) { keysUn[i].pt.x = xy[2 * i]; keysUn[i].pt.y = xy[2 * i + 1]; }
}

inline void computeImageBounds(const cv::Mat& K, const cv::Mat& distCoef, int cols, int rows, float& minX, float& maxX, float& minY, float& maxY) {
    const hvo_camera cam = cameraOf(K, distCoef);
    if (hvo_image_bounds(&cam, cols, rows, &minX, &maxX, &minY, &maxY) != HVO_OK) std::fprintf(stderr, "computeImageBounds: %s\n", hvo_last_error());
}

}  // namespace hvo_shim

#endif
