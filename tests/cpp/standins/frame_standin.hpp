// TEST INFRASTRUCTURE — stand-in for ORB_SLAM2::Frame (reference include/Frame.h) carrying exactly the members the extraction block
// of Frame::Frame fills (threads A-C, the grid threads, ComputeBoW) and the static image bounds of the first frame, with the
// reference's types (OpenCV / Eigen / DBoW2 / KeyLine through the stand-ins of oracle/cvshim and tests/cpp/standins), and
// SurfaceNormal (include/SurfaceNormal.h).  PlaneDetection is the shim of shim/PlaneExtractor.h, as after the header swap.
#pragma once
#include <cstddef>
#include <vector>

#include <opencv2/core/core.hpp>
#include <Eigen/Core>

#include "DBoW2/BowVector.h"
#include "DBoW2/FeatureVector.h"
#include "PlaneExtractor.h"
#include "keyline_standin.hpp"

#define FRAME_GRID_ROWS 48
#define FRAME_GRID_COLS 64

namespace ORB_SLAM2 {

struct SurfaceNormal {
    cv::Point3f normal;
    cv::Point3f cameraPosition;
    cv::Point2i FramePosition;
};

class Frame {
public:
    int N = 0;
    std::vector<cv::KeyPoint> mvKeys, mvKeysUn;
    cv::Mat mDescriptors;
    std::vector<float> mvuRight, mvDepth;

    int NL = 0;
    std::vector<cv::line_descriptor::KeyLine> mvKeylinesUn;
    cv::Mat mLdesc;
    std::vector<Eigen::Vector3d> mvKeyLineFunctions;

    PlaneDetection planeDetector;
    std::vector<SurfaceNormal> vSurfaceNormal;

    std::vector<std::size_t> mGrid[FRAME_GRID_COLS][FRAME_GRID_ROWS];
    std::vector<std::size_t> mGridForLine[FRAME_GRID_COLS][FRAME_GRID_ROWS];

    DBoW2::BowVector mBowVec;
    DBoW2::FeatureVector mFeatVec;

    static float mnMinX, mnMaxX, mnMinY, mnMaxY;
    static float mfGridElementWidthInv, mfGridElementHeightInv;
};

}  // namespace ORB_SLAM2
