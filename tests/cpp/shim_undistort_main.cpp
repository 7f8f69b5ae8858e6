// Test driver: the Frame::UndistortKeyPoints / Frame::ComputeImageBounds bridge (shim/UndistortGPU.h -> C ABI), called with the
// reference's types (cv::Mat mK, mDistCoef; std::vector<cv::KeyPoint>).  Host functions only: runs without a GPU.
//   in.bin : int32 magic, w, h, ndist, n ; float fx, fy, cx, cy ; ndist floats ; n x 28 B keypoints
//   out.bin: n x 28 B mvKeysUn ; 4 floats mnMinX, mnMaxX, mnMinY, mnMaxY
#include <cstdint>
#include <cstdio>
#include <vector>

#include "UndistortGPU.h"

int main(int argc, char** argv) {
    if (argc != 3) { std::fprintf(stderr, "usage: shim_undistort in.bin out.bin\n"); return 2; }
    FILE* fi = std::fopen(argv[1], "rb");
    FILE* fo = std::fopen(argv[2], "wb");
    if (!fi || !fo) return 2;
    int32_t hdr[5];
    if (std::fread(hdr, 4, 5, fi) != 5 || hdr[0] != 0x554e4453 || hdr[3] < 4 || hdr[3] > 5) return 3;
    const int w = hdr[1], h = hdr[2], nd = hdr[3], n = hdr[4];
    float k[4], d[5];
    std::vector<cv::KeyPoint> keys(n);
    if (std::fread(k, 4, 4, fi) != 4 || std::fread(d, 4, nd, fi) != (size_t)nd || std::fread(keys.data(), 28, n, fi) != (size_t)n) return 4;
    std::fclose(fi);

    cv::Mat K(3, 3, CV_32F), distCoef(nd, 1, CV_32F);   // as Tracking fills mK / mDistCoef from the settings file
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) K.at<float>(i, j) = 0.f;
    K.at<float>(0, 0) = k[0]; K.at<float>(1, 1) = k[1]; K.at<float>(0, 2) = k[2]; K.at<float>(1, 2) = k[3]; K.at<float>(2, 2) = 1.f;
    for (int i = 0; i < nd; ++i) distCoef.at<float>(i) = d[i];

    std::vector<cv::KeyPoint> keysUn;
    hvo_shim::undistortKeyPoints(keys, K, distCoef, keysUn);
    float b[4];
    hvo_shim::computeImageBounds(K, distCoef, w, h, b[0], b[1], b[2], b[3]);
    if (std::fwrite(keysUn.data(), 28, n, fo) != (size_t)n || std::fwrite(b, 4, 4, fo) != 4) return 5;
    std::fclose(fo);
    return 0;
}
