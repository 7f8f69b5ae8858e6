// Point undistortion of Frame::UndistortKeyPoints / Frame::ComputeImageBounds (reference src/Frame.cc:1701-1760):
// cv::undistortPoints(src, dst, mK, mDistCoef, noArray(), mK) of OpenCV 4.13 for one point, restated so that the device kernel
// (k_undistort_kps) and the host entries (hvo_undistort_points, hvo_image_bounds) share one implementation.
//
// Bit-exact with cv2 when every double operation rounds on its own: the device side uses explicit __d*_rn intrinsics, the host side
// relies on -ffp-contract=off (build.py).  The evaluation order of every expression is OpenCV's (cvUndistortPointsInternal), zero
// terms included: they are what makes the restatement match, e.g. 0*y + cx is not cx when y is -0 or not finite.
#ifndef HVO_UNDISTORT_CUH
#define HVO_UNDISTORT_CUH

#include <cuda_runtime.h>

#include "../../include/hvo_capi.h"

namespace hvo {

__host__ __device__ inline double und_mul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
__host__ __device__ inline double und_add(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
__host__ __device__ inline double und_sub(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
__host__ __device__ inline double und_div(double a, double b) {
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}
__host__ __device__ inline float und_narrow(double a) {
#ifdef __CUDA_ARCH__
    return __double2float_rn(a);
#else
    return (float)a;
#endif
}

// (u, v) -> (*xo, *yo) = cv::undistortPoints with P = K, R = I, TermCriteria(COUNT, 5, 0.01): K and the coefficients are the float
// values of mK / mDistCoef widened to double; of OpenCV's 14 coefficients only k1, k2, p1, p2, k3 can be non-zero.
__host__ __device__ inline void undistort_point(const hvo_camera& c, float u, float v, float* xo, float* yo) {
    const double fx = c.fx, fy = c.fy, cx = c.cx, cy = c.cy;
    const double k0 = c.k1, k1 = c.k2, k2 = c.p1, k3 = c.p2, k4 = c.k3, kz = 0.0;   // k[5] .. k[13] = 0
    const double ifx = und_div(1.0, fx), ify = und_div(1.0, fy);
    const double ud = u, vd = v;
    double x = und_mul(und_sub(ud, cx), ifx), y = und_mul(und_sub(vd, cy), ify);
    const double x0 = x, y0 = y;   // the tilt step of an untilted camera is the identity
    for (int j = 0; j < 5; ++j) {
        const double r2 = und_add(und_mul(x, x), und_mul(y, y));
        // icdist = (1 + ((k[7]*r2 + k[6])*r2 + k[5])*r2) / (1 + ((k[4]*r2 + k[1])*r2 + k[0])*r2)
        const double num = und_add(1.0, und_mul(und_add(und_mul(und_add(und_mul(kz, r2), kz), r2), kz), r2));
        const double den = und_add(1.0, und_mul(und_add(und_mul(und_add(und_mul(k4, r2), k1), r2), k0), r2));
        const double icdist = und_div(num, den);
        if (icdist < 0) {   // OpenCV gives up and keeps the distorted normalised point
            x = und_mul(und_sub(ud, cx), ifx);
            y = und_mul(und_sub(vd, cy), ify);
            break;
        }
        // deltaX = 2*k[2]*x*y + k[3]*(r2 + 2*x*x) + k[8]*r2 + k[9]*r2*r2
        const double dx = und_add(und_add(und_add(und_mul(und_mul(und_mul(2.0, k2), x), y),
                                                  und_mul(k3, und_add(r2, und_mul(und_mul(2.0, x), x)))),
                                          und_mul(kz, r2)),
                                  und_mul(und_mul(kz, r2), r2));
        // deltaY = k[2]*(r2 + 2*y*y) + 2*k[3]*x*y + k[10]*r2 + k[11]*r2*r2
        const double dy = und_add(und_add(und_add(und_mul(k2, und_add(r2, und_mul(und_mul(2.0, y), y))),
                                                  und_mul(und_mul(und_mul(2.0, k3), x), y)),
                                          und_mul(kz, r2)),
                                  und_mul(und_mul(kz, r2), r2));
        x = und_mul(und_sub(x0, dx), icdist);
        y = und_mul(und_sub(y0, dy), icdist);
    }
    // RR = P * R = K: xx = fx*x + 0*y + cx, yy = 0*x + fy*y + cy, ww = 1/(0*x + 0*y + 1)
    const double xx = und_add(und_add(und_mul(fx, x), und_mul(0.0, y)), cx);
    const double yy = und_add(und_add(und_mul(0.0, x), und_mul(fy, y)), cy);
    const double ww = und_div(1.0, und_add(und_add(und_mul(0.0, x), und_mul(0.0, y)), 1.0));
    *xo = und_narrow(und_mul(xx, ww));
    *yo = und_narrow(und_mul(yy, ww));
}

}  // namespace hvo

#endif
