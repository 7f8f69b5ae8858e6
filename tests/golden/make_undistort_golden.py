"""Generates tests/golden/undistort_cv2.npz (needs cv2 4.13.0, the project's pin for OpenCV behaviour):

    python tests/golden/make_undistort_golden.py

undistort_cv2.npz  cv2.undistortPoints(pts, K, dist, None, K) (what Frame::UndistortKeyPoints / ComputeImageBounds call, Frame.cc:1701-1760)
                   for the TUM1 and TUM2 cameras, a 4-coefficient set and a k1 = -3 set (OpenCV's icdist < 0 exit) on random points in
                   and around a 640x480 image, the four corners first.
"""
import os

import cv2
import numpy as np

OUT = os.path.dirname(os.path.abspath(__file__))

CASES = {   # name: (fx, fy, cx, cy), (k1, k2, p1, p2[, k3])
    'tum1': ((517.306408, 516.469215, 318.643040, 255.313989), (0.262383, -0.953104, -0.005358, 0.002628, 1.163314)),   # TUM1.yaml
    'tum2': ((520.908620, 521.007327, 325.141442, 249.701764), (0.231222, -0.784899, -0.003257, -0.000105, 0.917205)),  # TUM2.yaml
    'four': ((517.306408, 516.469215, 318.643040, 255.313989), (0.12, -0.31, 0.0021, -0.0017)),
    'k1neg3': ((517.306408, 516.469215, 318.643040, 255.313989), (-3.0, 0.0, 0.0, 0.0)),
}


def undistort():
    assert cv2.__version__ == '4.13.0', cv2.__version__
    r = np.random.RandomState(31)
    pts = np.concatenate([np.stack([r.uniform(-5, 645, 3000), r.uniform(-5, 485, 3000)], 1),
                          np.stack([r.uniform(-200, 840, 1000), r.uniform(-200, 680, 1000)], 1)]).astype(np.float32)
    pts[:4] = [[0, 0], [640, 0], [0, 480], [640, 480]]
    out = dict(pts=pts, cv2_version=np.array(cv2.__version__))
    for name, ((fx, fy, cx, cy), dist) in CASES.items():
        K = np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1]], np.float32)
        d = np.array(dist, np.float32)
        out[name + '_K'], out[name + '_dist'] = K, d
        out[name + '_un'] = cv2.undistortPoints(pts.reshape(-1, 1, 2), K, d, None, K).reshape(-1, 2)
    return out


if __name__ == '__main__':
    np.savez_compressed(os.path.join(OUT, 'undistort_cv2.npz'), **undistort())
    print('undistort_cv2.npz written')
