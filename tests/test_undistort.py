"""Keypoint undistortion (Frame::UndistortKeyPoints / ComputeImageBounds, reference src/Frame.cc:1701-1760): the host entries
(hvo_undistort_points, hvo_image_bounds) against cv2.undistortPoints of OpenCV 4.13 (committed fixture undistort_cv2.npz, and
live cv2 when it is importable), and the device path (k_undistort_kps through hvo_orb_undistort_batch_device and the frame handle)
against them."""
import os
import struct
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'a-low-texture-robust-hybrid-feature-based-visual-odometry_b200')
GOLDEN = np.load(os.path.join(ROOT, 'tests', 'golden', 'undistort_cv2.npz'))
CASES = ('tum1', 'tum2', 'four', 'k1neg3')
TUM1_K, TUM1_DIST = GOLDEN['tum1_K'], GOLDEN['tum1_dist']
K1ZERO_DIST = np.array([0.0, 0.05, 0.004, -0.003, 0.02], np.float32)   # k1 == 0: the reference does not undistort


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _bounds_formula(c):
    """Frame::ComputeImageBounds on the undistorted corners (0,0), (cols,0), (0,rows), (cols,rows)."""
    return (min(c[0, 0], c[2, 0]), max(c[1, 0], c[3, 0]), min(c[0, 1], c[1, 1]), max(c[2, 1], c[3, 1]))


def _host_un(hvo, kps, K, dist):
    """mvKeysUn as the reference forms it on the host: keypoint copies with pt from cv::undistortPoints (k1 == 0: unchanged)."""
    un = kps.copy()
    if np.float32(dist[0]) != 0 and len(kps):
        try:
            import cv2
            xy = cv2.undistortPoints(np.stack([kps['x'], kps['y']], 1).reshape(-1, 1, 2).astype(np.float32), K, dist, None, K).reshape(-1, 2)
        except ImportError:   # the host restatement equals cv2 bit for bit (CPU tests below)
            xy = hvo.undistort_points(np.stack([kps['x'], kps['y']], 1), K, dist)
        un['x'], un['y'] = xy[:, 0], xy[:, 1]
    return un


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('case', CASES)
def test_undistort_points_equals_cv2_fixture(hvo, case):
    got = hvo.undistort_points(GOLDEN['pts'], GOLDEN[case + '_K'], GOLDEN[case + '_dist'])
    assert np.array_equal(_bits(got), _bits(GOLDEN[case + '_un']))


@pytest.mark.parametrize('case', CASES)
def test_undistort_points_equals_live_cv2(hvo, case):
    cv2 = pytest.importorskip('cv2')
    K, dist = GOLDEN[case + '_K'], GOLDEN[case + '_dist']
    r = np.random.default_rng(7)
    pts = np.stack([r.uniform(-40, 680, 50000), r.uniform(-40, 520, 50000)], 1).astype(np.float32)
    ref = cv2.undistortPoints(pts.reshape(-1, 1, 2), K, dist, None, K).reshape(-1, 2)
    assert np.array_equal(_bits(hvo.undistort_points(pts, K, dist)), _bits(ref))


def test_icdist_exit_keeps_the_distorted_point(hvo):
    """k1 = -3: OpenCV's icdist < 0 exit returns the image corners unchanged."""
    corners = GOLDEN['pts'][:4]
    assert np.array_equal(GOLDEN['k1neg3_un'][:4], corners)
    assert np.array_equal(hvo.undistort_points(corners, GOLDEN['k1neg3_K'], GOLDEN['k1neg3_dist']), corners)


@pytest.mark.parametrize('case', CASES)
def test_image_bounds_equal_reference_formula_on_cv2_corners(hvo, case):
    K, dist = GOLDEN[case + '_K'], GOLDEN[case + '_dist']
    exp = _bounds_formula(GOLDEN[case + '_un'][:4])      # the fixture's first four points are the corners of 640 x 480
    got = hvo.image_bounds(K, dist, 640, 480)
    assert np.array_equal(_bits(np.array(got)), _bits(np.array(exp)))


def test_k1_zero_is_not_undistorted_by_the_frame_rules(hvo):
    """Frame::UndistortKeyPoints / ComputeImageBounds test k1 only: p1 != 0 with k1 == 0 gives the plain image bounds, while
    hvo_undistort_points (plain cv::undistortPoints) does move the points."""
    assert hvo.image_bounds(TUM1_K, K1ZERO_DIST, 640, 480) == (0.0, 640.0, 0.0, 480.0)
    assert hvo.image_bounds(TUM1_K, K1ZERO_DIST[:4], 320, 240) == (0.0, 320.0, 0.0, 240.0)
    moved = hvo.undistort_points(GOLDEN['pts'][:4], TUM1_K, K1ZERO_DIST)
    assert not np.array_equal(moved, GOLDEN['pts'][:4])
    try:
        import cv2
    except ImportError:
        return
    ref = cv2.undistortPoints(GOLDEN['pts'].reshape(-1, 1, 2), TUM1_K, K1ZERO_DIST, None, TUM1_K).reshape(-1, 2)
    assert np.array_equal(_bits(hvo.undistort_points(GOLDEN['pts'], TUM1_K, K1ZERO_DIST)), _bits(ref))


def test_four_coefficients_mean_k3_zero(hvo):
    d4 = GOLDEN['four_dist']
    assert len(d4) == 4
    d5 = np.concatenate([d4, [0]]).astype(np.float32)
    assert np.array_equal(hvo.undistort_points(GOLDEN['pts'], GOLDEN['four_K'], d4), hvo.undistort_points(GOLDEN['pts'], GOLDEN['four_K'], d5))


def test_undistort_argument_validation(hvo):
    with pytest.raises(hvo.HvoError) as e:
        hvo.undistort_points(GOLDEN['pts'][:4], TUM1_K, TUM1_DIST[:3])
    assert e.value.status == hvo.HVO_ERR_ARG
    K0 = TUM1_K.copy(); K0[0, 0] = 0
    with pytest.raises(hvo.HvoError) as e:
        hvo.undistort_points(GOLDEN['pts'][:4], K0, TUM1_DIST)
    assert e.value.status == hvo.HVO_ERR_ARG
    with pytest.raises(hvo.HvoError) as e:
        hvo.image_bounds(TUM1_K, TUM1_DIST, 0, 480)
    assert e.value.status == hvo.HVO_ERR_ARG


def test_binding_covers_the_new_entries(hvo):
    for name in ('hvo_undistort_points', 'hvo_image_bounds', 'hvo_orb_undistort_batch_device'):
        assert name in hvo.ABI
    names = [f[0] for f in hvo._FrameParams._fields_]
    assert names[-5:] == ['k1', 'k2', 'p1', 'p2', 'k3'] and hvo.FrameFrontEnd.FIELDS[-1] == 'kps_un'


def _build_shim(exe):
    if not os.path.exists(os.path.join(PKG, 'libhvofront.so')):
        import __graft_entry__
        __graft_entry__.build()
    subprocess.check_call(['g++', '-O2', '-std=c++14', '-I' + os.path.join(ROOT, 'oracle', 'cvshim'), '-I' + os.path.join(PKG, 'shim'),
                           '-I' + os.path.join(ROOT, 'include'), os.path.join(ROOT, 'tests', 'cpp', 'shim_undistort_main.cpp'), '-o', exe,
                           '-L' + PKG, '-lhvofront', '-Wl,-rpath,' + PKG])


@pytest.mark.parametrize('case', CASES + ('k1zero',))
def test_shim_bridge_equals_python_mirror(hvo, tmp_path, case):
    """shim/UndistortGPU.h called with cv::Mat mK / mDistCoef and std::vector<cv::KeyPoint> (host functions: no GPU needed)."""
    exe = str(tmp_path / 'shim_undistort')
    _build_shim(exe)
    K, dist = (TUM1_K, K1ZERO_DIST) if case == 'k1zero' else (GOLDEN[case + '_K'], GOLDEN[case + '_dist'])
    pts = GOLDEN['pts']
    kps = np.zeros(len(pts), hvo.KP_DTYPE)
    kps['x'], kps['y'] = pts[:, 0], pts[:, 1]
    kps['size'], kps['angle'], kps['response'] = 31.0, np.arange(len(pts)) % 360, 0.5
    kps['octave'], kps['class_id'] = np.arange(len(pts)) % 8, -1
    fi, fo = str(tmp_path / 'in.bin'), str(tmp_path / 'out.bin')
    with open(fi, 'wb') as f:
        f.write(struct.pack('<5i', 0x554e4453, 640, 480, len(dist), len(kps)) + np.array([K[0, 0], K[1, 1], K[0, 2], K[1, 2]], np.float32).tobytes()
                + np.asarray(dist, np.float32).tobytes() + kps.tobytes())
    subprocess.check_call([exe, fi, fo])
    raw = open(fo, 'rb').read()
    assert len(raw) == 28 * len(kps) + 16
    assert raw[:28 * len(kps)] == _host_un(hvo, kps, K, dist).tobytes()
    assert np.array_equal(np.frombuffer(raw, np.float32, 4, 28 * len(kps)), np.array(hvo.image_bounds(K, dist, 640, 480), np.float32))


# ---------------------------------------------------------------------------------------------------------------- GPU
def _tum1_cam():
    return float(TUM1_K[0, 0]), float(TUM1_K[1, 1]), float(TUM1_K[0, 2]), float(TUM1_K[1, 2])


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES + ('k1zero',))
def test_gpu_undistort_batch_device_on_fixture_points(hvo, case):
    """hvo_orb_undistort_batch_device on the fixture points packed as keypoints of three frames: x, y bit-equal to cv2, every other
    field copied, kp_uright = x_un - bf / d where d > 0, rows at or past counts[f] untouched."""
    import torch
    K, dist = (TUM1_K, K1ZERO_DIST) if case == 'k1zero' else (GOLDEN[case + '_K'], GOLDEN[case + '_dist'])
    pts = GOLDEN['pts']
    ex = hvo.ORBextractor(1000, 1.2, 8, 20, 7, width=640, height=480, max_batch=4)
    cap = ex.capacity
    counts = np.array([min(cap, 1500), 0, min(cap - 3, 1200), min(cap, len(pts))], np.int32)
    kps = np.zeros((4, cap), hvo.KP_DTYPE)
    r = np.random.default_rng(3)
    for f in range(4):
        sel = r.permutation(len(pts))[:cap]
        kps[f]['x'], kps[f]['y'] = pts[sel, 0], pts[sel, 1]
        kps[f]['size'], kps[f]['angle'], kps[f]['response'] = r.uniform(31, 100, cap), r.uniform(0, 360, cap), r.uniform(0, 1, cap)
        kps[f]['octave'], kps[f]['class_id'] = r.integers(0, 8, cap), -1
    depth = r.uniform(-1, 7, (4, cap)).astype(np.float32)
    depth[depth < 0.5] = -1
    bf = np.float32(40.0)
    dev = torch.device('cuda', 0)
    d_kps = torch.from_numpy(kps.view(np.uint8).reshape(4, -1).copy()).to(dev)
    d_counts, d_depth = torch.from_numpy(counts).to(dev), torch.from_numpy(depth).to(dev)
    d_un = torch.full((4, cap * 28), 0xAB, dtype=torch.uint8, device=dev)
    d_ur = torch.full((4, cap), 1234.5, dtype=torch.float32, device=dev)
    torch.cuda.synchronize()
    ex.undistort_batch_device((K, dist), d_kps.data_ptr(), d_counts.data_ptr(), 4, d_depth.data_ptr(), float(bf), d_un.data_ptr(), d_ur.data_ptr())
    ex.sync()
    un = d_un.cpu().numpy().view(hvo.KP_DTYPE).reshape(4, cap)
    ur = d_ur.cpu().numpy()
    for f in range(4):
        n = int(counts[f])
        exp = _host_un(hvo, kps[f, :n], K, dist)
        assert un[f, :n].tobytes() == exp.tobytes()
        with np.errstate(divide='ignore'):
            eur = np.where(depth[f, :n] > 0, exp['x'] - bf / depth[f, :n], np.float32(-1)).astype(np.float32)
        assert np.array_equal(_bits(ur[f, :n]), _bits(eur))
        assert (un[f, n:].view(np.uint8) == 0xAB).all() and (ur[f, n:] == 1234.5).all()
    # without kp_uright / kps_un: only the requested output is written
    d_un2 = torch.full_like(d_un, 0xCD)
    torch.cuda.synchronize()
    ex.undistort_batch_device((K, dist), d_kps.data_ptr(), d_counts.data_ptr(), 4, None, 0.0, d_un2.data_ptr(), None)
    ex.sync()
    un2 = d_un2.cpu().numpy()
    for f in range(4):
        n = int(counts[f])
        assert un2[f, :28 * n].tobytes() == un[f, :n].tobytes() and (un2[f, 28 * n:] == 0xCD).all()
    with pytest.raises(hvo.HvoError):   # kp_uright needs kp_depth
        ex.undistort_batch_device((K, dist), d_kps.data_ptr(), d_counts.data_ptr(), 4, None, 0.0, None, d_ur.data_ptr())
    ex.close()


def _frames(synth, n, start):
    return synth.sequence('S1', n, start=start)


def _fe(hvo, dist, **kw):
    fx, fy, cx, cy = _tum1_cam()
    return hvo.FrameFrontEnd(640, 480, fx, fy, cx, cy, 1.0 / 5000.0, bf=40.0, dist=dist, **kw)


def _check_distorted_against_plain(hvo, d, p, nframes, K, dist):
    """d: outputs of a handle with coefficients, p: the same handle without; both host dicts."""
    assert 'kps_un' in d and 'kps_un' not in p
    for f in range(nframes):
        n, nl, npl = int(p['kp_counts'][f]), int(p['line_counts'][f]), int(p['n_planes'][f])
        assert n == int(d['kp_counts'][f]) and n > 100
        for k in ('kps', 'desc', 'kp_depth'):
            assert d[k][f, :n].tobytes() == p[k][f, :n].tobytes(), k
        un = _host_un(hvo, d['kps'][f, :n], K, dist)
        assert d['kps_un'][f, :n].tobytes() == un.tobytes()
        ur = hvo.ORBextractor.stereo_uright_from_depth(un, d['kp_depth'][f, :n], 40.0)
        assert np.array_equal(_bits(d['kp_uright'][f, :n]), _bits(ur))
        assert nl == int(d['line_counts'][f]) and npl == int(d['n_planes'][f])
        for k in ('keylines', 'line_desc', 'linevec3'):
            assert d[k][f, :nl].tobytes() == p[k][f, :nl].tobytes(), k
        assert np.array_equal(d['planes7'][f, :npl], p['planes7'][f, :npl])
        for k in ('membership', 'membership8', 'membership4', 'normals8', 'normals3'):
            if k in p:
                assert np.array_equal(d[k][f], p[k][f], equal_nan=True), k
    if np.float32(dist[0]) != 0:
        moved = np.abs(d['kps_un'][0, :20]['x'] - d['kps'][0, :20]['x']) > 0.01
        assert moved.any()


@pytest.mark.gpu
def test_gpu_frame_front_end_undistorts_tum1(hvo, synth):
    gray, depth = _frames(synth, 3, 40)
    plain = _fe(hvo, None, max_batch=3)
    p = plain.extract_batch(gray, depth)
    plain.close()
    fe = _fe(hvo, TUM1_DIST, max_batch=3)
    assert fe.output_shapes(3)['kps_un'] == ((3, fe.orb_capacity), hvo.KP_DTYPE)
    d = fe.extract_batch(gray, depth)
    _check_distorted_against_plain(hvo, d, p, 3, TUM1_K, TUM1_DIST)
    # kps_un is optional on the host: without it the uright still comes from the undistorted keypoints
    out = {k: v for k, v in fe.alloc_host(3).items() if k != 'kps_un'}
    with pytest.raises(hvo.HvoError):           # a caller-supplied dict must hold every output of output_shapes
        fe.extract_batch(gray, depth, out=out)
    o = fe._outputs({k: v.ctypes.data for k, v in out.items()})
    import ctypes as C
    hvo._check(hvo.lib().hvo_frame_extract_batch(fe._h, hvo._np_ptr(gray), hvo._np_ptr(depth), 3, C.byref(o)))
    for f in range(3):
        n = int(d['kp_counts'][f])
        assert np.array_equal(out['kp_uright'][f, :n], d['kp_uright'][f, :n])
    fe.close()


@pytest.mark.gpu
def test_gpu_frame_undistort_launch_count_and_pinhole_handles(hvo, synth):
    """One extra launch per chunk; all-zero coefficients keep today's handle (no kps_un, kp_uright -1 when `distorted`), and a
    pinhole handle refuses a kps_un output."""
    gray, depth = _frames(synth, 2, 7)
    a, b = _fe(hvo, None, max_batch=2), _fe(hvo, TUM1_DIST, max_batch=2)
    a.extract_batch(gray, depth); b.extract_batch(gray, depth)
    assert b.last_launches() == a.last_launches() + 1
    a.close(); b.close()
    z = _fe(hvo, np.zeros(5, np.float32), max_batch=2, distorted=True)
    assert 'kps_un' not in z.output_shapes(2)
    o = z.extract_batch(gray, depth)
    for f in range(2):
        assert (o['kp_uright'][f, :int(o['kp_counts'][f])] == -1).all()
    out = z.alloc_host(2)
    out['kps_un'] = np.empty((2, z.orb_capacity), hvo.KP_DTYPE)
    c = z._outputs({k: v.ctypes.data for k, v in out.items()})
    import ctypes as C
    assert hvo.lib().hvo_frame_extract_batch(z._h, hvo._np_ptr(gray), hvo._np_ptr(depth), 2, C.byref(c)) == hvo.HVO_ERR_ARG
    z.close()


@pytest.mark.gpu
def test_gpu_frame_undistort_chunked_async_and_device_resident(hvo, synth):
    """The same frames through the two-lane chunked path (n larger than a chunk), queued async calls and the device-resident call."""
    import torch
    gray, depth = _frames(synth, 5, 23)
    ref = _fe(hvo, TUM1_DIST, max_batch=5, lanes=1)
    r = ref.extract_batch(gray, depth)
    ref.close()
    plain = _fe(hvo, None, max_batch=5, lanes=1)
    _check_distorted_against_plain(hvo, r, plain.extract_batch(gray, depth), 5, TUM1_K, TUM1_DIST)
    plain.close()
    keys = ('kps', 'kps_un', 'desc', 'kp_depth', 'kp_uright')

    def same(o, n):
        for f in range(n):
            k = int(r['kp_counts'][f])
            assert k == int(o['kp_counts'][f])
            for key in keys:
                assert o[key][f, :k].tobytes() == r[key][f, :k].tobytes(), key

    fe = _fe(hvo, TUM1_DIST, max_batch=4, lanes=2)
    assert fe.chunk == 2
    same(fe.extract_batch(gray, depth), 5)               # three chunks through two lanes
    outs = [fe.alloc_host(5) for _ in range(2)]
    for o in outs:
        fe.extract_batch(gray, depth, out=o, wait=False)
    fe.sync()
    for o in outs:
        same(o, 5)
    bad = fe.alloc_host(5)
    bad['kps_un'] = np.empty((5, fe.orb_capacity + 1), hvo.KP_DTYPE)
    with pytest.raises(hvo.HvoError):
        fe.extract_batch(gray, depth, out=bad)
    # device-resident: n <= max_batch
    dev = torch.device('cuda', 0)
    shapes = fe.output_shapes(4)
    d = {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
    g, dp = torch.from_numpy(gray[:4].copy()).to(dev), torch.from_numpy(depth[:4].copy()).to(dev)
    torch.cuda.synchronize()
    fe.extract_batch_device(g.data_ptr(), dp.data_ptr(), 4, {k: v.data_ptr() for k, v in d.items()})
    fe.sync()
    same({k: d[k].cpu().numpy().view(dt).reshape(s) for k, (s, dt) in shapes.items()}, 4)
    fe.close()


@pytest.mark.gpu
def test_gpu_frame_sequence_undistorts_like_the_frame_handle(hvo, synth):
    gray, depth = _frames(synth, 5, 23)
    fx, fy, cx, cy = _tum1_cam()
    ref = _fe(hvo, TUM1_DIST, max_batch=5, line_cull=True)
    r = ref.extract_batch(gray, depth)
    ref.close()
    seq = hvo.FrameSequence(640, 480, fx, fy, cx, cy, 1.0 / 5000.0, [0, 0], frames_per_call=2, bf=40.0, dist=TUM1_DIST)
    assert 'kps_un' in seq.output_shapes(5, device=False)
    o = seq.extract(gray, depth)
    for f in range(5):
        k, nl = int(r['kp_counts'][f]), int(r['line_counts'][f])
        assert k == int(o['kp_counts'][f]) and nl == int(o['line_counts'][f])
        for key in ('kps', 'kps_un', 'desc', 'kp_depth', 'kp_uright'):
            assert o[key][f, :k].tobytes() == r[key][f, :k].tobytes(), key
        assert o['keylines'][f, :nl].tobytes() == r['keylines'][f, :nl].tobytes()
    bad = seq.alloc_host(5)
    bad['kps_un'] = np.empty((4, seq.orb_capacity), hvo.KP_DTYPE)
    with pytest.raises(hvo.HvoError):
        seq.extract(gray, depth, out=bad)
    seq.close()


@pytest.mark.gpu
def test_gpu_k1_zero_keeps_the_keypoints(hvo, synth):
    """k1 == 0 with other coefficients: the reference leaves mvKeysUn = mvKeys, so kps_un == kps and kp_uright is the pinhole one."""
    gray, depth = _frames(synth, 2, 3)
    plain = _fe(hvo, None, max_batch=2)
    p = plain.extract_batch(gray, depth)
    plain.close()
    fe = _fe(hvo, K1ZERO_DIST, max_batch=2)
    o = fe.extract_batch(gray, depth)
    fe.close()
    for f in range(2):
        n = int(p['kp_counts'][f])
        assert o['kps_un'][f, :n].tobytes() == o['kps'][f, :n].tobytes() == p['kps'][f, :n].tobytes()
        assert np.array_equal(_bits(o['kp_uright'][f, :n]), _bits(p['kp_uright'][f, :n]))


@pytest.mark.gpu
def test_gpu_orb_extractor_extract_batch_with_camera(hvo, synth):
    gray, depth = _frames(synth, 2, 3)
    ex = hvo.ORBextractor(1000, 1.2, 8, 20, 7, width=640, height=480, max_batch=2)
    plain = ex.extract_batch(gray, depth16=depth, depth_factor=1.0 / 5000.0, bf=40.0, distorted=True)
    out = ex.extract_batch(gray, depth16=depth, depth_factor=1.0 / 5000.0, bf=40.0, camera=(TUM1_K, TUM1_DIST))
    for f in range(2):
        n = int(plain['counts'][f])
        assert int(out['counts'][f]) == n and out['kps'][f, :n].tobytes() == plain['kps'][f, :n].tobytes()
        assert np.array_equal(out['desc'][f, :n], plain['desc'][f, :n]) and np.array_equal(out['depth'][f, :n], plain['depth'][f, :n])
        un = _host_un(hvo, plain['kps'][f, :n], TUM1_K, TUM1_DIST)
        assert out['kps_un'][f, :n].tobytes() == un.tobytes()
        assert np.array_equal(out['uright'][f, :n], hvo.ORBextractor.stereo_uright_from_depth(un, plain['depth'][f, :n], 40.0))
    ex.close()


@pytest.mark.gpu
def test_gpu_kps_un_and_bounds_build_the_reference_grid(hvo, synth):
    """The first consumer of mvKeysUn: ProjectionMatcher.set_frame (Frame::AssignFeaturesToGrid with ComputeImageBounds' bounds) gives
    the same grid from the device's kps_un as from host-undistorted keypoints."""
    gray, depth = _frames(synth, 1, 11)
    fe = _fe(hvo, TUM1_DIST, max_batch=1)
    o = fe.extract_batch(gray, depth)
    fe.close()
    n = int(o['kp_counts'][0])
    bounds = hvo.image_bounds(TUM1_K, TUM1_DIST, 640, 480)
    min_x, max_x, min_y, max_y = bounds
    grids = []
    for keys in (o['kps_un'][0, :n], _host_un(hvo, o['kps'][0, :n], TUM1_K, TUM1_DIST)):
        pm = hvo.ProjectionMatcher()
        pm.set_frame(keys, o['kp_uright'][0, :n], o['desc'][0, :n], min_x, min_y, max_x, max_y)
        grids.append(pm.grid())
        pm.close()
    assert np.array_equal(grids[0][0], grids[1][0]) and np.array_equal(grids[0][1], grids[1][1])
    assert grids[0][0][-1] > n // 2                 # most keypoints land in a cell
    plain = hvo.ProjectionMatcher()                 # and the distortion changes the grid
    plain.set_frame(o['kps'][0, :n], None, o['desc'][0, :n], 0.0, 0.0, 640.0, 480.0)
    assert not np.array_equal(plain.grid()[1], grids[0][1])
    plain.close()
