"""The frame drop-in hvo_shim::FrameExtractorGPU (shim/FrameExtractorGPU.h): one frame call fills every member of Frame::Frame's
extraction block (threads A-C, the grid threads, ComputeBoW) and returns thread D's LPVO rows on request.

  CPU: the header and tests/cpp/shim_frame_main.cpp compile with g++ -std=c++14 against the stand-ins; a refused frame writes exactly
       the empty serialisation of this module's writer (the layout is pinned); without a device extract returns false with empty
       outputs and the library's message.
  GPU: for every case, frame (a) (FrameExtractorGPU::extract) equals frame (b) (the per-class drop-ins in the reference's order) member by
       member, byte for byte, and both equal the serialisation built here from FrameFrontEnd.extract_batch with the existing expanders."""
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'a-low-texture-robust-hybrid-feature-based-visual-odometry_b200')
MAGIC = 0x444d5246
TUM1_K = (517.306408, 516.469215, 318.643040, 255.313989)
TUM1_DIST = (0.262383, -0.953104, -0.005358, 0.002628, 1.163314)
KEYS = ('bounds', 'N', 'mvKeys', 'mvKeysUn', 'mDescriptors', 'mvDepth', 'mvuRight', 'NL', 'mvKeylinesUn', 'mLdesc', 'mvKeyLineFunctions',
        'plane_num_', 'planes', 'vSurfaceNormal', 'mGrid', 'mGridForLine', 'mBowVec', 'mFeatVec', 'lpvo')


def build_driver(out):
    """g++ -std=c++14 of tests/cpp/shim_frame_main.cpp against the stand-ins and the library, to the path out"""
    if not os.path.exists(os.path.join(PKG, 'libhvofront.so')):
        import __graft_entry__
        __graft_entry__.build()
    subprocess.check_call(['g++', '-O2', '-std=c++14', '-Wall', '-Werror', '-I' + os.path.join(ROOT, 'oracle', 'cvshim'),
                           '-I' + os.path.join(ROOT, 'tests', 'cpp', 'standins'), '-I' + os.path.join(PKG, 'shim'), '-I' + os.path.join(ROOT, 'include'),
                           os.path.join(ROOT, 'tests', 'cpp', 'shim_frame_main.cpp'), '-o', out, '-L' + PKG, '-lhvofront', '-Wl,-rpath,' + PKG])
    return out


@pytest.fixture(scope='module')
def exe(tmp_path_factory):
    return build_driver(str(tmp_path_factory.mktemp('shim_frame') / 'shim_frame'))


# ---- the canonical serialisation (the layout tests/cpp/shim_frame_main.cpp writes) ------------------------------------------------
def _grid_bytes(counts, items):
    return np.asarray(counts, '<i4').tobytes() + np.asarray(items, '<i4').tobytes()


def serialise(fr, lpvo):
    """fr: dict of one frame's members (see _empty / _expected) -> the bytes the driver writes for it"""
    b = np.asarray(fr['bounds'], '<f4').tobytes()
    n, nl = len(fr['desc']), len(fr['ldesc'])
    b += struct.pack('<i', n) + fr['kps'].tobytes() + fr['kps_un'].tobytes()
    b += struct.pack('<3i', n, 32 if n else 0, 0) + fr['desc'].tobytes() + np.asarray(fr['depth'], '<f4').tobytes()
    b += np.asarray(fr['uright'], '<f4').tobytes()
    b += struct.pack('<i', nl) + fr['keylines'].tobytes() + struct.pack('<3i', nl, 32 if nl else 0, 0) + fr['ldesc'].tobytes()
    b += np.asarray(fr['linevec'], '<f8').tobytes()
    b += struct.pack('<i', len(fr['planes']))
    for normal, center, support, idx, xyz in fr['planes']:
        b += np.asarray(normal, '<f8').tobytes() + np.asarray(center, '<f8').tobytes() + struct.pack('<2i', support, len(idx))
        b += np.asarray(idx, '<i4').tobytes() + np.asarray(xyz, '<f8').tobytes()
    sn = np.asarray(fr['normals8'], '<f4').reshape(-1, 8)
    rows = np.zeros(len(sn), [('xyz', '<f4', 6), ('pos', '<i4', 2)])   # FramePosition as the int it is
    rows['xyz'], rows['pos'] = sn[:, :6], sn[:, 6:].astype(np.int32)
    b += struct.pack('<i', len(sn)) + rows.tobytes()
    b += _grid_bytes(*fr['grid']) + _grid_bytes(*fr['lgrid'])
    (words, values), fv = fr['bow']
    b += struct.pack('<i', len(words)) + b''.join(struct.pack('<Id', int(w), float(v)) for w, v in zip(words, values))
    b += struct.pack('<i', len(fv)) + b''.join(struct.pack('<Ii', k, len(fv[k])) + np.asarray(fv[k], '<u4').tobytes() for k in sorted(fv))
    if lpvo:
        nrm, dep = fr['lpvo']
        b += struct.pack('<i', len(dep)) + np.asarray(nrm, '<f8').tobytes() + np.asarray(dep, '<f4').tobytes()
    return b


def parse(raw, off, lpvo):
    """One serialised frame at raw[off:] -> (member name -> its bytes, next offset)"""
    m = {}

    def take(key, nbytes):
        nonlocal off
        m[key] = m.get(key, b'') + raw[off:off + nbytes]
        off += nbytes

    def i32():
        return struct.unpack_from('<i', raw, off)[0]

    take('bounds', 24)
    n = i32(); take('N', 4); take('mvKeys', 28 * n); take('mvKeysUn', 28 * n)
    rows = i32(); take('mDescriptors', 12 + 32 * rows); take('mvDepth', 4 * n); take('mvuRight', 4 * n)
    nl = i32(); take('NL', 4); take('mvKeylinesUn', 68 * nl)
    rows = i32(); take('mLdesc', 12 + 32 * rows); take('mvKeyLineFunctions', 24 * nl)
    npl = i32(); take('plane_num_', 4)
    for _ in range(npl):
        nv = struct.unpack_from('<i', raw, off + 52)[0]
        take('planes', 56 + 4 * nv + 24 * nv)
    ns = i32(); take('vSurfaceNormal', 4 + 32 * ns)
    for key in ('mGrid', 'mGridForLine'):
        total = int(np.frombuffer(raw, '<i4', 3072, off).sum())
        take(key, 4 * (3072 + total))
    nw = i32(); take('mBowVec', 4 + 12 * nw)
    nn = i32(); take('mFeatVec', 4)
    for _ in range(nn):
        k = struct.unpack_from('<i', raw, off + 4)[0]
        take('mFeatVec', 8 + 4 * k)
    if lpvo:
        k = i32(); take('lpvo', 4 + 28 * k)
    m.setdefault('planes', b'')
    m.setdefault('lpvo', b'')
    return m, off


def _empty(hvo):
    z = np.zeros((0, 32), np.uint8)
    return dict(bounds=np.zeros(6, np.float32), kps=np.zeros(0, hvo.KP_DTYPE), kps_un=np.zeros(0, hvo.KP_DTYPE), desc=z, depth=[], uright=[],
                keylines=np.zeros(0, hvo.KL_DTYPE), ldesc=z, linevec=np.zeros((0, 3)), planes=[], normals8=np.zeros((0, 8), np.float32),
                grid=(np.zeros(3072, np.int32), []), lgrid=(np.zeros(3072, np.int32), []), bow=(([], []), {}), lpvo=([], []))


# ---- the driver's input --------------------------------------------------------------------------------------------------------
def _run(exe, tmp_path, gray, depth, cam, dist=(0, 0, 0, 0, 0), bf=40.0, nfeatures=1000, max_planes=64, lpvo=False, vocabulary=None,
         mode=0, reps=None):
    n, h, w = gray.shape
    fx, fy, cx, cy, df = cam
    voc = vocabulary
    nodes = len(voc['node_weight']) if voc is not None else 0
    fi, fo = str(tmp_path / 'in.bin'), str(tmp_path / 'out.bin')
    with open(fi, 'wb') as f:
        f.write(struct.pack('<14i', MAGIC, w, h, n, nfeatures, 8, 20, 7, 200, max_planes, int(lpvo), mode, nodes, voc['L'] if voc else 0))
        f.write(np.array([1.2, fx, fy, cx, cy, *dist, bf, df], '<f4').tobytes())
        for g, d in zip(gray, depth):
            f.write(np.ascontiguousarray(g, np.uint8).tobytes() + np.ascontiguousarray(d, '<u2').tobytes())
        if voc is not None:
            f.write(np.asarray(voc['child_start'], '<i4').tobytes() + struct.pack('<i', len(voc['child_ids'])))
            f.write(np.asarray(voc['child_ids'], '<i4').tobytes() + np.asarray(voc['node_desc'], np.uint8).tobytes())
            f.write(np.asarray(voc['node_weight'], '<f8').tobytes() + np.asarray(voc['node_word'], '<i4').tobytes())
    r = subprocess.run([exe, fi, fo] + ([str(reps)] if reps else []), capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return open(fo, 'rb').read(), r.stderr


def _records(raw, nframes, lpvo):
    """[(ok, frame a, frame b or None)] of a driver output"""
    off, recs = 0, []
    for _ in range(nframes):
        ok = struct.unpack_from('<i', raw, off)[0]
        a, off = parse(raw, off + 4, lpvo)
        b = None
        if ok:
            b, off = parse(raw, off, lpvo)
        recs.append((ok, a, b))
    assert off == len(raw)
    return recs


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_dropin_compiles_against_the_standin_frame(exe):
    assert os.path.exists(exe)


def test_empty_frame_layout_is_pinned(hvo):
    raw = serialise(_empty(hvo), lpvo=True)
    # 6 bounds, N, (rows, cols, type), NL, (rows, cols, type), planes, normals, 2 x 3072 cell sizes, words, nodes, lpvo rows
    assert len(raw) == 24 + 4 + 12 + 4 + 12 + 4 + 4 + 2 * 4 * 3072 + 4 + 4 + 4
    m, off = parse(raw, 0, True)
    assert off == len(raw) and b''.join(m[k] for k in KEYS) == raw
    fr = _empty(hvo)
    fr['kps'] = fr['kps_un'] = np.zeros(2, hvo.KP_DTYPE)
    fr['desc'] = np.arange(64, dtype=np.uint8).reshape(2, 32)
    fr['depth'], fr['uright'] = [1.5, -1.0], [3.0, -1.0]
    fr['planes'] = [((0, 0, 1), (0, 0, 2), 7, [3, 9], np.ones((2, 3)))]
    fr['grid'] = (np.eye(1, 3072, 5, dtype=np.int32)[0] * 2, [0, 1])
    fr['bow'] = (([4, 9], [0.25, 0.75]), {3: [0], 1: [1]})
    raw = serialise(fr, lpvo=False)
    m, off = parse(raw, 0, False)
    assert off == len(raw) and b''.join(m[k] for k in KEYS) == raw
    assert m['mDescriptors'] == struct.pack('<3i', 2, 32, 0) + fr['desc'].tobytes()
    assert m['planes'] == struct.pack('<3d3d2i2i', 0, 0, 1, 0, 0, 2, 7, 2, 3, 9) + np.ones(6).tobytes()
    assert m['mFeatVec'] == struct.pack('<iIiIIiI', 2, 1, 1, 1, 3, 1, 0)     # nodes ascending, as in the std::map


def _no_device(hvo):
    """None with a CUDA device, else the message hvo_frame_create leaves"""
    try:
        if hvo.device_count() > 0:
            return None
    except hvo.HvoError:
        pass
    with pytest.raises(hvo.HvoError) as e:
        hvo.FrameFrontEnd(64, 64, 50.0, 50.0, 32.0, 32.0, 0.001)
    assert e.value.status == hvo.HVO_ERR_CUDA
    return str(e.value).split(': ', 1)[1]


def test_without_a_device_extract_refuses_with_empty_outputs(hvo, exe, tmp_path):
    why = _no_device(hvo)
    if why is None:
        pytest.skip('a CUDA device is present: the GPU tests cover the refusals')
    gray = np.full((1, 64, 64), 100, np.uint8)
    raw, err = _run(exe, tmp_path, gray, np.zeros((1, 64, 64), np.uint16), (50.0, 50.0, 32.0, 32.0, 0.001), lpvo=True)
    (ok, a, b), = _records(raw, 1, True)
    assert ok == 0 and b is None
    assert b''.join(a[k] for k in KEYS) == serialise(_empty(hvo), lpvo=True)
    assert 'FrameExtractorGPU: ' + why in err


# ---------------------------------------------------------------------------------------------------------------- GPU
def _vocabulary():
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from test_frame_bow import _random_vocabulary
    return _random_vocabulary(11, 4, 8, 5)


def _expected(hvo, fe, out, f, depth, lpvo):
    """frame f of FrameFrontEnd.extract_batch as the members Frame::Frame holds, with the existing expanders"""
    n, nl = int(out['kp_counts'][f]), int(out['line_counts'][f])
    fx, fy, cx, cy, df = (float(np.float32(v)) for v in fe.cam)   # the handle's float camera, widened as PlaneDetection does
    mn_x, mx_x, mn_y, mx_y = fe.image_bounds()
    bounds = np.array([mn_x, mx_x, mn_y, mx_y, np.float32(64) / (mx_x - mn_x), np.float32(48) / (mx_y - mn_y)], np.float32)
    kps = out['kps'][f, :n]
    if fe.membership_mode == 'u4':
        lab = fe.membership4_expand(out['membership4'][f])
    else:
        lab = out['membership'][f]
    npl = min(int(out['n_planes'][f]), fe.max_planes)
    planes = []
    zall = depth.ravel().astype(np.float64) * df
    for i in range(npl):
        idx = np.flatnonzero(lab == i).astype(np.int32)
        row, col, z = (idx // fe.w).astype(np.float64), (idx % fe.w).astype(np.float64), zall[idx]
        xyz = np.stack([(col - cx) * z / fx, (row - cy) * z / fy, z], 1)
        p = out['planes7'][f, i]
        planes.append((p[:3], p[3:6], int(p[6]), idx, xyz))
    n8 = out['normals8'][f] if fe.normals_mode == 'n8' else fe.normals3_expand(out['normals3'][f], depth)
    fr = dict(bounds=bounds, kps=kps, kps_un=out['kps_un'][f, :n] if fe.undistorts else kps, desc=out['desc'][f, :n], depth=out['kp_depth'][f, :n],
              uright=out['kp_uright'][f, :n], keylines=out['keylines'][f, :nl], ldesc=out['line_desc'][f, :nl], linevec=out['linevec3'][f, :nl],
              planes=planes, normals8=n8, grid=fe.grid(out, f), lgrid=fe.line_grid(out, f),
              bow=fe.bow(out, f) if fe.vocabulary is not None else (([], []), {}), lpvo=fe.lpvo(out, f)[:2] if lpvo else None)
    return fr


def _check(hvo, exe, tmp_path, gray, depth, cam, dist=None, bf=40.0, nfeatures=1000, max_planes=64, lpvo=False, vocabulary=None,
           membership='i32', normals='n8'):
    h, w = gray.shape[1:]
    raw, err = _run(exe, tmp_path, gray, depth, cam, dist if dist is not None else (0, 0, 0, 0, 0), bf, nfeatures, max_planes, lpvo, vocabulary)
    fe = hvo.FrameFrontEnd(w, h, *cam, bf=bf, nfeatures=nfeatures, max_planes=max_planes, line_cull=True, grids=True, lpvo=lpvo,
                           dist=dist, vocabulary=vocabulary, membership=membership, normals=normals)
    stats = []
    try:
        for f, (ok, a, b) in enumerate(_records(raw, len(gray), lpvo)):
            assert ok == 1, err
            for k in KEYS:
                assert a[k] == b[k], f'frame {f}: {k} of the frame drop-in differs from the per-class drop-ins'
            out = fe.extract_batch(gray[f:f + 1], depth[f:f + 1])
            want, _ = parse(serialise(_expected(hvo, fe, out, 0, depth[f], lpvo), lpvo), 0, lpvo)
            for k in KEYS:
                assert a[k] == want[k], f'frame {f}: {k} differs from FrameFrontEnd.extract_batch'
            stats.append((int(out['kp_counts'][0]), int(out['line_counts'][0]), int(out['n_planes'][0]),
                          int(out['lpvo_counts'][0]) if lpvo else 0, int(out['bow_counts'][0]) if vocabulary is not None else 0))
    finally:
        fe.close()
    return stats


def _cam(c):
    return (c['fx'], c['fy'], c['cx'], c['cy'], float(np.float32(1.0 / c['factor'])))


@pytest.mark.gpu
def test_tum3_camera_with_vocabulary_and_lpvo(hvo, synth, exe, tmp_path):
    g, d = synth.sequence('S1', 2, 0)
    st = _check(hvo, exe, tmp_path, g, d, _cam(synth.CONFIGS['S1']), lpvo=True, vocabulary=_vocabulary())
    assert all(s[0] > 500 and s[1] > 20 and s[2] >= 3 and s[3] > 500 and s[4] > 50 for s in st), st


@pytest.mark.gpu
def test_icl_camera_negative_fy_compact_forms(hvo, synth, exe, tmp_path):
    """ICL intrinsics (fy < 0), no vocabulary, no LPVO; the reference side expands the 4-bit labels and the 3-float normals"""
    g, d = synth.sequence('S2', 2, 3)
    st = _check(hvo, exe, tmp_path, g, d, _cam(synth.CONFIGS['S2']), max_planes=15, membership='u4', normals='n3')
    assert all(s[0] > 0 and s[2] >= 1 for s in st), st


@pytest.mark.gpu
def test_distorted_tum1_camera(hvo, synth, exe, tmp_path):
    """mvKeysUn != mvKeys and the image bounds are not (0, W, 0, H)"""
    g, d = synth.sequence('S1', 2, 5)
    cam = TUM1_K + (float(np.float32(1.0 / 5000.0)),)
    raw, _ = _run(exe, tmp_path, g[:1], d[:1], cam, TUM1_DIST)
    (ok, a, b), = _records(raw, 1, False)
    assert ok and a['mvKeys'] != a['mvKeysUn'] and np.frombuffer(a['bounds'], '<f4')[0] != 0
    _check(hvo, exe, tmp_path, g, d, cam, dist=TUM1_DIST, lpvo=True, vocabulary=_vocabulary())


@pytest.mark.gpu
def test_720p_with_int32_labels(hvo, synth, exe, tmp_path):
    """S3 at 1280x720; max_planes 300 is past the one-byte labels, so the drop-in takes the int32 ones"""
    c = synth.CONFIGS['S3']
    g, d = synth.frame('S3', 1)
    _check(hvo, exe, tmp_path, g[None], d[None], _cam(c), bf=c['bf'], nfeatures=c['nfeatures'], max_planes=300, lpvo=True)


@pytest.mark.gpu
def test_1080p_frame(hvo, synth, exe, tmp_path):
    c = synth.CONFIGS['S6']
    g, d = synth.frame('S6', 0)
    _check(hvo, exe, tmp_path, g[None], d[None], _cam(c), bf=c['bf'], nfeatures=c['nfeatures'], lpvo=True, vocabulary=_vocabulary())


@pytest.mark.gpu
def test_zero_depth_and_flat_image(hvo, synth, exe, tmp_path):
    """all-zero depth: no planes, every surface normal NaN, no LPVO sample; a flat image: no keypoints, no lines"""
    g, d = synth.frame('S1', 2)
    cam = _cam(synth.CONFIGS['S1'])
    st = _check(hvo, exe, tmp_path, g[None], np.zeros_like(d)[None], cam, lpvo=True, vocabulary=_vocabulary())
    assert st[0][2] == 0 and st[0][3] == 0 and st[0][0] > 0
    st = _check(hvo, exe, tmp_path, np.full_like(g, 128)[None], d[None], cam, lpvo=True, vocabulary=_vocabulary())
    assert st[0][0] == 0 and st[0][1] == 0 and st[0][2] >= 3


@pytest.mark.gpu
def test_sixteen_planes(hvo, synth, exe, tmp_path):
    """max_planes = 16, where the 4-bit label form is refused: the drop-in takes the one-byte labels"""
    g, d = synth.sequence('S1', 2, 7)
    _check(hvo, exe, tmp_path, g, d, _cam(synth.CONFIGS['S1']), max_planes=16)


@pytest.mark.gpu
@pytest.mark.parametrize('mode, why', [(1, 'the depth CV_16UC1'), (2, 'size differs')])
def test_refused_inputs_leave_every_output_empty(hvo, synth, exe, tmp_path, mode, why):
    g, d = synth.frame('S1', 0)
    raw, err = _run(exe, tmp_path, g[None], d[None], _cam(synth.CONFIGS['S1']), lpvo=True, vocabulary=_vocabulary(), mode=mode)
    (ok, a, b), = _records(raw, 1, True)
    assert ok == 0 and b is None and why in err
    assert b''.join(a[k] for k in KEYS) == serialise(_empty(hvo), lpvo=True)
