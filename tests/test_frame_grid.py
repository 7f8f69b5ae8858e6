"""Frame grids from the frame pipeline: a frame handle (or a sequence) created with grids=True also returns, for every frame, what
Frame::AssignFeaturesToGrid / AssignFeaturesToGridForLine (reference src/Frame.cc:832-872) build, mGrid and mGridForLine, with the
handle's image bounds.

  CPU: the binding mirrors the header's hvo_frame_grid_outputs; the drop-in hvo_shim::fillGrid (shim/FrameGridGPU.h) builds from
       fabricated rows the grids FrameFrontEnd.grid() / line_grid() return
  GPU: frame f's grids == oracle.grid_build / oracle.line_grid_build on its rows == the single-frame hvo_proj / hvo_lproj grids, through
       every call path; every other output is byte-identical to the same call without grids."""
import ctypes as C
import os
import re
import struct
import subprocess

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'a-low-texture-robust-hybrid-feature-based-visual-odometry_b200')
GRID_KEYS = ('grid_counts', 'grid_items', 'lgrid_counts', 'lgrid_items')
TUM1 = np.array([0.262383, -0.953104, -0.005358, 0.002628, 1.163314], np.float32)
SENTINEL = 0xBEEF


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_grid_outputs_binding_mirrors_the_header(hvo):
    src = open(os.path.join(ROOT, 'include', 'hvo_capi.h')).read()
    body = re.search(r'typedef struct hvo_frame_grid_outputs \{(.*?)\} hvo_frame_grid_outputs;', src, re.S).group(1)
    body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)
    assert re.findall(r'uint16_t\*\s*(\w+)\s*;', body) == [f[0] for f in hvo._FrameGridOutputs._fields_] == hvo.FrameFrontEnd.GRID_FIELDS \
        == list(GRID_KEYS)
    for name in ('hvo_frame_extract_batch_grid', 'hvo_frame_extract_batch_async_grid', 'hvo_frame_extract_batch_device_grid', 'hvo_frame_image_bounds',
                 'hvo_frame_line_grid_capacity', 'hvo_seq_extract_grid', 'hvo_seq_image_bounds', 'hvo_seq_line_grid_capacity'):
        assert name in hvo.ABI
    # the existing output structs are unchanged
    assert hvo.FrameFrontEnd.FIELDS[-1] == 'kps_un' and len(hvo.FrameFrontEnd.FIELDS) == 17
    assert hvo.FrameFrontEnd.BOW_FIELDS == ['bow_counts', 'bow_words', 'bow_values', 'fv_order', 'fv_counts', 'node_of', 'word_of']


def _random_keys(hvo, n, seed, lo=(-40.0, -30.0), hi=(680.0, 510.0)):
    rng = np.random.default_rng(seed)
    k = np.zeros(n, hvo.KP_DTYPE)
    k['x'] = rng.uniform(lo[0], hi[0], n).astype(np.float32)
    k['y'] = rng.uniform(lo[1], hi[1], n).astype(np.float32)
    return k


def _random_keylines(hvo, n, seed):
    rng = np.random.default_rng(seed)
    kl = np.zeros(n, hvo.KL_DTYPE)
    kl['startPointX'], kl['startPointY'] = rng.uniform(-20, 660, n), rng.uniform(-20, 500, n)
    kl['endPointX'], kl['endPointY'] = rng.uniform(-20, 660, n), rng.uniform(-20, 500, n)
    return kl


def _rows(grids, cap):
    """[(counts, items)] -> ([n][3072] uint16, [n][cap] uint16) as a frame call lays them out, the tail of each items row a sentinel."""
    counts = np.zeros((len(grids), 64 * 48), np.uint16)
    items = np.full((len(grids), cap), SENTINEL, np.uint16)
    for f, (c, it) in enumerate(grids):
        counts[f], items[f, :len(it)] = c, it
    return counts, items


def _run_fill(exe, tmp_path, counts, items):
    fi, fo = str(tmp_path / 'in.bin'), str(tmp_path / 'out.bin')
    with open(fi, 'wb') as f:
        f.write(struct.pack('<3i', 0x44495247, len(counts), items.shape[1]) + counts.tobytes() + items.tobytes())
    subprocess.check_call([exe, fi, fo])
    raw, pos, res = open(fo, 'rb').read(), 0, []
    for _ in range(len(counts)):
        c = np.frombuffer(raw, np.int32, 64 * 48, pos); pos += 4 * 64 * 48
        it = np.frombuffer(raw, np.int32, int(c.sum()), pos); pos += 4 * int(c.sum())
        res.append((c, it))
    assert pos == len(raw)
    return res


def test_shim_fill_grid_equals_frame_front_end_grid(hvo, tmp_path):
    exe = str(tmp_path / 'shim_grid_fill')
    subprocess.check_call(['g++', '-O2', '-std=c++14', '-Wall', '-I' + os.path.join(PKG, 'shim'), os.path.join(ROOT, 'tests', 'cpp', 'shim_grid_fill_main.cpp'),
                           '-o', exe])
    bounds = (0.0, 0.0, 640.0, 480.0)   # oracle order: min_x, min_y, max_x, max_y
    cap = 300
    # points: an empty frame, one whose points partly fall outside the bounds (dropped), a full frame inside them (round(x / 10) < 64)
    pts = [oracle.grid_build(_random_keys(hvo, 0, 1), bounds), oracle.grid_build(_random_keys(hvo, 200, 2), bounds),
           oracle.grid_build(_random_keys(hvo, cap, 3, lo=(0.0, 0.0), hi=(634.0, 474.0)), bounds)]
    assert pts[1][0].sum() < 200 and pts[2][0].sum() == cap
    counts, items = _rows(pts, cap)
    out = dict(grid_counts=counts, grid_items=items)
    for f, (c, it) in enumerate(_run_fill(exe, tmp_path, counts, items)):
        want = hvo.FrameFrontEnd.grid(out, f)
        assert np.array_equal(c, want[0]) and np.array_equal(it, want[1]) and np.array_equal(it, pts[f][1])
    # lines: an empty frame and a frame of lines crossing many cells, some leaving the image
    lcap = 64 * 40
    lines = [oracle.line_grid_build(_random_keylines(hvo, 0, 4), bounds), oracle.line_grid_build(_random_keylines(hvo, 40, 5), bounds)]
    assert lines[1][0].sum() > 40 * 10
    counts, items = _rows(lines, lcap)
    out = dict(lgrid_counts=counts, lgrid_items=items)
    for f, (c, it) in enumerate(_run_fill(exe, tmp_path, counts, items)):
        want = hvo.FrameFrontEnd.line_grid(out, f)
        assert np.array_equal(c, want[0]) and np.array_equal(it, want[1]) and np.array_equal(it, lines[f][1])


# ---------------------------------------------------------------------------------------------------------------- GPU
def _cam(synth, config='S1'):
    c = synth.CONFIGS[config]
    return c['fx'], c['fy'], c['cx'], c['cy'], 1.0 / c['factor']


def _frames(synth, config='S1'):
    """Two frames of `config` and a constant image (no keypoints, no lines)."""
    g, d = synth.sequence(config, 2, start=31 if config == 'S1' else 9)
    return np.concatenate([g, np.full_like(g[:1], 128)]), np.concatenate([d, d[:1]])


def _fe(hvo, synth, config='S1', **kw):
    return hvo.FrameFrontEnd(640, 480, *_cam(synth, config), bf=40.0, **kw)


def _oracle_bounds(fe):
    min_x, max_x, min_y, max_y = fe.image_bounds()
    return float(min_x), float(min_y), float(max_x), float(max_y)


def _point_rows(fe, out, f):
    return (out['kps_un'] if fe.undistorts else out['kps'])[f, :int(out['kp_counts'][f])]


def _check_parity(hvo, fe, out, nframes, pm=None, lpm=None):
    """Frame f's grids == the oracle's on its rows (and == the single-frame device grids when pm / lpm are given)."""
    b = _oracle_bounds(fe)
    for f in range(nframes):
        if 'grid_counts' in out:
            rows = _point_rows(fe, out, f)
            got = hvo.FrameFrontEnd.grid(out, f)
            want = oracle.grid_build(rows, b)
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), f
            if pm is not None:
                pm.set_frame(rows, None, np.zeros((len(rows), 32), np.uint8), *b)
                cs, it = pm.grid()
                assert np.array_equal(np.diff(cs), got[0]) and np.array_equal(it, got[1]), f
        if 'lgrid_counts' in out:
            kl = out['keylines'][f, :int(out['line_counts'][f])]
            got = hvo.FrameFrontEnd.line_grid(out, f)
            want = oracle.line_grid_build(kl, b)
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), f
            if lpm is not None:
                lpm.set_frame(kl, np.zeros((len(kl), 3)), np.zeros((len(kl), 32), np.uint8), None, *b)
                c, it = lpm.grid()
                assert np.array_equal(c, got[0]) and np.array_equal(it, got[1]), f


def _check_same_as_plain(d, p, nframes):
    """Every output of the call without grids, byte for byte, in the rows a frame owns."""
    for f in range(nframes):
        n, nl, npl = int(p['kp_counts'][f]), int(p['line_counts'][f]), int(p['n_planes'][f])
        assert (n, nl, npl) == (int(d['kp_counts'][f]), int(d['line_counts'][f]), int(d['n_planes'][f]))
        for k in ('kps', 'desc', 'kp_depth', 'kp_uright', 'kps_un'):
            if k in p:
                assert d[k][f, :n].tobytes() == p[k][f, :n].tobytes(), k
        for k in ('keylines', 'line_desc', 'linevec3'):
            assert d[k][f, :nl].tobytes() == p[k][f, :nl].tobytes(), k
        assert d['planes7'][f, :npl].tobytes() == p['planes7'][f, :npl].tobytes()
        for k in ('membership', 'membership8', 'membership4', 'normals8', 'normals3'):
            if k in p:
                assert d[k][f].tobytes() == p[k][f].tobytes(), k


def _same_grids(hvo, o, r, n, frames=None):
    """Frame f of o has the grids of frame frames[f] (default f) of r."""
    for f in range(n):
        g = f if frames is None else frames[f]
        for key, fn in (('grid_counts', hvo.FrameFrontEnd.grid), ('lgrid_counts', hvo.FrameFrontEnd.line_grid)):
            if key in o:
                a, b = fn(o, f), fn(r, g)
                assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), (key, f)


@pytest.mark.gpu
@pytest.mark.parametrize('config,line_cull', [('S1', False), ('S1', True), ('S2', False), ('S2', True)])
def test_gpu_frame_grids_equal_oracle_and_single_frame_grids(hvo, synth, config, line_cull):
    gray, depth = _frames(synth, config)
    nf = len(gray)
    plain = _fe(hvo, synth, config, max_batch=nf, line_cull=line_cull)
    p = plain.extract_batch(gray, depth)
    launches = plain.last_launches()
    plain.close()
    assert int(p['kp_counts'][-1]) == 0 and min(p['kp_counts'][:-1]) > 100 and min(p['line_counts'][:-1]) > 5
    fe = _fe(hvo, synth, config, max_batch=nf, line_cull=line_cull, grids=True)
    assert fe.image_bounds() == (0.0, 640.0, 0.0, 480.0)
    assert fe.line_grid_capacity == 64 * fe.max_lines
    sh = fe.output_shapes(nf)
    assert sh['grid_items'] == ((nf, fe.orb_capacity), np.uint16) and sh['lgrid_items'] == ((nf, 64 * fe.max_lines), np.uint16)
    d = fe.extract_batch(gray, depth)
    assert fe.last_launches() == launches + 3                # k_proj_grid, k_lproj_grid + k_lproj_grid_compact
    _check_same_as_plain(d, p, nf)
    pm, lpm = hvo.ProjectionMatcher(), hvo.LineProjectionMatcher()
    _check_parity(hvo, fe, d, nf, pm, lpm)
    pm.close(); lpm.close(); fe.close()
    assert not d['grid_counts'][-1].any() and not d['lgrid_counts'][-1].any()
    assert int(d['grid_counts'][0].sum()) == int(d['kp_counts'][0])            # no undistortion: every keypoint is inside the grid


@pytest.mark.gpu
def test_gpu_frame_grids_on_the_undistorting_tum1_handle(hvo, synth):
    """Bounds == hvo_image_bounds of the camera; the point grid is built on kps_un, also when the host call does not ask for kps_un."""
    gray, depth = _frames(synth)
    nf = len(gray)
    fx, fy, cx, cy, _ = _cam(synth)
    K = np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1]], np.float32)
    fe = _fe(hvo, synth, max_batch=nf, dist=TUM1, grids=True)
    assert fe.image_bounds() == hvo.image_bounds(K, TUM1, 640, 480) and fe.image_bounds() != (0.0, 640.0, 0.0, 480.0)
    d = fe.extract_batch(gray, depth)
    pm, lpm = hvo.ProjectionMatcher(), hvo.LineProjectionMatcher()
    _check_parity(hvo, fe, d, nf, pm, lpm)
    pm.close(); lpm.close()
    for f in range(nf - 1):                                  # not the grid of the distorted keypoints
        assert not np.array_equal(hvo.FrameFrontEnd.grid(d, f)[1], oracle.grid_build(d['kps'][f, :int(d['kp_counts'][f])], _oracle_bounds(fe))[1])
    # host call without kps_un: the grid still comes from the undistorted rows
    part = {k: v for k, v in fe.alloc_host(nf).items() if k != 'kps_un'}
    ptrs = {k: v.ctypes.data for k, v in part.items()}
    hvo._check(hvo.lib().hvo_frame_extract_batch_grid(fe._h, hvo._np_ptr(gray), hvo._np_ptr(depth), nf, C.byref(fe._outputs(ptrs)), None,
                                                      fe._grid_outputs(ptrs)))
    _same_grids(hvo, part, d, nf)
    fe.close()


@pytest.mark.gpu
def test_gpu_frame_grids_through_every_call_path(hvo, synth):
    """Blocking, two queued wait=False calls, the device-resident call (untouched entries past each frame's total), several chunks
    through two lanes, two serial chunks of 2048 frames (device-resident), FrameSequence and grids with a vocabulary: the same grids
    as the blocking call."""
    import torch
    g1, d1 = _frames(synth)
    g2, d2 = _frames(synth, 'S2')
    gray, depth = np.concatenate([g1, g2[:2]]), np.concatenate([d1, d2[:2]])
    nf = len(gray)
    ref = _fe(hvo, synth, max_batch=nf, lanes=1, grids=True)
    r = ref.extract_batch(gray, depth)
    _check_parity(hvo, ref, r, nf)
    ref.close()

    fe = _fe(hvo, synth, max_batch=4, lanes=2, grids=True)
    assert fe.chunk == 2
    _same_grids(hvo, fe.extract_batch(gray, depth), r, nf)         # three chunks through two lanes (side by side)
    outs = [fe.alloc_host(nf) for _ in range(2)]
    for o in outs:
        fe.extract_batch(gray, depth, out=o, wait=False)
    fe.sync()
    for o in outs:
        _same_grids(hvo, o, r, nf)
    bad = fe.alloc_host(nf)
    bad['lgrid_items'] = np.empty((nf, fe.line_grid_capacity - 1), np.uint16)
    with pytest.raises(hvo.HvoError):
        fe.extract_batch(gray, depth, out=bad)
    # device-resident, on torch tensors prefilled with a sentinel: entries past each frame's total are not written
    dev = torch.device('cuda', 0)
    shapes = fe.output_shapes(4)
    d = {k: torch.full((int(np.prod(s)) * np.dtype(dt).itemsize,), 0xEF, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
    g, dp = torch.from_numpy(gray[:4].copy()).to(dev), torch.from_numpy(depth[:4].copy()).to(dev)
    torch.cuda.synchronize()
    fe.extract_batch_device(g.data_ptr(), dp.data_ptr(), 4, {k: v.data_ptr() for k, v in d.items()})
    fe.sync()
    o = {k: d[k].cpu().numpy().view(dt).reshape(s) for k, (s, dt) in shapes.items()}
    _same_grids(hvo, o, r, 4)
    for f in range(4):
        for c, i in (('grid_counts', 'grid_items'), ('lgrid_counts', 'lgrid_items')):
            assert (o[i][f, int(o[c][f].sum()):] == 0xEFEF).all(), (i, f)
    fe.close()
    del d

    # 4096 frames device-resident through two lanes: two chunks of 2048, each running its pipelines one after the other
    big = _fe(hvo, synth, max_batch=4096, lanes=2, grids=True, membership='u8', normals='n8')
    assert big.chunk == 2048
    n = 4096
    pick = np.arange(n) % nf
    g = torch.from_numpy(gray).to(dev)[torch.from_numpy(pick).to(dev)].contiguous()
    dp = torch.from_numpy(depth.view(np.int16)).to(dev)[torch.from_numpy(pick).to(dev)].contiguous()   # (no uint16 indexing on the device)
    shapes = big.output_shapes(n)
    d = {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
    torch.cuda.synchronize()
    big.extract_batch_device(g.data_ptr(), dp.data_ptr(), n, {k: v.data_ptr() for k, v in d.items()})
    big.sync()
    _same_grids(hvo, {k: d[k].cpu().numpy().view(shapes[k][1]).reshape(shapes[k][0]) for k in GRID_KEYS}, r, n, pick)
    big.close()
    del d, g, dp
    torch.cuda.empty_cache()

    # FrameSequence: two handles (the device list names cuda:0 twice), queued calls of two frames
    seq = hvo.FrameSequence(640, 480, *_cam(synth), [0, 0], frames_per_call=2, bf=40.0, line_cull=False, grids=True)
    assert set(GRID_KEYS) <= set(seq.output_shapes(nf, device=False)) and seq.image_bounds() == (0.0, 640.0, 0.0, 480.0)
    assert seq.line_grid_capacity == 64 * seq.max_lines
    _same_grids(hvo, seq.extract(gray, depth), r, nf)
    bad = seq.alloc_host(nf)
    bad['grid_counts'] = np.empty((nf, 64 * 48), np.int32)
    with pytest.raises(hvo.HvoError):
        seq.extract(gray, depth, out=bad)
    seq.close()

    # grids and BoW in one call
    gv = np.load(os.path.join(ROOT, 'tests', 'golden', 'bow_ref.npz'))
    voc = {k[4:]: gv[k] for k in gv.files if k.startswith('voc_')}
    voc['L'] = int(voc['L'])
    fb = _fe(hvo, synth, max_batch=nf, vocabulary=voc, grids=True)
    o = fb.extract_batch(gray, depth)
    _same_grids(hvo, o, r, nf)
    bt = hvo.ORBVocabulary(voc)
    ref_bow = bt.transform_batch([o['desc'][f, :int(o['kp_counts'][f])] for f in range(nf)], 4)
    bt.close()
    for f in range(nf):
        w = int(o['bow_counts'][f])
        assert np.array_equal(o['bow_words'][f, :w], ref_bow[f][0][0])
    fb.close()


@pytest.mark.gpu
def test_gpu_frame_grid_argument_errors(hvo, synth):
    gray, depth = _frames(synth)
    gray, depth = gray[:1], depth[:1]
    zeros16 = np.zeros(16, np.uint16)   # (refused calls write nothing)

    def grid_arg(points, lines):
        p = zeros16.ctypes.data
        return hvo._FrameGridOutputs(p if points else None, p if points else None, p if lines else None, p if lines else None)

    for stages, points, lines in ((hvo.STAGE_LINES, True, False), (hvo.STAGE_ORB, False, True)):
        fe = _fe(hvo, synth, stages=stages)
        out = fe.alloc_host(1)
        ptrs = {k: v.ctypes.data for k, v in out.items()}
        st = hvo.lib().hvo_frame_extract_batch_grid(fe._h, hvo._np_ptr(gray), hvo._np_ptr(depth), 1, C.byref(fe._outputs(ptrs)), None,
                                                     C.byref(grid_arg(points, lines)))
        assert st == hvo.HVO_ERR_ARG, stages
        fe.close()
    fe = _fe(hvo, synth, stages=hvo.STAGE_ORB)
    out = fe.alloc_host(1)
    ptrs = {k: v.ctypes.data for k, v in out.items()}
    half = hvo._FrameGridOutputs(zeros16.ctypes.data, None, None, None)
    assert hvo.lib().hvo_frame_extract_batch_grid(fe._h, hvo._np_ptr(gray), hvo._np_ptr(depth), 1, C.byref(fe._outputs(ptrs)), None,
                                                  C.byref(half)) == hvo.HVO_ERR_ARG          # counts without items
    fe.close()

    # the device call of an undistorting handle needs kps_un for point grids
    import torch
    fe = _fe(hvo, synth, dist=TUM1, grids=True)
    dev = torch.device('cuda', 0)
    shapes = fe.output_shapes(1)
    d = {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
    g, dp = torch.from_numpy(gray.copy()).to(dev), torch.from_numpy(depth.copy()).to(dev)
    dptr = {k: v.data_ptr() for k, v in d.items()}
    no_un = dict(dptr, kps_un=None)
    st = hvo.lib().hvo_frame_extract_batch_device_grid(fe._h, g.data_ptr(), dp.data_ptr(), 1, C.byref(fe._outputs(no_un)), None, fe._grid_outputs(dptr))
    assert st == hvo.HVO_ERR_ARG
    fe.extract_batch_device(g.data_ptr(), dp.data_ptr(), 1, dptr)
    fe.sync()
    fe.close()
