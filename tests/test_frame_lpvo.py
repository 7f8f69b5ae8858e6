"""LPVO normals from the frame pipeline: a frame handle (or a sequence) created with lpvo=True also returns, for every frame of a call,
what Manhattan::computeNormalsLPVO (reference src/Manhattan.cpp:237-393) computes on the frame's depth, the rows Frame::Frame gets from
ExtractMainImgPtNormals while the Manhattan axes are not initialised (src/Frame.cc:218-228).

  CPU: the binding mirrors the header's hvo_frame_lpvo_outputs (names, types, offsets) and the new entry points' argument lists; the
       flag is refused without the normals stage
  GPU: frame f's rows == hvo.Manhattan on the same depth == oracle.lpvo_normals (== the executed reference on its fixture cases), bytes
       of doubles, floats and int32, through every call path, at 640x480 and 1280x720; every other output is byte-identical to the same
       call without LPVO outputs."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, 'include', 'hvo_capi.h')
LPVO_KEYS = ('lpvo_normals3', 'lpvo_depth', 'lpvo_pix2', 'lpvo_counts')
TUM1 = np.array([0.262383, -0.953104, -0.005358, 0.002628, 1.163314], np.float32)
C_DTYPE = {'double': np.float64, 'float': np.float32, 'int32_t': np.int32}
NEW_CALLS = ('hvo_frame_extract_batch_lpvo', 'hvo_frame_extract_batch_async_lpvo', 'hvo_frame_extract_batch_device_lpvo', 'hvo_frame_lpvo_capacity',
             'hvo_seq_extract_lpvo', 'hvo_seq_lpvo_capacity')


def _header():
    return open(HEADER).read()


def _struct_fields():
    body = re.search(r'typedef struct hvo_frame_lpvo_outputs \{(.*?)\} hvo_frame_lpvo_outputs;', _header(), re.S).group(1)
    body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)
    return re.findall(r'(\w+)\*\s*(\w+)\s*;', body)


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_lpvo_outputs_binding_mirrors_the_header(hvo, tmp_path):
    fields = _struct_fields()
    assert [n for _, n in fields] == [f[0] for f in hvo._FrameLpvoOutputs._fields_] == ['normals3', 'depth', 'pix2', 'counts']
    assert hvo.FrameFrontEnd.LPVO_FIELDS == list(LPVO_KEYS)
    assert [t for t, _ in fields] == ['double', 'float', 'int32_t', 'int32_t']
    # offsets and size as a C compiler lays the header's struct out
    src = tmp_path / 'off.c'
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hvo_capi.h"\nint main(void) {\n'
                   + ''.join(f'    printf("%zu\\n", offsetof(hvo_frame_lpvo_outputs, {n}));\n' for _, n in fields)
                   + '    printf("%zu\\n", sizeof(hvo_frame_lpvo_outputs));\n    return 0;\n}\n')
    exe = str(tmp_path / 'off')
    subprocess.check_call(['gcc', '-std=c99', '-I' + os.path.join(ROOT, 'include'), str(src), '-o', exe])
    got = [int(v) for v in subprocess.check_output([exe], text=True).split()]
    assert got == [getattr(hvo._FrameLpvoOutputs, n).offset for _, n in fields] + [C.sizeof(hvo._FrameLpvoOutputs)]
    # the host arrays output_shapes asks for have the header's element types (a handle-free instance: shapes need no device)
    fe = object.__new__(hvo.FrameFrontEnd)
    fe.stages, fe.normals_mode, fe.normals_count, fe.with_lpvo, fe.lpvo_capacity = hvo.STAGE_NORMALS, 'n8', 7, True, 11
    sh = fe.output_shapes(3)
    assert [np.dtype(sh[k][1]) for k in LPVO_KEYS] == [np.dtype(C_DTYPE[t]) for t, _ in fields]
    assert [sh[k][0] for k in LPVO_KEYS] == [(3, 11, 3), (3, 11), (3, 11, 2), (3,)]
    # the existing output structs are unchanged
    assert len(hvo.FrameFrontEnd.FIELDS) == 17 and hvo.FrameFrontEnd.GRID_FIELDS == ['grid_counts', 'grid_items', 'lgrid_counts', 'lgrid_items']
    assert len(hvo.FrameFrontEnd.BOW_FIELDS) == 7


def test_lpvo_entry_points_are_bound_with_the_header_arguments(hvo):
    src = re.sub(r'/\*.*?\*/', '', _header(), flags=re.S)
    for name in NEW_CALLS:
        m = re.search(r'\bint\s+' + name + r'\s*\(([^)]*)\)\s*;', src)
        assert m, name
        params = [p.strip() for p in m.group(1).split(',')]
        want = [hvo._vp if '*' in p else C.c_int for p in params]
        restype, argtypes = hvo.ABI[name]
        assert restype is C.c_int and argtypes == want, name
    # the _lpvo calls take the _grid calls' arguments plus the LPVO outputs
    for kind in ('', '_async', '_device'):
        assert hvo.ABI[f'hvo_frame_extract_batch{kind}_lpvo'][1] == hvo.ABI[f'hvo_frame_extract_batch{kind}_grid'][1] + [hvo._vp]
    assert hvo.ABI['hvo_seq_extract_lpvo'][1] == hvo.ABI['hvo_seq_extract_grid'][1] + [hvo._vp]


def test_lpvo_capacity_of_no_handle_is_zero(hvo):
    assert hvo.lib().hvo_frame_lpvo_capacity(None) == 0 and hvo.lib().hvo_seq_lpvo_capacity(None) == 0


def test_lpvo_flag_is_refused_without_the_normals_stage(hvo):
    """Checked before any handle is created, so no device is needed."""
    for stages in (hvo.STAGE_ORB, hvo.STAGE_ALL & ~hvo.STAGE_NORMALS):
        with pytest.raises(hvo.HvoError) as ei:
            hvo.FrameFrontEnd(640, 480, 535.4, 539.2, 320.1, 247.6, 1 / 5000, stages=stages, lpvo=True)
        assert ei.value.status == hvo.HVO_ERR_ARG
        with pytest.raises(hvo.HvoError) as ei:
            hvo.FrameSequence(640, 480, 535.4, 539.2, 320.1, 247.6, 1 / 5000, [0], stages=stages, lpvo=True)
        assert ei.value.status == hvo.HVO_ERR_ARG


def _capacity(w, h):
    """the header's formula: the lattice u = 10, 25, .. < W - 1 by v = 10, 25, .. < H - 1"""
    assert -(-(w - 11) // 15) * -(-(h - 11) // 15) == len(range(10, w - 1, 15)) * len(range(10, h - 1, 15))
    return -(-(w - 11) // 15) * -(-(h - 11) // 15)


# ---------------------------------------------------------------------------------------------------------------- GPU
def _cam(synth, config='S1'):
    c = synth.CONFIGS[config]
    return c['fx'], c['fy'], c['cx'], c['cy'], np.float32(1.0 / c['factor'])


def _K(synth, config='S1'):
    fx, fy, cx, cy, _ = _cam(synth, config)
    return np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1]], np.float32)


def _oracle(synth, d, config='S1'):
    fx, fy, cx, cy, f = _cam(synth, config)
    return oracle.lpvo_normals(d, f, fx, fy, cx, cy)


def _frames(synth, config='S1', start=70):
    """Three frames of `config`, then an all-zero depth, a hole, and strips at z = 0.2 exactly and z = 8 > 7 (factor 1 / 5000)."""
    g, d = synth.sequence(config, 3, start=start)
    extra = np.repeat(d[:1], 3, axis=0).copy()
    extra[0] = 0
    extra[1, 100:300, 200:400] = 0
    extra[2, :, :320] = 1000
    extra[2, :, 320:] = 40000
    return np.concatenate([g, g[:3]]), np.concatenate([d, extra])


def _fe(hvo, synth, config='S1', **kw):
    c = synth.CONFIGS[config]
    return hvo.FrameFrontEnd(c['w'], c['h'], *_cam(synth, config), bf=c['bf'], nfeatures=c['nfeatures'], **kw)


def _same_rows(got, want):
    """(normals, depth, pix) byte for byte"""
    assert len(got[0]) == len(want[0])
    for a, b in zip(got, want):
        assert a.tobytes() == b.tobytes()


def _same_lpvo(hvo, o, r, n, frames=None):
    for f in range(n):
        g = f if frames is None else frames[f]
        assert int(o['lpvo_counts'][f]) == int(r['lpvo_counts'][g]), f
        _same_rows(hvo.FrameFrontEnd.lpvo(o, f), hvo.FrameFrontEnd.lpvo(r, g))


def _check_same_as_plain(d, p, nframes):
    """Every output of the call without LPVO outputs, byte for byte, in the rows a frame owns."""
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


@pytest.mark.gpu
@pytest.mark.parametrize('config', ['S1', 'S2'])
def test_gpu_frame_lpvo_equals_manhattan_and_oracle(hvo, synth, config):
    gray, depth = _frames(synth, config)
    nf = len(gray)
    plain = _fe(hvo, synth, config, max_batch=nf)
    p = plain.extract_batch(gray, depth)
    launches = plain.last_launches()
    plain.close()
    fe = _fe(hvo, synth, config, max_batch=nf, lpvo=True)
    m = hvo.Manhattan(_K(synth, config), 640, 480, _cam(synth, config)[4], max_batch=nf)
    assert fe.lpvo_capacity == m.capacity == _capacity(640, 480) == 32 * 42
    # the same handle without LPVO outputs: the launches of a handle without lpvo, and the same outputs
    fe.with_lpvo = False
    q = fe.extract_batch(gray, depth)
    assert fe.last_launches() == launches
    _check_same_as_plain(q, p, nf)
    fe.with_lpvo = True
    d = fe.extract_batch(gray, depth)
    assert fe.last_launches() == launches + 3                # k_lpvo_rows, k_lpvo_cols, k_lpvo_normals
    _check_same_as_plain(d, p, nf)
    ref = m.computeNormalsLPVO_batch(depth)
    m.close()
    for f in range(nf):
        got = hvo.FrameFrontEnd.lpvo(d, f)
        _same_rows(got, ref[f])
        _same_rows(got, _oracle(synth, depth[f], config))
    counts = d['lpvo_counts']
    assert min(counts[:3]) > 500 and counts[3] == 0 and 0 < counts[4] < counts[0]
    fe.close()


GOLDEN_REF = os.path.join(ROOT, 'tests', 'golden', 'lpvo_ref.npz')
REF_CASES = [('S1', 0), ('S2', 3), ('S1', 5)]


def _holes(d, k):
    """case k > 0 of a fixture frame: a hole, a strip at the range limits (z = 0.2 exactly; z = 8 > 7)"""
    d = d.copy()
    if k:
        d[100:300, 200:400] = 0
        d[:, :40] = 1000
        d[:, 600:] = 40000
    return d


@pytest.mark.gpu
@pytest.mark.parametrize('config', ['S1', 'S2'])
def test_gpu_frame_lpvo_equals_executed_reference(hvo, synth, config):
    """The fixture cases of the executed Manhattan::computeNormalsLPVO (tests/golden/lpvo_ref.npz) through the frame call."""
    g = np.load(GOLDEN_REF)
    cases = [(idx, k) for cfg, idx in REF_CASES if cfg == config for k in (0, 1)]
    gray = np.stack([synth.frame(config, idx)[0] for idx, _ in cases])
    depth = np.stack([_holes(synth.frame(config, idx)[1], k) for idx, k in cases])
    fe = _fe(hvo, synth, config, max_batch=len(cases), lpvo=True)
    d = fe.extract_batch(gray, depth)
    fe.close()
    for f, (idx, k) in enumerate(cases):
        n, z, _ = hvo.FrameFrontEnd.lpvo(d, f)
        rn, rz = g[f'{config}_{idx}_{k}_n'], g[f'{config}_{idx}_{k}_z']
        assert len(rn) > 300 and n.tobytes() == rn.tobytes() and z.tobytes() == rz.tobytes(), (idx, k)


@pytest.mark.gpu
def test_gpu_frame_lpvo_at_1280x720(hvo, synth):
    """The S3 camera (1280x720: 170 lattice columns): the frame call and hvo.Manhattan, which now accepts that width, equal the oracle."""
    gray, depth = synth.sequence('S3', 2, start=11)
    depth = np.concatenate([depth, depth[:1]])
    depth[2, 200:500, 300:900] = 0
    gray = np.concatenate([gray, gray[:1]])
    fe = _fe(hvo, synth, 'S3', max_batch=3, lpvo=True)
    m = hvo.Manhattan(_K(synth, 'S3'), 1280, 720, _cam(synth, 'S3')[4], max_batch=3)
    assert fe.lpvo_capacity == m.capacity == _capacity(1280, 720) == 48 * 85
    d = fe.extract_batch(gray, depth)
    ref = m.computeNormalsLPVO_batch(depth)
    fe.close(); m.close()
    for f in range(3):
        got = hvo.FrameFrontEnd.lpvo(d, f)
        want = _oracle(synth, depth[f], 'S3')
        _same_rows(got, want)
        _same_rows(ref[f], want)
        assert len(got[0]) > 1000 and got[2][:, 0].max() > 1000   # samples right of the old 730-px limit
    assert d['lpvo_counts'][2] < d['lpvo_counts'][0]


@pytest.mark.gpu
def test_gpu_frame_lpvo_on_the_undistorting_tum1_handle(hvo, synth):
    """LPVO reads the depth image, which undistortion does not touch: the same rows as the plain handle."""
    gray, depth = _frames(synth)
    nf = len(gray)
    a = _fe(hvo, synth, max_batch=nf, lpvo=True)
    b = _fe(hvo, synth, max_batch=nf, lpvo=True, dist=TUM1)
    assert b.undistorts
    _same_lpvo(hvo, b.extract_batch(gray, depth), a.extract_batch(gray, depth), nf)
    a.close(); b.close()


@pytest.mark.gpu
def test_gpu_frame_lpvo_through_every_call_path(hvo, synth):
    """Blocking, two queued wait=False calls, the device-resident call (rows past each count keep a sentinel), several chunks through
    two lanes, two serial chunks of 2048 frames (device-resident), FrameSequence, and LPVO with a vocabulary and grids: the same rows
    as the blocking call."""
    import torch
    g1, d1 = _frames(synth)
    g2, d2 = _frames(synth, 'S2', start=9)
    gray, depth = np.concatenate([g1[:4], g2[:2]]), np.concatenate([d1[:4], d2[:2]])
    nf = len(gray)
    ref = _fe(hvo, synth, max_batch=nf, lanes=1, lpvo=True)
    r = ref.extract_batch(gray, depth)
    ref.close()
    m = hvo.Manhattan(_K(synth), 640, 480, _cam(synth)[4], max_batch=nf)
    for f, want in enumerate(m.computeNormalsLPVO_batch(depth)):
        _same_rows(hvo.FrameFrontEnd.lpvo(r, f), want)
    m.close()

    fe = _fe(hvo, synth, max_batch=4, lanes=2, lpvo=True)
    assert fe.chunk == 2
    _same_lpvo(hvo, fe.extract_batch(gray, depth), r, nf)         # three chunks through two lanes (side by side)
    outs = [fe.alloc_host(nf) for _ in range(2)]
    for o in outs:
        fe.extract_batch(gray, depth, out=o, wait=False)
    fe.sync()
    for o in outs:
        _same_lpvo(hvo, o, r, nf)
    bad = fe.alloc_host(nf)
    bad['lpvo_normals3'] = np.empty((nf, fe.lpvo_capacity - 1, 3), np.float64)
    with pytest.raises(hvo.HvoError):
        fe.extract_batch(gray, depth, out=bad)
    # host call without pix2 (optional on the host)
    part = {k: v for k, v in fe.alloc_host(nf).items() if k != 'lpvo_pix2'}
    ptrs = {k: v.ctypes.data for k, v in part.items()}
    hvo._check(hvo.lib().hvo_frame_extract_batch_lpvo(fe._h, hvo._np_ptr(gray), hvo._np_ptr(depth), nf, C.byref(fe._outputs(ptrs)), None, None,
                                                      fe._lpvo_outputs(ptrs)))
    for f in range(nf):
        c = int(r['lpvo_counts'][f])
        assert int(part['lpvo_counts'][f]) == c
        assert part['lpvo_normals3'][f, :c].tobytes() == r['lpvo_normals3'][f, :c].tobytes()
        assert part['lpvo_depth'][f, :c].tobytes() == r['lpvo_depth'][f, :c].tobytes()
    # device-resident, on torch tensors prefilled with a sentinel: rows at or past each frame's count are not written
    dev = torch.device('cuda', 0)
    shapes = fe.output_shapes(4)
    d = {k: torch.full((int(np.prod(s)) * np.dtype(dt).itemsize,), 0xEF, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
    g, dp = torch.from_numpy(gray[:4].copy()).to(dev), torch.from_numpy(depth[:4].copy()).to(dev)
    torch.cuda.synchronize()
    fe.extract_batch_device(g.data_ptr(), dp.data_ptr(), 4, {k: v.data_ptr() for k, v in d.items()})
    fe.sync()
    raw = {k: d[k].cpu().numpy() for k in LPVO_KEYS}
    o = {k: raw[k].view(shapes[k][1]).reshape(shapes[k][0]) for k in LPVO_KEYS}
    _same_lpvo(hvo, o, r, 4)
    for f in range(4):
        c = int(o['lpvo_counts'][f])
        for k in ('lpvo_normals3', 'lpvo_depth', 'lpvo_pix2'):
            rows = raw[k].reshape(4, fe.lpvo_capacity, -1)
            assert (rows[f, c:] == 0xEF).all(), (k, f)
    fe.close()
    del d

    # 4096 frames device-resident through two lanes: two chunks of 2048, each running its pipelines one after the other, and the LPVO
    # chain in passes of 256 frames
    big = _fe(hvo, synth, max_batch=4096, lanes=2, lpvo=True, membership='u8', normals='n8')
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
    _same_lpvo(hvo, {k: d[k].cpu().numpy().view(shapes[k][1]).reshape(shapes[k][0]) for k in LPVO_KEYS}, r, n, pick)
    big.close()
    del d, g, dp
    torch.cuda.empty_cache()

    # FrameSequence: two handles (the device list names cuda:0 twice), queued calls of two frames
    seq = hvo.FrameSequence(640, 480, *_cam(synth), [0, 0], frames_per_call=2, bf=40.0, line_cull=False, lpvo=True)
    assert set(LPVO_KEYS) <= set(seq.output_shapes(nf, device=False)) and seq.lpvo_capacity == _capacity(640, 480)
    _same_lpvo(hvo, seq.extract(gray, depth), r, nf)
    bad = seq.alloc_host(nf)
    bad['lpvo_counts'] = np.empty(nf, np.int64)
    with pytest.raises(hvo.HvoError):
        seq.extract(gray, depth, out=bad)
    seq.close()

    # LPVO, BoW and grids in one call
    gv = np.load(os.path.join(ROOT, 'tests', 'golden', 'bow_ref.npz'))
    voc = {k[4:]: gv[k] for k in gv.files if k.startswith('voc_')}
    voc['L'] = int(voc['L'])
    fb = _fe(hvo, synth, max_batch=nf, vocabulary=voc, grids=True, lpvo=True)
    o = fb.extract_batch(gray, depth)
    fb.close()
    _same_lpvo(hvo, o, r, nf)
    bt = hvo.ORBVocabulary(voc)
    ref_bow = bt.transform_batch([o['desc'][f, :int(o['kp_counts'][f])] for f in range(nf)], 4)
    bt.close()
    for f in range(nf):
        w = int(o['bow_counts'][f])
        assert np.array_equal(o['bow_words'][f, :w], ref_bow[f][0][0])
        rows = o['kps'][f, :int(o['kp_counts'][f])]
        got = hvo.FrameFrontEnd.grid(o, f)
        want = oracle.grid_build(rows, (0.0, 0.0, 640.0, 480.0))
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


@pytest.mark.gpu
def test_gpu_frame_lpvo_argument_errors(hvo, synth):
    import torch
    gray, depth = _frames(synth)
    gray, depth = gray[:1], depth[:1]
    buf = np.zeros(64, np.float64)   # (refused calls write nothing)
    p = buf.ctypes.data

    def call(fe, lp, out=None):
        out = out if out is not None else fe.alloc_host(1)
        ptrs = {k: v.ctypes.data for k, v in out.items()}
        return hvo.lib().hvo_frame_extract_batch_lpvo(fe._h, hvo._np_ptr(gray), hvo._np_ptr(depth), 1, C.byref(fe._outputs(ptrs)), None, None,
                                                      C.byref(lp))

    fe = _fe(hvo, synth, stages=hvo.STAGE_ALL & ~hvo.STAGE_NORMALS)      # a handle without the normals stage
    assert fe.lpvo_capacity == 0
    assert call(fe, hvo._FrameLpvoOutputs(p, p, p, p)) == hvo.HVO_ERR_ARG
    fe.close()
    fe = _fe(hvo, synth, lpvo=True)
    out = fe.alloc_host(1)
    for missing in range(4):                                             # pix2 (index 2) is optional on the host
        args = [out[k].ctypes.data for k in LPVO_KEYS]
        args[missing] = None
        assert (call(fe, hvo._FrameLpvoOutputs(*args), out) == hvo.HVO_ERR_ARG) == (missing != 2), missing
    # the device call needs every array
    dev = torch.device('cuda', 0)
    shapes = fe.output_shapes(1)
    d = {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
    g, dp = torch.from_numpy(gray.copy()).to(dev), torch.from_numpy(depth.copy()).to(dev)
    dptr = {k: v.data_ptr() for k, v in d.items()}
    st = hvo.lib().hvo_frame_extract_batch_device_lpvo(fe._h, g.data_ptr(), dp.data_ptr(), 1, C.byref(fe._outputs(dptr)), None, None,
                                                       fe._lpvo_outputs(dict(dptr, lpvo_pix2=None)))
    assert st == hvo.HVO_ERR_ARG
    fe.extract_batch_device(g.data_ptr(), dp.data_ptr(), 1, dptr)
    fe.sync()
    fe.close()
