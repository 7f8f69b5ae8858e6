"""Frames above 1280x720: every stage of the frame handle, the sequence and the standalone handles at 1920x1080 (S6), 1920x1200,
1280x1024 and 1024x1024 (S7).  Two per-stage ceilings moved: the plane graph has a 24-word row instantiation of k_plane_cluster /
k_plane_merge for more than 9216 10x10 blocks (up to 24576), and k_line_keylines has a uint32_t index / rank path in global memory
for segment bounds above 65535 or shared-memory lists above 200 KB.

  CPU: S6 / S7 are deterministic and shaped as stated; the LSD oracle equals cv2 at 1920x1080; the plane oracle labels an S6 frame
       validly
  GPU: the same parity bars as at 640x480 (planes and ORB bit for bit, lines as tests/test_lsd.py, normals and LPVO as their tests),
       the kernel paths each size takes (launch timeline), the heap-key tie fallback at 15 id bits, libstdc++'s tie order through
       the uint32_t sort, every frame-handle call path, and the refusal of 2048x1536."""
import os

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL_PX = 1e-3
# image -> (seg_cap, 10x10 blocks) from the formulas of hvo_line_create / hvo_plane_create
LIMITS = {(1920, 1080): (73595, 20736), (1920, 1200): (81782, 23040), (1280, 1024): (49225, 13056), (1024, 1024): (39361, 10404),
          (1280, 720): (34602, 9216)}
# the two sizes without a synthetic config of their own: the S6 camera's shape at other resolutions
EXTRA = {'HD1200': dict(w=1920, h=1200, fx=1380.0, fy=1380.0, cx=959.5, cy=599.5, factor=1000.0, bf=69.0, textured=True, nfeatures=3000),
         'SXGA': dict(w=1280, h=1024, fx=920.0, fy=920.0, cx=639.5, cy=511.5, factor=1000.0, bf=46.0, textured=True, nfeatures=2000)}
HD = ['S6', 'HD1200', 'SXGA', 'S7']
KS_DIST = np.array([0.08, -0.11, 0.0007, -0.0004, 0.05], np.float32)   # a mildly distorted 1080p colour camera (synthetic)


@pytest.fixture
def cfgs(synth, monkeypatch):
    for k, v in EXTRA.items():
        monkeypatch.setitem(synth.CONFIGS, k, v)
    return synth.CONFIGS


def _cam(c):
    return c['fx'], c['fy'], c['cx'], c['cy'], np.float32(1.0 / c['factor'])


def _ocam(c):
    """the oracle's argument order: factor, fx, fy, cx, cy"""
    fx, fy, cx, cy, f = _cam(c)
    return f, fx, fy, cx, cy


def _K(c):
    return np.array([[c['fx'], 0, c['cx']], [0, c['fy'], c['cy']], [0, 0, 1]], np.float32)


def _seg_cap(w, h):
    """hvo_line_create's construction bound on the segments of one frame"""
    sw, sh = int(np.rint(w * 0.8)), int(np.rint(h * 0.8))
    log_nt = 5 * (np.log10(sw) + np.log10(sh)) / 2 + np.log10(11.0)
    return (sw - 1) * (sh - 1) // int(-log_nt / np.log10(22.5 / 180)) + 1


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_synth_hd_configs_are_deterministic_and_shaped(synth):
    assert (synth.CONFIGS['S6']['w'], synth.CONFIGS['S6']['h'], synth.CONFIGS['S6']['factor']) == (1920, 1080, 1000.0)
    assert (synth.CONFIGS['S7']['w'], synth.CONFIGS['S7']['h']) == (1024, 1024) and synth.CONFIGS['S6']['nfeatures'] == 3000
    for cfg, (w, h) in (('S6', (1920, 1080)), ('S7', (1024, 1024))):
        for i in (0, 7):
            g, d = synth.frame(cfg, i)
            g2, d2 = synth.frame(cfg, i)
            assert g.shape == d.shape == (h, w) and g.dtype == np.uint8 and d.dtype == np.uint16
            assert np.array_equal(g, g2) and np.array_equal(d, d2)
            assert 0.002 < (d == 0).mean() < 0.05 and 60 < g.mean() < 180
        assert not np.array_equal(synth.frame(cfg, 0)[0], synth.frame(cfg, 1)[0])


def test_limits_table_follows_the_create_formulas():
    for (w, h), (seg_cap, nb) in LIMITS.items():
        assert _seg_cap(w, h) == seg_cap and (w // 10) * (h // 10) == nb
    assert _seg_cap(2048, 1536) == 111680 and (2048 // 10) * (1536 // 10) == 31212


@pytest.mark.parametrize('cfg,idx', [('S6', 0), ('S6', 5)])
def test_oracle_lsd_equals_cv2_at_1080p(synth, cfg, idx):
    cv2 = pytest.importorskip('cv2')
    cv2.setNumThreads(1)
    g, _ = synth.frame(cfg, idx)
    ref = cv2.createLineSegmentDetector().detect(g)[0].reshape(-1, 4)
    seg = oracle.lsd_detect(g)
    assert seg.shape == ref.shape and np.array_equal(seg, ref) and len(seg) > 200


def test_oracle_plane_labelling_on_s6(synth):
    c = synth.CONFIGS['S6']
    for idx in (0, 4):
        _, d = synth.frame('S6', idx)
        n, planes, mem = oracle.plane_detect(d, *_ocam(c))
        assert 3 <= n <= 8 and mem.shape == (1920 * 1080,)
        assert mem.min() >= -1 and mem.max() < n
        assert all((mem == i).any() for i in range(n))
        assert np.all(np.diff(planes[:, 6]) <= 0) and planes[-1, 6] >= 3000


# ---------------------------------------------------------------------------------------------------------------- GPU
def _fe(hvo, c, **kw):
    return hvo.FrameFrontEnd(c['w'], c['h'], *_cam(c), bf=c['bf'], nfeatures=c['nfeatures'], **kw)


def _names(hvo, run):
    hvo.timeline(True)
    try:
        run()
    finally:
        names = {n for _, _, n in hvo.timeline_dump()}
        hvo.timeline(False)
    return names


@pytest.mark.gpu
@pytest.mark.parametrize('cfg', HD + ['S3'])
def test_gpu_hd_limits_and_kernel_paths(hvo, synth, cfgs, cfg):
    """seg_cap as the table; the 24-word plane kernels run exactly above 9216 blocks, the uint32_t KeyLine sort exactly above 65535
    segments or 200 KB of lists; the frame handle and the standalone handles launch the same ones."""
    c = cfgs[cfg]
    w, h = c['w'], c['h']
    seg_cap, nb = LIMITS[(w, h)]
    g, d = synth.frame(cfg, 2)
    ex = hvo.LINEextractor(1, 1.2, 200, 0.125, width=w, height=h)
    assert ex.segment_capacity == seg_cap
    wide = nb > 9216
    u32 = seg_cap > 65535 or seg_cap * 4 > 200 * 1024
    names = _names(hvo, lambda: ex(g))
    assert ('k_line_keylines<uint32_t>' in names) == u32 and ('k_line_keylines' in names) == (not u32)
    ex.close()
    pd = hvo.PlaneDetection(w, h)
    pd.readDepthImage(d, _K(c), _cam(c)[4])
    names = _names(hvo, lambda: pd.runPlaneDetection())
    assert ('k_plane_cluster<24>' in names) == wide and ('k_plane_merge<24>' in names) == wide
    assert ('k_plane_cluster' in names) == (not wide) and ('k_plane_merge' in names) == (not wide)
    pd.close()
    fe = _fe(hvo, c)
    names = _names(hvo, lambda: fe.extract_batch(g[None], d[None]))
    fe.close()
    assert ('k_plane_cluster<24>' in names) == wide and ('k_line_keylines<uint32_t>' in names) == u32
    assert {'k_fast_strips', 'k_lsd_grow', 'k_plane_flood', 'k_sn_normals'} <= names


@pytest.mark.gpu
@pytest.mark.parametrize('cfg', HD)
def test_gpu_hd_planes_equal_oracle(hvo, synth, cfgs, cfg):
    """PlaneDetection: count, planes7 bit for bit and membership, one frame and a batch of two."""
    c = cfgs[cfg]
    _, depths = synth.sequence(cfg, 2, start=3)
    pd = hvo.PlaneDetection(c['w'], c['h'], max_batch=2)
    assert pd.readDepthImage(depths[0], _K(c), _cam(c)[4])
    n1 = pd.runPlaneDetection()
    n, planes, mem = pd.detect_batch(depths)
    for f in range(2):
        on, op, om = oracle.plane_detect(depths[f], *_ocam(c))
        assert n[f] == on >= 3
        assert planes[f, :on].tobytes() == op.tobytes()
        assert np.array_equal(mem[f], om)
    assert n1 == n[0] and np.array_equal(pd.membership, mem[0])
    pd.close()


def _heap_keys(mse, nb):
    """heap_entry's key part (plane.cu) of every block MSE: 5 exponent bits, 27 - idbits mantissa bits"""
    idbits = int(nb - 1).bit_length()
    mbits = 27 - idbits
    b = np.asarray(mse, np.float64).view(np.int64)
    e = (b >> 52) - (1023 - 24)
    key = (e << mbits) | ((b & 0xfffffffffffff) >> (52 - mbits))
    return idbits, np.where(e < 0, 0, np.where(e >= 32, (1 << (mbits + 5)) - 1, key))


@pytest.mark.gpu
def test_gpu_hd_plane_key_ties_at_15_id_bits(hvo, synth):
    """A large exactly planar wall (one depth value) in front of the S6 room: thousands of blocks share a heap key, so the heap
    orders them by the exact double MSEs (the tie fallback), with 15 id bits and 12 mantissa bits.  The result equals the oracle."""
    c = synth.CONFIGS['S6']
    _, d = synth.frame('S6', 1)
    d = d.copy()
    d[100:1000, 200:1500] = 1800
    blocks = oracle.plane_blocks(d, *_ocam(c))
    queued = blocks[:, 0] == 1
    idbits, keys = _heap_keys(blocks[queued, 8], len(blocks))
    _, counts = np.unique(keys, return_counts=True)
    assert idbits == 15 and counts.max() > 2000
    pd = hvo.PlaneDetection(1920, 1080)
    pd.readDepthImage(d, _K(c), _cam(c)[4])
    n = pd.runPlaneDetection()
    on, op, om = oracle.plane_detect(d, *_ocam(c))
    assert n == on and np.array_equal(pd.membership, om)
    assert np.array_equal(pd.supports, op[:, 6].astype(np.int64)) and pd.normals.tobytes() == op[:, :3].copy().tobytes()
    pd.close()


def _check_lines(kl, desc, lv, okl, odesc, olv):
    """tests/test_lsd.py's bar for LINEextractor::operator()"""
    assert len(kl) == len(okl) and len(kl) > 10
    for name in ('class_id', 'octave', 'numOfPixels'):
        assert np.array_equal(kl[name], okl[name]), name
    for name in ('startPointX', 'startPointY', 'endPointX', 'endPointY', 'sPointInOctaveX', 'sPointInOctaveY', 'ePointInOctaveX',
                 'ePointInOctaveY', 'pt_x', 'pt_y'):
        assert np.abs(kl[name] - okl[name]).max() <= TOL_PX, name
    for name in ('angle', 'response', 'size', 'lineLength'):
        assert np.allclose(kl[name], okl[name], rtol=1e-5, atol=1e-4), name
    same = np.array([kl[i].tobytes() == okl[i].tobytes() for i in range(len(kl))])
    assert same.mean() > 0.9
    assert np.array_equal(desc[same], odesc[same])
    assert np.allclose(lv, olv, rtol=1e-9, atol=1e-9)


@pytest.mark.gpu
@pytest.mark.parametrize('cfg', HD)
def test_gpu_hd_lines_equal_oracle(hvo, synth, cfgs, cfg):
    """Segments, then LINEextractor with and without cullingLine: keylines, LBD and line functions."""
    c = cfgs[cfg]
    g, _ = synth.frame(cfg, 6)
    ex = hvo.LINEextractor(1, 1.2, 200, 0.125, width=c['w'], height=c['h'])
    (seg,) = ex.detect_segments(g)
    ref = oracle.lsd_detect(g)
    assert seg.shape == ref.shape and len(ref) > 200 and np.abs(seg - ref).max() <= TOL_PX
    _check_lines(*ex(g), *oracle.line_extract(g, n_features=200))
    ex.set_culling(True)
    kl, desc, lv = ex(g)
    okl, odesc, olv = oracle.line_extract_culled(g, 200)
    assert len(kl) == len(okl) and 10 < len(kl) < 200
    assert np.array_equal(kl['class_id'], okl['class_id']) and np.array_equal(kl['numOfPixels'], okl['numOfPixels'])
    for name in ('startPointX', 'startPointY', 'endPointX', 'endPointY'):
        assert np.abs(kl[name] - okl[name]).max() <= TOL_PX, name
    same = np.array([kl[i].tobytes() == okl[i].tobytes() for i in range(len(kl))])
    assert same.mean() > 0.9 and np.array_equal(desc[same], odesc[same])
    assert np.allclose(lv, olv, rtol=0, atol=1e-6 * max(1.0, np.abs(olv).max()))
    ex.close()


def _bars(w, h):
    """Dark 15x60 bars on a 40 x 120 px lattice: every segment has one of two lengths, so the response sort is all ties."""
    g = np.full((h, w), 200, np.uint8)
    for y in range(40, h - 100, 120):
        for x in range(40, w - 40, 40):
            g[y:y + 60, x:x + 15] = 40
    return g


@pytest.mark.gpu
@pytest.mark.parametrize('size', [(1920, 1080), (1920, 1200), (1280, 720)])
def test_gpu_hd_keyline_sort_tie_order(hvo, size):
    """Over a thousand equal responses at 1920 px (600 at 1280 px): which 200 lines survive, and their class_ids, follow libstdc++'s
    introsort through the uint32_t kernel (1920x1080, 1920x1200) exactly as through the uint16_t one (1280x720)."""
    w, h = size
    g = _bars(w, h)
    okl, odesc, olv = oracle.line_extract(g, n_features=200)
    allr = oracle.line_extract(g, n_features=100000)[0]['response']
    assert len(allr) > (1000 if w == 1920 else 500) and len(np.unique(allr)) <= 4
    ex = hvo.LINEextractor(1, 1.2, 200, 0.125, width=w, height=h)
    names = _names(hvo, lambda: ex(g))
    assert ('k_line_keylines<uint32_t>' in names) == (w == 1920)
    kl, desc, lv = ex(g)
    assert kl.tobytes() == okl.tobytes() and np.array_equal(desc, odesc) and np.array_equal(lv, olv)
    ex.close()


@pytest.mark.gpu
@pytest.mark.parametrize('cfg', HD)
def test_gpu_hd_orb_equals_oracle(hvo, synth, cfgs, cfg):
    c = cfgs[cfg]
    g, _ = synth.frame(cfg, 8)
    ex = hvo.ORBextractor(c['nfeatures'], 1.2, 8, 20, 7, width=c['w'], height=c['h'])
    kps, desc = ex(g)
    ok, od = oracle.OrbOracle(nfeatures=c['nfeatures']).extract(g)
    assert len(kps) == len(ok) > c['nfeatures'] * 0.9
    assert kps.tobytes() == ok.tobytes() and np.array_equal(desc, od)
    ex.close()


@pytest.mark.gpu
@pytest.mark.parametrize('cfg', HD)
def test_gpu_hd_normals_and_lpvo_equal_oracle(hvo, synth, cfgs, cfg):
    c = cfgs[cfg]
    fx, fy, cx, cy, f = _cam(c)
    _, d = synth.frame(cfg, 9)
    sn = hvo.SurfaceNormals(c['w'], c['h'], fx, fy, cx, cy, f)
    got = sn.compute(d)
    ref, rdist = oracle.surface_normals(d, f, fx, fy, cx, cy, want_dist=True)
    assert np.array_equal(sn.distance_map(), rdist) and got.shape == ref.shape
    assert np.array_equal(got[:, 3:], ref[:, 3:])
    nan_g, nan_r = np.isnan(got[:, 0]), np.isnan(ref[:, 0])
    assert np.array_equal(nan_g, nan_r) and (~nan_r).sum() > 10000
    assert np.all(np.arccos(np.clip(np.sum(got[~nan_r, :3] * ref[~nan_r, :3], axis=1), -1, 1)) < 1e-3)
    sn.close()
    m = hvo.Manhattan(_K(c), c['w'], c['h'], f)
    n, z, pix = m.computeNormalsLPVO(d)
    rn, rz, rpix = oracle.lpvo_normals(d, f, fx, fy, cx, cy)
    assert len(n) == len(rn) > 2000
    assert n.tobytes() == rn.tobytes() and z.tobytes() == rz.tobytes() and np.array_equal(pix, rpix)
    m.close()


def _vocabulary():
    gv = np.load(os.path.join(ROOT, 'tests', 'golden', 'bow_ref.npz'))
    voc = {k[4:]: gv[k] for k in gv.files if k.startswith('voc_')}
    voc['L'] = int(voc['L'])
    return voc


def _standalone(hvo, c, gray, depth, voc):
    """Every frame's outputs from the standalone handles (and the BoW / grid references on them)."""
    w, h = c['w'], c['h']
    fx, fy, cx, cy, f = _cam(c)
    n = len(gray)
    orb = hvo.ORBextractor(c['nfeatures'], 1.2, 8, 20, 7, width=w, height=h)
    ln = hvo.LINEextractor(1, 1.2, 200, 0.125, width=w, height=h)
    pd = hvo.PlaneDetection(w, h, max_batch=n)
    sn = hvo.SurfaceNormals(w, h, fx, fy, cx, cy, f, max_batch=n)
    m = hvo.Manhattan(_K(c), w, h, f, max_batch=n)
    bt = hvo.ORBVocabulary(voc)
    pd.readDepthImage(depth[0], _K(c), f)
    r = dict(orb=[orb(g) for g in gray], lines=[ln(g) for g in gray], planes=pd.detect_batch(depth),
             normals=[sn.compute(d) for d in depth], lpvo=m.computeNormalsLPVO_batch(depth))
    r['bow'] = bt.transform_batch([d for _, d in r['orb']], 4)
    for x in (orb, ln, pd, sn, m, bt):
        x.close()
    return r


def _same_as_standalone(hvo, o, r, n, bounds, frames=None):
    for i in range(n):
        f = i if frames is None else frames[i]
        kps, desc = r['orb'][f]
        k = int(o['kp_counts'][i])
        assert k == len(kps) and o['kps'][i, :k].tobytes() == kps.tobytes() and np.array_equal(o['desc'][i, :k], desc), i
        kl, ld, lv = r['lines'][f]
        nl = int(o['line_counts'][i])
        assert nl == len(kl) and o['keylines'][i, :nl].tobytes() == kl.tobytes()
        assert np.array_equal(o['line_desc'][i, :nl], ld) and np.array_equal(o['linevec3'][i, :nl], lv)
        pn, pl, pm = r['planes']
        npl = int(o['n_planes'][i])
        assert npl == pn[f] and o['planes7'][i, :npl].tobytes() == pl[f, :npl].tobytes()
        if 'membership' in o:
            assert np.array_equal(o['membership'][i], pm[f])
        else:
            assert np.array_equal(o['membership8'][i], np.where(pm[f] < 0, 255, pm[f]).astype(np.uint8))
        assert o['normals8'][i].tobytes() == r['normals'][f].tobytes()
        assert int(o['lpvo_counts'][i]) == len(r['lpvo'][f][0])
        for a, b in zip(hvo.FrameFrontEnd.lpvo(o, i), r['lpvo'][f]):
            assert a.tobytes() == b.tobytes()
        (bw, bv), fv = hvo.FrameFrontEnd.bow(o, i)
        (rw, rv), rfv = r['bow'][f][:2]
        assert np.array_equal(bw, rw) and bv.tobytes() == rv.tobytes() and fv == rfv
        gc, gi = hvo.FrameFrontEnd.grid(o, i)
        want = oracle.grid_build(kps, bounds)
        assert np.array_equal(gc, want[0]) and np.array_equal(gi, want[1])
        lc, li = hvo.FrameFrontEnd.line_grid(o, i)
        want = oracle.line_grid_build(kl, bounds)
        assert np.array_equal(lc, want[0]) and np.array_equal(li, want[1])


@pytest.mark.gpu
@pytest.mark.parametrize('cfg', ['S6', 'S7'])
def test_gpu_hd_frame_handle_equals_standalone(hvo, synth, cfgs, cfg):
    """Blocking, two queued calls, device-resident, chunked over two lanes and FrameSequence: every frame's outputs (with BoW, grids
    and LPVO) equal the standalone handles'."""
    import torch
    c = cfgs[cfg]
    gray, depth = synth.sequence(cfg, 3, start=20)
    nf = len(gray)
    voc = _vocabulary()
    r = _standalone(hvo, c, gray, depth, voc)
    bounds = (0.0, 0.0, float(c['w']), float(c['h']))
    kw = dict(vocabulary=voc, grids=True, lpvo=True)
    fe = _fe(hvo, c, max_batch=nf, lanes=1, **kw)
    _same_as_standalone(hvo, fe.extract_batch(gray, depth), r, nf, bounds)
    outs = [fe.alloc_host(nf) for _ in range(2)]
    for o in outs:
        fe.extract_batch(gray, depth, out=o, wait=False)
    fe.sync()
    for o in outs:
        _same_as_standalone(hvo, o, r, nf, bounds)
    dev = torch.device('cuda', 0)
    shapes = fe.output_shapes(nf)
    d = {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
    g, dp = torch.from_numpy(gray.copy()).to(dev), torch.from_numpy(depth.view(np.int16).copy()).to(dev)
    torch.cuda.synchronize()
    fe.extract_batch_device(g.data_ptr(), dp.data_ptr(), nf, {k: v.data_ptr() for k, v in d.items()})
    fe.sync()
    _same_as_standalone(hvo, {k: d[k].cpu().numpy().view(shapes[k][1]).reshape(shapes[k][0]) for k in shapes}, r, nf, bounds)
    fe.close()
    del d, g, dp
    torch.cuda.empty_cache()
    two = _fe(hvo, c, max_batch=2, lanes=2, membership='u8', **kw)
    assert (two.lanes, two.chunk) == (2, 1)
    _same_as_standalone(hvo, two.extract_batch(gray, depth), r, nf, bounds)   # three chunks through two lanes
    two.close()
    seq = hvo.FrameSequence(c['w'], c['h'], *_cam(c), [0, 0], frames_per_call=2, bf=c['bf'], nfeatures=c['nfeatures'], line_cull=False,
                            membership='u8', normals='n8', **kw)
    _same_as_standalone(hvo, seq.extract(gray, depth), r, nf, bounds)
    seq.close()


@pytest.mark.gpu
def test_gpu_hd_undistorting_s6_handle(hvo, synth):
    """A distorted 1080p camera: kps_un is cv::undistortPoints of the keypoints, kp_uright comes from them, the grid uses the
    undistorted rows and the handle's bounds; every other output equals the pinhole handle's."""
    c = synth.CONFIGS['S6']
    gray, depth = synth.sequence('S6', 2, start=30)
    K = _K(c)
    plain = _fe(hvo, c, max_batch=2)
    p = plain.extract_batch(gray, depth)
    plain.close()
    fe = _fe(hvo, c, max_batch=2, dist=KS_DIST, grids=True)
    assert fe.undistorts
    o = fe.extract_batch(gray, depth)
    bounds = fe.image_bounds()
    assert bounds == hvo.image_bounds(K, KS_DIST, 1920, 1080)
    fe.close()
    for f in range(2):
        n = int(p['kp_counts'][f])
        assert n == int(o['kp_counts'][f]) > 2000
        for k in ('kps', 'desc', 'kp_depth'):
            assert o[k][f, :n].tobytes() == p[k][f, :n].tobytes(), k
        kps = o['kps'][f, :n]
        un = kps.copy()
        try:
            import cv2
            xy = cv2.undistortPoints(np.stack([kps['x'], kps['y']], 1).reshape(-1, 1, 2).astype(np.float32), K, KS_DIST, None, K).reshape(-1, 2)
        except ImportError:
            xy = hvo.undistort_points(np.stack([kps['x'], kps['y']], 1), K, KS_DIST)
        un['x'], un['y'] = xy[:, 0], xy[:, 1]
        assert o['kps_un'][f, :n].tobytes() == un.tobytes()
        assert (np.abs(un['x'] - kps['x']) > 0.5).mean() > 0.5
        ur = hvo.ORBextractor.stereo_uright_from_depth(un, o['kp_depth'][f, :n], c['bf'])
        assert o['kp_uright'][f, :n].tobytes() == np.ascontiguousarray(ur, np.float32).tobytes()
        gc, gi = hvo.FrameFrontEnd.grid(o, f)
        want = oracle.grid_build(un, (bounds[0], bounds[2], bounds[1], bounds[3]))
        assert np.array_equal(gc, want[0]) and np.array_equal(gi, want[1])
        nl, npl = int(p['line_counts'][f]), int(p['n_planes'][f])
        assert o['keylines'][f, :nl].tobytes() == p['keylines'][f, :nl].tobytes()
        assert o['planes7'][f, :npl].tobytes() == p['planes7'][f, :npl].tobytes() and np.array_equal(o['membership'][f], p['membership'][f])


@pytest.mark.gpu
def test_gpu_hd_2048x1536_is_refused(hvo, synth):
    import torch
    c = synth.CONFIGS['S6']
    for make in (lambda: hvo.FrameFrontEnd(2048, 1536, *_cam(c)),
                 lambda: hvo.FrameSequence(2048, 1536, *_cam(c), [0], frames_per_call=2),
                 lambda: hvo.PlaneDetection(2048, 1536).readDepthImage(np.zeros((1536, 2048), np.uint16), _K(c), _cam(c)[4])):
        with pytest.raises(hvo.HvoError) as ei:
            make()
        assert ei.value.status == hvo.HVO_ERR_ARG and 'max 24576' in str(ei.value) and '1920x1200' in str(ei.value)
    # the largest accepted size still creates, and the refusal leaves the device as it found it
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(3):
        with pytest.raises(hvo.HvoError):
            hvo.FrameFrontEnd(2048, 1536, *_cam(c), max_batch=8)
    assert torch.cuda.mem_get_info()[0] >= free0 - (64 << 20)
    fe = hvo.FrameFrontEnd(1920, 1200, *_cam(c))
    fe.close()


@pytest.mark.gpu
def test_gpu_hd_oversized_batch_fails_cleanly(hvo, synth):
    """A max_batch that does not fit the device fails at create with HVO_ERR_CUDA and frees what it had allocated."""
    import torch
    c = synth.CONFIGS['S6']
    free0 = torch.cuda.mem_get_info()[0]
    with pytest.raises(hvo.HvoError) as ei:
        hvo.FrameFrontEnd(1920, 1080, *_cam(c), max_batch=20000, lanes=1)
    assert ei.value.status == hvo.HVO_ERR_CUDA
    assert torch.cuda.mem_get_info()[0] >= free0 - (64 << 20)
    fe = hvo.FrameFrontEnd(1920, 1080, *_cam(c), max_batch=2)
    g, d = synth.sequence('S6', 2)
    assert fe.extract_batch(g, d)['kp_counts'].min() > 0
    fe.close()


@pytest.mark.gpu
def test_gpu_hd_plane_handles_of_different_sizes_side_by_side(hvo, synth):
    """The kernels' shared-memory limit is per function, not per handle: a smaller handle created after a larger one must not make the
    larger one's launches fail.  1920x1080, then 1024x1024 (both on the 24-word kernels), then 640x480; every handle still runs."""
    sizes = [('S6', 4), ('S7', 4), ('S1', 0)]
    handles = []
    for cfg, idx in sizes:
        c = synth.CONFIGS[cfg]
        pd = hvo.PlaneDetection(c['w'], c['h'])
        _, d = synth.frame(cfg, idx)
        assert pd.readDepthImage(d, _K(c), _cam(c)[4])
        handles.append((pd, d, c))
    for pd, d, c in handles:
        n = pd.runPlaneDetection()
        on, op, om = oracle.plane_detect(d, *_ocam(c))
        assert n == on and np.array_equal(pd.membership, om)
        pd.close()


@pytest.mark.gpu
def test_gpu_hd_planes_at_the_block_limit(hvo, synth, monkeypatch):
    """2560x960 is exactly 24576 blocks (2.46 M pixels): the 24-word kernels take it and equal the oracle, standalone and inside a frame
    handle; 2570x960 (24672 blocks) is refused."""
    c = dict(w=2560, h=960, fx=1380.0, fy=1380.0, cx=1279.5, cy=479.5, factor=1000.0, bf=69.0, textured=True, nfeatures=3000)
    monkeypatch.setitem(synth.CONFIGS, 'W2560', c)
    gray, depth = synth.sequence('W2560', 1, start=2)
    pd = hvo.PlaneDetection(2560, 960)
    assert pd.readDepthImage(depth[0], _K(c), _cam(c)[4])
    names = _names(hvo, lambda: pd.runPlaneDetection())
    assert 'k_plane_cluster<24>' in names and 'k_plane_merge<24>' in names
    on, op, om = oracle.plane_detect(depth[0], *_ocam(c))
    assert pd.plane_num_ == on >= 3 and np.array_equal(pd.membership, om)
    assert np.array_equal(pd.supports, op[:, 6].astype(np.int64)) and pd.normals.tobytes() == op[:, :3].copy().tobytes()
    pd.close()
    fe = _fe(hvo, c)
    o = fe.extract_batch(gray, depth)
    fe.close()
    assert int(o['n_planes'][0]) == on and o['planes7'][0, :on].tobytes() == op.tobytes() and np.array_equal(o['membership'][0], om)
    assert int(o['kp_counts'][0]) > 2000 and int(o['line_counts'][0]) == 200
    with pytest.raises(hvo.HvoError) as ei:
        hvo.PlaneDetection(2570, 960).readDepthImage(np.zeros((960, 2570), np.uint16), _K(c), _cam(c)[4])
    assert ei.value.status == hvo.HVO_ERR_ARG and 'max 24576' in str(ei.value)
