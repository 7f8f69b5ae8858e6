"""Surface normals (csrc/normals.cu, the pcl::IntegralImageNormalEstimation block of Frame::ComputePlanes) against an
independent statement of PCL's AVERAGE_3D_GRADIENT path in numpy, written from the published algorithm
(integral_image_normal.hpp / integral_image2D.hpp), not from oracle/normals_oracle.cpp.

The reference does in float32 what PCL does in float, one IEEE operation at a time (back-projection, central differences,
depth-change mask, both chamfer passes, the flip test), and in float64 what PCL does in double: the window sums (taken
directly over the float32 differences, no summed-area table), the cross product and the normalisation.

Bar for the CUDA kernels: distance map identical, positions and pixels bit for bit, NaN pattern identical, normals within
1e-6 rad, at shapes that reach every tail of k_sn_rowscan (cw % 32) and of the unrolled chamfer scan (cw % 4), at the
non-default parameters, at batches that fill, overfill and partly fill the 8-frame chamfer blocks, and through the
device-pointer and frame-handle call paths.
"""
import functools

import numpy as np
import pytest

import oracle

F32 = np.float32
ONE = F32(1.0)
TOL = 1e-6                      # rad
DEPTH_FACTOR = 1.0 / 5000.0     # 16-bit depth in units of 0.2 mm


# ---- the reference ---------------------------------------------------------------------------------------------------

def _scan(x, diag_row):
    """One row of a chamfer pass, in place, in the order the pass visits it (x[0] first, not updated): every later element
    becomes min(x[c], diag_row[c - 1], x[c - 1] + 1) with every addition rounded to float32.  Jacobi sweeps of the whole row
    converge to the serial scan: x[c] depends on x[0..c] only, so the fixed point is unique."""
    x[1:] = np.minimum(x[1:], diag_row)
    while True:
        y = np.minimum(x[1:], x[:-1] + ONE)
        if np.array_equal(y, x[1:]):
            return
        x[1:] = y


def _chamfer(dist, diag):
    """PCL's two-pass 3-4 chamfer distance with float costs 1.0 / diag.  The passes read the flat buffer: the upper-right
    neighbour of the last column is the current row's first element, the lower-left neighbour of column 0 the current
    row's last element."""
    d = dist.copy()
    ch, cw = d.shape
    dg = F32(diag)
    for r in range(1, ch):                                   # forward: c = 1 .. cw-1, left to right
        prev, cur = d[r - 1], d[r]
        up_right = np.append(prev[2:], cur[0])
        taps = np.minimum(np.minimum(prev[:-1] + dg, prev[1:] + ONE), up_right + dg)
        _scan(cur, taps)
    for r in range(ch - 2, -1, -1):                          # backward: c = cw-2 .. 0, right to left
        nxt, cur = d[r + 1], d[r]
        low_left = np.append(cur[-1], nxt[:-2])
        taps = np.minimum(np.minimum(low_left + dg, nxt[:-1] + ONE), nxt[1:] + dg)
        _scan(cur[::-1], taps[::-1])
    return d


def reference(depth16, factor, fx, fy, cx, cy, max_depth_change=0.05, smoothing=10.0, shift=0, rw_delta=0, diag=1.4, border_delta=0,
              flip_away=False):
    """Frame::ComputePlanes' normals: cloud of every 3rd pixel (depth 0 -> the point (0,0,0)), IntegralImageNormalEstimation
    (AVERAGE_3D_GRADIENT, BORDER_POLICY_IGNORE, no depth-dependent smoothing, viewpoint at the origin), kept at odd (row, col)
    of the cloud.  Returns dict(out [n,8] float64 = normal, position, pixel; dist [ch,cw] float32; gx, gy [n,3] window sums).
    shift / rw_delta / diag / border_delta / flip_away give the mutants of the sensitivity test."""
    d = np.asarray(depth16, np.uint16)
    z = d[::3, ::3].astype(F32) * F32(factor)
    ch, cw = z.shape
    u = (np.arange(cw) * 3).astype(F32)
    v = (np.arange(ch) * 3).astype(F32)
    P = np.stack([(u[None, :] - F32(cx)) * z / F32(fx), (v[:, None] - F32(cy)) * z / F32(fy), z], -1)
    assert P.dtype == F32
    # central differences of interior points; the border keeps 0
    dx = np.zeros((ch, cw, 3), F32)
    dy = np.zeros((ch, cw, 3), F32)
    dx[1:-1, 1:-1] = P[1:-1, 2:] - P[1:-1, :-2]
    dy[1:-1, 1:-1] = P[2:, 1:-1] - P[:-2, 1:-1]
    dx, dy = dx.astype(np.float64), dy.astype(np.float64)
    # depth-change mask: a jump to the right / lower neighbour zeroes both points; the last row and column are not visited
    th = F32(max_depth_change) * (np.abs(z) + ONE) * F32(2.0)
    jr = np.abs(z[:-1, :-1] - z[:-1, 1:]) > th[:-1, :-1]
    jd = np.abs(z[:-1, :-1] - z[1:, :-1]) > th[:-1, :-1]
    edge = np.zeros((ch, cw), bool)
    edge[:-1, :-1] |= jr | jd
    edge[:-1, 1:] |= jr
    edge[1:, :-1] |= jd
    dist = _chamfer(np.where(edge, F32(0), F32(cw + ch)).astype(F32), diag)
    # kept points
    oh, ow = ch // 2, cw // 2
    m, n = (a.ravel() for a in np.mgrid[1:2 * oh:2, 1:2 * ow:2])
    out = np.full((len(m), 8), np.nan)
    out[:, 3:6] = P[m, n]
    out[:, 6], out[:, 7] = n * 3, m * 3
    gx, gy = np.full((len(m), 3), np.nan), np.full((len(m), 3), np.nan)
    border = int(smoothing) + border_delta
    s = np.minimum(dist[m, n], F32(smoothing))
    ok = (m >= border) & (m < ch - border) & (n >= border) & (n < cw - border) & (s > 2)
    rw = s.astype(np.int64) + rw_delta                         # setRectSize(int(smoothing)); s > 0, so truncation
    for w in np.unique(rw[ok]):
        idx = np.flatnonzero(ok & (rw == w))
        vx = np.lib.stride_tricks.sliding_window_view(dx, (w, w), axis=(0, 1))   # [top, left, xyz, w, w]
        vy = np.lib.stride_tricks.sliding_window_view(dy, (w, w), axis=(0, 1))
        for part in np.array_split(idx, -(-len(idx) // 4096)):
            sy, sx = m[part] - w // 2, n[part] - w // 2 + shift
            gx[part] = vx[sy, sx].sum(axis=(-2, -1))
            gy[part] = vy[sy, sx].sum(axis=(-2, -1))
    nv = np.cross(gy, gx)
    len2 = np.sum(nv * nv, axis=1)
    good = ok & (len2 != 0)
    nv = nv[good] / np.sqrt(len2[good])[:, None]
    # flipNormalTowardsViewpoint on the float normal: (vp - p) . n in float32, flip when < 0
    n32, p32 = nv.astype(F32), P[m[good], n[good]]
    cos_theta = (F32(0) - p32[:, 0]) * n32[:, 0] + (F32(0) - p32[:, 1]) * n32[:, 1] + (F32(0) - p32[:, 2]) * n32[:, 2]
    flip = cos_theta > 0 if flip_away else cos_theta < 0
    out[good, :3] = np.where(flip[:, None], -nv, nv)
    return dict(out=out, dist=dist, gx=gx, gy=gy)


def angles(a, b):
    """Angle in rad between the rows of a and b (float64, atan2: accurate near 0)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.arctan2(np.linalg.norm(np.cross(a, b), axis=1), np.sum(a * b, axis=1))


def mismatches(got, got_dist, ref, tol=TOL):
    """What separates a result (normals8 rows + distance map) from the reference; empty when it is within the bar."""
    bad = []
    out = ref['out']
    if got_dist is not None and not np.array_equal(got_dist, ref['dist']):
        bad.append(f'distance map: {int(np.sum(got_dist != ref["dist"]))} of {got_dist.size} differ')
    if got.shape != out.shape:
        return bad + [f'shape {got.shape} != {out.shape}']
    if not np.array_equal(got[:, 3:], out[:, 3:].astype(F32)):
        bad.append('positions / pixels differ')
    nan_g, nan_r = np.isnan(got[:, :3]).any(1), np.isnan(out[:, 0])
    if not np.array_equal(nan_g, nan_r):
        bad.append(f'NaN pattern: {int(np.sum(nan_g != nan_r))} rows differ')
    both = ~nan_g & ~nan_r
    if both.any():
        worst = angles(got[both, :3], out[both, :3]).max()
        if not worst <= tol:
            bad.append(f'normals: max angle {worst:.3g} rad > {tol:g}')
    return bad


# ---- scenes ----------------------------------------------------------------------------------------------------------

def _camera(W, H, fy_sign=1.0):
    f = 0.83 * W
    return dict(factor=F32(DEPTH_FACTOR), fx=f, fy=fy_sign * f, cx=W / 2 - 0.3, cy=H / 2 + 0.2)


def _rays(W, H, cam):
    u, v = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    return (u - cam['cx']) / cam['fx'], (v - cam['cy']) / cam['fy']


def _quantise(zm):
    return np.clip(np.floor(zm / DEPTH_FACTOR + 0.5), 0, 65535).astype(np.uint16)


def _curved(W, H, seed, fy_sign=1.0):
    """Smooth curved surface (sinusoid + quadratic in depth), an occluding box in front of it (depth steps), clustered holes
    (depth 0) and a saturated patch (65535)."""
    cam = _camera(W, H, fy_sign)
    r = np.random.RandomState(seed)
    X, Y = _rays(W, H, cam)
    ph = r.uniform(0, 2 * np.pi, 2)
    z = 2.5 + 0.3 * np.sin(7 * X + ph[0]) * np.cos(5 * Y + ph[1]) + 0.2 * X ** 2
    bx, by = r.randint(0, W // 2), r.randint(0, H // 2)
    z[by:by + H // 3, bx:bx + W // 3] -= 0.8
    raw = _quantise(z)
    yy, xx = np.mgrid[0:H, 0:W]
    for _ in range(4):
        hx, hy, rad = r.randint(0, W), r.randint(0, H), r.randint(2, max(3, W // 40))
        raw[(xx - hx) ** 2 + (yy - hy) ** 2 <= rad * rad] = 0
    sx, sy = r.randint(0, W - W // 6), r.randint(0, H - H // 6)
    raw[sy:sy + H // 6, sx:sx + W // 6] = 65535
    return raw, cam


def _wall(W, H, z=2.0):
    return np.full((H, W), _quantise(np.float64(z)), np.uint16), _camera(W, H)


def _step(W, H, c0, z1=1.0, z2=2.0):
    """Depth z1 left of cloud column c0 (pixels < 3*c0 - 1), z2 from there on."""
    d = np.full((H, W), _quantise(np.float64(z1)), np.uint16)
    d[:, 3 * c0 - 1:] = _quantise(np.float64(z2))
    return d, _camera(W, H)


def _tilted(W, H, theta=0.5, z0=2.0):
    """Plane through (0, 0, z0) rotated about the camera's y axis by theta: Z = z0 / (1 - X/Z * tan(theta))."""
    cam = _camera(W, H)
    X, _ = _rays(W, H, cam)
    zm = z0 / (1.0 - X * np.tan(theta))
    return _quantise(zm), cam, np.array([-np.sin(theta), 0.0, np.cos(theta)]), zm


def _synth_frame(cfg, idx):
    from hvo_b200 import synth
    c = synth.CONFIGS[cfg]
    return synth.frame(cfg, idx)[1], dict(factor=F32(1.0 / c['factor']), fx=c['fx'], fy=c['fy'], cx=c['cx'], cy=c['cy'])


@functools.lru_cache(maxsize=None)
def scene(kind, W=None, H=None, seed=0):
    if kind in ('S1', 'S2', 'S3'):
        return _synth_frame(kind, seed)
    if kind == 'curved':
        return _curved(W, H, seed)
    if kind == 'curved_neg_fy':
        return _curved(W, H, seed, fy_sign=-1.0)
    if kind == 'wall':
        return _wall(W, H)
    if kind == 'zeros':
        return np.zeros((H, W), np.uint16), _camera(W, H)
    if kind == 'step':
        return _step(W, H, c0=-(-W // 3) // 2 + 1)
    if kind == 'tilted':
        return _tilted(W, H)[:2]
    raise KeyError(kind)


@functools.lru_cache(maxsize=None)
def ref_case(sc, params=(), **mutant):
    d, cam = scene(*sc)
    return reference(d, **cam, **dict(params), **mutant)


# scene key, (parameter overrides).  Widths give cw = ceil(W/3) = 22, 31, 32, 33, 64, 65, 214, 214, 427, 534, 640, 2421: every
# cw % 4 and both sides of every multiple of 32 up to 65; heights are not multiples of 3 or 6, down to the 64-px minimum.
SHAPE_CASES = [
    (('curved', 64, 64, 1), (('smoothing', 3.0),)),
    (('curved', 91, 65, 2), (('smoothing', 3.0),)),
    (('curved', 94, 67, 3), (('smoothing', 4.5),)),
    (('curved', 97, 100, 4), (('smoothing', 6.5),)),
    (('curved', 190, 71, 5), ()),
    (('curved', 193, 203, 6), (('max_depth_change', 0.01),)),
    (('curved', 640, 481, 7), ()),
    (('curved_neg_fy', 641, 479, 8), ()),
    (('curved', 1280, 722, 9), (('smoothing', 20.0),)),
    (('curved', 1600, 640, 10), ()),
    (('curved', 1920, 1080, 11), ()),
    (('curved', 7263, 64, 12), (('smoothing', 3.0),)),       # the widest image the chamfer block fits (96 * 2421 B of 227 KB)
]
PARAM_CASES = [
    (('S1', None, None, 0), ()),
    (('S2', None, None, 3), ()),                              # fy < 0
    (('S3', None, None, 1), ()),
    (('S1', None, None, 0), (('smoothing', 6.5),)),
    (('S1', None, None, 0), (('smoothing', 3.0),)),
    (('S1', None, None, 0), (('smoothing', 2.0),)),           # min(dist, 2) > 2 never holds: all NaN
    (('S1', None, None, 0), (('smoothing', 20.0), ('max_depth_change', 0.01))),
    (('S2', None, None, 3), (('max_depth_change', 0.0),)),
    (('S1', None, None, 0), (('max_depth_change', 1.0),)),
    (('curved', 640, 481, 7), (('smoothing', 2.5), ('max_depth_change', 0.0))),
    (('wall', 190, 71, 0), ()),
    (('wall', 190, 71, 0), (('max_depth_change', 0.0),)),     # no depth change at all: a zero factor masks nothing
    (('step', 193, 203, 0), ()),
    (('zeros', 97, 100, 0), ()),
    (('tilted', 640, 480, 0), ()),
]
CASES = SHAPE_CASES + PARAM_CASES


def _case_id(case):
    (kind, W, H, seed), params = case
    s = kind + (f'-{W}x{H}' if W else '') + f'-{seed}'
    return s + ''.join(f'-{k}{v:g}' for k, v in params)


CASE_IDS = [_case_id(c) for c in CASES]


# ---- CPU: the reference against the oracle, closed forms, sensitivity ------------------------------------------------

@pytest.mark.parametrize('case', CASES, ids=CASE_IDS)
def test_reference_equals_oracle(case):
    """First independent check of oracle/normals_oracle.cpp: identical distance map and NaN pattern, normals within 1e-6 rad."""
    sc, params = case
    d, cam = scene(*sc)
    ref = ref_case(sc, params)
    got, dist = oracle.surface_normals(d, **cam, want_dist=True, **dict(params))
    assert mismatches(got, dist, ref) == []
    p = dict(params)
    all_nan = p.get('smoothing', 10.0) <= 2.0 or sc[0] == 'zeros' or (sc[0] == 'S2' and p.get('max_depth_change') == 0.0)
    assert np.isnan(ref['out'][:, 0]).all() if all_nan else np.isfinite(ref['out'][:, 0]).any()


def test_fronto_parallel_wall_is_exactly_minus_z():
    """Constant depth: dz = 0, dx.y = 0 and dy.x = 0 hold exactly, so every finite normal is exactly (0, 0, -1)."""
    ref = ref_case(('wall', 190, 71, 0))
    n = ref['out'][np.isfinite(ref['out'][:, 0]), :3]
    assert len(n) > 40 and np.array_equal(n, np.tile([0.0, 0.0, -1.0], (len(n), 1)))
    assert np.array_equal(ref['dist'], np.full_like(ref['dist'], 64 + 24))    # no depth change: cw + ch everywhere


def test_depth_step_distance_is_the_closed_form_chamfer_distance():
    """A step between cloud columns c0-1 and c0: the mask zeroes both columns in every row but the last (the mask loop does
    not visit it).  Rows 1 .. ch-2 hold the column distance k to the nearer zero column, an integer and exact in float.  The
    passes leave the edge rows their own closed forms: the forward pass skips row 0, so right of the step row 0 is one
    diagonal plus straight steps (k + 0.4); the backward pass skips the last row, so there the left side is j diagonal steps
    (1.4 j) and the right side k + 0.4; the top-right and bottom-left corners are visited by neither pass and keep cw + ch."""
    W, H = 193, 203
    d, cam = scene('step', W, H, 0)
    dist = reference(d, **cam)['dist']
    ch, cw = dist.shape
    c0 = -(-W // 3) // 2 + 1
    c = np.arange(cw)
    k = np.minimum(np.abs(c - (c0 - 1)), np.abs(c - c0)).astype(np.float64)
    exp = np.tile(k, (ch, 1))
    exp[0, c > c0] = k[c > c0] + 0.4
    exp[-1] = np.where(c < c0 - 1, 1.4 * k, np.where(c > c0, k + 0.4, 1.0))
    exp[0, -1] = exp[-1, 0] = cw + ch
    assert np.array_equal(dist[1:-1], exp[1:-1])
    assert np.allclose(dist[[0, -1]], exp[[0, -1]], rtol=0, atol=1e-4)     # float rounding of the running sums of 1.0 and 1.4
    assert np.array_equal(oracle.surface_normals(d, **cam, want_dist=True)[1], dist)


def test_all_zero_depth_gives_all_nan():
    ref = ref_case(('zeros', 97, 100, 0))
    assert np.isnan(ref['out'][:, :3]).all()
    assert np.array_equal(ref['out'][:, 3:6], np.zeros((len(ref['out']), 3)))     # depth 0 is the point (0, 0, 0)


def test_tilted_plane_within_the_quantisation_bound():
    """A plane Z = z0 + X tan(theta), depth quantised to 0.2 mm.  The window sums telescope: per window row, gx is
    P[e] + P[e-1] - P[s] - P[s-1], so the quantisation enters gx (and gy) through 4 rw points, each off by ray * dZ with
    |dZ| <= 0.1 mm.  |delta gx| <= eps_x = 4 rw |ray|max 1e-4 m, and the normal gy x gx turns by at most
    asin((eps_x / |gx| + eps_y / |gy| + their product) / sin(gx, gy)), which the test doubles for the neglected float32 rounding."""
    W, H = 640, 480
    d, cam, n_true, _ = _tilted(W, H)
    ref = reference(d, **cam)
    ok = np.isfinite(ref['out'][:, 0])
    assert ok.mean() > 0.75
    gx, gy = ref['gx'][ok], ref['gy'][ok]
    X, Y = _rays(W, H, cam)
    ray_max = np.sqrt(X ** 2 + Y ** 2 + 1).max()
    rw = np.minimum(ref['dist'].max(), 10.0)
    eps = 4 * rw * ray_max * 0.5 * DEPTH_FACTOR
    ex, ey = eps / np.linalg.norm(gx, axis=1), eps / np.linalg.norm(gy, axis=1)
    sin_xy = np.linalg.norm(np.cross(gx, gy), axis=1) / np.linalg.norm(gx, axis=1) / np.linalg.norm(gy, axis=1)
    bound = 2 * np.arcsin(np.minimum(1.0, (ex + ey + ex * ey) / sin_xy))
    err = angles(ref['out'][ok, :3], np.tile(-n_true, (int(ok.sum()), 1)))      # the plane faces the camera: -n_true
    assert np.all(err <= bound), (err.max(), bound.min())
    assert bound.max() < 2e-2 and err.max() > 1e-5       # the bound is tight enough to mean something, and the test is not vacuous


SENSITIVITY_SCENES = [(('S1', None, None, 0), ()), (('curved', 640, 481, 7), ())]
MUTANTS = {'window one column right': dict(shift=1), 'window rw - 1': dict(rw_delta=-1), 'chamfer diagonal 1.5': dict(diag=1.5),
           'border one less': dict(border_delta=-1), 'flip inverted': dict(flip_away=True)}


@pytest.mark.parametrize('name', list(MUTANTS))
def test_sensitivity_mutants_break_the_gpu_bar(name):
    """Each slightly wrong statement of the algorithm fails the bar the GPU tests apply, on every scene here: the scenes and
    the tolerance can tell a subtly wrong kernel from a right one."""
    for sc, params in SENSITIVITY_SCENES:
        ref = ref_case(sc, params)
        mut = ref_case(sc, params, **MUTANTS[name])
        assert mismatches(mut['out'].astype(F32), mut['dist'], ref) != [], (name, sc)


def test_create_refuses_a_batch_the_grid_cannot_hold(hvo):
    """The frame index is a grid y / z coordinate (<= 65535): such a handle could never run its full batch.  No device needed."""
    with pytest.raises(hvo.HvoError) as e:
        hvo.SurfaceNormals(64, 64, 50.0, 50.0, 32.0, 32.0, DEPTH_FACTOR, max_batch=65536)
    assert e.value.status == hvo.HVO_ERR_ARG and 'max_batch' in str(e.value)


# ---- GPU: the CUDA kernels against the reference ---------------------------------------------------------------------

def _normals(hvo, W, H, cam, params=(), max_batch=1):
    return hvo.SurfaceNormals(W, H, cam['fx'], cam['fy'], cam['cx'], cam['cy'], cam['factor'], max_batch=max_batch, **dict(params))


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES, ids=CASE_IDS)
def test_gpu_normals_equal_reference(hvo, case):
    sc, params = case
    d, cam = scene(*sc)
    H, W = d.shape
    sn = _normals(hvo, W, H, cam, params)
    try:
        got = sn.compute(d)
        assert mismatches(got, sn.distance_map(), ref_case(sc, params)) == []
        # the summed-area tables add the same float differences in another order than PCL's recurrence: record whether
        # that changes a bit of the result against the oracle (it does not on these scenes)
        assert got.tobytes() == oracle.surface_normals(d, **cam, **dict(params)).tobytes()
    finally:
        sn.close()


def _batch_frames(n, W=193, H=203):
    return np.stack([scene('curved', W, H, 100 + i)[0] for i in range(n)]), _camera(W, H)


@pytest.mark.gpu
def test_gpu_batches_equal_single_frames(hvo):
    """nf in {1, 7, 8, 9, 17}: one chamfer block partly filled, exactly filled, a second block with one live warp, three
    blocks.  Every frame of a batch equals its single-frame result byte for byte (NaN included), the single-frame results
    equal the reference, and a full batch followed by shorter ones on the same handle leaves nothing behind."""
    depths, cam = _batch_frames(17)
    H, W = depths.shape[1:]
    sn = _normals(hvo, W, H, cam, max_batch=17)
    try:
        refs = [reference(depths[f], **cam) for f in range(17)]
        single = []
        for f in range(17):
            single.append(sn.compute(depths[f]))
            assert mismatches(single[-1], sn.distance_map(), refs[f]) == [], f
        for nf in (17, 9, 8, 7, 1):
            got = sn.compute(depths[:nf])
            assert got.shape == (nf, sn.count, 8)
            for f in range(nf):
                assert got[f].tobytes() == single[f].tobytes(), (nf, f)
                assert np.array_equal(sn.distance_map(f), refs[f]['dist']), (nf, f)
        with pytest.raises(hvo.HvoError):
            sn.compute(np.concatenate([depths, depths[:1]]))          # 18 > max_batch
    finally:
        sn.close()


@pytest.mark.gpu
def test_gpu_compute_device_equals_compute(hvo):
    """hvo_normals_compute_batch_device on torch tensors returns the bytes the host call returns."""
    import torch
    depths = np.stack([scene('curved', 641, 479, s)[0] for s in (21, 22, 23)])
    cam = _camera(641, 479)
    sn = _normals(hvo, 641, 479, cam, max_batch=3)
    try:
        host = sn.compute(depths)
        d_depth = torch.from_numpy(depths.view(np.int16)).cuda()          # the same bytes
        d_out = torch.full((3, sn.count, 8), -7.0, dtype=torch.float32, device='cuda')
        torch.cuda.synchronize()
        sn.compute_device(d_depth.data_ptr(), 3, d_out.data_ptr())
        sn.sync()
        assert d_out.cpu().numpy().tobytes() == host.tobytes()
        assert np.array_equal(sn.distance_map(2), reference(depths[2], **cam)['dist'])
    finally:
        sn.close()


@pytest.mark.gpu
def test_gpu_frame_handle_normals_at_1600x640(hvo):
    """A frame handle with the normals stage at 1600 x 640 (over 48 KB of chamfer shared memory): normals8, and normals3
    through normals3_expand, equal the standalone result, which equals the reference."""
    depths = np.stack([scene('curved', 1600, 640, s)[0] for s in (10, 31)])
    cam = _camera(1600, 640)
    gray = np.zeros(depths.shape, np.uint8)
    sn = _normals(hvo, 1600, 640, cam, max_batch=2)
    try:
        alone = sn.compute(depths)
    finally:
        sn.close()
    assert mismatches(alone[0], None, ref_case(('curved', 1600, 640, 10))) == []
    args = (1600, 640, cam['fx'], cam['fy'], cam['cx'], cam['cy'], cam['factor'])
    fe = hvo.FrameFrontEnd(*args, stages=hvo.STAGE_NORMALS, max_batch=2)
    try:
        out = fe.extract_batch(gray, depths)
        assert out['normals8'].tobytes() == alone.tobytes()
    finally:
        fe.close()
    fe = hvo.FrameFrontEnd(*args, stages=hvo.STAGE_NORMALS, max_batch=2, normals='n3')
    try:
        out = fe.extract_batch(gray, depths)
        for f in range(2):
            assert fe.normals3_expand(out['normals3'][f], depths[f]).tobytes() == alone[f].tobytes()
    finally:
        fe.close()


@pytest.mark.gpu
def test_gpu_create_refuses_widths_the_chamfer_block_cannot_hold(hvo):
    """96 * ceil(W/3) bytes of shared memory per chamfer block: 7263 fits the B200's 227 KB opt-in limit, 7264 does not."""
    cam = _camera(7264, 64)
    with pytest.raises(hvo.HvoError) as e:
        _normals(hvo, 7264, 64, cam)
    assert e.value.status == hvo.HVO_ERR_ARG and 'width 7264' in str(e.value) and 'width <= 7263' in str(e.value)
    _normals(hvo, 7263, 64, cam).close()
