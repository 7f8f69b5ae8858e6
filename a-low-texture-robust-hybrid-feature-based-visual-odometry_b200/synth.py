"""Synthetic RGB-D inputs shaped like the reference's datasets (SURVEY.md section 8d).  numpy only.

S1  TUM-fr3-shaped, textured 640x480 (TUM3.yaml intrinsics, depth factor 5000)
S2  ICL-NUIM-shaped, low texture 640x480 (ICL.yaml intrinsics, fy < 0)
S3  RealSense-shaped 1280x720, 2000 ORB
S6  1080p-colour-shaped 1920x1080 (depth aligned to a 1080p colour stream), 3000 ORB
S7  wide-FOV-depth-shaped 1024x1024 (Azure-Kinect-class WFOV depth mode), 2000 ORB
S4  matching stress descriptors (2000 x 50 000 ORB, 200 x 5 000 LBD)

Every frame is a ray-cast box room (floor, ceiling, two side walls, back wall) seen from a camera on a
smooth path; frame i of a sequence uses seed 1000+i for its pixel noise and (clustered) depth holes, so the same
(config, index) always yields the same bytes on every machine.
"""
import numpy as np

CONFIGS = {
    'S1': dict(w=640, h=480, fx=535.4, fy=539.2, cx=320.1, cy=247.6, factor=5000.0, bf=40.0, textured=True, nfeatures=1000),
    'S2': dict(w=640, h=480, fx=481.2, fy=-480.0, cx=319.5, cy=239.5, factor=5000.0, bf=40.0, textured=False, nfeatures=1000),
    'S3': dict(w=1280, h=720, fx=910.0, fy=910.0, cx=640.0, cy=360.0, factor=1000.0, bf=45.0, textured=True, nfeatures=2000),
    'S6': dict(w=1920, h=1080, fx=1380.0, fy=1380.0, cx=959.5, cy=539.5, factor=1000.0, bf=69.0, textured=True, nfeatures=3000),
    'S7': dict(w=1024, h=1024, fx=504.0, fy=504.0, cx=511.5, cy=511.5, factor=1000.0, bf=25.2, textured=True, nfeatures=2000),
}

_ROOM = dict(x=(-2.6, 2.6), y=(-1.4, 1.4), z=4.5)  # metres; camera near the origin looking down +z
_TEX = 1024


def _wall_textures(textured, seed=7):
    """One 1024x1024 albedo map per wall (5 walls)."""
    r = np.random.RandomState(seed)
    tex = []
    for wall in range(5):
        base = r.randint(90, 170)
        t = np.full((_TEX, _TEX), base, np.float32)
        if textured:
            for _ in range(80):
                x, y = r.randint(0, _TEX - 8), r.randint(0, _TEX - 8)
                ww, hh = r.randint(8, 160), r.randint(8, 160)
                t[y:y + hh, x:x + ww] = r.randint(10, 246)
            t += r.randn(_TEX, _TEX).astype(np.float32) * 6.0  # fine grain
        else:
            t += (r.rand() - 0.5) * 4.0
            for _ in range(r.randint(2, 4)):  # door / window frames: long thin edges
                x, y = r.randint(60, _TEX - 400), r.randint(60, _TEX - 400)
                ww, hh = r.randint(150, 350), r.randint(200, 380)
                v = base + r.choice([-45, -30, 30, 45])
                t[y:y + hh, x:x + 6] = v
                t[y:y + hh, x + ww:x + ww + 6] = v
                t[y:y + 6, x:x + ww + 6] = v
                t[y + hh:y + hh + 6, x:x + ww + 6] = v
        tex.append(np.clip(t, 0, 255))
    return tex


_TEX_CACHE = {}


def _blur3(img):
    """3x3 Gaussian, sigma 0.8, reflect-101 (separable, float)."""
    k = np.exp(-0.5 * (np.arange(-1, 2) / 0.8) ** 2)
    k /= k.sum()
    p = np.pad(img, 1, mode='reflect')
    t = k[0] * p[:, :-2] + k[1] * p[:, 1:-1] + k[2] * p[:, 2:]
    return k[0] * t[:-2] + k[1] * t[1:-1] + k[2] * t[2:]


def frame(config='S1', index=0):
    """Returns (gray uint8 [h,w], depth16 uint16 [h,w]) for frame `index` of the synthetic sequence."""
    c = CONFIGS[config]
    w, h = c['w'], c['h']
    key = (c['textured'],)
    if key not in _TEX_CACHE:
        _TEX_CACHE[key] = _wall_textures(c['textured'])
    tex = _TEX_CACHE[key]
    # smooth camera path
    t = index * 0.02
    yaw, pitch = 0.25 * np.sin(0.7 * t), 0.08 * np.sin(0.9 * t + 1.0)
    o = np.array([0.6 * np.sin(0.5 * t), 0.15 * np.sin(0.8 * t), 0.5 * np.sin(0.3 * t)])
    cyw, syw, cp, sp = np.cos(yaw), np.sin(yaw), np.cos(pitch), np.sin(pitch)
    R = np.array([[cyw, 0, syw], [0, 1, 0], [-syw, 0, cyw]]) @ np.array([[1, 0, 0], [0, cp, -sp], [0, sp, cp]])
    u, v = np.meshgrid(np.arange(w, dtype=np.float64), np.arange(h, dtype=np.float64))
    dc = np.stack([(u - c['cx']) / c['fx'], (v - c['cy']) / c['fy'], np.ones_like(u)], -1)
    d = dc @ R.T
    best_t = np.full((h, w), np.inf)
    wall = np.zeros((h, w), np.int32)
    planes = [(0, _ROOM['x'][0]), (0, _ROOM['x'][1]), (1, _ROOM['y'][0]), (1, _ROOM['y'][1]), (2, _ROOM['z'])]
    with np.errstate(divide='ignore', invalid='ignore'):
        for i, (ax, val) in enumerate(planes):
            tt = (val - o[ax]) / d[..., ax]
            ok = (tt > 1e-6) & (tt < best_t)
            best_t = np.where(ok, tt, best_t)
            wall = np.where(ok, i, wall)
    hit = o + d * best_t[..., None]
    # wall-plane coordinates -> texture lookup (nearest)
    a = np.where(wall < 2, hit[..., 2] + 1.5, hit[..., 0] + 3.0)
    b = np.where((wall == 2) | (wall == 3), hit[..., 2] + 1.5, hit[..., 1] + 1.5)
    b = np.where(wall < 2, hit[..., 1] + 1.5, b)
    ti = np.clip((a * 160).astype(np.int64), 0, _TEX - 1)
    tj = np.clip((b * 300).astype(np.int64) % _TEX, 0, _TEX - 1)
    gray = np.zeros((h, w), np.float32)
    for i in range(5):
        m = wall == i
        gray[m] = tex[i][tj[m], ti[m]]
    shade = np.clip(1.15 - 0.07 * best_t, 0.55, 1.1).astype(np.float32)
    r = np.random.RandomState(1000 + index)
    gray = gray * shade + r.randn(h, w).astype(np.float32) * 2.0
    gray = np.clip(_blur3(gray) + 0.5, 0, 255).astype(np.uint8)
    z = best_t  # camera-frame ray has unit z, so depth == ray parameter
    # structured-light style depth: disparity (fb / z, fb = 42.75 m px) with Gaussian noise, quantised to 1/8 px
    with np.errstate(divide='ignore', invalid='ignore'):
        disp = 42.75 / z + r.randn(h, w) * 0.06
        z = 42.75 / (np.round(disp * 8.0) / 8.0)
    raw = np.floor(z * c['factor'] + 0.5)
    raw = np.where(np.isfinite(raw) & (raw < 65535), raw, 0).astype(np.uint16)
    # ~1 % holes, clustered as on a real structured-light sensor (blobs), not i.i.d. pixels
    yy, xx = np.mgrid[0:h, 0:w]
    for _ in range(max(8, (w * h) // 12000)):
        cxh, cyh, rad = r.randint(0, w), r.randint(0, h), r.randint(2, 9)
        raw[(xx - cxh) ** 2 + (yy - cyh) ** 2 <= rad * rad] = 0
    return gray, raw


def sequence(config='S1', n=8, start=0):
    """gray [n,h,w] uint8, depth16 [n,h,w] uint16."""
    g, d = zip(*[frame(config, start + i) for i in range(n)])
    return np.stack(g), np.stack(d)


def noise_frame(w, h, seed):
    """Structured random image (blurred noise + rectangles): dense FAST corners, many t=7 fallbacks."""
    r = np.random.RandomState(seed)
    a = r.randint(0, 256, (h, w)).astype(np.float32)
    a = _blur3(_blur3(a))
    a = (a - a.min()) / max(a.max() - a.min(), 1e-6) * 255.0
    for _ in range(60):
        x, y = r.randint(0, w - 40), r.randint(0, h - 40)
        a[y:y + r.randint(5, 80), x:x + r.randint(5, 80)] = r.randint(0, 256)
    return a.astype(np.uint8)


def descriptors_S4(nq=2000, nt=50000, seed=4, planted=200, ties=20):
    """Matching stress set: i.i.d. uniform descriptors with planted near-duplicates and exact ties."""
    r = np.random.RandomState(seed)
    q = r.randint(0, 256, (nq, 32)).astype(np.uint8)
    t = r.randint(0, 256, (nt, 32)).astype(np.uint8)
    qi = r.choice(nq, planted, replace=False)
    ti = r.choice(nt, planted, replace=False)
    for a, b in zip(qi, ti):
        d = q[a].copy()
        bits = r.choice(256, r.randint(0, 21), replace=False)
        for bit in bits:
            d[bit >> 3] ^= 1 << (bit & 7)
        t[b] = d
    # exact ties: the same train row twice for some queries (lowest train index must win)
    for k in range(ties):
        a = qi[k]
        src = ti[k]
        dst = (src + 1 + r.randint(0, nt - 1)) % nt
        t[dst] = t[src]
    return q, t
