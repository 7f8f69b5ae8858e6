"""Cost of on-device keypoint undistortion (k_undistort_kps) in the whole front-end, in one process:

  step     the C5-shaped step (one device-resident call of --call S1 frames, every stage, cullingLine, 4-bit labels / normals-only as
           bench.py runs it) with the TUM3 camera (no distortion), the TUM1 camera (k1..k3 != 0) and the TUM1 intrinsics without the
           coefficients (the planes and normals depend on K, so this pair isolates the undistortion), rotated --rounds times,
           --steps timed steps each after --warmup; CUDA events on the frame handle's master stream
  kernel   k_undistort_kps alone on the TUM1 step's outputs (keypoints, counts, depth of --call frames), CUDA events around --launches
           launches on an ORB handle's stream
  latency  one frame per blocking host call (hvo_frame_extract_batch), the three cameras alternated, median of --lat-calls
Prints one JSON object (and writes it to --out) with the card name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import hvo_b200 as hvo  # noqa: E402
from bench import BF, CAM, DEPTH_FACTOR, MAX_PLANES, NLINES, ORB, make_frames  # noqa: E402

TUM1 = dict(fx=517.306408, fy=516.469215, cx=318.643040, cy=255.313989)                        # TUM1.yaml
TUM1_DIST = np.array([0.262383, -0.953104, -0.005358, 0.002628, 1.163314], np.float32)


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.returncode == 0 else q.stderr.strip())


def frontend(cam, dist, max_batch, **kw):
    return hvo.FrameFrontEnd(640, 480, cam['fx'], cam['fy'], cam['cx'], cam['cy'], DEPTH_FACTOR, bf=BF, n_lines=NLINES, line_cull=True,
                             membership='u4', normals='n3', max_planes=MAX_PLANES, max_batch=max_batch, dist=dist,
                             nfeatures=ORB['nfeatures'], scale_factor=ORB['scale_factor'], nlevels=ORB['nlevels'], ini_th=ORB['ini_th'],
                             min_th=ORB['min_th'], **kw)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--call', type=int, default=4096)
    ap.add_argument('--distinct', type=int, default=256)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--launches', type=int, default=50)
    ap.add_argument('--lat-calls', type=int, default=60)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    n = a.call
    gray, depth = make_frames(a.distinct)
    reps = (n + len(gray) - 1) // len(gray)
    dev = torch.device('cuda', 0)
    d_gray = torch.from_numpy(gray).to(dev).repeat(reps, 1, 1)[:n].contiguous()
    d_depth = torch.from_numpy(depth.view(np.int16)).to(dev).repeat(reps, 1, 1)[:n].contiguous()
    res = dict(card=card(), call_frames=n, distinct_frames=a.distinct, rounds=a.rounds, steps_per_round=a.steps,
               step_ms={'tum3': [], 'tum1': [], 'tum1_pinhole': []})
    cams = (('tum3', CAM, None), ('tum1', TUM1, TUM1_DIST), ('tum1_pinhole', TUM1, None))
    keep = {}
    for r in range(a.rounds):
        for name, cam, dist in cams[r % 3:] + cams[:r % 3]:
            fe = frontend(cam, dist, n, lanes=1)
            shapes = fe.output_shapes(n)
            d_out = {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
            ptrs = {k: v.data_ptr() for k, v in d_out.items()}
            torch.cuda.synchronize()
            for _ in range(a.warmup):
                fe.extract_batch_device(d_gray.data_ptr(), d_depth.data_ptr(), n, ptrs)
            fe.sync()
            fe.timer_start()
            for _ in range(a.steps):
                fe.extract_batch_device(d_gray.data_ptr(), d_depth.data_ptr(), n, ptrs)
            res['step_ms'][name].append(fe.timer_stop() / a.steps)
            res.setdefault('launches_per_step', {})[name] = fe.last_launches()
            if name == 'tum1' and r == a.rounds - 1:
                keep = dict(d_out=d_out, shapes=shapes, cap=fe.orb_capacity)
            fe.close()
            torch.cuda.synchronize()
    for name, _, _ in cams:
        v = res['step_ms'][name]
        res[f'{name}_step_ms_median'] = float(np.median(v))
        res[f'{name}_frames_per_s'] = n / (float(np.median(v)) / 1e3)
    res['tum1_minus_tum3_step_ms'] = res['tum1_step_ms_median'] - res['tum3_step_ms_median']
    res['tum1_minus_tum1_pinhole_step_ms'] = res['tum1_step_ms_median'] - res['tum1_pinhole_step_ms_median']

    # k_undistort_kps alone on the TUM1 outputs of the last round
    d_out, shapes, cap = keep['d_out'], keep['shapes'], keep['cap']
    ex = hvo.ORBextractor(ORB['nfeatures'], ORB['scale_factor'], ORB['nlevels'], ORB['ini_th'], ORB['min_th'], width=640, height=480, max_batch=1)
    assert ex.capacity == cap
    camera = (np.array([[TUM1['fx'], 0, TUM1['cx']], [0, TUM1['fy'], TUM1['cy']], [0, 0, 1]], np.float32), TUM1_DIST)
    un2 = d_out['kps_un'].clone()        # rows past the counts are not written: start from the frame handle's buffers
    ur2 = d_out['kp_uright'].clone()
    k0 = int(d_out['kp_counts'].view(torch.int32)[0].item())
    un2.view(n, -1)[0, :28 * k0].zero_()     # frame 0's rows must be rewritten for the comparison to mean anything
    torch.cuda.synchronize()

    def launch():
        ex.undistort_batch_device(camera, d_out['kps'].data_ptr(), d_out['kp_counts'].data_ptr(), n, d_out['kp_depth'].data_ptr(), BF,
                                  un2.data_ptr(), ur2.data_ptr())
    for _ in range(5):
        launch()
    ex.sync()
    ex.timer_start()
    for _ in range(a.launches):
        launch()
    kms = ex.timer_stop() / a.launches
    ex.close()
    counts = d_out['kp_counts'].view(torch.int32).cpu().numpy()
    nkp = int(counts.sum())
    res['kernel'] = dict(ms_per_call=kms, us_per_call=kms * 1e3, keypoints=nkp, rows=n * cap,
                         same_as_frame_handle=bool(torch.equal(un2, d_out['kps_un']) and torch.equal(ur2, d_out['kp_uright'])),
                         bytes_min=nkp * (28 + 4 + 28 + 4) + n * 4,
                         note='bytes_min = keypoint read + depth read + kps_un write + uright write per valid row, counts')
    res['kernel']['achieved_GBps'] = res['kernel']['bytes_min'] / (kms / 1e3) / 1e9
    kps = d_out['kps'].cpu().numpy().view(hvo.KP_DTYPE).reshape(n, cap)
    un = d_out['kps_un'].cpu().numpy().view(hvo.KP_DTYPE).reshape(n, cap)
    f0 = int(counts[0])
    ref = hvo.undistort_points(np.stack([kps[0, :f0]['x'], kps[0, :f0]['y']], 1), *camera)
    res['kernel']['frame0_equals_host'] = bool(np.array_equal(ref[:, 0], un[0, :f0]['x']) and np.array_equal(ref[:, 1], un[0, :f0]['y']))
    del d_out, keep, un2, ur2
    torch.cuda.empty_cache()

    # single-frame latency, host arrays, the three cameras alternated
    lat = {name: [] for name, _, _ in cams}
    fes = {name: frontend(cam, dist, 1) for name, cam, dist in cams}
    g1, dp1 = np.ascontiguousarray(gray[:1]), np.ascontiguousarray(depth[:1])
    outs = {name: fe.alloc_host(1) for name, fe in fes.items()}
    for name, fe in fes.items():
        for _ in range(5):
            fe.extract_batch(g1, dp1, out=outs[name])
    for i in range(a.lat_calls):
        for name, _, _ in cams[i % 3:] + cams[:i % 3]:
            t0 = time.perf_counter()
            fes[name].extract_batch(g1, dp1, out=outs[name])
            lat[name].append(1e3 * (time.perf_counter() - t0))
    for name, fe in fes.items():
        fe.close()
    res['latency_ms_median'] = {k: float(np.median(v)) for k, v in lat.items()}
    res['latency_ms_p10_p90'] = {k: [float(np.percentile(v, 10)), float(np.percentile(v, 90))] for k, v in lat.items()}
    res['card_after'] = card()
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(s + '\n')


if __name__ == '__main__':
    main()
