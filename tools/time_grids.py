"""Cost of the frame grids (Frame::AssignFeaturesToGrid / AssignFeaturesToGridForLine on the device: k_proj_grid, k_lproj_grid +
k_lproj_grid_compact) in the whole front-end, in one process:

  step      the C5-shaped step (one device-resident call of --call S1 frames, every stage, cullingLine, 4-bit labels / normals-only as
            bench.py runs it, one lane) without and with grid outputs, alternated on one handle over --rounds rounds, --steps timed steps
            each after --warmup; CUDA events on the frame handle's master stream
  kernels   the grid kernels of one more step with grids (after the timed ones), from torch.profiler (CUDA activity)
  e2e       host arrays (pinned) through the blocking host call, --e2e-frames frames per call, without and with grid outputs alternated,
            host clock; plus the bytes copied back per frame
  latency   one frame per blocking host call, without and with grids alternated, median of --lat-calls
Prints one JSON object (and writes it to --out) with the card name, power limit and max SM clock read in the same run."""
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


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.returncode == 0 else q.stderr.strip())


def frontend(max_batch, **kw):
    return hvo.FrameFrontEnd(640, 480, CAM['fx'], CAM['fy'], CAM['cx'], CAM['cy'], DEPTH_FACTOR, bf=BF, n_lines=NLINES, line_cull=True,
                             membership='u4', normals='n3', max_planes=MAX_PLANES, max_batch=max_batch, nfeatures=ORB['nfeatures'],
                             scale_factor=ORB['scale_factor'], nlevels=ORB['nlevels'], ini_th=ORB['ini_th'], min_th=ORB['min_th'], grids=True, **kw)


def pinned(shapes):
    return {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, pin_memory=True).numpy().view(dt).reshape(s)
            for k, (s, dt) in shapes.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--call', type=int, default=4096)
    ap.add_argument('--distinct', type=int, default=256)
    ap.add_argument('--rounds', type=int, default=6)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--e2e-frames', type=int, default=1024)
    ap.add_argument('--e2e-calls', type=int, default=6)
    ap.add_argument('--lat-calls', type=int, default=60)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    n = a.call
    gray, depth = make_frames(a.distinct)
    reps = (n + len(gray) - 1) // len(gray)
    dev = torch.device('cuda', 0)
    d_gray = torch.from_numpy(gray).to(dev).repeat(reps, 1, 1)[:n].contiguous()
    d_depth = torch.from_numpy(depth.view(np.int16)).to(dev).repeat(reps, 1, 1)[:n].contiguous()
    res = dict(card=card(), call_frames=n, distinct_frames=a.distinct, rounds=a.rounds, steps_per_round=a.steps, step_ms={'plain': [], 'grids': []})
    order = ['plain', 'grids']

    # ---- whole-front-end step on one handle, with and without grid outputs alternated; then one profiled step with grids
    fe = frontend(n, lanes=1)
    shapes = fe.output_shapes(n)
    d_out = {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
    ptrs = {k: v.data_ptr() for k, v in d_out.items()}
    launches = {}
    for r in range(a.rounds):
        for name in order[r % 2:] + order[:r % 2]:
            fe.grids = name == 'grids'
            torch.cuda.synchronize()
            for _ in range(a.warmup):
                fe.extract_batch_device(d_gray.data_ptr(), d_depth.data_ptr(), n, ptrs)
            fe.sync()
            fe.timer_start()
            for _ in range(a.steps):
                fe.extract_batch_device(d_gray.data_ptr(), d_depth.data_ptr(), n, ptrs)
            res['step_ms'][name].append(fe.timer_stop() / a.steps)
            launches[name] = fe.last_launches()
    res['launches_per_step'] = launches
    fe.grids = True
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fe.extract_batch_device(d_gray.data_ptr(), d_depth.data_ptr(), n, ptrs)
        fe.sync()
    kern = {}
    for e in prof.key_averages():
        if 'grid' in e.key:
            t = getattr(e, 'device_time_total', None)
            kern[e.key] = (t if t is not None else e.cuda_time_total) / 1e3
    host = {k: d_out[k].cpu().numpy().view(shapes[k][1]).reshape(shapes[k][0]) for k in ('kp_counts', 'line_counts', 'grid_counts', 'lgrid_counts')}
    fe.close()
    del d_out
    torch.cuda.empty_cache()
    for name in order:
        v = res['step_ms'][name]
        res[f'{name}_step_ms_median'] = float(np.median(v))
        res[f'{name}_frames_per_s'] = n / (float(np.median(v)) / 1e3)
    res['grids_minus_plain_step_ms'] = res['grids_step_ms_median'] - res['plain_step_ms_median']
    res['grids_over_plain_percent'] = 100.0 * res['grids_minus_plain_step_ms'] / res['plain_step_ms_median']
    res['grid_kernels_ms_per_step'] = kern
    res['grid_kernels_ms_total'] = float(sum(kern.values()))
    res['grid_kernels_over_plain_step_percent'] = 100.0 * res['grid_kernels_ms_total'] / res['plain_step_ms_median']
    res['grid_entries_per_frame_mean'] = dict(points=float(host['grid_counts'].sum(1).mean()), keypoints=float(host['kp_counts'].mean()),
                                              line_cells=float(host['lgrid_counts'].sum(1).mean()), lines=float(host['line_counts'].mean()))

    # ---- end to end: pinned host arrays through the blocking host call, with and without grid outputs alternated
    m = a.e2e_frames
    fe = frontend(m)
    hg, hd = pinned({'g': ((m, 480, 640), np.uint8), 'd': ((m, 480, 640), np.uint16)}).values()
    idx = np.arange(m) % len(gray)
    hg[:] = gray[idx]
    hd[:] = depth[idx]
    fe.grids = True
    outs = {'grids': pinned(fe.output_shapes(m, device=False))}
    fe.grids = False
    outs['plain'] = pinned(fe.output_shapes(m, device=False))
    nbytes = {k: int(sum(v.nbytes for v in o.values())) // m for k, o in outs.items()}
    e2e = {'plain': [], 'grids': []}
    for name in order:
        fe.grids = name == 'grids'
        fe.extract_batch(hg, hd, out=outs[name])
    for i in range(a.e2e_calls):
        for name in order[i % 2:] + order[:i % 2]:
            fe.grids = name == 'grids'
            t0 = time.perf_counter()
            fe.extract_batch(hg, hd, out=outs[name])
            e2e[name].append(m / (time.perf_counter() - t0))
    fe.close()
    res['e2e'] = dict(frames_per_call=m, lanes_default=True, frames_per_s_median={k: float(np.median(v)) for k, v in e2e.items()},
                      frames_per_s_all=e2e, output_bytes_per_frame=nbytes, grid_bytes_per_frame=nbytes['grids'] - nbytes['plain'],
                      note='blocking hvo_frame_extract_batch_grid, pinned input and output arrays, host clock')

    # ---- single-frame latency, host arrays, with and without grids alternated on one handle
    fe = frontend(1)
    g1, dp1 = np.ascontiguousarray(gray[:1]), np.ascontiguousarray(depth[:1])
    fe.grids = True
    lo = {'grids': fe.alloc_host(1)}
    fe.grids = False
    lo['plain'] = fe.alloc_host(1)
    lat = {'plain': [], 'grids': []}
    for name in order:
        fe.grids = name == 'grids'
        for _ in range(5):
            fe.extract_batch(g1, dp1, out=lo[name])
    for i in range(a.lat_calls):
        for name in order[i % 2:] + order[:i % 2]:
            fe.grids = name == 'grids'
            t0 = time.perf_counter()
            fe.extract_batch(g1, dp1, out=lo[name])
            lat[name].append(1e3 * (time.perf_counter() - t0))
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
