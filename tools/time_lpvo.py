"""Cost of the LPVO normals in the frame pipeline (Manhattan::computeNormalsLPVO on the device: k_lpvo_rows, k_lpvo_cols,
k_lpvo_normals after the surface normals), in one process:

  step       the C5-shaped step (one device-resident call of --call S1 frames, every stage, cullingLine, 4-bit labels / normals-only as
             bench.py runs it, one lane) without and with LPVO outputs, alternated on one handle over --rounds rounds, --steps timed steps
             each after --warmup; CUDA events on the frame handle's master stream
  kernels    the LPVO kernels of one more step with LPVO outputs (after the timed ones), from torch.profiler (CUDA activity)
  scratch    device memory the first call with LPVO outputs allocates (cudaMemGetInfo before / after), and the formula's value
  standalone hvo_lpvo (hvo.Manhattan) on the same device-resident depth, one call of --call frames, CUDA events on its stream
  latency    one frame per blocking host call, without and with LPVO outputs alternated, p10 / p50 / p90 of --lat-calls
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

SUB_BATCH = 256   # kLpvoFrames in csrc/frame.cu


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.returncode == 0 else q.stderr.strip())


def frontend(max_batch, **kw):
    return hvo.FrameFrontEnd(640, 480, CAM['fx'], CAM['fy'], CAM['cx'], CAM['cy'], DEPTH_FACTOR, bf=BF, n_lines=NLINES, line_cull=True,
                             membership='u4', normals='n3', max_planes=MAX_PLANES, max_batch=max_batch, nfeatures=ORB['nfeatures'],
                             scale_factor=ORB['scale_factor'], nlevels=ORB['nlevels'], ini_th=ORB['ini_th'], min_th=ORB['min_th'], lpvo=True, **kw)


def scratch_bytes(w, h, frames):
    nsu, nsv = -(-(w - 11) // 15), -(-(h - 11) // 15)
    return dict(rowsum=frames * 7 * h * 2 * nsu * 8, integrals=frames * 7 * 2 * nsv * 2 * nsu * 8)


def spread(v):
    return dict(median=float(np.median(v)), min=float(np.min(v)), max=float(np.max(v)), p10=float(np.percentile(v, 10)),
                p90=float(np.percentile(v, 90)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--call', type=int, default=4096)
    ap.add_argument('--distinct', type=int, default=256)
    ap.add_argument('--rounds', type=int, default=6)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--lat-calls', type=int, default=60)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    n = a.call
    gray, depth = make_frames(a.distinct)
    reps = (n + len(gray) - 1) // len(gray)
    dev = torch.device('cuda', 0)
    d_gray = torch.from_numpy(gray).to(dev).repeat(reps, 1, 1)[:n].contiguous()
    d_depth = torch.from_numpy(depth.view(np.int16)).to(dev).repeat(reps, 1, 1)[:n].contiguous()
    res = dict(card=card(), call_frames=n, distinct_frames=a.distinct, rounds=a.rounds, steps_per_round=a.steps, lpvo_sub_batch=SUB_BATCH,
               step_ms={'plain': [], 'lpvo': []})
    order = ['plain', 'lpvo']

    # ---- whole-front-end step on one handle, with and without LPVO outputs alternated; then one profiled step with them
    fe = frontend(n, lanes=1)
    fe.with_lpvo = True
    shapes = fe.output_shapes(n)
    d_out = {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
    ptrs = {k: v.data_ptr() for k, v in d_out.items()}
    torch.cuda.synchronize()
    fe.with_lpvo = False
    fe.extract_batch_device(d_gray.data_ptr(), d_depth.data_ptr(), n, ptrs)
    fe.sync()
    free0 = torch.cuda.mem_get_info(0)[0]
    fe.with_lpvo = True
    fe.extract_batch_device(d_gray.data_ptr(), d_depth.data_ptr(), n, ptrs)   # allocates the LPVO scratch
    fe.sync()
    free1 = torch.cuda.mem_get_info(0)[0]
    res['scratch'] = dict(measured_bytes=int(free0 - free1), formula_bytes=scratch_bytes(640, 480, SUB_BATCH),
                          formula_bytes_1280x720=scratch_bytes(1280, 720, SUB_BATCH),
                          chunk_sized_bytes_at_call=scratch_bytes(640, 480, n),
                          note='cudaMemGetInfo difference around the first call with LPVO outputs (allocation granularity included)')
    launches = {}
    for r in range(a.rounds):
        for name in order[r % 2:] + order[:r % 2]:
            fe.with_lpvo = name == 'lpvo'
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
    fe.with_lpvo = True
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fe.extract_batch_device(d_gray.data_ptr(), d_depth.data_ptr(), n, ptrs)
        fe.sync()
    kern = {}
    for e in prof.key_averages():
        if 'lpvo' in e.key:
            t = getattr(e, 'device_time_total', None)
            kern[e.key] = (t if t is not None else e.cuda_time_total) / 1e3
    counts = d_out['lpvo_counts'].cpu().numpy().view(np.int32)
    frame_rows = {k: d_out[k].cpu().numpy().view(shapes[k][1]).reshape(shapes[k][0])[:a.distinct].copy() for k in ('lpvo_normals3', 'lpvo_counts')}
    fe.close()
    del d_out
    torch.cuda.empty_cache()
    for name in order:
        res[f'{name}_step_ms'] = spread(res['step_ms'][name])
        res[f'{name}_frames_per_s'] = n / (float(np.median(res['step_ms'][name])) / 1e3)
    res['lpvo_minus_plain_step_ms'] = res['lpvo_step_ms']['median'] - res['plain_step_ms']['median']
    res['lpvo_over_plain_percent'] = 100.0 * res['lpvo_minus_plain_step_ms'] / res['plain_step_ms']['median']
    res['lpvo_kernels_ms_per_step'] = kern
    res['lpvo_kernels_ms_total'] = float(sum(kern.values()))
    res['lpvo_samples_per_frame_mean'] = float(counts.mean())

    # ---- standalone hvo_lpvo on the same device-resident depth (one pass of n frames: chunk-sized scratch)
    m = hvo.Manhattan(np.array([[CAM['fx'], 0, CAM['cx']], [0, CAM['fy'], CAM['cy']], [0, 0, 1]], np.float32), 640, 480, DEPTH_FACTOR, max_batch=n)
    c = m.capacity
    so = dict(nrm=torch.empty(n * c * 3, dtype=torch.float64, device=dev), z=torch.empty(n * c, dtype=torch.float32, device=dev),
              pix=torch.empty(n * c * 2, dtype=torch.int32, device=dev), cnt=torch.empty(n, dtype=torch.int32, device=dev))
    args = (d_depth.data_ptr(), n, so['nrm'].data_ptr(), so['z'].data_ptr(), so['pix'].data_ptr(), so['cnt'].data_ptr())
    for _ in range(a.warmup):
        m.compute_device(*args)
    m.sync()
    alone = []
    for _ in range(a.rounds):
        m.timer_start()
        for _ in range(a.steps):
            m.compute_device(*args)
        alone.append(m.timer_stop() / a.steps)
    sn = so['nrm'].cpu().numpy().reshape(n, c, 3)[:a.distinct]
    sc = so['cnt'].cpu().numpy()[:a.distinct]
    same = bool(np.array_equal(sc, frame_rows['lpvo_counts']) and all(
        sn[f, :sc[f]].tobytes() == frame_rows['lpvo_normals3'][f, :sc[f]].tobytes() for f in range(a.distinct)))
    m.close()
    del so
    torch.cuda.empty_cache()
    res['standalone_hvo_lpvo_ms'] = spread(alone)
    res['standalone_rows_equal_frame_call'] = same

    # ---- single-frame latency, host arrays, with and without LPVO outputs alternated on one handle
    fe = frontend(1)
    g1, dp1 = np.ascontiguousarray(gray[:1]), np.ascontiguousarray(depth[:1])
    lo = {'lpvo': fe.alloc_host(1)}
    fe.with_lpvo = False
    lo['plain'] = fe.alloc_host(1)
    lat = {'plain': [], 'lpvo': []}
    for name in order:
        fe.with_lpvo = name == 'lpvo'
        for _ in range(5):
            fe.extract_batch(g1, dp1, out=lo[name])
    for i in range(a.lat_calls):
        for name in order[i % 2:] + order[:i % 2]:
            fe.with_lpvo = name == 'lpvo'
            t0 = time.perf_counter()
            fe.extract_batch(g1, dp1, out=lo[name])
            lat[name].append(1e3 * (time.perf_counter() - t0))
    fe.close()
    res['latency_ms'] = {k: dict(p10=float(np.percentile(v, 10)), p50=float(np.median(v)), p90=float(np.percentile(v, 90))) for k, v in lat.items()}
    res['card_after'] = card()
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(s + '\n')


if __name__ == '__main__':
    main()
