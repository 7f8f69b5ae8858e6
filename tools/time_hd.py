"""Front-end throughput and latency above 1280x720 (synthetic S6 = 1920x1080, S7 = 1024x1024, and S3 = 1280x720 for reference), in one
process:

  memory     device bytes per frame of a frame handle (cudaMemGetInfo around hvo_frame_create with --probe frames, every stage,
             lpvo / grids off) and the largest chunk the free memory of this device holds at that rate
  device     frames/s of device-resident calls of up to --call frames (fewer where a quarter of the free memory holds fewer; every
             stage, cullingLine, one lane), CUDA events on the handle's master
             stream; --rounds rounds of --steps timed calls after --warmup, the configurations alternated in a rotating order
  e2e        the same calls through the host API with pinned host buffers (uploads and downloads inside the timed region), host clock
  pipelines  at 1920x1080: the device step of a handle with only one stage (ORB, lines, planes, normals); with --profile (a run of its
             own, after the timed one) the kernel time of one all-stage step per kernel from torch.profiler (CUDA activity), merged
             into --out
  latency    one frame per blocking host call, p10 / p50 / p90 of --lat-calls, the configurations alternated
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
from hvo_b200 import synth  # noqa: E402

CONFIGS = ['S6', 'S7', 'S3']
PIPELINES = {'orb': hvo.STAGE_ORB, 'lines': hvo.STAGE_LINES, 'planes': hvo.STAGE_PLANES, 'normals': hvo.STAGE_NORMALS}
# kernel name prefix -> pipeline (every other kernel is the ORB pipeline's)
KERNEL_PIPELINE = (('k_plane', 'planes'), ('k_pack_membership', 'planes'), ('k_lsd', 'lines'), ('k_line', 'lines'), ('k_lbd', 'lines'),
                   ('k_lproj', 'lines'), ('k_sn', 'normals'), ('k_lpvo', 'normals'), ('k_pack_normals', 'normals'), ('k_frame', 'frame'))


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.returncode == 0 else q.stderr.strip())


def frontend(cfg, max_batch, stages=hvo.STAGE_ALL, lanes=1):
    c = synth.CONFIGS[cfg]
    return hvo.FrameFrontEnd(c['w'], c['h'], c['fx'], c['fy'], c['cx'], c['cy'], np.float32(1.0 / c['factor']), bf=c['bf'],
                             nfeatures=c['nfeatures'], line_cull=True, membership='u4' if stages & hvo.STAGE_PLANES else 'i32',
                             normals='n3', max_planes=15, max_batch=max_batch, stages=stages, lanes=lanes)


def spread(v):
    return dict(median=float(np.median(v)), min=float(np.min(v)), max=float(np.max(v)), p10=float(np.percentile(v, 10)),
                p90=float(np.percentile(v, 90)), n=len(v))


def pinned(shape, dt):
    n = int(np.prod(shape)) * np.dtype(dt).itemsize
    return torch.empty(max(n, 1), dtype=torch.uint8, pin_memory=True).numpy()[:n].view(dt).reshape(shape)


class Run:
    """One handle of one configuration with its device-resident and pinned host buffers."""

    def __init__(self, cfg, gray, depth, n, dev, stages=hvo.STAGE_ALL):
        self.cfg, self.n = cfg, n
        reps = -(-n // len(gray))
        self.fe = frontend(cfg, n, stages)
        self.d_gray = torch.from_numpy(gray).to(dev).repeat(reps, 1, 1)[:n].contiguous()
        self.d_depth = torch.from_numpy(depth.view(np.int16)).to(dev).repeat(reps, 1, 1)[:n].contiguous()
        shapes = self.fe.output_shapes(n)
        self.d_out = {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
        self.ptrs = {k: v.data_ptr() for k, v in self.d_out.items()}
        self.h_gray, self.h_depth = pinned((n,) + gray.shape[1:], np.uint8), pinned((n,) + depth.shape[1:], np.uint16)
        self.h_gray[:] = np.resize(gray, self.h_gray.shape)
        self.h_depth[:] = np.resize(depth, self.h_depth.shape)
        self.h_out = {k: pinned(s, dt) for k, (s, dt) in self.fe.output_shapes(n, device=False).items()}
        torch.cuda.synchronize()

    def device_step(self):
        self.fe.extract_batch_device(self.d_gray.data_ptr(), self.d_depth.data_ptr(), self.n, self.ptrs)

    def host_step(self):
        self.fe.extract_batch(self.h_gray, self.h_depth, out=self.h_out)

    def time_device(self, warmup, steps):
        for _ in range(warmup):
            self.device_step()
        self.fe.sync()
        self.fe.timer_start()
        for _ in range(steps):
            self.device_step()
        return self.fe.timer_stop() / steps

    def time_host(self, warmup, steps):
        for _ in range(warmup):
            self.host_step()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.host_step()
        return 1e3 * (time.perf_counter() - t0) / steps

    def close(self):
        self.fe.close()
        del self.d_out, self.d_gray, self.d_depth
        torch.cuda.empty_cache()


def per_frame_bytes(cfg, probe):
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    fe = frontend(cfg, probe)
    free1 = torch.cuda.mem_get_info(0)[0]
    fe.close()
    return (free0 - free1) / probe


def profile_kernels(a, dev):
    """Kernel time per kernel and per pipeline of one all-stage 1920x1080 device-resident call, after --warmup untimed calls."""
    from torch.profiler import ProfilerActivity, profile
    gray, depth = synth.sequence('S6', a.distinct)
    n = min(a.call, int(torch.cuda.mem_get_info(0)[0] // per_frame_bytes('S6', a.probe)) // 4)
    r = Run('S6', gray, depth, n, dev)
    for _ in range(a.warmup):
        r.device_step()
    r.fe.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r.device_step()
        r.fe.sync()
    r.close()
    kern = {}
    for e in prof.key_averages():
        if e.key.startswith('k_') or '::k_' in e.key:
            t = getattr(e, 'device_time_total', None)
            kern[e.key] = (t if t is not None else e.cuda_time_total) / 1e3
    by_pipe = {}
    for name, t in kern.items():
        pipe = next((p for pre, p in KERNEL_PIPELINE if pre in name), 'orb')
        by_pipe[pipe] = by_pipe.get(pipe, 0.0) + t
    return dict(s6_profiled_call_frames=n, s6_kernel_ms_per_call=kern, s6_kernel_ms_per_call_by_pipeline=by_pipe)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--call', type=int, default=512, help='frames per device-resident / host call')
    ap.add_argument('--distinct', type=int, default=16, help='distinct synthetic frames per configuration (repeated to fill a call)')
    ap.add_argument('--probe', type=int, default=64, help='frames of the handle the memory probe creates')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--lat-calls', type=int, default=30)
    ap.add_argument('--profile', action='store_true', help='only the torch.profiler pass, merged into --out (run it after the timed run)')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    dev = torch.device('cuda', 0)
    if a.profile:
        res = json.load(open(a.out)) if a.out and os.path.exists(a.out) else {}
        res.update(profile_kernels(a, dev))
        res['card_profile_run'] = card()
        s = json.dumps(res, indent=1)
        print(s)
        if a.out:
            with open(a.out, 'w') as f:
                f.write(s + '\n')
        return
    res = dict(card=card(), call_frames=a.call, distinct_frames=a.distinct, rounds=a.rounds, steps_per_round=a.steps, warmup=a.warmup,
               configs={k: {kk: synth.CONFIGS[k][kk] for kk in ('w', 'h', 'nfeatures', 'factor')} for k in CONFIGS})
    frames = {k: synth.sequence(k, a.distinct) for k in CONFIGS}

    # ---- memory per frame
    total = torch.cuda.mem_get_info(0)[1]
    mem = {}
    for k in CONFIGS:
        b = per_frame_bytes(k, a.probe)
        free = torch.cuda.mem_get_info(0)[0]
        mem[k] = dict(bytes_per_frame=int(b), mb_per_frame=b / 2**20, largest_chunk_in_free_memory=int(free // b), device_total_bytes=int(total))
    res['memory'] = mem
    calls = {k: int(min(a.call, mem[k]['largest_chunk_in_free_memory'] // 4)) for k in CONFIGS}
    res['call_frames_per_config'] = calls

    # ---- whole front end: device-resident and host calls, the configurations alternated
    runs = {k: Run(k, *frames[k], calls[k], dev) for k in CONFIGS}
    dev_ms = {k: [] for k in CONFIGS}
    e2e_ms = {k: [] for k in CONFIGS}
    for r in range(a.rounds):
        order = CONFIGS[r % len(CONFIGS):] + CONFIGS[:r % len(CONFIGS)]
        for k in order:
            dev_ms[k].append(runs[k].time_device(a.warmup, a.steps))
        for k in order:
            e2e_ms[k].append(runs[k].time_host(a.warmup, a.steps))
    res['launches_per_call'] = {k: runs[k].fe.last_launches() for k in CONFIGS}
    for r in runs.values():
        r.close()
    res['device_call_ms'] = {k: spread(v) for k, v in dev_ms.items()}
    res['e2e_call_ms'] = {k: spread(v) for k, v in e2e_ms.items()}
    res['timed_window_s'] = {k: dict(device=a.steps * float(np.median(dev_ms[k])) / 1e3, e2e=a.steps * float(np.median(e2e_ms[k])) / 1e3)
                             for k in CONFIGS}
    res['device_frames_per_s'] = {k: calls[k] / (float(np.median(v)) / 1e3) for k, v in dev_ms.items()}
    res['e2e_frames_per_s'] = {k: calls[k] / (float(np.median(v)) / 1e3) for k, v in e2e_ms.items()}

    # ---- one pipeline at a time at 1920x1080 (device-resident, same call size)
    pipe_ms = {}
    for p, st in PIPELINES.items():
        r = Run('S6', *frames['S6'], calls['S6'], dev, stages=st)
        pipe_ms[p] = [r.time_device(a.warmup, a.steps) for _ in range(a.rounds)]
        r.close()
    res['s6_single_pipeline_call_ms'] = {p: spread(v) for p, v in pipe_ms.items()}

    # ---- single-frame blocking latency (host arrays), the configurations alternated
    lat_runs = {k: (frontend(k, 1), np.ascontiguousarray(frames[k][0][:1]), np.ascontiguousarray(frames[k][1][:1])) for k in CONFIGS}
    outs = {k: fe.alloc_host(1) for k, (fe, _, _) in lat_runs.items()}
    lat = {k: [] for k in CONFIGS}
    for k, (fe, g, d) in lat_runs.items():
        for _ in range(3):
            fe.extract_batch(g, d, out=outs[k])
    for i in range(a.lat_calls):
        for k in CONFIGS[i % len(CONFIGS):] + CONFIGS[:i % len(CONFIGS)]:
            fe, g, d = lat_runs[k]
            t0 = time.perf_counter()
            fe.extract_batch(g, d, out=outs[k])
            lat[k].append(1e3 * (time.perf_counter() - t0))
    for fe, _, _ in lat_runs.values():
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
