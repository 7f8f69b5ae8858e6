#!/usr/bin/env python
"""bench.py — front-end frames/s at 640x480 (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over the C5 sequence of BASELINE.json: 8192 synthetic TUM-fr3-shaped 640x480 RGB-D frames,
frame-sharded across the N GPUs in contiguous ranges (8192 / N frames per GPU per step: "scaling": "strong").  Frames are
independent, so there is no data-path collective; torch.distributed carries only the barrier and the max-over-ranks of the time.
A GPU processes its share as calls of at most 4096 frames; a call of >= 2048 frames is one chunk whose pipelines run one after the
other, each at its saturating batch (DESIGN.md section 4, scheduling); two lanes of staging overlap the copies of neighbouring calls.

  value     whole-job frames/s with the inputs already resident in HBM (CUDA events on the library's master stream, max over ranks)
  e2e       the same through the reference-facing C-ABI call with HOST (pinned) buffers: host->device copy of gray + depth and
            device->host read of every output inside the timed region (compact outputs: 4-bit plane labels, normal-only normals)
  weak      the round-1 line for comparison: every GPU processes one call (<= 4096 frames) per step, whatever N is
  configs   sub-records for the other BASELINE.json configs: C2 (ICL-shaped low texture), C3 (1280x720, 2000 ORB), C4 (matching
            stress 2000 x 50 000 ORB + 200 x 5 000 LBD with cv2.BFMatcher beside it)
  roofline / cpu_baseline (throughput AND per-frame latency in the reference's 3-thread shape) / clocks / gpu_launches /
  p50_latency_ms_single_frame: see DESIGN.md section "Measurement"

--impl reference times the reference's CPU implementation of the same path on the host cores: the oracle port (oracle/), which is
pinned by execution to the reference's own sources compiled in oracle/_ref (ORBextractor.cc, PlaneExtractor.cpp + peac, the vendored
line_descriptor, Frame::cullingLine); the reference binary itself cannot be built (OpenCV / PCL / Eigen / Pangolin are absent).
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner at the WARN / VERSION debug levels) write to
# file descriptor 1 directly, so descriptor 1 is pointed at stderr for the whole run and the result line goes to the real stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(obj):
    os.write(_REAL_STDOUT, (json.dumps(obj) + '\n').encode())


METRIC = 'front-end frames/s @640x480'
C5_FRAMES = 8192                                                               # BASELINE.json configs[4]
CALL_FRAMES = 4096                                                             # frames per library call = one chunk (serial pipeline schedule)
ORB = dict(nfeatures=1000, scale_factor=1.2, nlevels=8, ini_th=20, min_th=7)  # TUM3.yaml:41-54
CAM = dict(fx=535.4, fy=539.2, cx=320.1, cy=247.6)                             # TUM3.yaml:8-11
DEPTH_FACTOR, BF, NLINES = 1.0 / 5000.0, 40.0, 200                             # TUM3.yaml:34, Camera.bf, LINE.nFeatures
MAX_PLANES = 15                                                                # rows of planes7 (4-bit labels on the wire)
ORACLE_CAM = (DEPTH_FACTOR, CAM['fx'], CAM['fy'], CAM['cx'], CAM['cy'])
ORACLE_STAGES = 15 | 16  # ORB | lines | planes | normals | cullingLine after the line extractor (what Frame::Frame runs)
STAGES = ['orb: 8-level pyramid + per-cell FAST + quadtree + IC_Angle + 7x7 blur (per keypoint patch) + rBRIEF + RGB-D depth lookup',
          'lines: LSD (blur, 0.8 resize, gradient, ordered region growing, rectangles) + KeyLines + top-200 + LBD + line functions + '
          'Frame::cullingLine (merge, rebuild, LBD again)',
          'planes: depth back-projection + 10x10 block fits + AHC merging + block erosion + ordered pixel flood fill + last merge',
          'normals: 3x subsampled cloud + integral-image normals (PCL AVERAGE_3D_GRADIENT restatement)']
# algorithmic bytes per 640x480 frame of the HBM-bound kernels (SURVEY.md section 8d; DESIGN.md section 4)
# (k_describe: the 43 x 43 level patch of ~1000 keypoints + the outputs; the reference's blurred pyramid, 1 901 064 B written and read
# back, is no longer materialised: the 7 x 7 blur is computed per patch inside k_describe)
ALG_BYTES = {'k_resize x7': 1569878, 'k_fast_strips': 950532, 'k_describe': 1000 * 43 * 43 + 60000,
             'k_lsd_prep': 307200 + 16 * 512 * 384, 'k_plane_blocks': 614400 + 3072 * 96}
# whole front-end: ORB 6 403 474 + LBD pre 2 150 400 + LBD gather 2 x 3 024 000 + LSD 3 452 928 + seed order / regions 2 359 296 +
# planes 909 312 + membership 1 536 000 + normals 2 054 400 (SURVEY.md section 8d)
ALG_BYTES_FRAME = 6403474 + 2150400 + 2 * 3024000 + 3452928 + 2359296 + 909312 + 1536000 + 2054400
# dram__bytes_read.sum + dram__bytes_write.sum per frame of the same kernels, from this round's committed ncu capture
# (profiles/r2b_ncu_full_orb_kernels_b296.csv for the ORB kernels; profiles/r1d_* for the others, unchanged kernels)
NCU_DRAM_BYTES = {'k_resize x7': 1555000, 'k_fast_strips': 968000, 'k_describe': 1102000, 'k_lsd_prep': 3592000, 'k_plane_blocks': 857000}
DUMP_BYTES = 64 * 10 ** 6                                                      # --dump-outputs writes at most this much
DUMP_SEED = 0                                                                  # which frames of the last call --dump-outputs writes
# rows past the frame's count in these outputs are scratch, not results: --dump-outputs writes the valid rows of the sampled frames one
# after the other (the count outputs say how many belong to each frame)
DUMP_ROWS = dict(kps='kp_counts', desc='kp_counts', kp_depth='kp_counts', kp_uright='kp_counts', keylines='line_counts',
                 line_desc='line_counts', linevec3='line_counts', planes7='n_planes')


def _gen(args):
    from hvo_b200 import synth
    cfg, i = args
    return synth.frame(cfg, i)


def make_frames(n, start=0, cfg='S1'):
    """n distinct synthetic frames (gray u8, depth u16); generated in parallel, cached under /tmp."""
    cache = f'/tmp/hvo_bench_{cfg}_{start}_{n}.npz'
    if os.path.exists(cache):
        z = np.load(cache)
        return z['gray'], z['depth']
    import hvo_b200  # noqa: F401  (registers the package alias for the workers)
    procs = max(1, min(32, (os.cpu_count() or 2) - 1))
    with mp.get_context('fork').Pool(procs) as pool:
        res = pool.map(_gen, [(cfg, start + i) for i in range(n)], chunksize=max(1, n // (4 * procs)))
    gray = np.stack([r[0] for r in res])
    depth = np.stack([r[1] for r in res])
    try:
        np.savez(cache, gray=gray, depth=depth)
    except OSError:
        pass
    return gray, depth


def bind_to_gpu_numa_node(gpu_index):
    """N > 1: run this rank on the CPUs NVML reports as local to its GPU, BEFORE the pinned host buffers are allocated, so that the
    pages the copy engines read and write (first touch) and the thread that queues the copies sit on the GPU's own NUMA node; eight
    ranks then do not funnel 8 x 1.3 MB per frame through one socket's memory.  Returns the CPU list, or None where NVML / the
    affinity call is unavailable or the box has one node (nothing is changed then)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        try:
            ncpu = os.cpu_count() or 1
            words = pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(gpu_index), (ncpu + 63) // 64)
        finally:
            pynvml.nvmlShutdown()
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = sorted(set(cpus) & allowed)
        if len(cpus) < 4 or len(cpus) >= len(allowed):   # one node, or a cpuset that leaves this GPU next to no local CPUs: stay unbound
            return None
        os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:   # a placement hint must never take the bench down
        return None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100',
                                          '-i', str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=3)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            self.proc.wait()
        sm, smax, reasons = [], None, set()
        for ts, line in self.lines:
            p = [x.strip() for x in line.split(',')]
            if len(p) < 9:
                continue
            try:
                smax = float(p[2])
                if t0 - 0.05 <= ts <= t1 + 0.15:
                    sm.append(float(p[1]))
                    for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), p[5:9]):
                        if v.lower().startswith('active'):
                            reasons.add(name)
            except ValueError:
                continue
        if not sm:  # region shorter than the sampling period: take every sample we have
            for ts, line in self.lines:
                p = [x.strip() for x in line.split(',')]
                try:
                    sm.append(float(p[1]))
                except (ValueError, IndexError):
                    pass
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=smax, reasons=sorted(reasons), samples=len(sm))


def measured_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def cpu_baseline(gray, depth, target_s=15.0):
    """The oracle port of the whole front-end timed on the host cores: frame-parallel over all cores."""
    import oracle
    cores = os.cpu_count() or 1
    ns = min(len(gray), 2 * cores)
    g, d = gray[:ns], depth[:ns]
    oracle.frontend_batch(g[:cores], d[:cores], ORACLE_CAM, stages=ORACLE_STAGES, nthreads=cores, nlines=NLINES, **ORB)  # warm-up / page-in
    n, dt, counts = 0, 0.0, []
    t0 = time.perf_counter()
    while dt < target_s:  # bounded sample: whole passes over the same frames until ~target_s of CPU work
        counts.append(oracle.frontend_batch(g, d, ORACLE_CAM, stages=ORACLE_STAGES, nthreads=cores, nlines=NLINES, **ORB).mean(axis=0))
        n += ns
        dt = time.perf_counter() - t0
    c = np.mean(counts, axis=0)
    return dict(value=n / dt, unit='frames/s', cores=cores, kind='port',
                sample=f'{n} frames ({n // ns} passes over the same {ns} synthetic 640x480 RGB-D frames), whole front-end (ORB + LSD/LBD lines '
                       f'+ PEAC planes + surface normals), oracle C++ port (-O3), one frame per thread on {cores} threads, {dt:.1f} s; '
                       f'mean per frame: {c[0]:.0f} keypoints, {c[1]:.0f} lines, {c[2]:.1f} planes, {c[3]:.0f} normals')


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (oracle port of the whole front-end) on all host cores; rank 0 only."""
    if rank != 0:
        return
    import oracle
    cores = os.cpu_count() or 1
    sample = max(cores, min(2368, 2 * cores))
    gray, depth = make_frames(sample)
    for _ in range(args.warmup):
        oracle.frontend_batch(gray, depth, ORACLE_CAM, stages=ORACLE_STAGES, nthreads=cores, nlines=NLINES, **ORB)
    t = time.perf_counter()
    for _ in range(args.steps):
        oracle.frontend_batch(gray, depth, ORACLE_CAM, stages=ORACLE_STAGES, nthreads=cores, nlines=NLINES, **ORB)
    dt = time.perf_counter() - t
    v = sample * args.steps / dt
    emit({
        'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': 'frames/s', 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'strong',
        'vs_baseline': None, 'dtype': 'u8', 'data': 'synthetic',
        'config': {'workload': f'C5/C1: synthetic TUM-fr3-shaped 640x480 RGB-D frames (TUM3.yaml: ORB 1000 features 8 levels x1.2, LINE 200), whole '
                               f'front-end of Frame::Frame; bounded sample of {sample} frames/step of the 8192-frame sequence',
                   'stages': STAGES, 'note': 'reference CPU path = oracle port, pinned by execution to the reference sources compiled in oracle/_ref '
                                             '(ORBextractor.cc, PlaneExtractor.cpp + peac, vendored line_descriptor, Frame::cullingLine; LSD to cv2 4.13.0); '
                                             'the reference binary needs OpenCV/PCL/Eigen/Pangolin, absent here'},
        'cpu_baseline': {'value': v, 'unit': 'frames/s', 'cores': cores, 'kind': 'port', 'sample': f'{sample} frames x {args.steps} steps'},
        'e2e': {'value': v, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    })


def cpu_latency(gray, depth, nframes=60, warm=5):
    """Per-frame latency of the CPU front-end in the reference's own shape (src/Frame.cc:208-233): three concurrent threads per frame,
    ORB || LSD + cullingLine + LBD || PEAC + normals, joined; time around the join as MTimeFeatExtract does."""
    import oracle
    groups = (1, 2 | 16, 4 | 8)
    lat = []
    for i in range(warm + nframes):
        g, d = gray[i % len(gray)][None], depth[i % len(depth)][None]
        th = [threading.Thread(target=oracle.frontend_batch, args=(g, d, ORACLE_CAM), kwargs=dict(stages=s, nthreads=1, nlines=NLINES, **ORB)) for s in groups]
        t0 = time.perf_counter()
        for t in th:
            t.start()
        for t in th:
            t.join()
        if i >= warm:
            lat.append(1e3 * (time.perf_counter() - t0))
    lat = np.array(lat)
    return dict(mean=float(lat.mean()), p50=float(np.median(lat)), p95=float(np.percentile(lat, 95)), frames=nframes, threads_per_frame=3,
                shape='ORB || LSD + cullingLine + LBD x2 || PEAC + normals, joined (Frame.cc:208-233)')


def shard(n, world, rank):
    """(first frame, frame count) of rank's contiguous range of the sequence: the package's partition (sharding.shard_range, the one
    hvo_seq_* uses below the C ABI and tests/test_sharding_cpu.py checks under gloo)"""
    from hvo_b200.sharding import shard_range
    lo, hi = shard_range(n, rank, world)
    return lo, hi - lo


def _float_dtype(dt):
    """the float type that holds every value of dt exactly: floats stay, 8- / 16-bit integers -> float32, wider -> float64"""
    return dt if dt.kind == 'f' else np.dtype(np.float32 if dt.itemsize <= 2 else np.float64)


def _float_bytes(dt):
    """bytes --dump-outputs may write per element of dt: the float copy, and a float32 finite mask for float outputs"""
    if dt.names:
        return sum(_float_bytes(dt.fields[f][0]) for f in dt.names)
    return _float_dtype(dt).itemsize + (4 if dt.kind == 'f' else 0)


def dump_outputs(out_dir, shapes, d_out, n, frames):
    """--dump-outputs: the outputs of the first n frames held in d_out (output_shapes layout), sampled to at most DUMP_BYTES, as
    out_dir/<name>.npy in float32 / float64, every value finite.  A structured output gives one file per field (kps_x,
    keylines_class_id, ...); the outputs of DUMP_ROWS keep only the valid rows.  Where an output holds NaN or inf (surface normals
    that have none), those entries are written as 0 and <name>_finite.npy is 1 where the value is finite, 0 where it is not.
    frames: the sequence index of each of the n frames (frame.npy)."""
    import torch
    per_frame = sum(int(np.prod(sh[1:])) * _float_bytes(np.dtype(dt)) for sh, dt in shapes.values()) + 8
    k = max(1, min(n, (DUMP_BYTES - (1 << 16)) // per_frame))              # 64 KB for the .npy headers
    pick = np.sort(np.random.RandomState(DUMP_SEED).choice(n, k, replace=False))
    sel = torch.from_numpy(pick).to(next(iter(d_out.values())).device)
    host = {}
    for name, (sh, dt) in shapes.items():
        rows = d_out[name].view(sh[0], -1).index_select(0, sel).cpu().numpy()
        host[name] = rows.view(dt).reshape((k,) + tuple(sh[1:]))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'frame.npy'), np.asarray(frames, np.float64)[pick])
    for name, a in host.items():
        for key, v in ({f'{name}_{f}': a[f] for f in a.dtype.names} if a.dtype.names else {name: a}).items():
            v = v.astype(_float_dtype(v.dtype))
            if name in DUMP_ROWS:
                v = v[np.arange(v.shape[1])[None, :] < host[DUMP_ROWS[name]][:, None]]
            finite = np.isfinite(v)
            if not finite.all():
                np.save(os.path.join(out_dir, key + '_finite.npy'), finite.astype(np.float32))
                v = np.where(finite, v, 0).astype(v.dtype)
            np.save(os.path.join(out_dir, key + '.npy'), v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--frames', type=int, default=C5_FRAMES, help='frames per step over all GPUs (default: the C5 sequence, 8192)')
    ap.add_argument('--batch', type=int, default=CALL_FRAMES, help='frames per library call (default 4096 = one chunk)')
    ap.add_argument('--stages', type=int, default=15, help='bit 0 ORB, 1 lines, 2 planes, 3 normals (profiling aid; the metric is 15)')
    ap.add_argument('--lanes', type=int, default=0, help='pipeline lanes of the frame handle (0 = library default)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-configs', action='store_true', help='skip the C2 / C3 / C4 sub-records')
    ap.add_argument('--device-only', action='store_true', help='profiling aid: only the device-resident loop')
    ap.add_argument('--as-shard', default='', help='profiling aid: R/W = process the range rank R of W would get (single process)')
    ap.add_argument('--e2e-only', action='store_true', help='profiling aid: skip the per-stage passes, the latency probe and the CPU baseline')
    ap.add_argument('--dump-outputs', metavar='DIR', default='',
                    help='after the timed steps, write the outputs of the last call of the last step (rank 0; a fixed, seeded sample of '
                         f'its frames, at most {DUMP_BYTES // 10 ** 6} MB) as DIR/<name>.npy in float32 / float64, to compare two builds')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours')
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup

    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import hvo_b200 as hvo
    from hvo_b200 import synth
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)')
    W, H = 640, 480
    px = W * H
    first, count = shard(args.frames, world, rank)            # this rank's contiguous range of the sequence
    if args.as_shard and world == 1:
        first, count = shard(args.frames, int(args.as_shard.split('/')[1]), int(args.as_shard.split('/')[0]))
    call = min(args.batch, count)
    # distinct synthetic frames of this rank's range (seeds 1000 + first ...): up to 1024, repeated to fill the range.  Generated
    # (forked worker pool) before this process touches CUDA or NCCL.
    n_distinct = min(count, 1024)
    gray, depth = make_frames(n_distinct, start=first)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    torch.cuda.set_device(local_rank)
    if world > 1 or os.environ.get('HVO_BENCH_FORCE_DIST'):   # (the switch: profiling aid, a process group of one)
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        os.environ.setdefault('MASTER_PORT', '29540')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank), rank=rank, world_size=world)
    reps = (count + n_distinct - 1) // n_distinct
    dev = torch.device('cuda', local_rank)
    d_gray = torch.from_numpy(gray).to(dev).repeat(reps, 1, 1)[:count].contiguous()
    d_depth = torch.from_numpy(depth.view(np.int16)).to(dev).repeat(reps, 1, 1)[:count].contiguous()
    # Two lanes of `call` frames each (the lanes share the pipelines' scratch; a lane is the input / output staging of one call in flight):
    # consecutive calls alternate lanes, so the upload of call k + 1 and the download of call k - 1 run beside the kernels of call k.
    nl = args.lanes if args.lanes > 0 else 2
    fe = hvo.FrameFrontEnd(W, H, CAM['fx'], CAM['fy'], CAM['cx'], CAM['cy'], DEPTH_FACTOR, bf=BF, n_lines=NLINES, stages=args.stages, line_cull=True,
                           lanes=nl, membership='u4', normals='n3', max_planes=MAX_PLANES, max_batch=nl * call, device=local_rank,
                           nfeatures=ORB['nfeatures'], scale_factor=ORB['scale_factor'], nlevels=ORB['nlevels'], ini_th=ORB['ini_th'], min_th=ORB['min_th'])
    # one set of device outputs for a call, reused by every call of a step (the bench keeps no results)
    shapes = fe.output_shapes(call)
    d_out = {k: torch.empty(int(np.prod(sh)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (sh, dt) in shapes.items()}
    d_ptrs = {k: v.data_ptr() for k, v in d_out.items()}
    torch.cuda.synchronize()

    fe_open = [True]

    def close_fe():
        if fe_open[0]:
            torch.cuda.synchronize()
            fe.close()
            fe_open[0] = False

    def teardown():
        # leave the device idle and release everything in a fixed order (handles before the process group)
        torch.cuda.synchronize()
        close_fe()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()

    def step_device(nfr=count):
        for off in range(0, nfr, call):
            fe.extract_batch_device(d_gray.data_ptr() + off * px, d_depth.data_ptr() + off * px * 2, min(call, nfr - off), d_ptrs)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def d_counts(name):
        return d_out[name].view(torch.int32).float().mean().item() if name in d_out else None

    # ---- value: strong scaling on the C5 sequence, inputs resident in HBM ----
    for _ in range(args.warmup):
        step_device()
    fe.sync()
    clocks = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get('HVO_BENCH_NO_CLOCKS'):  # one sampler per job (rank 0's GPU): N concurrent nvidia-smi loops would only load the driver
        clocks.start()
    time.sleep(0.25)
    barrier()
    t0 = time.time()
    if os.environ.get('HVO_BENCH_TIMELINE'):   # profiling aid: per-stream kernel start times of the timed steps (hvo_timeline_*)
        hvo.timeline(True)
    fe.timer_start()
    th0 = time.perf_counter()
    for _ in range(args.steps):
        step_device()
    host_enqueue_ms = 1e3 * (time.perf_counter() - th0) / args.steps   # host time to queue one step (the device runs behind)
    ms = fe.timer_stop()
    if os.environ.get('HVO_BENCH_TIMELINE'):
        by = {}
        for t, s_, n_ in hvo.timeline_dump():
            by.setdefault(s_, []).append((t, n_))
        hvo.timeline(False)
        with open(os.path.join(ROOT, 'gpurun_out', f'timeline_rank{rank}.txt'), 'w') as fh:
            fh.write(f'rank {rank}/{world}: {ms / args.steps:.2f} ms/step\n')
            for s_ in sorted(by):
                fh.write(f'stream {s_}: ' + '  '.join(f'{n_}@{t:.1f}' for t, n_ in by[s_]) + '\n')
    t1 = time.time()
    barrier()
    clk = clocks.stop(t0, t1)
    ms_rank = ms
    ms = max_over_ranks(ms)
    calls_per_step = (count + call - 1) // call
    launches_per_step = fe.last_launches() * calls_per_step
    value = args.frames * args.steps / (ms * 1e-3)
    means = dict(keypoints=d_counts('kp_counts'), lines=d_counts('line_counts'), planes=d_counts('n_planes'))
    if args.dump_outputs and rank == 0:
        last = (count - 1) // call * call                     # d_out holds what the last call of the step wrote: frames last .. count - 1
        dump_outputs(args.dump_outputs, shapes, d_out, count - last, np.arange(first + last, first + count))

    if args.device_only:
        emit({'metric': METRIC, 'value': value, 'unit': 'frames/s', 'ms_per_step': ms / args.steps, 'rank': rank, 'ms_per_step_this_rank': ms_rank / args.steps, 'host_enqueue_ms_per_step': host_enqueue_ms, 'device_only': True, 'frames_per_step': args.frames,
              'stages': args.stages, 'lanes': fe.lanes, 'chunk': fe.chunk, 'means': means})
        teardown()
        return

    # ---- weak scaling (the round-1 line): every GPU processes one call of 2368 frames per step ----
    wn = min(call, count)
    for _ in range(2):
        step_device(wn)
    barrier()
    fe.timer_start()
    for _ in range(5):
        step_device(wn)
    weak_ms = max_over_ranks(fe.timer_stop())
    barrier()
    weak = dict(value=world * wn * 5 / (weak_ms * 1e-3), unit='frames/s', frames_per_gpu_per_step=wn, steps=5, ms_per_step=weak_ms / 5, scaling='weak')

    roofline = None
    if not args.e2e_only:
        # ---- per-stage device times: every pipeline alone at the chunk size the frame handle runs (standalone handles) ----
        Bs = min(count, call)
        stage_ms, kern_ms = {}, {}
        ex = hvo.ORBextractor(ORB['nfeatures'], ORB['scale_factor'], ORB['nlevels'], ORB['ini_th'], ORB['min_th'], width=W, height=H,
                              max_batch=Bs, device=local_rank)
        kp = d_ptrs

        def orb_step():
            ex.extract_batch_device(d_gray.data_ptr(), Bs, kp['kps'], kp['desc'], kp['kp_counts'], d_depth.data_ptr(), DEPTH_FACTOR, BF,
                                    kp['kp_depth'], kp['kp_uright'])
        for _ in range(2):
            orb_step()
        ex.sync()
        ex.timer_start()
        for _ in range(5):
            orb_step()
        stage_ms['orb'] = ex.timer_stop() / 5
        ex.set_profiling(True)
        acc = {}
        for _ in range(5):
            orb_step()
            ex.sync()
            for k, v in ex.stage_times().items():
                acc[k] = acc.get(k, 0.0) + v / 5
        ex.close()
        kern_ms.update({'k_resize x7': acc['pyramid'], 'k_fast_strips': acc['fast'], 'k_octree': acc['octree'], 'k_describe': acc['describe']})

        le = hvo.LINEextractor(1, 1.2, NLINES, 0.125, width=W, height=H, max_batch=Bs, device=local_rank)
        le.set_culling(True)

        def line_step():
            le.extract_batch_device(d_gray.data_ptr(), Bs, kp['keylines'], kp['line_desc'], kp['linevec3'], kp['line_counts'])
        line_step()
        le.sync()
        le.timer_start()
        for _ in range(3):
            line_step()
        stage_ms['lines'] = le.timer_stop() / 3
        le.set_profiling(True)
        line_step()
        le.sync()
        lt = le.stage_times()
        le.close()
        kern_ms.update({'k_lsd_prep': lt['prep'], 'k_lsd_order': lt['order'], 'k_lsd_grow': lt['grow'], 'k_line_keylines + k_line_cull + k_lbd_*': lt['keylines_lbd']})

        pd = hvo.PlaneDetection(W, H, max_batch=Bs, device=local_rank)
        pd.readDepthImage(depth[0], np.array([[CAM['fx'], 0, CAM['cx']], [0, CAM['fy'], CAM['cy']], [0, 0, 1]], np.float32), np.float32(DEPTH_FACTOR))

        def plane_step():
            pd.detect_batch_device(d_depth.data_ptr(), Bs, kp['n_planes'], kp['planes7'], fe.max_planes, kp['membership'])
        plane_step()
        pd.sync()
        pd.timer_start()
        for _ in range(3):
            plane_step()
        stage_ms['planes'] = pd.timer_stop() / 3
        pd.timer_start()
        for _ in range(5):
            pd.blocks_device(d_depth.data_ptr(), Bs)
        kern_ms['k_plane_blocks'] = pd.timer_stop() / 5
        cyc = pd.phase_cycles(0)
        rest = stage_ms['planes'] - kern_ms['k_plane_blocks']
        # split of the ordered chain by its own cycle counters (frame 0) x the waves each kernel needs for Bs frames: k_plane_cluster keeps
        # 16 frames resident per SM (one warp each, 128 registers), k_plane_flood 4 (one CTA of 256 each), the last merge 16; the ncu launch
        # list of the same chunk (profiles/r2b_launch_summary.txt) gives the same split
        waves = lambda per_sm: -(-Bs // (per_sm * 148))
        wc = dict(cluster=cyc.get('cluster', 0) * waves(16), flood=(cyc.get('seeds', 0) + cyc.get('flood', 0)) * waves(4),
                  merge=cyc.get('merge_relabel', 0) * waves(16))
        tot_c = float(sum(wc.values())) or 1.0
        kern_ms['k_plane_cluster'] = rest * wc['cluster'] / tot_c
        kern_ms['k_plane_flood'] = rest * wc['flood'] / tot_c
        kern_ms['k_plane_merge + k_plane_relabel'] = rest * wc['merge'] / tot_c
        pd.close()

        sn = hvo.SurfaceNormals(W, H, CAM['fx'], CAM['fy'], CAM['cx'], CAM['cy'], DEPTH_FACTOR, max_batch=Bs, device=local_rank)
        sn.compute_device(d_depth.data_ptr(), Bs, kp['normals8'])
        sn.sync()
        sn.timer_start()
        for _ in range(5):
            sn.compute_device(d_depth.data_ptr(), Bs, kp['normals8'])
        stage_ms['normals'] = sn.timer_stop() / 5
        kern_ms['k_sn_* x5'] = stage_ms['normals']
        sn.close()

        # roofline: the HBM-bound (stencil / streaming) kernels against the measured copy bandwidth; beside it the step as a whole and the
        # kernel that really dominates it (an ordered graph kernel: latency-bound by construction, no bandwidth roofline applies)
        peak, peak_src = measured_peak()
        dom = max(ALG_BYTES, key=lambda k: kern_ms[k])
        achieved = ALG_BYTES[dom] * Bs / (kern_ms[dom] * 1e-3) / 1e9
        serial_sum = sum(kern_ms.values())
        top = max(kern_ms, key=lambda k: kern_ms[k])
        step_gbs = ALG_BYTES_FRAME * count / ((ms / args.steps) * 1e-3) / 1e9
        roofline = dict(bound='hbm', kernel=dom, achieved=achieved, peak=peak, unit='GB/s', frac=achieved / peak,
                        traffic=NCU_DRAM_BYTES[dom] * Bs, traffic_source='ncu dram__bytes_read.sum + dram__bytes_write.sum per frame (profiles/'
                        'r2b_ncu_full_orb_kernels_b296.csv) x frames per launch',
                        peak_source=peak_src, algorithmic_bytes_per_launch=ALG_BYTES[dom] * Bs, batch=Bs,
                        kernel_ms={k: round(v, 4) for k, v in kern_ms.items()},
                        frac_of_hbm={k: round(ALG_BYTES[k] * Bs / (kern_ms[k] * 1e-3) / 1e9 / peak, 4) for k in ALG_BYTES},
                        stage_ms_alone={k: round(v, 3) for k, v in stage_ms.items()},
                        step_frac=step_gbs / peak, step_achieved_gbs=step_gbs, step_algorithmic_bytes_per_frame=ALG_BYTES_FRAME,
                        dominant_kernel=dict(name=top, ms=round(kern_ms[top], 3), share_of_serialised_kernels=round(kern_ms[top] / serial_sum, 3),
                                             note='the step is dominated by the ordered graph kernels (k_lsd_grow, k_plane_cluster, k_plane_flood): the '
                                                  'reference sequential algorithms, one warp / CTA per frame, latency-bound; their throughput comes from the '
                                                  'frames in flight, not from bandwidth'),
                        serialised_kernel_ms_per_chunk=round(serial_sum, 2))

    # ---- e2e: host (pinned) buffers through the C-ABI call, copies inside the timed region ----
    def pinned(shape, dtype):
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        t = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        return t.numpy().view(dtype).reshape(shape)
    h_gray = pinned((call, H, W), np.uint8)
    h_depth = pinned((call, H, W), np.uint16)
    rep = (call + n_distinct - 1) // n_distinct
    h_gray[:] = np.concatenate([gray] * rep)[:call]
    h_depth[:] = np.concatenate([depth] * rep)[:call]
    # two sets of pinned output buffers, used alternately: call k+1 is queued (hvo_frame_extract_batch_async) while call k still
    # runs, so its uploads overlap the tail of call k; the timer stops after every download has landed
    outs = [{k: pinned(sh, dt) for k, (sh, dt) in fe.output_shapes(call, device=False).items()} for _ in range(2)]

    def step_host(wait):
        for i, off in enumerate(range(0, count, call)):
            n = min(call, count - off)
            o = outs[i % 2] if n == call else {k: v[:n] for k, v in outs[i % 2].items()}
            fe.extract_batch(h_gray[:n], h_depth[:n], out=o, wait=wait)
    step_host(True)
    barrier()
    e2e_steps = max(3, args.steps // 2)
    fe.timer_start()
    for i in range(e2e_steps):
        step_host(False)
    e2e_ms = max_over_ranks(fe.timer_stop())
    barrier()
    # the same with blocking calls (what a caller without double buffering sees)
    fe.timer_start()
    for i in range(2):
        step_host(True)
    e2e_blocking_ms = max_over_ranks(fe.timer_stop())
    barrier()
    out_bytes_frame = sum(v.nbytes for v in outs[0].values()) // call
    e2e = dict(value=args.frames * e2e_steps / (e2e_ms * 1e-3), unit='frames/s',
               h2d_bytes_per_step=int(count * px * 3), d2h_bytes_per_step=int(count * out_bytes_frame), d2h_bytes_per_frame=int(out_bytes_frame),
               bytes_are='per GPU', host_cpus=(f'{len(numa)} CPUs local to the GPU (NVML affinity)' if numa else 'unbound'), ms_per_step=e2e_ms / e2e_steps, steps=e2e_steps,
               call=f'hvo_frame_extract_batch_async per {call} frames + hvo_frame_timer_stop (pinned host buffers, two output sets alternating; outputs: '
                    'keypoints, descriptors, depth / uRight, keylines, LBD, line functions, planes, 4-bit plane labels, surface normals)',
               blocking_calls_value=args.frames * 2 / (e2e_blocking_ms * 1e-3))

    if args.e2e_only:
        if rank == 0:
            emit({'metric': METRIC, 'value': value, 'ms_per_step': ms / args.steps, 'e2e': e2e, 'weak': weak, 'lanes': fe.lanes, 'chunk': fe.chunk})
        teardown()
        return

    # ---- single-frame latency through the host call (p50) ----
    fe1 = hvo.FrameFrontEnd(W, H, CAM['fx'], CAM['fy'], CAM['cx'], CAM['cy'], DEPTH_FACTOR, bf=BF, n_lines=NLINES, stages=args.stages, line_cull=True,
                            max_batch=1, device=local_rank, max_planes=MAX_PLANES, membership='u4', normals='n3')
    out1 = fe1.alloc_host(1)
    lat = []
    for i in range(24):
        t = time.perf_counter()
        fe1.extract_batch(gray[i % n_distinct][None], depth[i % n_distinct][None], out=out1)
        lat.append(1e3 * (time.perf_counter() - t))
    p50 = float(np.median(lat[4:]))
    fe1.close()

    # ---- the other BASELINE.json configs (rank 0): device-resident throughput of C2 / C3, matching stress C4 ----
    fe_lanes, fe_chunk = fe.lanes, fe.chunk
    close_fe()                       # the C5 handle and its buffers make room for the C2 / C3 handles
    del d_gray, d_depth, d_out
    torch.cuda.empty_cache()
    configs = None
    if rank == 0 and not args.no_configs:
        configs = {}
        for name, cfg, w2, h2, nfeat, nb in (('C2', 'S2', 640, 480, 1000, 4096), ('C3', 'S3', 1280, 720, 2000, 2048)):
            c = synth.CONFIGS[cfg]
            g2, dp2 = make_frames(64, cfg=cfg)
            fe2 = hvo.FrameFrontEnd(w2, h2, c['fx'], c['fy'], c['cx'], c['cy'], 1.0 / c['factor'], bf=BF, n_lines=NLINES, line_cull=True, lanes=1,
                                    membership='u4', normals='n3', max_planes=MAX_PLANES, max_batch=nb, device=local_rank, nfeatures=nfeat)
            r2 = (nb + 63) // 64
            dg = torch.from_numpy(g2).to(dev).repeat(r2, 1, 1)[:nb].contiguous()
            dd = torch.from_numpy(dp2.view(np.int16)).to(dev).repeat(r2, 1, 1)[:nb].contiguous()
            sh2 = fe2.output_shapes(nb)
            do = {k: torch.empty(int(np.prod(s_)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s_, dt) in sh2.items()}
            dp = {k: v.data_ptr() for k, v in do.items()}
            for _ in range(2):
                fe2.extract_batch_device(dg.data_ptr(), dd.data_ptr(), nb, dp)
            fe2.sync()
            fe2.timer_start()
            for _ in range(3):
                fe2.extract_batch_device(dg.data_ptr(), dd.data_ptr(), nb, dp)
            m2 = fe2.timer_stop() / 3
            configs[name] = dict(workload=f'{cfg}: {w2}x{h2}, {nfeat} ORB features, whole front-end, {nb} frames per step (64 distinct), device-resident',
                                 value=nb / m2 * 1e3, unit='frames/s', ms_per_step=m2,
                                 mean_per_frame=dict(keypoints=do['kp_counts'].view(torch.int32).float().mean().item(),
                                                     lines=do['line_counts'].view(torch.int32).float().mean().item(),
                                                     planes=do['n_planes'].view(torch.int32).float().mean().item()))
            fe2.close()
            del dg, dd, do
        bfm = hvo.BFMatcherHamming(local_rank)
        c4 = {}
        for name, nq, nt, seed in (('orb_2000x50000', 2000, 50000, 4), ('lbd_200x5000', 200, 5000, 5)):
            q, t = synth.descriptors_S4(nq=nq, nt=nt, seed=seed)
            dq, dt_ = torch.from_numpy(q).to(dev), torch.from_numpy(t).to(dev)
            di = torch.empty((nq, 2), dtype=torch.int32, device=dev); dd_ = torch.empty((nq, 2), dtype=torch.int32, device=dev)
            for _ in range(3):
                bfm.knn2_device(dq.data_ptr(), nq, dt_.data_ptr(), nt, di.data_ptr(), dd_.data_ptr())
            bfm.sync()
            bfm.timer_start()
            for _ in range(50):
                bfm.knn2_device(dq.data_ptr(), nq, dt_.data_ptr(), nt, di.data_ptr(), dd_.data_ptr())
            mm = bfm.timer_stop() / 50
            peak_popc = 148 * 16 * (clk.get('sm_mhz') or 1965.0) * 1e6           # 16 POPC lanes per SM per clock (XU pipe)
            r = dict(ms=mm, pairs_per_s=nq * nt / mm * 1e3, popc32_per_s=nq * nt * 8 / mm * 1e3, xu_pipe_frac=nq * nt * 8 / (mm * 1e-3) / peak_popc)
            t0c = time.perf_counter()
            idx, _ = bfm.knnMatch2(q, t)
            r['host_call_ms'] = 1e3 * (time.perf_counter() - t0c)
            try:
                import cv2
                t0c = time.perf_counter()
                cvm = cv2.BFMatcher(cv2.NORM_HAMMING, False).knnMatch(q, t, k=2)
                r['cv2_bfmatcher_ms'] = 1e3 * (time.perf_counter() - t0c)
                r['cv2_threads'] = cv2.getNumThreads()
                r['same_as_cv2'] = bool(np.array_equal(idx, np.array([[a.trainIdx, b.trainIdx] for a, b in cvm], np.int32)))
            except ImportError:
                pass
            c4[name] = r
        bfm.close()
        configs['C4'] = dict(workload='matching stress: brute-force Hamming knn-2 + ratio test inputs, device-resident', **c4)

        # ---- tracking-time path (host call, host buffers in / out): Tracking::SearchLocalPoints as one call (isInFrustum over the local map +
        #      SearchByProjection) for a 2000-keypoint frame against 10^4 / 5 x 10^4 map points, and Frame::ComputeBoW on a synthetic k = 10, L = 6
        #      vocabulary (10^6 words, random descriptors: the reference's ORBvoc.bin is not in the tree) ----
        try:
            rng = np.random.RandomState(7)
            nk = 2000
            keys = np.zeros(nk, hvo.KP_DTYPE)
            keys['x'] = rng.uniform(20, W - 20, nk); keys['y'] = rng.uniform(20, H - 20, nk); keys['octave'] = rng.randint(0, 8, nk)
            kdesc = rng.randint(0, 256, (nk, 32)).astype(np.uint8)
            sf = (np.float32(1.2) ** np.arange(8, dtype=np.float32)).astype(np.float32)
            cam = hvo.frustum_cam(np.eye(3, dtype=np.float32), np.zeros(3, np.float32), CAM['fx'], CAM['fy'], CAM['cx'], CAM['cy'], 40.0, (0.0, 0.0, float(W), float(H)))
            pmh = hvo.ProjectionMatcher(local_rank)
            pmh.set_frame(keys, None, kdesc, 0.0, 0.0, float(W), float(H))
            track = {}
            for M in (10000, 50000):
                z = rng.uniform(0.5, 6.0, M)
                src = rng.randint(0, nk, M)
                pts = np.zeros(M, hvo.MAP_POINT_DTYPE)
                u = keys['x'][src] + rng.normal(0, 1.5, M); v = keys['y'][src] + rng.normal(0, 1.5, M)
                pts['pos'] = np.stack([(u - CAM['cx']) * z / CAM['fx'], (v - CAM['cy']) * z / CAM['fy'], z], 1).astype(np.float32)
                nrm = -pts['pos'] / np.linalg.norm(pts['pos'], axis=1)[:, None]
                pts['normal'] = -nrm
                d = np.linalg.norm(pts['pos'], axis=1)
                pts['max_distance'] = (d * sf[keys['octave'][src]]).astype(np.float32); pts['min_distance'] = pts['max_distance'] / sf[7]
                pdesc = kdesc[src].copy()
                flip = rng.randint(0, 256, M)
                pdesc[np.arange(M), flip // 8] ^= (1 << (flip % 8)).astype(np.uint8)
                for _ in range(2):
                    res = pmh.search_local_map(cam, pts, pdesc, sf, th=3.0, th_dist=100, nnratio=0.8)
                t0c = time.perf_counter()
                for _ in range(5):
                    res = pmh.search_local_map(cam, pts, pdesc, sf, th=3.0, th_dist=100, nnratio=0.8)
                ms_c = 1e3 * (time.perf_counter() - t0c) / 5
                track[f'search_local_points_{M}'] = dict(host_call_ms=ms_c, map_points_per_s=M / ms_c * 1e3, in_view=int(res[3]), matches=int(res[4]),
                                                         rounds=int(pmh.rounds()))
            pmh.close()
            kk, LL = 10, 6
            nn = (kk ** (LL + 1) - 1) // (kk - 1)
            first_leaf = (kk ** LL - 1) // (kk - 1)
            child_start = np.minimum(np.arange(nn + 1, dtype=np.int64) * kk, (first_leaf) * kk).astype(np.int32)
            child_ids = np.arange(1, first_leaf * kk + 1, dtype=np.int32)
            voc = dict(child_start=child_start, child_ids=child_ids, node_desc=rng.randint(0, 256, (nn, 32)).astype(np.uint8),
                       node_weight=np.where(np.arange(nn) >= first_leaf, rng.uniform(0.5, 8.0, nn), 0.0),
                       node_word=np.where(np.arange(nn) >= first_leaf, np.arange(nn) - first_leaf, -1).astype(np.int32), L=LL)
            vv = hvo.ORBVocabulary(voc, local_rank)
            frames_d = [rng.randint(0, 256, (1000, 32)).astype(np.uint8) for _ in range(64)]
            for _ in range(2):
                vv.transform_batch(frames_d, 4)
            t0c = time.perf_counter()
            for _ in range(3):
                vv.transform_batch(frames_d, 4)
            ms_c = 1e3 * (time.perf_counter() - t0c) / 3
            vv.close()
            track['compute_bow_64x1000'] = dict(host_call_ms=ms_c, frames_per_s=64 / ms_c * 1e3, vocabulary=f'synthetic k={kk} L={LL}, {nn - first_leaf} words')
            configs['track'] = dict(workload='tracking-time path through the C ABI with host buffers, wall clock around the mirror call (uploads, downloads and the '
                                             'Python-side unpacking included): isInFrustum + SearchByProjection over a local map; ComputeBoW', **track)
        except Exception as e:   # a profiling extra must never take the bench line down
            configs['track'] = dict(error=repr(e))

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(gray, depth)
        cpu['latency_ms'] = cpu_latency(gray, depth)

    if rank == 0:
        emit({
            'metric': METRIC, 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'u8',
            'data': 'synthetic',
            'config': {'workload': f'C5/C1: {args.frames} synthetic TUM-fr3-shaped 640x480 RGB-D frames per step (TUM3.yaml: ORB 1000 features 8 levels x1.2, '
                                   f'LINE 200), whole front-end of Frame::Frame, frame-sharded over {world} GPU(s) in contiguous ranges: {count} frames per GPU '
                                   f'per step ({n_distinct} distinct per GPU), {calls_per_step} call(s) of <= {call} frames',
                       'stages': STAGES, 'frames_per_step': args.frames, 'frames_per_gpu': count, 'frames_per_call': call, 'lanes': fe_lanes,
                       'chunk_frames': fe_chunk, 'schedule': 'pipelines one after the other (planes, lines, ORB, normals)' if min(call, count) >= 2048 else 'pipelines side by side',
                       'mean_per_frame': means,
                       'outputs': 'keypoints + descriptors + depth/uRight, keylines + LBD + line functions, planes + plane labels, surface normals',
                       'l2': f'inputs larger than L2: per-step inputs {count} x 0.92 MB and working set ~{min(count, call)} x 17 MB >> 126 MB'},
            'roofline': roofline, 'cpu_baseline': cpu, 'e2e': e2e, 'weak': weak, 'configs': configs, 'gpu_launches': launches_per_step * args.steps,
            'gpu_launches_per_step': launches_per_step, 'clocks': clk, 'p50_latency_ms_single_frame': p50,
        })
    teardown()


if __name__ == '__main__':
    main()
