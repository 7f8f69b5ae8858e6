"""Cost of the bag-of-words stage (Frame::ComputeBoW on the device, k_bow_descend + k_bow_frame) in the whole front-end, in one process:

  step      the C5-shaped step (one device-resident call of --call S1 frames, every stage, cullingLine, 4-bit labels / normals-only as
            bench.py runs it, one lane) without and with a full-size synthetic vocabulary (K = 10, L = 6: 1 111 111 nodes, random node
            descriptors, seeded), alternated over --rounds rounds, --steps timed steps each after --warmup; CUDA events on the frame
            handle's master stream
  kernels   the BoW kernels of one more step with the vocabulary (after the timed ones), from torch.profiler (CUDA activity)
  transform hvo_bow_transform of the same descriptors (the valid rows of every frame, concatenated) including their upload and the
            download of its results, host clock around the blocking call; its results are compared with the frame handle's
  oracle    the CPU oracle's transform (oracle.bow_transform: DBoW2's algorithm, one frame at a time) per frame, the baseline
  latency   one frame per blocking host call (hvo_frame_extract_batch), without and with the vocabulary alternated, median of --lat-calls
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
import oracle  # noqa: E402
from bench import BF, CAM, DEPTH_FACTOR, MAX_PLANES, NLINES, ORB, make_frames  # noqa: E402

LEVELSUP = 4   # Frame::ComputeBoW


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.returncode == 0 else q.stderr.strip())


def full_vocabulary(k=10, levels=6, seed=10):
    """A complete k-ary tree of `levels` levels in DBoW2's node order (the children of node i are k*i+1 .. k*i+k), random node
    descriptors, positive random leaf weights (idf-like)."""
    n = (k ** (levels + 1) - 1) // (k - 1)
    inner = (k ** levels - 1) // (k - 1)
    rng = np.random.default_rng(seed)
    nch = np.zeros(n, np.int32)
    nch[:inner] = k
    desc = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    desc[0] = 0
    weight = np.zeros(n)
    weight[inner:] = rng.uniform(0.5, 3.0, n - inner)
    word = np.full(n, -1, np.int32)
    word[inner:] = np.arange(n - inner, dtype=np.int32)
    return dict(child_start=np.concatenate([[0], np.cumsum(nch)]).astype(np.int32), child_ids=np.arange(1, n, dtype=np.int32), node_desc=desc,
                node_weight=weight, node_word=word, L=levels)


def frontend(max_batch, voc, **kw):
    return hvo.FrameFrontEnd(640, 480, CAM['fx'], CAM['fy'], CAM['cx'], CAM['cy'], DEPTH_FACTOR, bf=BF, n_lines=NLINES, line_cull=True,
                             membership='u4', normals='n3', max_planes=MAX_PLANES, max_batch=max_batch, nfeatures=ORB['nfeatures'],
                             scale_factor=ORB['scale_factor'], nlevels=ORB['nlevels'], ini_th=ORB['ini_th'], min_th=ORB['min_th'], vocabulary=voc,
                             levelsup=LEVELSUP, **kw)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--call', type=int, default=4096)
    ap.add_argument('--distinct', type=int, default=256)
    ap.add_argument('--rounds', type=int, default=4)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--oracle-frames', type=int, default=16)
    ap.add_argument('--lat-calls', type=int, default=60)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    n = a.call
    voc = full_vocabulary()
    gray, depth = make_frames(a.distinct)
    reps = (n + len(gray) - 1) // len(gray)
    dev = torch.device('cuda', 0)
    d_gray = torch.from_numpy(gray).to(dev).repeat(reps, 1, 1)[:n].contiguous()
    d_depth = torch.from_numpy(depth.view(np.int16)).to(dev).repeat(reps, 1, 1)[:n].contiguous()
    res = dict(card=card(), call_frames=n, distinct_frames=a.distinct, rounds=a.rounds, steps_per_round=a.steps,
               vocabulary=dict(K=10, L=6, nodes=len(voc['node_weight']), node_desc_MB=voc['node_desc'].nbytes / 1e6, levelsup=LEVELSUP),
               step_ms={'plain': [], 'bow': []})

    # ---- whole-front-end step, with and without the vocabulary, alternated; one handle at a time (each holds the scratch of 4096 frames);
    # the last round also profiles one step with the vocabulary (the BoW kernels)
    bufs = {}
    order = ['plain', 'bow']
    kern = {}
    for r in range(a.rounds):
        for name in order[r % 2:] + order[:r % 2]:
            fe = frontend(n, voc if name == 'bow' else None, lanes=1)
            if name not in bufs:
                shapes = fe.output_shapes(n)
                d_out = {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
                bufs[name] = (d_out, {k: v.data_ptr() for k, v in d_out.items()}, shapes)
            ptrs = bufs[name][1]
            torch.cuda.synchronize()
            for _ in range(a.warmup):
                fe.extract_batch_device(d_gray.data_ptr(), d_depth.data_ptr(), n, ptrs)
            fe.sync()
            fe.timer_start()
            for _ in range(a.steps):
                fe.extract_batch_device(d_gray.data_ptr(), d_depth.data_ptr(), n, ptrs)
            res['step_ms'][name].append(fe.timer_stop() / a.steps)
            res.setdefault('launches_per_step', {})[name] = fe.last_launches()
            if name == 'bow' and r == a.rounds - 1:
                from torch.profiler import ProfilerActivity, profile
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    fe.extract_batch_device(d_gray.data_ptr(), d_depth.data_ptr(), n, ptrs)
                    fe.sync()
                for e in prof.key_averages():
                    if 'k_bow' in e.key:
                        t = getattr(e, 'device_time_total', None)
                        kern[e.key] = (t if t is not None else e.cuda_time_total) / 1e3
            fe.close()
            torch.cuda.synchronize()
    for name in order:
        v = res['step_ms'][name]
        res[f'{name}_step_ms_median'] = float(np.median(v))
        res[f'{name}_frames_per_s'] = n / (float(np.median(v)) / 1e3)
    res['bow_minus_plain_step_ms'] = res['bow_step_ms_median'] - res['plain_step_ms_median']
    res['bow_over_plain_percent'] = 100.0 * res['bow_minus_plain_step_ms'] / res['plain_step_ms_median']
    res['bow_kernels_ms_per_step'] = kern
    res['bow_kernels_ms_total'] = float(sum(kern.values()))

    # ---- outputs of the last step: hvo_bow_transform of the same descriptors, and the CPU oracle
    d_out, _, shapes = bufs['bow']
    host = {k: d_out[k].cpu().numpy().view(shapes[k][1]).reshape(shapes[k][0]) for k in ('kp_counts', 'desc') + tuple(hvo.FrameFrontEnd.BOW_FIELDS)}
    del bufs, d_out
    torch.cuda.empty_cache()
    counts = host['kp_counts'].astype(np.int64)
    cap = host['desc'].shape[1]
    valid = np.arange(cap)[None, :] < counts[:, None]
    desc = np.ascontiguousarray(host['desc'][valid])
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    total = int(off[-1])
    bt = hvo.ORBVocabulary(voc)
    word = np.empty(total, np.int32); node = np.empty(total, np.int32); bw = np.empty(total, np.int32); bv = np.empty(total, np.float64)
    fo = np.empty(total, np.int32); bc = np.empty(n, np.int32); fc = np.empty(n, np.int32)

    def transform():
        hvo._check(hvo.lib().hvo_bow_transform(bt._h, hvo._np_ptr(desc), hvo._np_ptr(off), n, LEVELSUP, hvo._np_ptr(word), hvo._np_ptr(node),
                                               hvo._np_ptr(bc), hvo._np_ptr(bw), hvo._np_ptr(bv), hvo._np_ptr(fo), hvo._np_ptr(fc)))
    transform()
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        transform()
        ts.append(1e3 * (time.perf_counter() - t0))
    same = bool(np.array_equal(bc, host['bow_counts']) and np.array_equal(fc, host['fv_counts']) and np.array_equal(word, host['word_of'][valid])
                and np.array_equal(node, host['node_of'][valid]))
    for f in range(n):
        a0, w = int(off[f]), int(bc[f])
        same = same and bw[a0:a0 + w].tobytes() == host['bow_words'][f, :w].tobytes() and bv[a0:a0 + w].tobytes() == host['bow_values'][f, :w].tobytes() \
            and fo[a0:a0 + int(fc[f])].tobytes() == host['fv_order'][f, :int(fc[f])].tobytes()
    bt.close()
    res['hvo_bow_transform'] = dict(ms_median=float(np.median(ts)), ms_all=ts, descriptors=total, pageable_host_arrays=True,
                                    same_as_frame_handle=same, note='one blocking call: descriptor upload, both kernels, downloads of every output')
    ot = []
    for f in range(a.oracle_frames):
        d = host['desc'][f, :int(counts[f])]
        t0 = time.perf_counter()
        o = oracle.bow_transform(voc, d, LEVELSUP)
        ot.append(1e3 * (time.perf_counter() - t0))
        assert np.array_equal(o[0][0], host['bow_words'][f, :len(o[0][0])]) and o[0][1].tobytes() == host['bow_values'][f, :len(o[0][1])].tobytes()
    res['cpu_oracle'] = dict(ms_per_frame_median=float(np.median(ot)), frames=a.oracle_frames, descriptors_per_frame_mean=float(counts[:a.oracle_frames].mean()),
                             same_as_frame_handle=True, note='oracle.bow_transform, one CPU thread, includes its ctypes call overhead')

    # ---- single-frame latency, host arrays, both handles alternated
    lat = {'plain': [], 'bow': []}
    fes = {'plain': frontend(1, None), 'bow': frontend(1, voc)}
    g1, dp1 = np.ascontiguousarray(gray[:1]), np.ascontiguousarray(depth[:1])
    outs = {name: fe.alloc_host(1) for name, fe in fes.items()}
    for name, fe in fes.items():
        for _ in range(5):
            fe.extract_batch(g1, dp1, out=outs[name])
    for i in range(a.lat_calls):
        for name in order[i % 2:] + order[:i % 2]:
            t0 = time.perf_counter()
            fes[name].extract_batch(g1, dp1, out=outs[name])
            lat[name].append(1e3 * (time.perf_counter() - t0))
    for fe in fes.values():
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
