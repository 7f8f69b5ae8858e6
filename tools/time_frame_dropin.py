"""Single-frame latency of the frame drop-in hvo_shim::FrameExtractorGPU::extract (shim/FrameExtractorGPU.h), in one process per image
size (tests/cpp/shim_frame_main.cpp with a repetition count):

  extract     host clock around FrameExtractorGPU::extract into a fresh stand-in Frame: the blocking frame call plus the host fill
  fill        the host part of extract alone (FrameExtractorGPU::lastFillSeconds: normals3 expansion, plane members and their cloud
              points, grids, BoW maps, LPVO rows, keypoint / line copies)
  call        host clock around the bare blocking hvo_frame_extract_batch_lpvo of the same frame, with the same outputs, on the same handle

The two calls alternate, --reps times after --warmup pairs, at 640x480 (synthetic S1) and 1280x720 (S3), every stage with cullingLine,
a vocabulary attached and LPVO rows requested.  Prints one JSON object (and writes it to --out) with the card name and power limit read
in the same run."""
import argparse
import json
import os
import pathlib
import struct
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from hvo_b200 import synth  # noqa: E402
import test_frame_dropin as tfd  # noqa: E402

CASES = (('640x480', 'S1', 0), ('1280x720', 'S3', 1))


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else q.stderr.strip()


def pct(v):
    v = np.asarray(v) * 1e3
    return {f'p{p}': round(float(np.percentile(v, p)), 3) for p in (10, 50, 90)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    tmp = pathlib.Path(tempfile.mkdtemp())
    exe = tfd.build_driver(str(tmp / 'shim_frame'))
    voc = tfd._vocabulary()
    res = dict(card=card(), reps=a.reps, warmup=a.warmup, clock='host steady_clock, ms', sizes={})
    for name, cfg, idx in CASES:
        c = synth.CONFIGS[cfg]
        g, d = synth.frame(cfg, idx)
        raw, _ = tfd._run(exe, tmp, g[None], d[None], tfd._cam(c), bf=c['bf'], nfeatures=c['nfeatures'], lpvo=True, vocabulary=voc,
                          reps=a.warmup + a.reps)
        n = struct.unpack_from('<i', raw, 0)[0]
        t = np.frombuffer(raw, '<f8', 3 * n, 4).reshape(3, n)[:, a.warmup:]
        res['sizes'][name] = dict(config=cfg, nfeatures=c['nfeatures'], extract=pct(t[0]), fill=pct(t[1]), call=pct(t[2]),
                                  extract_minus_call_p50=round(float(np.median(t[0] - t[2])) * 1e3, 3))
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, 'w').write(s + '\n')


if __name__ == '__main__':
    main()
