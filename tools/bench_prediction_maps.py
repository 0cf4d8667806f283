#!/usr/bin/env python3
"""python tools/bench_prediction_maps.py [--reps R] [--warmup W] [--no-files] [--out FILE]

The prediction maps (``ops.volumes_to_grid``, ``CryoEMPredictor(save_maps=)``) on one GPU.

(a) Kernel: random probability volumes in cube space (standard axis order) resampled to a target grid, CUDA-event time
    per launch, median over R repetitions after W warm-ups, for
      1.2A      bench.py's map: a 400^3 input at 1.2 A, so 480^3 working -> 400^3 ('input');
      identity  480^3 -> 480^3 (a 1 A input, or 'working');
      0.83A     a 578^3 input at 0.83 A: 480^3 working -> 578^3.
    Algorithmic bytes: 88 N_w read (22 channels; the stitched label is not read) + 92 N_s written (23 channels), over
    kernel time, against a device-to-device copy (torch copy_ of 4 GiB, read + write bytes) timed the same way in this
    run.  Every working set is larger than L2 (126 MB).
(b) The whole map writing of ``save_maps='input'`` at 1.2A (``CryoEMPredictor._write_maps``: kernel, device-to-host
    copies one kind at a time, 23 MRC files into a temporary directory), wall seconds split as the predictor records
    them.  Skipped with --no-files.
Prints one JSON line that names the card and its power limit."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from mica_b200 import ops
from mica_b200.pipeline import MapHeader
from mica_b200.predict import CryoEMPredictor

PERM = ops.STANDARD_PERM
CASES = {'1.2A': ((480,) * 3, (400,) * 3), 'identity': ((480,) * 3, (480,) * 3), '0.83A': ((480,) * 3, (578,) * 3)}


def _card(index):
    name = torch.cuda.get_device_name(index)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i',
                            str(index)], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unknown'
    return name, q


def _time(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def _volumes(working, dev):
    cube = ops.cube_space_shape(working, PERM)
    sv = ops.StitchedVolumes(cube, dev)
    g = torch.Generator(device=dev).manual_seed(2022)
    for k, v in sv.as_dict().items():
        v.uniform_(generator=g)
    return sv


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--no-files', action='store_true')
    ap.add_argument('--out')
    a = ap.parse_args()
    ops.require_gpu()
    dev = torch.device('cuda:0')
    name, power = _card(0)
    res = {'card': name, 'power_limit,max_sm_clock': power, 'reps': a.reps, 'warmup': a.warmup}

    src = torch.empty(1 << 30, dtype=torch.float32, device=dev)
    dst = torch.empty_like(src)
    ms = _time(lambda: dst.copy_(src), a.reps, a.warmup)
    copy_peak = 2 * src.numel() * 4 / (ms * 1e-3)
    res['copy_GBps'] = copy_peak / 1e9
    del src, dst

    vols = {}
    for case, (working, target) in CASES.items():
        if working not in vols:
            vols = {working: _volumes(working, dev)}
        sv = vols[working]
        out = {}

        def run():
            out['maps'] = ops.volumes_to_grid(sv, PERM, working, target)
        ms = _time(run, a.reps, a.warmup)
        n_w, n_s = int(np.prod(working)), int(np.prod(target))
        gbps = (88 * n_w + 92 * n_s) / (ms * 1e-3) / 1e9
        res[case] = {'working': working, 'target': target, 'kernel_ms': ms, 'GBps': gbps,
                     'of_copy': gbps * 1e9 / copy_peak}
        out.clear()
        torch.cuda.empty_cache()

    if not a.no_files:
        working, target = CASES['1.2A']
        sv = vols.get(working) or _volumes(working, dev)
        with tempfile.TemporaryDirectory() as td:
            pr = CryoEMPredictor('unused', os.path.join(td, 'g') + '/', td, save_output=False, quiet=True)
            pr.reconstruction_path = td
            hdr = MapHeader(voxel_size=(np.float32(1.2),) * 3)
            pr._maps_target = ('input', PERM, working, target, hdr)
            pr._write_maps(sv)                               # warm-up: page cache, pinned allocator
            t0 = time.time()
            pr._write_maps(sv)
            res['save_maps_1.2A_s'] = dict(pr.maps_timing, total=time.time() - t0)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
