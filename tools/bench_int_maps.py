"""Integer maps (DESIGN.md D12) at the headline shape: resample, order statistics and normalise of int8, int16 and
uint16 maps, each beside the float32 map of the same values in the same run, and the host -> device upload of each.

    python tools/bench_int_maps.py [--shape 400] [--voxel 1.2] [--reps 20] [--out FILE]

Times are CUDA-event means over --reps calls after two warm-up calls (upload: host clock around a synchronised
copy).  Prints one JSON line that names the card and its power limit."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mica_b200 import ops, synthetic  # noqa: E402
from mica_b200.preprocessing import upload_map  # noqa: E402


def _card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unknown'
    return name, q


def _time(fn, reps):
    for _ in range(2):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def _upload_ms(host, dev, reps):
    upload_map(host, dev)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        upload_map(host, dev)
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--shape', type=int, default=400)
    ap.add_argument('--voxel', type=float, default=1.2)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    dev = torch.device('cuda:0')
    n = args.shape
    zf = [np.float32(args.voxel)] * 3
    out_shape = ops.zoom_output_shape((n, n, n), zf)
    d = synthetic.synthetic_map_device((n, n, n), dev, voxel=args.voxel, seed=5)
    d = (d - d.min()) / (d.max() - d.min())
    card, power = _card()
    rows = {}
    for name, tdt, lo, hi in (('int8', torch.int8, -128, 127), ('int16', torch.int16, -32768, 32767),
                              ('uint16', torch.uint16, 0, 65535)):
        src_i = torch.round(d.double() * (0.9 * (hi - lo)) + lo).to(torch.int32).to(tdt)
        src_f = src_i.to(torch.int32).float()                    # the same values as a float32 map
        res_i = ops.resample(src_i, out_shape)
        res_f = ops.resample(src_f, out_shape)
        ist, fst = ops.IntOrderStats(dev), ops.OrderStats(dev, n_hint=res_f.numel())
        ist.run(res_i)
        fst.run(res_f)
        y = torch.empty(out_shape, dtype=torch.float32, device=dev)
        row = {
            'resample_ms': _time(lambda: ops.resample(src_i, out_shape), args.reps),
            'resample_f32_ms': _time(lambda: ops.resample(src_f, out_shape), args.reps),
            'order_stats_ms': _time(lambda: ist.run(res_i), args.reps),
            'order_stats_f32_ms': _time(lambda: fst.run(res_f), args.reps),
            'normalize_ms': _time(lambda: ist.apply(res_i, y), args.reps),
            'normalize_f32_ms': _time(lambda: fst.apply(res_f, y), args.reps),
        }
        host_i = src_i.cpu().numpy() if tdt is not torch.uint16 else src_i.view(torch.int16).cpu().numpy().view(np.uint16)
        host_f = src_f.cpu().numpy()
        row['upload_ms'] = _upload_ms(host_i, dev, 5)
        row['upload_f32_ms'] = _upload_ms(host_f, dev, 5)
        row['upload_bytes'], row['upload_f32_bytes'] = int(host_i.nbytes), int(host_f.nbytes)
        rows[name] = {k: round(v, 4) if isinstance(v, float) else v for k, v in row.items()}
        del src_i, src_f, res_i, res_f
    line = json.dumps({'card': card, 'power_limit': power, 'shape_in': [n] * 3, 'shape_out': list(out_shape),
                       'voxel': args.voxel, 'reps': args.reps, 'results': rows})
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
