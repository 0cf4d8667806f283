#!/usr/bin/env python3
"""python tools/bench_stitch_host.py [--tree DIR] [--maps N] [--out FILE]

Host cost of the stitch calls of ``MapPipeline.predict_and_stitch`` on one GPU.  A synthetic 480^3 working map at
1 A (normalised; no atoms, so the AF3 channels are zero), grid_size 48 / padding 8: 1000 cubes of 64^3, cut in
super-batches of 64 (16 per map, so the prefetch path runs and sets ``last_loop_enqueue_ms``).  The model computes
nothing: every call hands out the next of two preallocated float32 logits batches, so the host side of the batch loop
is the cut, the stitch and the loop itself.  For the paste (default), ``overlap_window='uniform'`` and ``tta='flips'``,
each at ``model_batch`` 1 and 8:
  host_us_per_model_call  ``last_loop_enqueue_ms`` / the model calls of the map;
  device_ms_per_map       CUDA events around ``predict_and_stitch`` (the map synchronised after it).
Medians over ``--maps`` maps after one warm-up map per case.  ``--tree DIR`` imports ``mica_b200`` from DIR instead of
this checkout, so the same script measures another version of the package in the same session.  Prints one JSON line
that names the card and its power limit."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

EDGE, GS, PAD, SUPER = 480, 48, 8, 64
W = GS + 2 * PAD
MODES = {'paste': {}, 'uniform': {'overlap_window': 'uniform'}, 'flips': {'tta': 'flips'}}


def _card(index):
    import torch
    name = torch.cuda.get_device_name(index)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i',
                            str(index)], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unknown'
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--tree', default=ROOT, help='directory holding the mica_b200 package to measure')
    ap.add_argument('--maps', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.tree))
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        sys.exit('bench_stitch_host needs a CUDA device')
    import mica_b200
    from mica_b200 import synthetic
    from mica_b200.pipeline import MapHeader, MapPipeline

    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    out = {'tool': 'bench_stitch_host', 'package': os.path.dirname(os.path.abspath(mica_b200.__file__)),
           'map': [EDGE] * 3, 'grid_size': GS, 'padding': PAD, 'super_batch': SUPER, 'maps': args.maps}
    out['card'], out['power_limit_max_sm_clock'] = _card(0)
    pipe = MapPipeline(dev, GS, PAD, batch_cubes=SUPER)
    src = synthetic.synthetic_map_device((EDGE,) * 3, dev, voxel=1.0, seed=2022)
    assert pipe.resample_and_normalize(src, MapHeader(voxel_size=(np.float32(1.0),) * 3))
    del src
    g = torch.Generator(device=dev).manual_seed(7)
    ring = [[torch.randn((8, c, W, W, W), device=dev, generator=g) for c in (4, 4, 21)] for _ in range(2)]
    calls = [0]

    def model(x, af):
        lg = ring[calls[0] & 1]
        calls[0] += 1
        B = x.shape[0]
        return lg[0][:B], lg[1][:B], lg[2][:B]

    rows = {}
    with torch.no_grad():
        for mode, kw in MODES.items():
            for mb in (1, 8):
                host, device = [], []
                for rep in range(args.maps + 1):
                    calls[0] = 0
                    torch.cuda.synchronize()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    vols = pipe.predict_and_stitch(model, model_batch=mb, d8='none', **kw)
                    b.record()
                    torch.cuda.synchronize()
                    del vols
                    if rep:                                         # the first map warms up
                        host.append(pipe.last_loop_enqueue_ms * 1e3 / calls[0])
                        device.append(a.elapsed_time(b))
                rows[f'{mode}_mb{mb}'] = {'model_calls_per_map': calls[0],
                                          'host_us_per_model_call': round(float(np.median(host)), 2),
                                          'host_us_per_model_call_all': [round(v, 2) for v in host],
                                          'device_ms_per_map': round(float(np.median(device)), 3)}
                torch.cuda.empty_cache()
    out['cases'] = rows
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
