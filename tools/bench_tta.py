#!/usr/bin/env python3
"""python tools/bench_tta.py [--reps R] [--warmup W] [--out FILE]

Test-time augmentation kernels on one GPU, at bench.py's workload: a synthetic 400^3 map at 1.2 A resampled to the
480^3 working grid, 64^3 windows at stride 32 (grid_size 32, padding 16), batches of 512 cubes.  CUDA-event time per
launch, median over R repetitions after W warm-ups, for orientation 0, 4 (the fastest axis reversed) and 40 (axes
(2, 1, 0): the fastest axis moved):
  extract_map   ops.extract_cubes of the normalised map into [512, 1, 64^3];
  af3_fill      Af3CubeFiller.fill, alternating two batches so that every call clears one cube set and sets another;
  accumulate    ops.Stitcher ('triangle' window, every window voxel contributes), 512 cubes of logits.
Algorithmic bytes: extract = window bytes read + written; accumulate = 26 logit channels read + 22 uint32 sums
added per window voxel; the fill moves a few bytes per atom voxel and is reported as time only.  ``copy_peak``: a
2 GiB device-to-device copy in the same run (read + write bytes / time), the reference for ``frac_copy``.
Then ``predict_and_stitch`` of the whole map with an elementwise stand-in model (logits = x * A + P) for
tta = None / 'flips' / 'rot90', one map per repetition.  Prints one JSON line that names the card and its power
limit; the working set is larger than L2 (126 MB) in every case."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from mica_b200 import ops, synthetic
from mica_b200.pdb import channel_codes
from mica_b200.pipeline import MapHeader, MapPipeline

GS, PAD, B = 32, 16, 512
W = GS + 2 * PAD
CODES = (0, 4, 40)


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--map-reps', type=int, default=2)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_tta needs a CUDA device')
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    out = {'tool': 'bench_tta', 'grid_size': GS, 'padding': PAD, 'batch_cubes': B, 'codes': list(CODES)}
    out['card'], out['power_limit_max_sm_clock'] = _card(0)

    buf = torch.empty(1 << 29, dtype=torch.float32, device=dev)           # 2 GiB
    dst = torch.empty_like(buf)
    ms = _time(lambda: dst.copy_(buf), args.reps, args.warmup)
    peak = 2 * buf.numel() * 4 / (ms * 1e-3)
    out['copy_peak_GBps'] = round(peak / 1e9, 1)
    del buf, dst

    src = synthetic.synthetic_map((400,) * 3, voxel=1.2, seed=2022)
    hdr = MapHeader(voxel_size=(np.float32(1.2),) * 3)
    pipe = MapPipeline(dev, GS, PAD, batch_cubes=B)
    assert pipe.resample_and_normalize(torch.from_numpy(src).to(dev), hdr)
    n_out = tuple(pipe.normalized.shape)
    st = synthetic.synthetic_structure(int(np.prod(n_out)) // 5500, n_out[::-1], seed=2022)
    bb_ch, aa_ch = channel_codes(st['atom_names'], st['res_names'])
    atoms = tuple(torch.from_numpy(a).to(dev) for a in (st['coords'], bb_ch, aa_ch))
    assert pipe.encode_af3(*atoms)
    pipe.cube_index()
    ijk = pipe.ijk[:B]
    ijk2 = pipe.ijk[B:2 * B]
    out['map'] = {'src': [400] * 3, 'grid': list(n_out), 'cubes': len(pipe.ijk_host), 'atoms': len(st['coords'])}

    cases = {}
    x = torch.empty((B, 1, W, W, W), dtype=torch.float32, device=dev)
    ext_bytes = 2 * B * W ** 3 * 4
    filler = pipe._fillers[0]
    bb = torch.randn((B, 4, W, W, W), device=dev)
    ca = torch.randn((B, 4, W, W, W), device=dev)
    aa = torch.randn((B, 21, W, W, W), device=dev)
    acc = ops.Stitcher(pipe.cube_shape, dev, GS, PAD, 'triangle', tta='all')
    acc_bytes = B * W ** 3 * (26 + 22) * 4
    for g in CODES:
        ms = _time(lambda: ops.extract_cubes(pipe.normalized, ijk, GS, PAD, pipe.perm, out=x, orient=g),
                   args.reps, args.warmup)
        c = {'extract_map_ms': round(ms, 4), 'extract_map_GBps': round(ext_bytes / (ms * 1e-3) / 1e9, 1),
             'extract_map_frac_copy': round(ext_bytes / (ms * 1e-3) / peak, 3)}
        turn = [0]

        def fill():
            turn[0] ^= 1
            filler.fill(ijk if turn[0] else ijk2, orient=g)
        c['af3_fill_ms'] = round(_time(fill, args.reps, args.warmup), 4)
        ms = _time(lambda: acc(bb, ca, aa, ijk, orient=g), args.reps, args.warmup)
        c.update({'accumulate_ms': round(ms, 4), 'accumulate_GBps': round(acc_bytes / (ms * 1e-3) / 1e9, 1),
                  'accumulate_frac_copy': round(acc_bytes / (ms * 1e-3) / peak, 3)})
        cases[str(g)] = c
    out['kernels'] = cases
    for g in CODES[1:]:
        for k in ('extract_map_ms', 'af3_fill_ms', 'accumulate_ms'):
            cases[str(g)][k.replace('_ms', '_vs_code0')] = round(cases[str(g)][k] / cases['0'][k], 3)
    del bb, ca, aa, acc, x
    filler.clear()

    gen = torch.Generator().manual_seed(5)
    ap_ = [(torch.randn((c, W, W, W), generator=gen).to(dev), 2 * torch.randn((c, W, W, W), generator=gen).to(dev))
           for c in (4, 4, 21)]

    def model(xx, af):
        return tuple(xx * a + p for a, p in ap_)
    maps = {}
    for tta in (None, 'flips', 'rot90'):
        def run():
            with torch.no_grad():
                pipe.predict_and_stitch(model, tta=tta)
        maps[str(tta)] = {'ms_per_map': round(_time(run, args.map_reps, 1), 1),
                          'orientations': 1 if tta is None else len(ops.tta_orientations(tta))}
    out['predict_and_stitch'] = maps
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
