#!/usr/bin/env python3
"""python tools/bench_cube_select.py [--reps R] [--warmup W] [--out FILE]

The inference keep rule (``min_max=``) on one GPU:
  window_max  ops.cube_window_max over every cube of a normalised map, CUDA-event time per call, median over R after W
              warm-ups: 480^3 with 64^3 windows at stride 32 (grid_size 32, padding 16: bench.py's workload) and
              720^3 with grid_size 48, padding 8.  ``gbps`` = algorithmic reads (W^3 floats per cube; windows overlap,
              so much of it is served by L2) over time; ``map_gbps`` = the map's own bytes over time.
  kept        the fraction of cubes kept at min_max = 0.01 on a synthetic map times a spherical mask (radius 0.35 of
              the edge, exact zeros outside), both geometries.
  dropin      DataPreprocessor -> GridCreator(min_max=) -> CryoEMPredictor on that masked map (256^3 at 1 A, cubes
              48 / 8), the model a Conv3d stand-in (25 -> 29 channels, 3^3 kernel, float32); wall clock of the grid
              creation + prediction with and without min_max, alternated, median over R.
Prints one JSON line that names the card and its power limit."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from mica_b200 import mrc, ops, session, synthetic
from mica_b200.create_grids import GridCreator
from mica_b200.pipeline import MapHeader, MapPipeline
from mica_b200.predict import CryoEMPredictor
from mica_b200.preprocessing import DataPreprocessor


def _card(index):
    name = torch.cuda.get_device_name(index)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', str(index)],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unknown'
    return name, q


def _masked(edge, seed, dev):
    """|synthetic map| (built on the device) times a sphere of radius 0.35 edge: exact zeros outside it."""
    m = synthetic.synthetic_map_device((edge,) * 3, dev, voxel=1.0, seed=seed).abs_()
    r = torch.arange(edge, device=dev, dtype=torch.float32) - (edge - 1) / 2
    r2 = r[:, None, None] ** 2 + r[None, :, None] ** 2 + r[None, None, :] ** 2
    return m.mul_(r2 <= (0.35 * edge) ** 2).contiguous()


def window_max(edge, gs, pad, reps, warmup, dev):
    pipe = MapPipeline(dev, gs, pad)
    assert pipe.resample_and_normalize(_masked(edge, 7, dev), MapHeader())
    pipe.cube_index()
    n, W = len(pipe.ijk_host), gs + 2 * pad
    out = torch.empty(n, dtype=torch.float32, device=dev)
    for _ in range(warmup):
        ops.cube_window_max(pipe.normalized, pipe.ijk, gs, pad, pipe.perm, out=out)
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ops.cube_window_max(pipe.normalized, pipe.ijk, gs, pad, pipe.perm, out=out)
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ms = float(np.median(ts))
    kept = len(ops.select_cubes(out, 0.01))
    return {'edge': edge, 'grid_size': gs, 'padding': pad, 'cubes': n, 'ms': ms,
            'gbps': n * W ** 3 * 4 / ms / 1e6, 'map_gbps': edge ** 3 * 4 / ms / 1e6,
            'kept_at_0.01': kept, 'kept_fraction': kept / n}


class Conv3dStandIn(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.conv = torch.nn.Conv3d(25, 29, 3, padding=1)

    def forward(self, x, af):
        y = self.conv(torch.cat([x, af], 1))
        return y[:, :4], y[:, 4:8], y[:, 8:]


def dropin(edge, reps, dev):
    work = tempfile.mkdtemp(prefix='bench_cube_select_')
    case = os.path.join(work, 'ID')
    os.makedirs(os.path.join(case, 'AF3_results'))
    map_path = os.path.join(case, 'map.mrc')
    mrc.write_mrc(map_path, mrc.MrcMap(data=_masked(edge, 5, dev).cpu().numpy(), voxel_size=(np.float32(1.0),) * 3))
    model = Conv3dStandIn().to(dev).eval()

    def once(min_max, tag):
        session.clear()
        dp = DataPreprocessor(map_path=map_path, AF3_results=os.path.join(case, 'AF3_results'), quiet=True)
        dp.resample_and_normalize_map()
        grids = os.path.join(case, f'grids_{tag}') + '/'
        t1 = time.perf_counter()
        r = GridCreator(quiet=True, min_max=min_max).create_normalized_map_grids(
            dp.normalized_map_path, os.path.join(grids, 'normalized_map_grids'), 48, 8)
        pr = CryoEMPredictor('unused', grids, os.path.join(work, 'out'), save_output=False, quiet=True, model=model)
        ok, _ = pr.run_prediction()
        torch.cuda.synchronize()
        assert ok and r['success']
        return time.perf_counter() - t1, r['grid_count']

    once(None, 'w')
    once(0.01, 'w')
    t_all, t_sel = [], []
    for _ in range(reps):
        t, n_all = once(None, 'a')
        t_all.append(t)
        t, n_sel = once(0.01, 's')
        t_sel.append(t)
    session.clear()
    shutil.rmtree(work, ignore_errors=True)
    return {'edge': edge, 'grid_size': 48, 'padding': 8, 'cubes_all': n_all, 'cubes_kept': n_sel,
            's_all': float(np.median(t_all)), 's_min_max_0.01': float(np.median(t_sel)),
            'speedup': float(np.median(t_all) / np.median(t_sel))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--dropin-reps', type=int, default=3)
    ap.add_argument('--dropin-edge', type=int, default=256)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    dev = torch.device('cuda', torch.cuda.current_device())
    name, power = _card(dev.index)
    res = {'card': name, 'power_limit': power,
           'window_max': [window_max(480, 32, 16, args.reps, args.warmup, dev),
                          window_max(720, 48, 8, args.reps, args.warmup, dev)],
           'dropin': dropin(args.dropin_edge, args.dropin_reps, dev)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
