#!/usr/bin/env python3
"""torchrun --standalone --nproc_per_node=N tools/bench_overlap_split.py [--edge E] [--reps R] [--warmup W] [--out FILE]

Overlap-weighted stitching ('triangle' window, grid_size 32 / padding 16) of one E^3 map at 1.0 A split over N GPUs:
  slab      SlabPipeline: z-slabs, every window contribution added into the block of the rank that owns its plane
            (the windows reach 16 planes into the neighbours' slabs, over NVLink);
  balanced  BalancedCubePipeline: cubes dealt out evenly, contributions added into the x-owner's block.
The stand-in model is elementwise (logits = x * A + P, A and P fixed per window position), so the time is the
pipeline's, not a network's.  Per case: CUDA-event time of ``run`` + ``finish_map`` per map, median over the timed
repetitions, then the slowest rank.  Every rank also stitches the whole map on its own GPU with MapPipeline and checks
that its block is bit-equal to its part of that; the flags are AND-reduced over the ranks.  Prints one JSON line
(rank 0) that names the card and its power limit."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from mica_b200 import synthetic
from mica_b200.pipeline import MapHeader, MapPipeline
from mica_b200.slab import BalancedCubePipeline, SlabPipeline

GS, PAD, WINDOW = 32, 16, 'triangle'


def _card(index):
    name = torch.cuda.get_device_name(index)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', str(index)],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unknown'
    return name, q


def _model(dev):
    W = GS + 2 * PAD
    g = torch.Generator().manual_seed(5)
    ap = [(torch.randn((c, W, W, W), generator=g).to(dev), 2 * torch.randn((c, W, W, W), generator=g).to(dev))
          for c in (4, 4, 21)]

    def fn(x, af):
        return tuple(x * a + p for a, p in ap)
    return fn


def _time(step, dev, reps, warmup):
    times = []
    for i in range(warmup + reps):
        dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = step()
        b.record()
        torch.cuda.synchronize(dev)
        if i >= warmup:
            times.append(a.elapsed_time(b))
    return out, float(np.median(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--edge', type=int, default=256)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    ok = False
    try:
        hdr = MapHeader(voxel_size=(np.float32(1.0),) * 3)
        full = synthetic.synthetic_map_device((args.edge,) * 3, dev, voxel=1.0, seed=2024)
        model = _model(dev)
        with torch.no_grad():
            single = MapPipeline(dev, GS, PAD, batch_cubes=64)
            want = {k: v.clone() for k, v in
                    single.run(full, hdr, None, model, overlap_window=WINDOW).as_dict().items()}
            del single
            out = {'tool': 'bench_overlap_split', 'world': world, 'window': WINDOW, 'grid_size': GS, 'padding': PAD,
                   'map': [args.edge] * 3, 'cases': {}}
            out['card'], out['power_limit'] = _card(local)
            flags = []

            slab = SlabPipeline(dev, rank, world, GS, PAD, batch_cubes=64, global_src_shape=tuple(full.shape))
            me = slab.make_plan(tuple(full.shape), hdr).ranks[rank]
            own = full[me.own_lo:me.own_hi].contiguous()

            def slab_step():
                v = slab.run(own, hdr, None, model, overlap_window=WINDOW)
                slab.finish_map()
                return v
            v, ms = _time(slab_step, dev, args.reps, args.warmup)
            (_, _, o2), (_, _, e2) = slab.box
            flags.append(all(torch.equal(t, want[k][..., o2:o2 + e2]) for k, t in v.as_dict().items()))
            out['cases']['slab'] = {'ms_per_map': ms}

            bal = BalancedCubePipeline(dev, rank, world, GS, PAD, batch_cubes=64)

            def bal_step():
                v = bal.run(full, hdr, None, model, overlap_window=WINDOW)
                bal.finish_map()
                return v
            v, ms = _time(bal_step, dev, args.reps, args.warmup)
            x0, x1 = bal.x_bounds[rank], bal.x_bounds[rank + 1]
            flags.append(all(torch.equal(t, want[k][:, x0:x1] if t.dim() == 4 else want[k][x0:x1])
                             for k, t in v.as_dict().items()))
            out['cases']['balanced'] = {'ms_per_map': ms}

        t = torch.tensor([out['cases'][c]['ms_per_map'] for c in ('slab', 'balanced')], dtype=torch.float64,
                         device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)                 # the slowest rank sets the pace
        for c, v in zip(('slab', 'balanced'), t.tolist()):
            out['cases'][c]['ms_per_map'] = round(v, 3)
        flag = torch.tensor([int(all(flags))], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = bool(flag.item())
        out['bit_identical_all_ranks'] = ok
        if rank == 0:
            line = json.dumps(out)
            print(line, flush=True)
            if args.out:
                os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
                with open(args.out, 'w') as f:
                    f.write(line + '\n')
        slab.peer_volumes and slab.peer_volumes.close()
        bal.peer_volumes and bal.peer_volumes.close()
    finally:
        dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == '__main__':
    main()
