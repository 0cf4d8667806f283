#!/usr/bin/env python3
"""torchrun --standalone --nproc_per_node=N tools/bench_int_slab.py [--reps R] [--warmup W] [--out FILE]

Integer maps (DESIGN.md D12) split over N GPUs in z-slabs (SlabPipeline, peer-memory halo and histogram exchange):
  int16 679^3 at 1.06 A -> 720^3   (resample on the general path, every rank's block on the whole line's segments)
  int16 720^3 at 1.0 A             (the D10 copy: halo of the cube padding only)
  int8  679^3 at 1.06 A -> 720^3
Per case and rank: CUDA-event times of the stages of ``resample_and_normalize`` (halo exchange, resample, order
statistics, normalise), median over the timed repetitions, then the slowest rank.  Every rank also runs the whole map
on its own GPU with MapPipeline and checks that its resampled slab, the thresholds and its normalised owned planes
are bit-equal to it; the flags are AND-reduced over the ranks.  Prints one JSON line (rank 0) that names the card and
its power limit."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from mica_b200 import ops, synthetic
from mica_b200.pipeline import MapHeader, MapPipeline, StageTimer
from mica_b200.slab import SlabPipeline

CASES = [('int16_679_to_720', torch.int16, 679, 1.06), ('int16_720_copy', torch.int16, 720, 1.0),
         ('int8_679_to_720', torch.int8, 679, 1.06)]
STAGES = ('halo_exchange', 'resample', 'order_stats', 'normalize_apply')


def _card(index):
    name = torch.cuda.get_device_name(index)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', str(index)],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unknown'
    return name, q


def _int_map(n, dtype, voxel, dev):
    """The same density-like map on every rank, scaled to 90 % of the type's range."""
    d = synthetic.synthetic_map_device((n, n, n), dev, voxel=voxel, seed=2024)
    d = (d - d.min()) / (d.max() - d.min())
    info = torch.iinfo(dtype)
    return torch.round(info.min + d.double() * (float(info.max) - info.min) * 0.9).to(dtype)


def run_case(name, dtype, n, voxel, rank, world, dev, reps, warmup):
    hdr = MapHeader(voxel_size=(np.float32(voxel),) * 3)
    full = _int_map(n, dtype, voxel, dev)
    pipe = SlabPipeline(dev, rank, world, 48, 8, global_src_shape=tuple(full.shape))
    plan = pipe.make_plan(tuple(full.shape), hdr, dtype)
    me = plan.ranks[rank]
    own = full[me.own_lo:me.own_hi].contiguous()
    plane_bytes = full.shape[1] * full.shape[2] * full.element_size()
    halo_bytes = {str(p): (b - a) * plane_bytes for p, a, b in plan.transfers(rank)[1]}

    # the whole map on this GPU
    single = MapPipeline(dev, 48, 8)
    ok = bool(single.resample_and_normalize(full, hdr))
    want_res = full.clone() if plan.identity else ops.resample(full, plan.out_shape)
    res, _ = pipe.slab_resample(own, hdr)
    ok &= torch.equal(res, want_res[me.ext_lo:me.ext_hi])
    del res, want_res

    per_rep = {s: [] for s in STAGES + ('step',)}
    for i in range(warmup + reps):
        timer = StageTimer()
        pipe.timer = timer
        dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ok &= bool(pipe.resample_and_normalize(own, hdr, defer_status=True))
        b.record()
        ok &= bool(pipe.check_status())
        torch.cuda.synchronize(dev)
        if i >= warmup:
            summ = timer.summary()
            for s in STAGES:
                per_rep[s].append(summ.get(s, (0, 0.0))[1])
            per_rep['step'].append(a.elapsed_time(b))
    pipe.timer = StageTimer()
    ok &= pipe.median == single.median and pipe.p999 == single.p999
    ok &= torch.equal(pipe.normalized[me.out_lo - me.ext_lo:me.out_hi - me.ext_lo],
                      single.normalized[me.out_lo:me.out_hi])
    med = {s: float(np.median(v)) for s, v in per_rep.items()}
    t = torch.tensor([med[s] for s in STAGES + ('step',)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)                 # the slowest rank sets the pace
    flag = torch.tensor([int(ok)], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    hb = torch.tensor([max(halo_bytes.values(), default=0)], dtype=torch.int64, device=dev)
    dist.all_reduce(hb, op=dist.ReduceOp.MAX)
    return {'dtype': str(dtype).split('.')[1], 'shape_in': [n] * 3, 'voxel': voxel, 'shape_out': list(plan.out_shape),
            'stage_ms_max_over_ranks': {s: round(v, 4) for s, v in zip(STAGES + ('step',), t.tolist())},
            'halo_bytes_per_neighbour_rank0': halo_bytes, 'halo_bytes_per_neighbour_max': int(hb.item()),
            'halo_via': 'peer' if pipe.peer_halo is not None else 'nccl',
            'bit_identical_all_ranks': bool(flag.item())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    try:
        out = {'tool': 'bench_int_slab', 'world': world}
        out['card'], out['power_limit'] = _card(local)
        out['cases'] = {}
        for name, dtype, n, voxel in CASES:
            out['cases'][name] = run_case(name, dtype, n, voxel, rank, world, dev, args.reps, args.warmup)
            torch.cuda.empty_cache()
        ok = all(c['bit_identical_all_ranks'] for c in out['cases'].values())
        if rank == 0:
            line = json.dumps(out)
            print(line, flush=True)
            if args.out:
                os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
                with open(args.out, 'w') as f:
                    f.write(line + '\n')
    finally:
        dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == '__main__':
    main()
