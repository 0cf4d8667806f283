#!/usr/bin/env python3
"""bench.py -- GVox/s of the map -> cubes -> stitched-volume hot path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A step = one pass of the whole hot path over one synthetic map: B-spline resample to
the 1 A grid, exact median/p99.9 normalisation, 24-channel AF3 rasterisation, 64^3 cube
extraction into the model's input batch, and softmax/argmax + stitching of the model's
logits into the four output volumes.  The model itself (models/model.py, PyTorch
convolutions) is out of scope per north_star and is replaced by a ring of pre-generated
logits larger than L2, so every byte the post-processing reads comes from HBM.

Headline (`value`), N = 1: BASELINE.json configs[1] -- synthetic 400^3 map at 1.2 A -> 480^3
working grid, 64^3 cubes at stride 32 (grid_size=32, padding=16), ~167 k atoms.  N > 1: the same
per-GPU slab (weak scaling): a (400 N) x 400 x 400 map z-slab partitioned over N ranks.

Further blocks of the same JSON line (each a different BASELINE config, never the headline):
  variant / variant_48_8   the reference's dense-AF3 dataflow and its default geometry (48 / 8)
  strong_720               configs[3]: ONE 679^3 @ 1.06 A -> 720^3 map z-slab partitioned over the N
                           ranks (strong scaling), with a built-in N-rank == 1-GPU parity check
  config5                  configs[4]: a 512^3 map through the REAL models/model.py::MICA, cubes dealt
                           out evenly over the ranks, cores stored into the owner's volume over NVLink
  e2e / e2e_aa_prob_resident / e2e_dropin
                           host buffers in, host volumes out; the last one through the reference-named
                           classes (DataPreprocessor -> GridCreator -> CryoEMPredictor), MRC + PDB on tmpfs

`--dump-outputs DIR` writes the four stitched volumes of the headline's last timed step (dump_outputs: a
fixed, seeded sample of voxels, float32) so that two builds can be compared output for output.  With
N > 1 it holds rank 0's slab only; the other ranks' slabs are not written.

Prints ONE JSON line (rank 0).  `--impl reference` times the UNMODIFIED reference (staged by
oracle/make_ref.py) as it is -- its .mrc / .npz files on tmpfs, its worker pools -- on a bounded
sample of the same workload, on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'map_to_stitched_volume_throughput'
UNIT = 'GVox/s'


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--src-edge', type=int, default=400)
    ap.add_argument('--voxel', type=float, default=1.2)
    ap.add_argument('--grid-size', type=int, default=32)
    ap.add_argument('--padding', type=int, default=16)
    ap.add_argument('--batch-cubes', type=int, default=512)
    ap.add_argument('--cpu-edge', type=int, default=0, help='source edge of the CPU sample (0 = auto)')
    ap.add_argument('--e2e-steps', type=int, default=5)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--af3-mode', default='sparse', choices=['sparse', 'dense'],
                    help='sparse: AF3 cube channels written from per-cube atom bins (default); dense: the '
                         "reference's dataflow (24-channel volume, then window extraction)")
    ap.add_argument('--no-variant', action='store_true', help='skip the dense / 48-8 variants')
    ap.add_argument('--no-strong', action='store_true', help='skip the strong_720 block (configs[3])')
    ap.add_argument('--no-config5', action='store_true', help='skip the config5 block (configs[4], real MICA)')
    ap.add_argument('--no-dropin', action='store_true', help='skip e2e_dropin')
    ap.add_argument('--config5-cubes', type=int, default=-1,
                    help='cubes of the 512^3 map pushed through MICA (-1 = all 1331; the model costs ~7.4 TFLOP '
                         'per cube, ~26 ms on a B200)')
    ap.add_argument('--maps-in-flight', type=int, default=0,
                    help='also time K steps with this many maps in flight (one pipeline + stream each); 0 = skip')
    ap.add_argument('--cpu-kind', default='as_is', choices=['as_is', 'port'],
                    help='reference arm: the unmodified reference with its file I/O (default) or the in-memory port')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the four volumes of the last timed step as DIR/<name>.npy (rank 0; a fixed sample '
                         'of voxels when the volumes exceed DUMP_VOXELS), to compare two builds output for output')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if args.dump_outputs and args.impl == 'reference':
        # the reference arm times a smaller CPU sample of the workload, so its volumes are not comparable
        ap.error('--dump-outputs writes the GPU path (--impl ours) only')
    return args


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        return float(json.load(open(path))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def algorithmic_bytes(n_src, n_vox, n_atoms, f):
    """SURVEY.md 8(d): B(N) = 4 Ns + N (420 + 100 f) (+16 per atom)."""
    return {
        'resample': 4 * n_src + 4 * n_vox,
        'normalize': 12 * n_vox,
        'af3_encode': 96 * n_vox + 16 * n_atoms,
        'extract': 100 * n_vox * (1 + f),
        'postproc_stitch': 208 * n_vox,
    }


def sparse_bytes(n_src, n_vox, n_atoms, f):
    """The bytes the sparse-AF3 dataflow has to move: as B(N) but the 24 AF3 channels are never
    materialised (neither the dense volume nor its windows) -- atoms in, map-channel windows out."""
    return {
        'resample': 4 * n_src + 4 * n_vox,
        'normalize': 12 * n_vox,
        'af3_encode': 16 * n_atoms,
        'extract': 4 * n_vox * (1 + f),
        'postproc_stitch': 208 * n_vox,
    }


# ----------------------------------------------------------------------------- CPU arm
def cpu_threads():
    """All host threads the reference can use -- torchrun exports OMP_NUM_THREADS=1, which made the
    N >= 2 reference arm three times slower than N = 1 in round 1."""
    import torch
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        pass
    torch.set_num_threads(n)
    return n


def cpu_sample_edge(args, kind):
    if args.cpu_edge:
        return args.cpu_edge
    runs = args.steps + args.warmup if args.impl == 'reference' else 1
    per_run = 150.0 / runs                      # seconds of CPU work one run may cost
    if kind == 'as_is':
        # ~0.17 s per cube at stride 32 (25 input + 4 output .npz per cube), cubes = ceil(1.2 e / 32)^3
        cubes = max(8.0, per_run / 0.17)
        edge = (cubes ** (1.0 / 3.0)) * args.grid_size / args.voxel
        return int(max(40, min(120, edge // 10 * 10)))
    edge = 100.0 * (per_run / 1.75) ** (1.0 / 3.0)
    return int(max(60, min(240 if runs > 1 else 200, edge // 20 * 20)))


def cpu_workload(edge, args):
    from mica_b200 import synthetic
    from oracle import mica_oracle as orc
    src = synthetic.synthetic_map((edge,) * 3, voxel=args.voxel, seed=2022)
    voxel = (np.float32(args.voxel),) * 3
    n_out = orc.zoom_output_shape(src.shape, orc.zoom_factors(voxel))
    st = synthetic.synthetic_structure(max(50, int(np.prod(n_out)) // 5500), n_out[::-1], seed=2022)
    bb_ch, aa_ch = orc.channel_codes(st['atom_names'], st['res_names'])
    n_cubes = int(np.prod([-(-n // args.grid_size) for n in n_out]))
    # 16 cubes of stand-in logits, reused for every chunk (the GPU arm reuses its ring the same way)
    ring = synthetic.synthetic_logits(16, args.grid_size + 2 * args.padding, seed=2022)
    return dict(src=src, voxel=voxel, coords=st['coords'], bb_ch=bb_ch, aa_ch=aa_ch, ring=ring,
                n_out=n_out, n_cubes=n_cubes, structure=st)


def cpu_port_step(w, args):
    """The reference's arithmetic for the whole path, in memory (no .mrc/.npz I/O)."""
    from oracle import mica_oracle as orc
    t0 = time.perf_counter()
    vols, nvox, ncubes = orc.pipeline_whole_streamed(
        w['src'], w['voxel'], w['coords'], w['bb_ch'], w['aa_ch'], (0.0, 0.0, 0.0), w['ring'],
        args.grid_size, args.padding)
    dt = time.perf_counter() - t0
    assert ncubes == w['n_cubes']
    return dt, nvox


def cpu_baseline(args, steps=1, warmup=0, kind=None):
    """kind 'as_is': the UNMODIFIED reference (oracle/_ref or /root/reference) run as Solver.getData +
    Solver.nnPred run it, files on tmpfs and worker pools included (`kind: reference`); 'port': the
    oracle's in-memory restatement (`kind: port`).  Falls back to the port when no reference is staged."""
    from oracle import ref_harness
    kind = kind or args.cpu_kind
    if kind == 'as_is' and not ref_harness.available():
        kind = 'port'
    threads = cpu_threads()
    edge = cpu_sample_edge(args, kind)
    w = cpu_workload(edge, args)
    nvox = int(np.prod(w['n_out']))
    extra = {}
    if kind == 'as_is':
        from oracle import ref_pipeline
        wd = ref_pipeline.make_workdir()
        try:
            paths = ref_pipeline.prepare(wd, w['src'], w['voxel'], w['structure'])
            times = []
            for i in range(warmup + steps):
                dt, _, ncubes = ref_pipeline.run_as_is(paths, w['ring'], args.grid_size, args.padding)
                assert ncubes == w['n_cubes']
                if i >= warmup:
                    times.append(dt)
            if args.impl != 'reference' or steps <= 2:
                # the same sample at the reference's own default geometry, and the arithmetic alone
                dt48, _, n48 = ref_pipeline.run_as_is(paths, synth_ring(48 + 16), 48, 8)
                extra['as_is_grid48_pad8'] = {'value': nvox / dt48 / 1e9, 'unit': UNIT, 's_per_step': dt48, 'cubes': n48}
        finally:
            shutil.rmtree(wd, ignore_errors=True)
        dtp, _ = cpu_port_step(w, args)
        extra['arithmetic_only_in_memory'] = {'value': nvox / dtp / 1e9, 'unit': UNIT, 's_per_step': dtp,
                                              'what': "oracle port: the same arithmetic without the reference's files"}
        how = ('UNMODIFIED reference (DataPreprocessor -> GridCreator -> CryoEMPredictor as Solver.getData/nnPred '
               'drive them, utils/modeler.py:673-760), its .mrc/.npz files on tmpfs, its mp.Pool / '
               'ProcessPoolExecutor workers, model = logits ring')
    else:
        for _ in range(warmup):
            cpu_port_step(w, args)
        times = [cpu_port_step(w, args)[0] for _ in range(steps)]
        how = 'oracle port (scipy zoom + numpy + torch-CPU softmax) in memory, no file I/O'
    t = float(np.mean(times))
    note = ''
    if kind == 'as_is' and (args.grid_size, args.padding) != (48, 8):
        note = ("; the reference's stitcher hard-codes padding=8 (utils/predict.py:438,547), so at this geometry it "
                'pastes shifted cores -- same work, timing only')
    return dict({
        'value': nvox / t / 1e9, 'unit': UNIT, 'cores': threads, 'kind': 'reference' if kind == 'as_is' else 'port',
        'host_cpus': os.cpu_count(),
        'sample': f'{edge}^3 map @ {args.voxel} A -> {"x".join(map(str, w["n_out"]))} grid, {w["n_cubes"]} cubes '
                  f'(grid_size={args.grid_size}, padding={args.padding}), {len(w["coords"])} atoms; {how}; '
                  f'{t:.2f} s/step{note}',
    }, **extra), t


def synth_ring(window):
    from mica_b200 import synthetic
    return synthetic.synthetic_logits(16, window, seed=2022)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cb, t = cpu_baseline(args, steps=args.steps, warmup=args.warmup)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': cb['value'], 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': t * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args, 1) | {'sampled': cb['sample']},
        'cpu_baseline': cb,
        'e2e': {'value': cb['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- GPU arm
def workload_config(args, n_gpus):
    e = args.src_edge
    return {
        'workload': f'BASELINE configs[1]: synthetic {e}^3 map @ {args.voxel} A -> 1 A grid, 64^3 cubes at stride '
                    f'{args.grid_size} (grid_size={args.grid_size}, padding={args.padding})'
                    + (f'; weak scaling: ({e}x{n_gpus})x{e}x{e} map z-slab partitioned over {n_gpus} GPUs'
                       if n_gpus > 1 else ''),
        'resample': 'cubic B-spline (scipy.ndimage.zoom order=3 semantics)',
        'model': 'excluded (north_star): logits come from a pre-generated HBM ring',
        'batch_cubes': args.batch_cubes,
        'l2': 'no flush needed: every stage streams buffers far larger than the 126 MB L2',
    }


class ClockSampler:
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', f'--id={index}', f'--query-gpu={self.FIELDS}',
                                       '--format=csv,noheader,nounits', '-lms', '20'],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        if self.p is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [r.split(',') for r in open(self.f.name).read().strip().splitlines() if r.count(',') >= 6]
        os.unlink(self.f.name)
        if not rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        sm = [float(r[0]) for r in rows]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].strip().lower() == 'active' for r in rows)]
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(rows[0][1]), 'samples': len(rows),
                'power_w_max': max(float(r[2]) for r in rows), 'reasons': reasons}


def bind_to_gpu_numa(local_rank):
    """Run this rank's host threads on the CPUs nearest its GPU before any pinned buffer is allocated
    (first touch places the pages): `nvidia-smi topo -m` names the CPU affinity of every GPU."""
    try:
        out = subprocess.run(['nvidia-smi', 'topo', '-m'], capture_output=True, text=True, timeout=20).stdout
        for ln in out.splitlines():
            parts = ln.split()
            if parts and parts[0] == f'GPU{local_rank}':
                for tok in parts[1:]:
                    if tok[0].isdigit() and ('-' in tok or ',' in tok) and not tok.endswith('X'):
                        cpus = set()
                        for rng in tok.split(','):
                            a, _, b = rng.partition('-')
                            cpus.update(range(int(a), int(b or a) + 1))
                        os.sched_setaffinity(0, cpus)
                        numa = parts[parts.index(tok) + 1] if parts.index(tok) + 1 < len(parts) else '?'
                        return {'cpus': tok, 'numa': numa}
    except Exception as e:                      # diagnostics only
        return {'error': str(e)[:80]}
    return None


class Ctx:
    """What every block of run_ours needs."""
    pass


def make_measure(ctx):
    import torch
    from mica_b200 import ops
    from mica_b200.pipeline import StageTimer, _no_timer
    args, dist, world, rank, dev = ctx.args, ctx.dist, ctx.world, ctx.rank, ctx.dev

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(pipe, inputs, model_fn, with_clocks=False, only=None, steps=None, warmup=None):
        """W warm-up steps, then exactly K timed steps between barrier+synchronize, CUDA events on the
        launching stream, max over ranks.  ``only``: the stages whose launches are bracketed by events
        inside the timed region (every event pair costs ~4 us of stream time; 81 launches per step)."""
        src, header, atoms = inputs
        steps = args.steps if steps is None else steps
        warmup = args.warmup if warmup is None else warmup
        vols = None
        for _ in range(warmup):
            # next_src: a stream of maps -- a z-slab rank exchanges the next map's source halo under this map's
            # cube loop (one exchange per step either way; no-op on one GPU)
            vols = pipe.run(src, header, atoms, model_fn, vols, next_src=src)      # checked at once: a broken setup fails here
        sync()
        timer = StageTimer(only)
        pipe.timer = timer
        if os.environ.get('MICA_NO_PREFETCH'):            # experiment knob
            pipe.prefetch = False
        launches0 = ops.launch_count()
        clocks = ClockSampler(ctx.local_rank) if (with_clocks and rank == 0) else None
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync()
        ev0.record()
        t_host = time.perf_counter()
        for _ in range(steps):
            # status words go to pinned memory in stream order and are checked after the loop (finish()):
            # no host synchronisation between the maps of the stream
            vols = pipe.run(src, header, atoms, model_fn, vols, defer_check=True, next_src=src)
        ev1.record()
        t_host = (time.perf_counter() - t_host) / steps * 1e3      # host time spent enqueueing one step
        sync()
        pipe.finish()
        ms = ev0.elapsed_time(ev1)
        launches = ops.launch_count() - launches0
        clk = clocks.stop() if clocks else None
        stages = timer.summary()
        pipe.timer = _no_timer
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, stages, launches, clk, vols, t_host

    return sync, measure


def stage_table(stages, steps):
    return {k: round(v[1] / steps, 4) for k, v in stages.items()}


DUMP_VOXELS = 1 << 19      # 23 float32 channels + a float64 index a voxel: 50 MiB, under 64 MB


def dump_outputs(out_dir, vols):
    """The four volumes ``pipe.run`` returned as out_dir/<name>.npy, float32, channels first.  Volumes larger
    than DUMP_VOXELS are sampled at the same voxels on every run (a seeded choice, independent of the build);
    sample_voxel_index.npy holds their flat C-order indices into the volume, as float64."""
    import torch
    n = vols.backbone_probability.numel()
    if n > DUMP_VOXELS:
        idx = np.sort(np.random.default_rng(2022).choice(n, DUMP_VOXELS, replace=False))
    else:
        idx = np.arange(n)
    os.makedirs(out_dir, exist_ok=True)
    idx_dev = torch.from_numpy(idx).to(vols.device)
    for k, v in vols.as_dict().items():
        flat = v.reshape(-1, n) if v.dim() == 4 else v.reshape(n)
        np.save(os.path.join(out_dir, f'{k}.npy'), flat[..., idx_dev].cpu().numpy())
    np.save(os.path.join(out_dir, 'sample_voxel_index.npy'), idx.astype(np.float64))


# ------------------------------------------------------------------ configs[3]: strong scaling of ONE 720^3 map
def strong_720(ctx, identity):
    """ONE map z-slab partitioned over the ranks (SlabPlan(global_src_shape)), reference-default geometry
    48 / 8.  identity=False: 679^3 @ 1.06 A -> 720^3 (resampler exercised); True: 720^3 @ 1.0 A (SciPy's copy
    path, D10).  Returns the block for the JSON line, parity included: every rank ALSO runs the whole map on
    its own GPU with a deterministic pointwise model and compares thresholds (bit-equal) and its owned slab of
    the four volumes with that run."""
    import torch
    from mica_b200 import ops, synthetic
    from mica_b200.pdb import channel_codes
    from mica_b200.pipeline import MapHeader, MapPipeline
    from mica_b200.slab import SlabPipeline, SlabPlan
    args, dist, world, rank, dev = ctx.args, ctx.dist, ctx.world, ctx.rank, ctx.dev
    edge, voxel = (720, 1.0) if identity else (679, 1.06)
    gs, pad, B = 48, 8, args.batch_cubes
    src_full = synthetic.synthetic_map_device((edge,) * 3, dev, voxel=voxel, seed=2022)    # identical on every rank
    header = MapHeader(voxel_size=(np.float32(voxel),) * 3)
    n_out = ops.zoom_output_shape(src_full.shape, [np.float32(voxel)] * 3)
    st = synthetic.synthetic_structure(30000, n_out[::-1], seed=2023)
    bb_ch, aa_ch = channel_codes(st['atom_names'], st['res_names'])
    atoms = tuple(torch.from_numpy(a).to(dev) for a in (st['coords'], bb_ch, aa_ch))
    if world == 1:
        pipe, own = MapPipeline(dev, gs, pad, batch_cubes=B), src_full
    else:
        plan = SlabPlan(tuple(src_full.shape), header.voxel_size, gs, pad, world)
        me = plan.ranks[rank]
        own = src_full[me.own_lo:me.own_hi].contiguous()
        pipe = SlabPipeline(dev, rank, world, gs, pad, batch_cubes=B, global_src_shape=tuple(src_full.shape))
    inputs = (own, header, atoms)
    steps, warmup = max(5, min(args.steps, 10)), max(3, min(args.warmup, 3))
    _, stages_all, _, _, vols, _ = ctx.measure(pipe, inputs, ctx.ring_model, steps=steps, warmup=warmup)
    del vols
    ms, _, launches, _, vols, host_ms = ctx.measure(pipe, inputs, ctx.ring_model, only=set(), steps=steps, warmup=warmup)
    n_vox = int(np.prod(n_out))
    f = ((gs + 2 * pad) / gs) ** 3
    peak, _ = peaks()
    nbytes = sum(sparse_bytes(src_full.numel(), n_vox, atoms[0].shape[0], f).values())
    block = {
        'workload': f'BASELINE configs[3]: ONE synthetic {edge}^3 map @ {voxel} A -> {"x".join(map(str, n_out))} grid'
                    f'{" (zoom 1: SciPy copy path, D10)" if identity else ""}, z-slab partitioned over {world} GPU(s), '
                    f'grid_size={gs}, padding={pad} (reference default), {atoms[0].shape[0]} atoms, sparse AF3',
        'scaling': 'strong', 'ms_per_step': ms, 'value': n_vox / (ms * 1e-3) / 1e9, 'unit': UNIT,
        'steps': steps, 'warmup': warmup, 'cubes_this_rank': len(pipe.ijk_host), 'gpu_launches': int(launches),
        'host_enqueue_ms_per_step': host_ms,
        'stage_ms_per_step_rank0': stage_table(stages_all, steps),
        'bytes_moved_frac_of_peak': nbytes / world / (ms * 1e-3) / 1e9 / peak,
        'halo_exchange': getattr(pipe, 'halo_exchange', None), 'hist_exchange': getattr(pipe, 'hist_exchange', None),
        'halo_prefetch': ('the source halo of map k+1 is exchanged on a side stream under the cube loop of map k '
                          '(SlabPipeline.prefetch_source): one exchange per timed step, off the critical path'
                          if world > 1 else None),
    }
    del vols
    # ---- parity: N-rank slab run == whole-map run on one GPU (same deterministic pointwise model)
    if world > 1:
        Bp = 64
        pipe.configure(batch_cubes=Bp)
        with torch.no_grad():
            v_slab = pipe.run(own, header, atoms, synthetic.pointwise_model)
            med_s, p_s = pipe.median, pipe.p999
            single = MapPipeline(dev, gs, pad, batch_cubes=Bp)
            v_full = single.run(src_full, header, atoms, synthetic.pointwise_model)
        (o0, o1, o2), (e0, e1, e2) = pipe.box
        diffs = {}
        for k, t in v_slab.as_dict().items():
            ref_t = v_full.as_dict()[k][..., o2:o2 + e2]
            if k == 'amino_acid_prediction':
                diffs[k + '_mismatch_frac'] = float((t != ref_t).float().mean())
            else:
                diffs[k] = float((t - ref_t).abs().max())
        me = pipe.plan.ranks[rank]
        norm_diff = float((pipe.normalized[me.out_lo - me.ext_lo:me.out_hi - me.ext_lo]
                           - single.normalized[me.out_lo:me.out_hi]).abs().max())
        thr_equal = bool(med_s == single.median and p_s == single.p999)
        worst = max([norm_diff] + [v for k, v in diffs.items() if not k.endswith('_frac')])
        t = torch.tensor([worst, diffs['amino_acid_prediction_mismatch_frac'], 0.0 if thr_equal else 1.0],
                         device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        worst_all, mism_all, thr_bad = (float(v) for v in t.tolist())
        block['parity'] = {
            'against': 'the whole map on ONE GPU (run on every rank), pointwise stand-in model',
            'thresholds_bit_equal_all_ranks': thr_bad == 0.0, 'median': float(med_s), 'p999': float(p_s),
            'median_one_gpu': float(single.median), 'p999_one_gpu': float(single.p999),
            'owned_slab_max_abs_all_ranks': worst_all, 'argmax_mismatch_frac_max': mism_all,
            'rank0': dict(diffs, normalized=norm_diff),
            'bit_identical_all_ranks': bool(thr_bad == 0.0 and worst_all == 0.0 and mism_all == 0.0),
            'ok': bool(thr_bad == 0.0 and worst_all <= 1e-6 and mism_all <= 1e-6),
            'tolerance': 'thresholds bit-equal; normalised planes and probability volumes <= 1e-6; argmax '
                         'mismatches <= 1e-6 of the voxels.  A rank holds whole prefilter windows of its planes '
                         '(SlabPlan aligned=True), so the expected difference is exactly 0 (bit_identical_all_ranks)',
        }
        del v_slab, v_full, single
    del pipe, src_full, own
    torch.cuda.empty_cache()
    return block


# ------------------------------------------------------------------ configs[4]: the real model loop
def load_mica():
    """models/model.py::MICA, unmodified: from the reference on sys.path, else the staged archive."""
    try:
        from models.model import MICA
        return MICA, 'models.model on sys.path'
    except Exception:
        pass
    for root in ('/root/reference', os.path.join(ROOT, 'oracle', '_ref', 'reference_py.zip')):
        if os.path.exists(root):
            sys.path.insert(0, root)
            try:
                from models.model import MICA
                return MICA, root
            except Exception:
                sys.path.remove(root)
    return None, None


def config5(ctx):
    """512^3 map through models/model.py::MICA (random weights, torch.manual_seed(2022), fp32), cubes dealt
    out evenly over the ranks, every core stored into its owner's volume block over NVLink peer memory."""
    import torch
    from mica_b200 import synthetic
    from mica_b200.pdb import channel_codes
    from mica_b200.pipeline import MapHeader, MapPipeline, StageTimer, _no_timer
    from mica_b200.slab import BalancedCubePipeline
    args, dist, world, rank, dev = ctx.args, ctx.dist, ctx.world, ctx.rank, ctx.dev
    MICA, where = load_mica()
    if MICA is None:
        return {'unavailable': 'models/model.py not importable (no reference on sys.path, no oracle/_ref archive)'}
    torch.manual_seed(2022)                                   # run.py:86
    model = MICA().to(dev).eval()
    gs, pad = 48, 8
    src = synthetic.synthetic_map_device((512,) * 3, dev, voxel=1.0, seed=2022)
    header = MapHeader(voxel_size=(np.float32(1.0),) * 3)
    st = synthetic.synthetic_structure(6400, (512, 512, 512), seed=2022)       # ~50 k atoms
    bb_ch, aa_ch = channel_codes(st['atom_names'], st['res_names'])
    atoms = tuple(torch.from_numpy(a).to(dev) for a in (st['coords'], bb_ch, aa_ch))
    n_all = 11 ** 3
    # which cubes: all 1331 (measured: ~26 ms of convolutions per cube on a B200 with TF32 convolutions, i.e.
    # ~35 s on one GPU, ~4.5 s on eight); --config5-cubes bounds the run to whole x-columns of cubes
    n_cubes = n_all if args.config5_cubes < 0 else min(n_all, args.config5_cubes)
    ijk_all = np.stack(np.meshgrid(*[np.arange(11)] * 3, indexing='ij'), -1).reshape(-1, 3)

    def subset(n):
        if n >= n_all:
            return None
        # whole x-columns (all 11 i for a (j,k) pair), columns spread over the map: touches every owner's x range
        cols = np.linspace(0, 120, max(1, n // 11), dtype=np.int64)
        sel = np.flatnonzero(np.isin(ijk_all[:, 1] * 11 + ijk_all[:, 2], cols))
        return sel[:n]
    sel = subset(n_cubes)
    spans = []

    def timed_model(x, af):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = model(x, af)
        b.record()
        spans.append((a, b))
        return out

    kw = dict(model_batch=8, d8='split')
    grp = None if world > 1 else False

    def run(pipe, fn):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        with torch.no_grad():
            vols = pipe.run(src, header, atoms, fn, **kw)
        e1.record()
        pipe.finish_map()
        return vols, e0.elapsed_time(e1)

    # warm-up: cuDNN algorithm selection, allocator, peer-volume mapping; the reference caps the model batch
    # at 8 (utils/predict.py:174) -- halve it if this GPU cannot hold the activations next to everything else
    all_or_sel = sel if sel is not None else np.arange(n_all)
    warm = BalancedCubePipeline(dev, rank, world, gs, pad, batch_cubes=8, group=grp, cube_subset=all_or_sel[:8 * world])
    while True:
        try:
            run(warm, model)
            break
        except torch.cuda.OutOfMemoryError:
            if world > 1 or kw['model_batch'] == 1:
                raise
            kw['model_batch'] //= 2
            torch.cuda.empty_cache()
    pipe = BalancedCubePipeline(dev, rank, world, gs, pad, batch_cubes=64, group=grp, cube_subset=sel,
                                _peer_volumes=warm.peer_volumes)
    del warm
    vols, total_ms = run(pipe, timed_model)
    m_ms = sum(a.elapsed_time(b) for a, b in spans)
    t = torch.tensor([total_ms, m_ms, total_ms - m_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_max, model_max, exposed_max = (float(v) for v in t.tolist())
    n_vox_done = int(len(sel) if sel is not None else n_all) * gs ** 3
    block = {
        'workload': 'BASELINE configs[4]: synthetic 512^3 map @ 1.0 A, 11^3 = 1331 cubes of 64^3 (grid 48 / pad 8) '
                    f'through models/model.py::MICA ({where}), random weights seed 2022, fp32 '
                    f'(cudnn.allow_tf32={torch.backends.cudnn.allow_tf32}), model batches of <= {kw["model_batch"]}, D8 split; '
                    f'{n_cubes} of 1331 cubes run' + ('' if sel is None else ' (bounded subset: whole x-columns)'),
        'cubes_run': int(n_cubes), 'cubes_per_rank': pipe.cubes_per_rank,
        'cube_balance_min_over_max': min(pipe.cubes_per_rank) / max(1, max(pipe.cubes_per_rank)),
        'x_bounds': pipe.x_bounds,
        'ms_total_max_rank': total_max, 'ms_model_max_rank': model_max, 'ms_exposed_hot_path_max_rank': exposed_max,
        'rank0': {'ms_total': total_ms, 'ms_model': m_ms, 'ms_exposed_hot_path': total_ms - m_ms,
                  'model_calls': len(spans)},
        'exposed_over_model': exposed_max / max(model_max, 1e-9),
        'model_ms_per_cube_rank0': m_ms / max(1, pipe.cubes_per_rank[rank]),
        'core_voxels_per_s': n_vox_done / (total_max * 1e-3),
        'stitch': 'ops.postproc_stitch_peer: cores stored into the owning rank\'s exported volume block '
                  '(local or NVLink peer memory), no NCCL on the data path',
    }
    # ---- parity: the same cubes on ONE GPU, on a small subset whose x-columns touch every owner's range.
    # One cube per model call on both sides: with TF32 convolutions the logits of a cube depend on the batch
    # it is convolved in (cuDNN picks its algorithm per shape; measured 6e-4 on the probabilities between a
    # batch of 8 and a batch of 3), so only equal batches isolate what is being checked -- the dataflow.
    kw = dict(model_batch=1, d8='split')
    par_sel = subset(22) if sel is None or len(sel) > 22 else sel
    pipe_n = BalancedCubePipeline(dev, rank, world, gs, pad, batch_cubes=22, group=grp, cube_subset=par_sel,
                                  _peer_volumes=pipe.peer_volumes)
    del vols
    v_n, _ = run(pipe_n, model)
    single = MapPipeline(dev, gs, pad, batch_cubes=22)
    with torch.no_grad():
        single.resample_and_normalize(src, header)
        single.encode_af3(*atoms)
        v_1 = single.predict_and_stitch(model, order=par_sel, **kw)
    torch.cuda.synchronize()
    x0, x1 = pipe_n.x_bounds[rank], pipe_n.x_bounds[rank + 1]
    # voxels covered by the subset's cores only (the rest is zero in both)
    worst, mism = 0.0, 0.0
    for k, tn in v_n.as_dict().items():
        t1 = v_1.as_dict()[k][..., x0:x1, :, :] if tn.dim() == 4 else v_1.as_dict()[k][x0:x1]
        if k == 'amino_acid_prediction':
            mism = float((tn != t1).float().mean())
        else:
            worst = max(worst, float((tn - t1).abs().max()))
    t = torch.tensor([worst, mism], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    block['parity'] = {'against': f'the same {len(par_sel)} cubes through the same model on ONE GPU (every rank checks '
                                  'its own x range)', 'max_abs_all_ranks': float(t[0]), 'argmax_mismatch_frac_max': float(t[1]),
                       'ok': bool(float(t[0]) <= 1e-5 and float(t[1]) <= 1e-5),
                       'model_batch': 1,
                       'tolerance': 'probabilities <= 1e-5; argmax mismatches <= 1e-5 of the voxels (same cube, same '
                                    'model call shape on both sides)'}
    if pipe.peer_volumes is not None:
        pipe.peer_volumes.close()
    del pipe, pipe_n, single, v_n, v_1, model
    torch.cuda.empty_cache()
    return block


# ------------------------------------------------------------------ e2e through the reference-named classes
def e2e_dropin(ctx, src_np, header, st, n_vox, host_volumes, steps):
    """utils/modeler.py:673-734 with the drop-in classes: MRC + PDB on tmpfs -> DataPreprocessor ->
    GridCreator -> CryoEMPredictor(model = logits ring) -> host volumes."""
    import torch
    from mica_b200 import mrc, session, synthetic
    from mica_b200.create_grids import GridCreator
    from mica_b200.predict import CryoEMPredictor, HostPool
    from mica_b200.preprocessing import DataPreprocessor
    args = ctx.args
    base = '/dev/shm' if os.path.isdir('/dev/shm') and os.access('/dev/shm', os.W_OK) else None
    wd = tempfile.mkdtemp(prefix='mica_dropin_', dir=base)
    try:
        case = os.path.join(wd, 'input', 'ID')
        os.makedirs(os.path.join(case, 'AF3_results'))
        map_path, pdb_path = os.path.join(case, 'map.mrc'), os.path.join(case, 'ID_af3_docked.pdb')
        mrc.write_mrc(map_path, mrc.MrcMap(data=src_np, voxel_size=header.voxel_size))
        synthetic.write_pdb(pdb_path, dict(st, hetero=np.zeros(len(st['coords']), bool)))
        af3_results, grids = os.path.join(case, 'AF3_results') + '/', os.path.join(case, 'grids') + '/'
        pool = HostPool()
        ring = ctx.ring

        class RingModel:
            """Stand-in for MICA.forward: logits of the first b cubes of the ring (views made once per size)."""

            def __init__(self):
                self.views = {}

            def eval(self):
                return self

            def __call__(self, x, af):
                b = x.shape[0]
                v = self.views.get(b)
                if v is None:
                    bb, ca, aa = ring[0]
                    v = self.views[b] = (bb[:b], ca[:b], aa[:b])
                return v

        phase = {}

        def once():
            t = [time.perf_counter()]

            def lap(name):
                t.append(time.perf_counter())
                phase[name] = phase.get(name, 0.0) + (t[-1] - t[-2]) * 1e3
            dp = DataPreprocessor(map_path=map_path, AF3_results=af3_results, quiet=True)
            dp.resample_and_normalize_map()
            lap('resample_and_normalize_map (MRC read + upload + GPU + status)')
            ok = dp.create_AF3_encodings(pdb_path)
            lap('create_AF3_encodings (PDB parse + upload + atom bins)')
            gc = GridCreator(quiet=True)
            r1 = gc.create_normalized_map_grids(dp.normalized_map_path, os.path.join(grids, 'normalized_map_grids'),
                                                args.grid_size, args.padding)
            r2 = gc.create_AF3_encodings_grids(dp.AF3_encodings, os.path.join(grids, 'AF3_encoding_grids'),
                                               args.grid_size, args.padding)
            lap('GridCreator x2 (index only)')
            pr = CryoEMPredictor(model_path='unused', grids_path=grids, output_path=os.path.join(wd, 'out'),
                                 save_output=False, device=str(ctx.dev), quiet=True, model=RingModel(),
                                 host_volumes=host_volumes, host_pool=pool, super_batch=args.batch_cubes)
            good, vols = pr.run_prediction()
            lap('CryoEMPredictor.run_prediction (cut + model ring + stitch + D2H)')
            assert ok and r1['success'] and r2['success'] and good, 'drop-in sequence failed'
            return vols, pr
        vols, pr = once()                                   # warm: pinned pool, buffers
        torch.cuda.synchronize()
        phase.clear()
        t0 = time.perf_counter()
        for _ in range(steps):
            vols, pr = once()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        d2h = sum(int(np.prod(v.shape)) * 4 for k, v in vols.items() if isinstance(v, np.ndarray))
        h2d = src_np.nbytes + st['coords'].nbytes + 2 * len(st['coords'])
        session.clear()
        return {'value': n_vox / dt / 1e9, 'unit': UNIT, 'ms_per_step': dt * 1e3, 'steps': steps,
                'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                'model_batch': pr._model_batch(), 'host_volumes': list(host_volumes),
                'phase_ms_per_step': {k: round(v / steps, 2) for k, v in phase.items()},
                'timing_stats_last': {k: round(float(v), 4) for k, v in pr.timing_stats.items()},
                'note': 'the utils/modeler.py:673-734 sequence through mica_b200.{DataPreprocessor, GridCreator, '
                        'CryoEMPredictor}: MRC map + PDB model read from tmpfs, model = logits ring fed in the '
                        "reference's batches, volumes returned as host arrays (a DeviceVolume for the ones not "
                        'listed in host_volumes)'}
    finally:
        shutil.rmtree(wd, ignore_errors=True)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from mica_b200 import ops, synthetic
    from mica_b200.pdb import channel_codes
    from mica_b200.pipeline import MapHeader, MapPipeline, _no_timer, run_map_pipeline_host

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit('launch with torch.distributed.run for --gpus > 1')
    ops.require_gpu()
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    numa = bind_to_gpu_numa(local_rank) if world > 1 else None
    saved_stdout = None
    if world > 1:
        # NCCL prints its version banner on stdout; the contract is ONE JSON line there
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group('nccl', device_id=dev)

    ctx = Ctx()
    ctx.args, ctx.dist, ctx.world, ctx.rank, ctx.local_rank, ctx.dev = args, dist, world, rank, local_rank, dev
    sync, measure = make_measure(ctx)
    ctx.measure = measure

    # ---------------- synthetic inputs (host), seed 2022
    e = args.src_edge
    src_np = synthetic.synthetic_map((e, e, e), voxel=args.voxel, seed=2022 + rank)
    header = MapHeader(voxel_size=(np.float32(args.voxel),) * 3)
    n_out = ops.zoom_output_shape(src_np.shape, [np.float32(args.voxel)] * 3)
    # atoms are replicated on every rank (a few MB) and span the whole (stacked) working grid: one
    # 20 k-residue chain per slab, so that every rank has the same AF3 work (weak scaling)
    parts = [synthetic.synthetic_structure(20000, (n_out[2], n_out[1], n_out[0]), seed=2022 + r) for r in range(world)]
    st1 = {k: (v.copy() if isinstance(v, np.ndarray) else list(v)) for k, v in parts[0].items()}
    for r, part in enumerate(parts):
        part['coords'][:, 2] += np.float32(r * n_out[0])
    st = {k: (np.concatenate([p_[k] for p_ in parts]) if isinstance(parts[0][k], np.ndarray)
              else sum((list(p_[k]) for p_ in parts), [])) for k in parts[0]}
    bb_ch, aa_ch = channel_codes(st['atom_names'], st['res_names'])
    src_host = torch.from_numpy(src_np).pin_memory()
    atoms_host = (torch.from_numpy(st['coords']).pin_memory(), torch.from_numpy(bb_ch).pin_memory(),
                  torch.from_numpy(aa_ch).pin_memory())
    src = src_host.to(dev)
    atoms = tuple(t.to(dev) for t in atoms_host)
    inputs = (src, header, atoms)

    def make_pipe(af3_mode, gs=args.grid_size, pad=args.padding):
        if world > 1:
            from mica_b200.slab import SlabPipeline
            p = SlabPipeline(dev, rank, world, grid_size=gs, padding=pad, batch_cubes=args.batch_cubes, af3_mode=af3_mode)
            # the stacked map is not cubic: use the geometrically meant clip bounds instead of the
            # reference's (z,y,x)-vs-(x,y,z) mix-up (D7), which would squash every atom onto z <= nx-1
            p.af3_clip = (n_out[2] - 1, n_out[1] - 1, n_out[0] * world - 1)
            return p
        return MapPipeline(dev, grid_size=gs, padding=pad, batch_cubes=args.batch_cubes, af3_mode=af3_mode)

    # ---------------- logits ring (stands where MICA.forward stands), >> L2
    W, B = args.grid_size + 2 * args.padding, args.batch_cubes
    gen = torch.Generator(device=dev).manual_seed(2022)
    ring = [tuple(torch.randn((B, c, W, W, W), generator=gen, device=dev) * 2 for c in (4, 4, 21)) for _ in range(2)]
    state = {'i': 0}

    def model_fn(x, af):
        bb, ca, aa = ring[state['i'] % len(ring)]
        state['i'] += 1
        b = x.shape[0]
        return bb[:b], ca[:b], aa[:b]
    ctx.ring, ctx.ring_model = ring, model_fn

    pipe = make_pipe(args.af3_mode)
    # pass 1 (not the headline): every stage bracketed by events -> the per-stage breakdown and which
    # single-kernel stage dominates.  pass 2 (the headline): the K timed steps with events around the
    # dominant kernel's launches only, as the roofline line needs its live launch duration.
    _, stages_all, _, _, vols, _ = measure(pipe, inputs, model_fn)
    single_kernel_stages = ('postproc_stitch', 'extract_af3', 'extract_map', 'normalize_apply')
    dom_stage = max((k for k in single_kernel_stages if k in stages_all), key=lambda k: stages_all[k][1])
    del vols
    ms_per_step, stages, launches, clk, vols, host_ms = measure(pipe, inputs, model_fn, True, only={dom_stage})
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, vols)
    n_vox_rank = int(np.prod(pipe.normalized.shape)) if world == 1 else pipe.owned_voxels
    n_vox = n_vox_rank * world
    value = n_vox / (ms_per_step * 1e-3) / 1e9
    n_cubes = len(pipe.ijk_host)
    peak, peak_src = peaks()
    S = args.grid_size
    f = (W / S) ** 3
    n_src = src.numel()
    n_atoms = atoms[0].shape[0]

    # ---------------- variants (never the headline): the reference's dense-AF3 dataflow, and its default geometry
    variant, variant_48_8 = None, None
    if not args.no_variant and world == 1:
        other = 'dense' if args.af3_mode == 'sparse' else 'sparse'
        del vols
        vols = None
        pipe2 = make_pipe(other)
        ms2, stages2, _, _, vols2, _ = measure(pipe2, inputs, model_fn, steps=min(args.steps, 10))
        bn = sum(algorithmic_bytes(n_src, n_vox_rank, n_atoms, f).values())
        variant = {'af3_mode': other, 'ms_per_step': ms2, 'value': n_vox / (ms2 * 1e-3) / 1e9, 'unit': UNIT,
                   'stage_ms_per_step': stage_table(stages2, min(args.steps, 10))}
        if other == 'dense':
            variant['dense_path_frac'] = bn / (ms2 * 1e-3) / 1e9 / peak
            variant['dense_path_note'] = ('SURVEY 8(d) B(N) = 4 Ns + N (420 + 100 f) bytes -- the dataflow the reference '
                                          'materialises -- over this variant\'s step time and the measured HBM peak')
        del pipe2, vols2
        torch.cuda.empty_cache()
        # reference-default geometry: grid_size 48, padding 8 (utils/create_grids.py:89), 661 B/voxel
        f48 = (64 / 48) ** 3
        v48 = {'geometry': 'grid_size=48, padding=8 (reference default; the unmodified reference stitcher '
                           'supports only this padding)', 'cubes': int(np.prod([-(-n // 48) for n in n_out]))}
        for mode in ('sparse', 'dense'):
            p48 = make_pipe(mode, 48, 8)
            ms48, st48, _, _, vv, _ = measure(p48, inputs, model_fn, steps=min(args.steps, 10))
            b48 = sum((algorithmic_bytes if mode == 'dense' else sparse_bytes)(n_src, n_vox_rank, n_atoms, f48).values())
            v48[mode] = {'ms_per_step': ms48, 'value': n_vox / (ms48 * 1e-3) / 1e9, 'unit': UNIT,
                         'bytes_per_voxel': b48 / n_vox_rank, 'frac_of_peak': b48 / (ms48 * 1e-3) / 1e9 / peak,
                         'stage_ms_per_step': stage_table(st48, min(args.steps, 10))}
            del p48, vv
            torch.cuda.empty_cache()
        v48['dense_path_frac'] = v48['dense']['frac_of_peak']
        v48['note'] = ('dense: B(N) = 661 B/voxel of SURVEY 8(d) over the dense-AF3 step time; sparse: the bytes the '
                       'sparse dataflow moves over its step time')
        variant_48_8 = v48
        # north_star's overlap-weighted stitching (NOT the reference's arithmetic, DESIGN.md D2): every voxel of
        # every 64^3 window is post-processed and accumulated with its weight, then divided
        po = make_pipe(args.af3_mode)
        for _ in range(2):
            po.run(src, header, atoms, model_fn, None, overlap_window='uniform')
        sync()
        eo0, eo1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        eo0.record()
        for _ in range(5):
            po.run(src, header, atoms, model_fn, None, defer_check=True, overlap_window='uniform')
        eo1.record()
        sync()
        po.finish()
        ms_o = eo0.elapsed_time(eo1) / 5
        variant['overlap_weighted_stitch'] = {
            'window': 'uniform', 'ms_per_step': ms_o, 'value': n_vox / (ms_o * 1e-3) / 1e9, 'unit': UNIT,
            'note': "BASELINE north_star's wording of the stitch (accumulate prediction x weight and weight volumes, "
                    'divide); the reference pastes disjoint cores, which is what every other number in this line '
                    'does.  8x the voxels of the core-only mode go through softmax and 23 float atomics each'}
        del po
        torch.cuda.empty_cache()
        vols = pipe.run(src, header, atoms, model_fn, None)

    # ---------------- several maps in flight (a stream of maps).  Reported as a variant.
    in_flight = None
    if args.maps_in_flight > 1 and world == 1:
        n_f = args.maps_in_flight
        pipes = [pipe] + [make_pipe(args.af3_mode) for _ in range(n_f - 1)]
        streams = [torch.cuda.Stream(dev) for _ in range(n_f)]
        fv = [vols] + [None] * (n_f - 1)
        for p_ in pipes:
            p_.timer = _no_timer

        def run_many(k):
            start = torch.cuda.Event(enable_timing=True)
            start.record()
            for st_ in streams:
                st_.wait_event(start)
            for s_ in range(k):
                i_ = s_ % n_f
                with torch.cuda.stream(streams[i_]):
                    fv[i_] = pipes[i_].run(src, header, atoms, model_fn, fv[i_], defer_check=True)
            for st_ in streams:
                torch.cuda.current_stream().wait_stream(st_)
            end = torch.cuda.Event(enable_timing=True)
            end.record()
            return start, end

        run_many(max(args.warmup, args.steps))
        sync()
        for p_ in pipes:
            p_.finish()
        a_, b_ = run_many(args.steps)
        sync()
        for p_ in pipes:
            p_.finish()
        ms_f = a_.elapsed_time(b_) / args.steps
        in_flight = {'maps_in_flight': n_f, 'ms_per_step': ms_f, 'value': n_vox / (ms_f * 1e-3) / 1e9, 'unit': UNIT,
                     'note': 'K steps issued round-robin on %d independent pipelines/streams; throughput of a stream of '
                             'maps, not the latency of one' % n_f}
        vols = fv[0]
        del pipes, fv
        torch.cuda.empty_cache()

    # ---------------- end to end through the public API with host buffers
    # (every rank copies its own source block in and its own slab of the four volumes out)
    out_host = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in vols.as_dict().items()}
    dev_vols = vols                                                 # device volumes reused by every e2e step

    def time_e2e(out):
        if world > 1:
            dist.barrier()      # ranks leave the pinned allocation above seconds apart; the halo exchange waits, but not forever
        run_map_pipeline_host(src_host, header, atoms_host, model_fn, pipe, out, dev_vols)       # warm
        sync()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            _, h2d_, d2h_ = run_map_pipeline_host(src_host, header, atoms_host, model_fn, pipe, out, dev_vols)
        sync()
        dt_ = (time.perf_counter() - t0) / args.e2e_steps
        if world > 1:
            t_ = torch.tensor([dt_], device=dev, dtype=torch.float64)
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
            dt_ = float(t_.item())
        return dt_, h2d_, d2h_

    dt, h2d, d2h = time_e2e(out_host)
    e2e = {'value': n_vox / dt / 1e9, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d) * world,
           'd2h_bytes_per_step': int(d2h) * world, 'ms_per_step': dt * 1e3, 'steps': args.e2e_steps,
           'd2h_gb_per_s_aggregate': d2h * world / dt / 1e9, 'cpu_binding': numa,
           'note': 'pinned host map + atoms -> device -> four stitched volumes -> pinned host (finished x-layers are '
                   'copied out on side streams while later cube batches run); '
                   'host wall clock between device synchronisations, max over ranks'}
    # the same call with amino_acid_probability (20 of the 23 channels) left in HBM: what the drop-in for the
    # head of Solver.clustering (mica_b200/candidates.py, SURVEY 8f N1) makes possible -- its only consumer in
    # the reference (utils/modeler.py:850) then runs on the device.  This is the drop-in's default hand-over
    # (CryoEMPredictor returns that volume as a DeviceVolume).  Reported next to e2e, never instead of it.
    out3 = {k: v for k, v in out_host.items() if k != 'amino_acid_probability'}
    dt3, h2d3, d2h3 = time_e2e(out3)
    e2e3 = {'value': n_vox / dt3 / 1e9, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d3) * world,
            'd2h_bytes_per_step': int(d2h3) * world, 'ms_per_step': dt3 * 1e3, 'steps': args.e2e_steps,
            'd2h_gb_per_s_aggregate': d2h3 * world / dt3 / 1e9,
            'note': 'as e2e, but amino_acid_probability stays on the device for mica_b200.candidates '
                    '(utils/modeler.py:767-860 on the GPU); backbone / C-alpha / amino_acid_prediction go to the host'}
    del out_host, out3, dev_vols, vols
    torch.cuda.empty_cache()

    dropin = None
    if world == 1 and not args.no_dropin:
        from mica_b200.predict import MAP_TYPES, SMALL_VOLUMES
        try:
            dropin = {'all_four_to_host': e2e_dropin(ctx, src_np, header, st1, n_vox, MAP_TYPES, max(2, args.e2e_steps - 2)),
                      'default': e2e_dropin(ctx, src_np, header, st1, n_vox, SMALL_VOLUMES, args.e2e_steps)}
            dropin['ratio_to_e2e'] = dropin['all_four_to_host']['ms_per_step'] / e2e['ms_per_step']
            dropin['default_ratio_to_e2e_aa_prob_resident'] = dropin['default']['ms_per_step'] / e2e3['ms_per_step']
        except Exception as ex:                                   # a broken optional block must not lose the line
            dropin = {'error': f'{type(ex).__name__}: {ex}'[:300]}

    # free the headline's buffers before the large blocks
    del pipe
    torch.cuda.empty_cache()

    strong = None
    if not args.no_strong:
        try:
            strong = {'resampled': strong_720(ctx, identity=False), 'copy_path_d10': strong_720(ctx, identity=True)}
        except Exception as ex:
            strong = {'error': f'{type(ex).__name__}: {ex}'[:300]}
            if world > 1:
                raise
    c5 = None
    if not args.no_config5:
        del ring
        ctx.ring = None
        torch.cuda.empty_cache()
        try:
            c5 = config5(ctx)
        except Exception as ex:
            c5 = {'error': f'{type(ex).__name__}: {ex}'[:300]}
            if world > 1:
                raise

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel (the single-kernel stage with the most time)
    sparse = args.af3_mode == 'sparse'
    alg = algorithmic_bytes(n_src, n_vox_rank, n_atoms, f)
    moved = sparse_bytes(n_src, n_vox_rank, n_atoms, f) if sparse else alg
    stage_ms = stage_table(stages_all, args.steps)
    # stage -> (kernel, SURVEY 8(d) algorithmic bytes per step of that kernel)
    single = {
        'postproc_stitch': ('postproc_stitch_kernel', alg['postproc_stitch'], '208 B/voxel: 29 logit channels of '
                            'each core voxel read (116 B), 23 output channels written (92 B)'),
        'extract_af3': ('extract_tma_kernel<4> (24 AF3 channels)', 96 * n_vox_rank * (1 + f),
                        '96 B/voxel x (1 + f): 24 channels read once, written f = (W/S)^3 times'),
        'extract_map': ('extract_tma_kernel<4> (map channel)', 4 * n_vox_rank * (1 + f),
                        '4 B/voxel x (1 + f): map read once, written f = (W/S)^3 times'),
        'normalize_apply': ('normalize_apply_kernel', 8 * n_vox_rank, '8 B/voxel: read + write in place'),
    }
    dom = dom_stage
    calls, tot_ms = stages[dom]
    launches_per_step = calls / args.steps
    per_launch_bytes = single[dom][1] / launches_per_step
    dur_ms = tot_ms / calls
    achieved = per_launch_bytes / (dur_ms * 1e-3) / 1e9
    traffic, traffic_note = None, None
    tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tpath):      # dram bytes per launch from the committed `ncu --set full` capture
        t = json.load(open(tpath)).get(single[dom][0].split(' ')[0])
        if t and t.get('batch_cubes') == args.batch_cubes and t.get('grid_size') == S:
            # the capture is a FULL batch_cubes launch; the live figure is the average launch of the step
            # (the last batch is short): scale the captured traffic to the same number of cubes
            avg_cubes = n_cubes / launches_per_step
            traffic = t['dram_bytes_per_launch'] * avg_cubes / args.batch_cubes
            traffic_note = (f'ncu dram bytes of a full {args.batch_cubes}-cube launch ({t["dram_bytes_per_launch"]:.4g}) '
                            f'scaled to the average live launch of {avg_cubes:.1f} cubes, like algorithmic_bytes_per_launch')
    stage_frac = {}
    for name, keys in (('resample', ['resample']), ('normalize', ['order_stats', 'normalize_apply']),
                       ('af3_encode', ['af3_encode', 'af3_bin_atoms']),
                       ('extract', ['extract_map', 'extract_af3', 'af3_fill_cubes']),
                       ('postproc_stitch', ['postproc_stitch'])):
        t_ms = sum(stage_ms.get(k, 0.0) for k in keys)
        if t_ms:
            stage_frac[name] = round(moved[name] / (t_ms * 1e-3) / 1e9 / peak, 4)
    total_moved = sum(moved.values())
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic (seed 2022; random-init stand-in logits)',
        'config': workload_config(args, world) | {'working_grid': list(n_out) if world == 1 else
                                                  [n_out[0] * world, n_out[1], n_out[2]], 'cubes': n_cubes,
                                                  'atoms': int(n_atoms)},
        'roofline': {
            'bound': 'hbm', 'kernel': single[dom][0], 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
            'frac': achieved / peak, 'traffic': traffic, 'traffic_note': traffic_note,
            'peak_source': peak_src, 'launch_ms': dur_ms, 'launches_per_step': launches_per_step,
            'algorithmic_bytes_per_launch': per_launch_bytes, 'algorithmic_bytes_rule': single[dom][2],
            'share_of_step': tot_ms / args.steps / ms_per_step,
            # the whole path against the bytes THIS dataflow moves (sparse AF3: the 24 channels are never
            # materialised, so SURVEY 8(d)'s B(N) does not apply to it; the dense variant's B(N) fraction is
            # variant.dense_path_frac / variant_48_8.dense_path_frac)
            'whole_path': {'dataflow': args.af3_mode, 'bytes_moved_per_voxel': total_moved / n_vox_rank,
                           'achieved': total_moved / (ms_per_step * 1e-3) / 1e9,
                           'frac': total_moved / (ms_per_step * 1e-3) / 1e9 / peak,
                           'survey_B_N_bytes_per_voxel': sum(alg.values()) / n_vox_rank},
            'stage_ms_per_step': stage_ms, 'stage_frac_of_peak': stage_frac,
            'stage_note': 'stage times come from a separate fully instrumented pass of the same K steps; with the '
                          'prefetch stream extract / fill overlap the stitch, so they do not add up to ms_per_step; '
                          'fractions use the bytes the ' + args.af3_mode + ' dataflow moves per stage',
        },
        'af3_mode': args.af3_mode, 'variant': variant, 'variant_48_8': variant_48_8,
        'clocks': clk, 'gpu_launches': int(launches), 'host_enqueue_ms_per_step': host_ms,
        'e2e': e2e, 'e2e_aa_prob_resident': e2e3, 'e2e_dropin': dropin, 'variant_maps_in_flight': in_flight,
        'strong_720': strong, 'config5': c5,
    }
    if not args.no_cpu_baseline:
        if world == 1:
            line['cpu_baseline'], _ = cpu_baseline(args)
        else:
            line['cpu_baseline'] = {'note': 'timed at N = 1 only (rank 0 of the 1-GPU run); see that line'}
    if saved_stdout is not None:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
