#!/usr/bin/env python3
"""python tools/bench_bf16.py [--reps R] [--warmup W] [--out FILE]

float32 against bfloat16 model-facing buffers on one GPU (``cube_dtype`` / ``CryoEMPredictor(precision='bf16')``).

(a) Kernels at bench.py's workload: a synthetic 400^3 map at 1.2 A resampled to the 480^3 working grid, 64^3 windows
    at stride 32 (grid_size 32, padding 16), batches of 512 cubes.  CUDA-event time per launch, median over R
    repetitions after W warm-ups, the two dtypes alternated launch by launch in this process:
      extract_map   ops.extract_cubes of the normalised map into [512, 1, 64^3];
      af3_fill      Af3CubeFiller.fill, alternating two batches (every call clears one cube set and sets another);
      paste         ops.postproc_stitch of 512 cubes of logits (the cores);
      accumulate    the weighted ops.Stitcher, 'triangle' window (every window voxel).
    Algorithmic bytes from the shapes: extract = float32 window read + window written in the dtype; paste = 26 logit
    channels read per core voxel + 23 float32 written; accumulate = 26 logit channels read + 22 uint32 sums added per
    window voxel; the fill moves a few bytes per atom voxel and is reported as time only.  Every working set is larger
    than L2 (126 MB).
(b) models/model.py::MICA when importable (bench.load_mica), random weights after torch.manual_seed(2022): 64 cubes
    of bench.py's config5 map (512^3 at 1.0 A, grid_size 48, padding 8, its atoms), model batch 8; ms per cube in
    float32 (cudnn.allow_tf32 as it is, recorded) against bfloat16 inputs under torch.autocast, and the largest power
    of two model batch (8..256) that runs for each.
(c) With that model: the four volumes of a 192^3 synthetic map (64 cubes, seed 2022, with atoms) from a float32 and a
    bfloat16 pipeline; max |dp| of backbone / carbon_alpha and the fraction of equal amino_acid_prediction.  Random
    weights: this says nothing about the accuracy of the trained model in bf16.
Prints one JSON line that names the card and its power limit."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from mica_b200 import ops, synthetic
from mica_b200.pdb import channel_codes
from mica_b200.pipeline import MapHeader, MapPipeline

GS, PAD, B = 32, 16, 512
W = GS + 2 * PAD
DTYPES = {'fp32': torch.float32, 'bf16': torch.bfloat16}


def _card(index):
    name = torch.cuda.get_device_name(index)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i',
                            str(index)], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unknown'
    return name, q


def _alternate(fns, reps, warmup):
    """{name: median ms} of each fn, the fns run in turn within every repetition."""
    for _ in range(warmup):
        for fn in fns.values():
            fn()
    ts = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts[k].append(a.elapsed_time(b))
    return {k: float(np.median(v)) for k, v in ts.items()}


def _atoms(shape_zyx, dev, per=5500, seed=2022):
    st = synthetic.synthetic_structure(int(np.prod(shape_zyx)) // per, shape_zyx[::-1], seed=seed)
    bb_ch, aa_ch = channel_codes(st['atom_names'], st['res_names'])
    return tuple(torch.from_numpy(a).to(dev) for a in (st['coords'], bb_ch, aa_ch))


def kernels(dev, reps, warmup):
    src = synthetic.synthetic_map((400,) * 3, voxel=1.2, seed=2022)
    pipe = MapPipeline(dev, GS, PAD, batch_cubes=B)
    assert pipe.resample_and_normalize(torch.from_numpy(src).to(dev), MapHeader(voxel_size=(np.float32(1.2),) * 3))
    n_out = tuple(pipe.normalized.shape)
    assert pipe.encode_af3(*_atoms(n_out, dev))
    pipe.cube_index()
    ijk, ijk2 = pipe.ijk[:B], pipe.ijk[B:2 * B]
    res = {'map': {'grid': list(n_out), 'cubes': len(pipe.ijk_host)}}
    fillers = {'fp32': pipe._fillers[0]}
    fillers['bf16'] = ops.Af3CubeFiller(dev, B, GS, PAD, pipe.perm, dtype=torch.bfloat16)
    fillers['bf16'].share_bins(pipe._fillers[0])
    xs = {k: torch.empty((B, 1, W, W, W), dtype=dt, device=dev) for k, dt in DTYPES.items()}
    g = torch.Generator(device=dev).manual_seed(7)
    logits32 = [torch.randn((B, c, W, W, W), device=dev, generator=g) for c in (4, 4, 21)]
    logits = {'fp32': logits32, 'bf16': [t.to(torch.bfloat16) for t in logits32]}
    vols = ops.StitchedVolumes(pipe.cube_shape, dev)
    acc = ops.Stitcher(pipe.cube_shape, dev, GS, PAD, 'triangle')
    turn = {k: 0 for k in DTYPES}

    def fill(k):
        turn[k] ^= 1
        fillers[k].fill(ijk if turn[k] else ijk2)
    fns = {}
    for k in DTYPES:
        fns['extract_map', k] = (lambda k=k: ops.extract_cubes(pipe.normalized, ijk, GS, PAD, pipe.perm, out=xs[k]))
        fns['af3_fill', k] = (lambda k=k: fill(k))
        fns['paste', k] = (lambda k=k: ops.postproc_stitch(*logits[k], ijk, vols, GS, PAD))
        fns['accumulate', k] = (lambda k=k: acc(*logits[k], ijk))
    ms = _alternate(fns, reps, warmup)
    for (name, k), t in ms.items():
        e = 4 if k == 'fp32' else 2
        nbytes = {'extract_map': B * W ** 3 * (4 + e), 'paste': B * GS ** 3 * (26 * e + 23 * 4),
                  'accumulate': B * W ** 3 * (26 * e + 22 * 4)}.get(name)
        row = res.setdefault(name, {})
        row[f'{k}_ms'] = round(t, 4)
        if nbytes is not None:
            row[f'{k}_GBps'] = round(nbytes / (t * 1e-3) / 1e9, 1)
    for name in ('extract_map', 'af3_fill', 'paste', 'accumulate'):
        res[name]['bf16_over_fp32'] = round(res[name]['bf16_ms'] / res[name]['fp32_ms'], 3)
    fillers['bf16'].clear()
    return res


def _model_call(model, dt):
    if dt == torch.float32:
        return model

    def call(x, af):
        with torch.autocast('cuda', dtype=torch.bfloat16):
            return model(x, af)
    return call


def model_section(dev, reps):
    sys.path.insert(0, ROOT)
    import bench
    MICA, where = bench.load_mica()
    if MICA is None:
        return {'unavailable': 'models/model.py not importable'}
    torch.manual_seed(2022)
    model = MICA().to(dev).eval()
    out = {'model_from': where, 'cudnn_allow_tf32': bool(torch.backends.cudnn.allow_tf32),
           'matmul_allow_tf32': bool(torch.backends.cuda.matmul.allow_tf32)}
    src = synthetic.synthetic_map_device((512,) * 3, dev, voxel=1.0, seed=2022)
    st = synthetic.synthetic_structure(6400, (512, 512, 512), seed=2022)
    bb_ch, aa_ch = channel_codes(st['atom_names'], st['res_names'])
    atoms = tuple(torch.from_numpy(a).to(dev) for a in (st['coords'], bb_ch, aa_ch))
    hdr = MapHeader(voxel_size=(np.float32(1.0),) * 3)
    cubes = {}
    for k, dt in DTYPES.items():
        p = MapPipeline(dev, 48, 8, batch_cubes=64, cube_dtype=dt)
        assert p.resample_and_normalize(src, hdr) and p.encode_af3(*atoms)
        p.cube_index()
        x, af = p.extract_batch(600, 664)
        cubes[k] = (x.clone(), af.clone())
    per_cube = {}
    with torch.no_grad():
        fns = {k: (lambda k=k: [_model_call(model, DTYPES[k])(cubes[k][0][b:b + 8], cubes[k][1][b:b + 8])
                                for b in range(0, 64, 8)]) for k in DTYPES}
        ms = _alternate(fns, reps, 1)
        for k in DTYPES:
            per_cube[k] = round(ms[k] / 64, 3)
        out['ms_per_cube'] = per_cube
        out['bf16_speedup'] = round(per_cube['fp32'] / per_cube['bf16'], 3)
        biggest = {}
        for k, dt in DTYPES.items():
            fits = None
            for mb in (8, 16, 32, 64, 128, 256):
                try:
                    x = cubes[k][0][:1].expand(mb, -1, -1, -1, -1).contiguous()
                    af = cubes[k][1][:1].expand(mb, -1, -1, -1, -1).contiguous()
                    _model_call(model, dt)(x, af)
                    torch.cuda.synchronize()
                    fits = mb
                    del x, af
                except torch.cuda.OutOfMemoryError:
                    break
                finally:
                    torch.cuda.empty_cache()
            biggest[k] = fits
        out['largest_model_batch'] = biggest

        # (c) agreement on a 192^3 map, random weights
        small = synthetic.synthetic_map((192,) * 3, voxel=1.0, seed=2022)
        vols = {}
        for k, dt in DTYPES.items():
            p = MapPipeline(dev, 48, 8, batch_cubes=16, cube_dtype=dt)
            assert p.resample_and_normalize(torch.from_numpy(small).to(dev), hdr)
            assert p.encode_af3(*_atoms((192,) * 3, dev))
            v = p.predict_and_stitch(_model_call(model, dt), model_batch=8, d8='split')
            vols[k] = {n: t.cpu().numpy() for n, t in v.as_dict().items()}
    a, b = vols['fp32'], vols['bf16']
    out['agreement_192'] = {
        'cubes': 64,
        'max_abs_dp_backbone': float(np.abs(a['backbone_probability'] - b['backbone_probability']).max()),
        'max_abs_dp_carbon_alpha': float(np.abs(a['carbon_alpha_probability'] - b['carbon_alpha_probability']).max()),
        'equal_amino_acid_prediction': float((a['amino_acid_prediction'] == b['amino_acid_prediction']).mean()),
        'note': 'random weights: not a statement about the trained model'}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--model-reps', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_bf16 needs a CUDA device')
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    out = {'tool': 'bench_bf16', 'grid_size': GS, 'padding': PAD, 'batch_cubes': B}
    out['card'], out['power_limit_max_sm_clock'] = _card(0)
    out['kernels'] = kernels(dev, args.reps, args.warmup)
    torch.cuda.empty_cache()
    out['model'] = model_section(dev, args.model_reps)
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
