"""Wall time of the drop-in sequence with one map's cubes dealt over 1, 2, 4, 8 GPUs of one process.

Each run is what a MICA user's script does: DataPreprocessor -> GridCreator -> CryoEMPredictor.run_prediction()
on the config-5 input (512^3 map at 1.0 A, ``synthetic_map_device`` seed 2022, ~50 k atoms, grid 48 / pad 8:
1331 cubes), with ``devices=`` listing the first n visible GPUs.  The model is models/model.py::MICA (random
weights, seed 2022) when it can be imported, else a Conv3d stand-in; the output says which ran and its time per
cube.  One warm-up run on every device count comes first (cuDNN algorithm choice, allocations, peer access).
Prints one JSON line per device count: wall time of ``run_prediction``, model time per worker (CUDA events),
cubes per worker, whether the four volumes equal the 1-device run bit for bit, and the GPU name and power limit
read in the same run.  Writes only to a temporary directory.

    python tools/bench_dropin_devices.py [--max-devices N]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mica_b200 import mrc, session, synthetic  # noqa: E402
from mica_b200.create_grids import GridCreator  # noqa: E402
from mica_b200.predict import CryoEMPredictor, HostPool  # noqa: E402
from mica_b200.preprocessing import DataPreprocessor  # noqa: E402


def load_mica():
    """models/model.py::MICA, unmodified: from sys.path, else the staged archive of the reference (as bench.py)."""
    try:
        from models.model import MICA
        return MICA, 'models.model on sys.path'
    except Exception:
        pass
    root = os.path.join(ROOT, 'oracle', '_ref', 'reference_py.zip')
    if os.path.exists(root):
        sys.path.insert(0, root)
        try:
            from models.model import MICA
            return MICA, root
        except Exception:
            sys.path.remove(root)
    return None, None


class StandIn(torch.nn.Module):
    """Three 3x3x3 convolutions (25 -> width -> width -> 29 channels) with MICA's signature."""

    def __init__(self, width):
        super().__init__()
        self.net = torch.nn.Sequential(torch.nn.Conv3d(25, width, 3, padding=1), torch.nn.ReLU(),
                                       torch.nn.Conv3d(width, width, 3, padding=1), torch.nn.ReLU(),
                                       torch.nn.Conv3d(width, 29, 3, padding=1))

    def forward(self, x, af):
        y = self.net(torch.cat([x, af], dim=1))
        return y[:, :4], y[:, 4:8], y[:, 8:]


class Timed:
    """Model call timed with CUDA events on the calling stream."""

    def __init__(self, model):
        self.model, self.spans, self.cubes = model, [], 0

    def eval(self):
        self.model.eval()
        return self

    def __call__(self, x, af):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = self.model(x, af)
        b.record()
        self.spans.append((a, b))
        self.cubes += int(x.shape[0])
        return out

    def take_ms(self):
        ms = sum(a.elapsed_time(b) for a, b in self.spans)
        self.spans, self.cubes = [], 0
        return ms


def gpu_info():
    out = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=index,name,power.limit', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        out['gpus'] = [line.strip() for line in q]
    except Exception as e:
        out['gpus'] = f'nvidia-smi unavailable: {e}'
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--max-devices', type=int, default=8)
    ap.add_argument('--edge', type=int, default=512, help='map edge (voxels); 512 = config 5')
    ap.add_argument('--emulate', action='store_true',
                    help='n workers on GPU 0 instead of n GPUs (the host cost of the worker threads, not a speed-up)')
    ap.add_argument('--width', type=int, default=32, help='hidden channels of the stand-in model')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this measurement runs on the GPU only')
    visible = 8 if args.emulate else torch.cuda.device_count()
    counts = [n for n in (1, 2, 4, 8) if n <= min(visible, args.max_devices)]
    gpu_of = (lambda w: 0) if args.emulate else (lambda w: w)
    info = gpu_info()
    MICA, where = load_mica()
    models = {}
    for d in sorted({gpu_of(w) for w in range(max(counts))}):
        torch.manual_seed(2022)                           # run.py:86: the same weights on every device
        m = (MICA() if MICA is not None else StandIn(args.width)).to(f'cuda:{d}').eval()
        models[torch.device('cuda', d)] = Timed(m)
    model_name = f'models.model.MICA ({where})' if MICA is not None else f'Conv3d stand-in (25-{args.width}-{args.width}-29, 3^3 kernels)'
    with tempfile.TemporaryDirectory() as td:
        case = os.path.join(td, 'input', 'ID')
        os.makedirs(os.path.join(case, 'AF3_results'))
        src = synthetic.synthetic_map_device((args.edge,) * 3, 'cuda:0', voxel=1.0, seed=2022).cpu().numpy()
        map_path = os.path.join(case, 'map.mrc')
        mrc.write_mrc(map_path, mrc.MrcMap(data=src, voxel_size=(np.float32(1.0),) * 3))
        del src
        n_res = max(1, round(6400 * (args.edge / 512) ** 3))
        pdb_path = os.path.join(case, 'ID_af3_docked.pdb')
        synthetic.write_pdb(pdb_path, synthetic.synthetic_structure(n_res, (args.edge,) * 3, seed=2022))
        pool = HostPool()

        def run(n_dev):
            session.clear()
            dp = DataPreprocessor(map_path=map_path, AF3_results=os.path.join(case, 'AF3_results'), quiet=True)
            dp.resample_and_normalize_map()
            assert dp.create_AF3_encodings(pdb_path)
            grids = os.path.join(case, 'grids') + '/'
            gc = GridCreator(quiet=True)
            assert gc.create_normalized_map_grids(dp.normalized_map_path, grids + 'normalized_map_grids')['success']
            assert gc.create_AF3_encodings_grids(dp.AF3_encodings, grids + 'AF3_encoding_grids')['success']
            out = os.path.join(td, 'out')
            pr = CryoEMPredictor('unused', grids, out, save_output=False, quiet=True, host_pool=pool,
                                 model=models[torch.device('cuda', 0)] if n_dev == 1 else models,
                                 devices=None if n_dev == 1 else [gpu_of(w) for w in range(n_dev)])
            for m in models.values():
                m.take_ms()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ok, _ = pr.run_prediction()
            wall = time.perf_counter() - t0
            assert ok, 'run_prediction failed'
            if args.emulate:                              # one model object serves every worker on GPU 0
                m = models[torch.device('cuda', 0)]
                cubes, model_ms = pr.worker_cubes or [m.cubes], [m.take_ms()]
            else:
                per_worker = [models[torch.device('cuda', d)] for d in range(n_dev)]
                cubes = [m.cubes for m in per_worker]
                model_ms = [m.take_ms() for m in per_worker]
            vols = session.get(os.path.join(out, 'results', 'device_volumes'))
            return wall, model_ms, cubes, pr, vols

        for n in sorted(set(counts), reverse=True):       # warm-up: every device count once
            run(n)
        ref = None
        for n in counts:
            wall, model_ms, cubes, pr, vols = run(n)
            if ref is None:
                ref = {k: v.clone() for k, v in vols.items()}
                same = True
            else:
                same = all(torch.equal(ref[k], vols[k]) for k in ref)
            rec = {'devices': n, 'emulated_on_gpu0': args.emulate, 'model': model_name, 'map_edge': args.edge, 'cubes': int(sum(cubes)),
                   'model_batch': pr._model_batch(), 'wall_s_run_prediction': round(wall, 4),
                   'model_ms_per_worker': [round(v, 2) for v in model_ms], 'cubes_per_worker': cubes,
                   'model_ms_per_cube': round(sum(model_ms) / max(1, sum(cubes)), 3),
                   'bit_identical_to_1_device': bool(same), 'gpu': info}
            if n == counts[0]:
                base = wall
            rec['speedup_vs_1_device'] = round(base / wall, 3)
            print(json.dumps(rec), flush=True)
            del vols
        session.clear()


if __name__ == '__main__':
    main()
