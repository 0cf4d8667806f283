"""Drop-in for the reference's ``utils/predict.py::CryoEMPredictor``.

Same constructor and ``run_prediction() -> (bool, {four volumes})`` contract
(utils/predict.py:48,589; consumer: Solver.nnPred, utils/modeler.py:722-734).  The
model (models/model.py::MICA, PyTorch convolutions) is used as it is; everything
around it -- cube assembly, softmax/argmax, stitching -- runs in libmica_b200.so on the
``MapPipeline`` that DataPreprocessor / GridCreator prepared (``MapPipeline.predict_and_stitch``,
the path ``bench.py`` measures): cubes are cut 256 at a time on a side stream into reused
buffers, the AF3 channels are rasterised straight from the docked atoms, the model is fed in the
reference's batches (1, or <= 8 above 200 cubes), its logits are post-processed and their cores
pasted into the four volumes, and finished layers of the volumes stream to pinned host memory
while later cubes are still in the model.  When only the reference's ``.npz`` files exist on
disk, the cubes are uploaded from them instead.

With ``devices=`` (or ``MICA_DEVICES``) the cubes of one map are dealt over several GPUs of this process:
one thread, ``MapPipeline``, stream and model replica per device, every model call the same as on one
device, every core stored into one volume block on the predictor's ``device`` over NVLink."""
from __future__ import annotations

import copy
import glob
import logging
import os
import re
import threading
import time
from collections.abc import Mapping

import numpy as np
import torch

from . import ops, pdb, session
from ._lib import check, lib
from .pipeline import (MapPipeline, _SlabDrain, deal_cubes, run_model_chunks, shared_pipeline, worker_batches,
                       worker_pipeline)

MAP_TYPES = ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_prediction',
             'amino_acid_probability')
SMALL_VOLUMES = MAP_TYPES[:3]


def parse_devices(spec, n_visible: int, allow_repeats: bool = True):
    """``devices=`` / ``MICA_DEVICES`` -> a list of CUDA device indices, or None for the one-device path.

    None or '' -> None; 'all' -> every visible device; '0,2,3' or a list of ints, 'N' or 'cuda:N' strings or
    ``torch.device`` -> those devices.  Repeats (several workers on one GPU) only with ``allow_repeats``.
    Anything else raises ValueError."""
    if spec is None:
        return None
    if isinstance(spec, str):
        text = spec.strip()
        if not text:
            return None
        if text.lower() == 'all':
            if n_visible < 1:
                raise ValueError('devices=all: no CUDA device is visible')
            return list(range(n_visible))
        items = text.split(',')
    else:
        items = list(spec)
        if not items:
            return None
    out = []
    for it in items:
        try:
            if isinstance(it, torch.device):
                d = it
            elif isinstance(it, (int, np.integer)) and not isinstance(it, bool):
                d = torch.device('cuda', int(it))
            elif isinstance(it, str) and it.strip().isdigit():
                d = torch.device('cuda', int(it.strip()))
            elif isinstance(it, str):
                d = torch.device(it.strip())
            else:
                raise ValueError
        except (ValueError, RuntimeError):
            raise ValueError(f'devices: cannot read {it!r} as a CUDA device (in {spec!r})') from None
        if d.type != 'cuda' or d.index is None or not 0 <= d.index < n_visible:
            raise ValueError(f'devices: {it!r} is not one of the {n_visible} visible CUDA devices (in {spec!r})')
        out.append(d.index)
    if not allow_repeats and len(set(out)) != len(out):
        raise ValueError(f'devices: {spec!r} lists a device twice')
    return out


class HostPool:
    """Pinned host buffers for the stitched volumes, reused from map to map (``cudaHostAlloc`` of the
    10 GB a 480^3 map returns costs seconds and synchronises the device).  Arrays handed out for one
    map are overwritten by the next map that uses the same pool -- pass a pool only when the previous
    map's volumes are no longer needed; without one every predictor allocates its own buffers."""

    def __init__(self):
        self._bufs = {}

    def get(self, name, shape, dtype=torch.float32):
        shape = tuple(int(v) for v in shape)
        t = self._bufs.get(name)
        if t is None or tuple(t.shape) != shape or t.dtype != dtype:
            t = self._bufs[name] = torch.empty(shape, dtype=dtype).pin_memory()
        return t


class DeviceVolume:
    """A stitched volume that stayed in HBM, usable where the reference expects the NumPy array:
    ``shape`` / ``dtype`` / indexing / ``np.asarray`` work, a full host copy is made (once) only when
    something asks for all of it.  ``mica_b200.candidates`` takes ``.tensor`` and never copies --
    ``amino_acid_probability`` is 20 of the 23 output channels and its only consumer in the reference is a
    gather at the picked C-alpha voxels (utils/modeler.py:850)."""

    #: item reads served by device gathers before the volume is downloaded once and for all: an unmodified
    #: Solver.clustering reads 27 voxels per picked C-alpha one at a time (utils/modeler.py:846-851)
    GATHERS_BEFORE_DOWNLOAD = 32

    def __init__(self, tensor: torch.Tensor):
        self.tensor = tensor
        self._host = None
        self._gathers = 0

    shape = property(lambda self: tuple(self.tensor.shape))
    ndim = property(lambda self: self.tensor.dim())
    size = property(lambda self: self.tensor.numel())
    dtype = property(lambda self: np.dtype(np.float32))

    def __len__(self):
        return self.tensor.shape[0]

    def numpy(self):
        if self._host is None:
            self._host = self.tensor.cpu().numpy()
        return self._host

    def __array__(self, dtype=None, copy=None):
        a = self.numpy()
        return a if dtype is None else a.astype(dtype, copy=False)

    def __getitem__(self, idx):
        if self._host is None:
            self._gathers += 1
            if self._gathers > self.GATHERS_BEFORE_DOWNLOAD:
                self.numpy()
        if self._host is not None:
            return self._host[idx]
        dev = self.tensor.device

        def conv(i):
            if isinstance(i, np.ndarray):
                return torch.from_numpy(np.ascontiguousarray(i)).to(dev)
            if isinstance(i, (list,)):
                return torch.as_tensor(i, device=dev)
            if isinstance(i, np.integer):
                return int(i)
            return i
        tidx = tuple(conv(i) for i in idx) if isinstance(idx, tuple) else conv(idx)
        out = self.tensor[tidx]
        return out.cpu().numpy() if out.dim() else np.float32(out.item())


class CryoEMPredictor:
    def __init__(self, model_path, grids_path, output_path, save_output=True, device='cuda', quiet=False,
                 model=None, keep_on_device=True, host_volumes=None, host_pool=None, reference_batching=False,
                 super_batch=256, release_inputs=True, devices=None, *, overlap_window=None):
        """Additions to the reference signature (all optional):

        ``model``               an already loaded model (callable ``(exp_map, af_features) -> (bb, ca, aa)``).
        ``host_volumes``        the volumes copied to the host as NumPy arrays.  Default: the three
                                single-channel volumes; ``amino_acid_probability`` is returned as a
                                ``DeviceVolume`` (array-like, downloads itself when read as a whole).
                                ``MAP_TYPES`` returns four NumPy arrays exactly as the reference does.
        ``keep_on_device``      keep the four device volumes registered (``session`` key
                                ``<output_path>/results/device_volumes``) for ``mica_b200.candidates``.
        ``host_pool``           a ``HostPool`` whose pinned buffers receive the host volumes (reused from map
                                to map); default: fresh pinned buffers per predictor.
        ``reference_batching``  D8: False (default) never lets a cube without AF3 signal share a model call
                                with one that has some, so every cube gets the logits of the reference's
                                single-sample mode whatever the batch size; True reproduces the reference's
                                batched mode literally -- cubes in ``glob`` order (utils/predict.py:269) when
                                the grid files exist, mixed batches of ``optimal_batch_size``.
        ``super_batch``         cubes cut / stitched per kernel launch.
        ``release_inputs``      drop the consumed session entries (normalised map, atoms, cube indices) when
                                done, as Solver.nnPred deletes the files (utils/modeler.py:753-758).
        ``devices``             deal the map's cubes over several GPUs of this process: 'all', '0,2,3', or a list
                                of ints / 'cuda:N'; None reads ``MICA_DEVICES`` when ``run_prediction`` is called
                                (unset or empty: one device).  ``device`` is always worker 0 and receives the
                                volumes.  A device listed n times in ``devices`` runs n workers, each with its
                                own stream.  Every model call sees the cubes, in the order, it sees on one device
                                with the same options, so the volumes do not depend on the device count.  The
                                model is loaded once per GPU; an ``nn.Module`` given as ``model`` is deep-copied
                                to the other GPUs, or ``model`` may be a {device: callable} mapping.
        ``overlap_window``      (keyword only) None: the reference's paste of the cube cores.  'uniform',
                                'triangle' or W = grid_size + 2 * padding weights: overlap-weighted stitching
                                (``ops.OverlapStitcher``; NOT the reference's arithmetic, DESIGN.md D2), the same bits
                                on one device and with ``devices=``.  'core' is the paste."""
        self.devices = devices
        self.overlap_window = overlap_window
        self.worker_cubes = None                        # cubes each worker ran (several devices only)
        self._workers = None
        self._models = None
        self.keep_on_device = bool(keep_on_device)
        self.host_volumes = SMALL_VOLUMES if host_volumes is None else tuple(host_volumes)
        self.host_pool = host_pool
        self.reference_batching = bool(reference_batching)
        self.super_batch = int(super_batch)
        self.release_inputs = bool(release_inputs)
        self.model_path = model_path
        self.grids_path = grids_path
        self.output_path = output_path
        self.temp_output_path = os.path.join(output_path, 'results', 'predicted_grids')
        parts = str(grids_path).split('/')
        self.reconstruction_path = os.path.join(output_path, 'results', parts[-2] if len(parts) > 1 else parts[-1])
        self.save_output = save_output.lower() == 'true' if isinstance(save_output, str) else bool(save_output)
        self.device = device
        self.quiet = quiet
        self.batch_threshold = 200                      # utils/predict.py:72
        self.model = model
        self.use_optimized_batching = False
        self.sample_count = 0
        self.optimal_batch_size = 1
        self.timing_stats = {k: 0 for k in ('strategy_selection', 'model_loading', 'data_loading', 'inference',
                                            'reconstruction', 'saving', 'total')}
        self.logger = logging.getLogger(__name__)
        self._source = None

    def _print_status(self, message):
        if not self.quiet:
            print(message)

    # ------------------------------------------------------------------ data source
    def _map_dir(self):
        return os.path.join(str(self.grids_path).rstrip('/'), 'normalized_map_grids')

    def _af3_dir(self):
        return os.path.join(str(self.grids_path).rstrip('/'), 'AF3_encoding_grids')

    def _resolve_source(self):
        """Resident volumes registered by GridCreator, else the reference's files on disk."""
        m = session.get(self._map_dir())
        if m is not None:
            a = session.get(self._af3_dir())
            self._source = {'kind': 'resident', 'map': m, 'af3': a, 'ijk': m['ijk'], 'cube_shape': m['cube_shape'],
                            'grid_size': m['grid_size'], 'padding': m['padding']}
            return len(m['ijk'])
        files = sorted(glob.glob(os.path.join(self._map_dir(), '*.npz')))
        if not files:
            return 0
        first = np.load(files[0])
        gs, pad = int(first['grid_size']), int(first['padding'])
        ijk = np.array([[int(np.load(f)[k]) for k in ('i', 'j', 'k')] for f in files], dtype=np.int32)
        self._source = {'kind': 'files', 'files': files, 'ijk': ijk,
                        'cube_shape': tuple(int(v) for v in np.asarray(first['orig_shape']).ravel()),
                        'grid_size': gs, 'padding': pad}
        return len(files)

    # utils/predict.py:156-215
    def _calculate_optimal_batch_size(self):
        per_sample_gb = (64 ** 3 * 25 * 5) / 1024 ** 3
        try:
            free = torch.cuda.get_device_properties(torch.device(self.device)).total_memory / 1024 ** 3 * 0.7
        except Exception:
            return 1
        return int(min(max(1, free / per_sample_gb), 8))      # capped at 8 as in the reference (:174)

    def select_processing_strategy(self):
        t0 = time.time()
        try:
            self.sample_count = self._resolve_source()
            if self.sample_count == 0:
                self.logger.error(f'No grid files found in: {self._map_dir()}/')
                return False
            self.use_optimized_batching = self.sample_count > self.batch_threshold
            if self.use_optimized_batching:
                self.optimal_batch_size = self._calculate_optimal_batch_size()
            return True
        except Exception as e:
            self.logger.error(f'Strategy selection failed: {e}')
            return False
        finally:
            self.timing_stats['strategy_selection'] = time.time() - t0

    # ------------------------------------------------------------------ several devices
    def _resolve_workers(self):
        """The worker devices (worker 0 = ``device``), or None for the one-device path."""
        from_env = self.devices is None
        spec = os.environ.get('MICA_DEVICES') if from_env else self.devices
        if spec is None or (isinstance(spec, str) and not spec.strip()):
            return None
        idx = parse_devices(spec, torch.cuda.device_count(), allow_repeats=not from_env)
        if idx is None:
            return None
        primary = torch.device(self.device)
        if primary.type != 'cuda':
            raise ops._lib.MicaError(f'devices= needs a CUDA device, got device={self.device!r}')
        if primary.index is None:
            primary = torch.device('cuda', torch.cuda.current_device())
        if primary.index in idx:
            idx.remove(primary.index)                   # its first listing is worker 0
        workers = [primary] + [torch.device('cuda', i) for i in idx]
        return workers if len(workers) > 1 else None

    def _replicate_model(self, devs):
        """{device: callable} for every distinct worker device; False (logged) if the model cannot be placed."""
        model = self.model
        if isinstance(model, Mapping):
            given = {}
            for k, v in model.items():
                d = torch.device('cuda', k) if isinstance(k, int) else torch.device(k)
                given[torch.device('cuda', torch.cuda.current_device()) if d.index is None else d] = v
            missing = [str(d) for d in devs if d not in given]
            if missing:
                self.logger.error(f'model mapping has no entry for {", ".join(missing)}')
                return False
            self._models = {d: given[d] for d in devs}
            return True
        if len(devs) > 1 and not isinstance(model, torch.nn.Module):
            self.logger.error('a model that is not an nn.Module cannot be copied to several devices: '
                              'pass model={device: callable}')
            return False
        self._models = {devs[0]: model}
        for d in devs[1:]:
            self._models[d] = copy.deepcopy(model).to(d)
        return True

    # utils/predict.py:217-258
    def load_model(self):
        t0 = time.time()
        try:
            devs = list(dict.fromkeys(self._workers)) if self._workers else None
            if self.model is not None:
                return True if devs is None else self._replicate_model(devs)
            if not os.path.exists(self.model_path):
                self.logger.error(f'Model file not found: {self.model_path}')
                return False
            if devs is None:
                self.model = self._load_checkpoint(self.device)
                return True
            self._models = {d: self._load_checkpoint(d) for d in devs}
            self.model = self._models[devs[0]]
            return True
        except Exception as e:
            self.logger.error(f'Model loading failed: {e}')
            return False
        finally:
            self.timing_stats['model_loading'] = time.time() - t0

    def _load_checkpoint(self, device):
        from models.model import MICA                           # the reference's model, unchanged
        model = MICA().to(device)
        checkpoint = torch.load(self.model_path, map_location=device)
        state = {k.replace('module.', ''): v.to(device) for k, v in checkpoint['model_state_dict'].items()}
        model.load_state_dict(state, strict=False)
        model.eval()
        return model

    # ------------------------------------------------------------------ inference + stitch
    def _model_batch(self):
        return self.optimal_batch_size if self.use_optimized_batching else 1

    def _reference_order(self):
        """The cube order of the reference's DataLoader: ``glob.glob`` over the grid files
        (utils/predict.py:269, shuffle=False) -- directory order, when the files exist; the creation
        (loop) order otherwise.  Returns indices into the pipeline's cube list, or None."""
        files = glob.glob(os.path.join(self._map_dir(), '*.npz'))
        if not files:
            return None
        where = {tuple(int(v) for v in row): n for n, row in enumerate(self._source['ijk'])}
        order = []
        for f in files:
            mt = re.search(r'_i(-?\d+)_j(-?\d+)_k(-?\d+)\.npz$', os.path.basename(f))
            if mt is None or tuple(int(g) for g in mt.groups()) not in where:
                return None
            order.append(where[tuple(int(g) for g in mt.groups())])
        return order if sorted(order) == list(range(len(where))) else None

    def _pipeline(self, dev):
        """The MapPipeline holding this map: the one DataPreprocessor started, else a fresh one around
        the registered volume."""
        s = self._source
        m, a = s['map'], s['af3']
        pipe = m.get('pipe') or shared_pipeline(m['volume'].device)
        n = len(s['ijk'])
        pipe.configure(grid_size=s['grid_size'], padding=s['padding'], batch_cubes=max(1, min(self.super_batch, n)))
        pipe.set_normalized(m['volume'], m['header'])
        if a is not None and a.get('atoms') is not None:
            if not pipe.encode_af3(*a['atoms']):            # bins for the final geometry; cannot fail if
                raise IndexError('atom index outside the grid')    # create_AF3_encodings succeeded
        elif a is not None:
            vol = a['volume']
            pipe.af3, pipe._atoms_binned = (vol.get() if hasattr(vol, 'get') else vol), False
        else:
            pipe.af3, pipe._atoms_binned = None, False      # dataset/dataset.py:218-219: zeros
        return pipe

    def _host_buffers(self, vols):
        out = {}
        for k, v in vols.as_dict().items():
            if k in self.host_volumes:
                out[k] = (self.host_pool.get(k, v.shape) if self.host_pool is not None
                          else torch.empty(tuple(v.shape), dtype=v.dtype).pin_memory())
        return out

    def _fetch_files(self, b0, b1, dev):
        """dataset/dataset.py:194-224 for the reference's .npz files: (exp_map, af_features, flags)."""
        s = self._source
        W = s['grid_size'] + 2 * s['padding']
        B = b1 - b0
        xs, afs = [], []
        for f in s['files'][b0:b1]:
            xs.append(np.load(f)['grid'])
            try:
                feats = []
                for name in pdb.CHANNEL_NAMES:
                    p = f.replace('normalized_map_grids', f'AF3_encoding_grids/{name}_grids')
                    feats.append(np.load(p.replace('normalized_map', name))['grid'])
                afs.append(np.stack(feats))
            except Exception:
                afs.append(np.zeros((24, W, W, W), np.float32))
        x = torch.from_numpy(np.stack(xs)[:, None].astype(np.float32)).to(dev)
        af = torch.from_numpy(np.stack(afs).astype(np.float32)).to(dev)
        flags = (af.abs().reshape(B, -1).sum(1) > 0).to(torch.int32)
        return x, af, flags

    def _download(self, vols):
        """The host volumes of finished device volumes (one synchronisation)."""
        out_host = self._host_buffers(vols)
        with torch.cuda.device(vols.device):
            for k, t in out_host.items():
                t.copy_(getattr(vols, k), non_blocking=True)
            torch.cuda.current_stream(vols.device).synchronize()
        return out_host

    def _overlap_weights(self):
        """The window of an overlap-weighted map (checked before any launch), or None for the paste."""
        if self.overlap_window is None:
            return None
        gs, pad = self._source['grid_size'], self._source['padding']
        w1 = ops.overlap_window(self.overlap_window, gs, pad)
        return None if ops.is_core_window(w1, gs, pad) else w1

    def run_inference_and_reconstruct(self):
        """run_inference + reconstruct_volume (utils/predict.py:307-512) fused.  Returns
        (device volumes, {name: pinned host tensor})."""
        w1 = self._overlap_weights()
        if self._workers:
            return self._run_on_devices(self._workers, w1)
        dev = torch.device(self.device)
        s = self._source
        gs, pad = s['grid_size'], s['padding']
        model = self.model
        if hasattr(model, 'eval'):
            model.eval()
        d8 = 'reference' if self.reference_batching else 'split'
        with torch.no_grad():
            if s['kind'] == 'resident':
                pipe = self._pipeline(dev)
                order = self._reference_order() if self.reference_batching else None
                self._pipe = pipe
                if w1 is not None:                          # nothing is final before the last cube: no drain
                    vols = pipe.predict_and_stitch(model, None, model_batch=self._model_batch(), d8=d8, order=order,
                                                   overlap_window=w1)
                    return vols, self._download(vols)
                pipe.cube_index()
                vols = pipe._new_volumes()
                out_host = self._host_buffers(vols)
                drain = _SlabDrain(pipe, out_host)
                vols = pipe.predict_and_stitch(model, vols, on_batch=drain, model_batch=self._model_batch(),
                                               d8=d8, order=order)
                drain.finish()
                torch.cuda.current_stream(pipe.device).synchronize()
                self._pipe = pipe
                return vols, out_host
            # the reference's per-cube files: upload, then the same model feeding and stitching
            if dev.type != 'cuda':
                raise ops._lib.MicaError('mica_b200 has no CPU path')
            ijk_dev = torch.from_numpy(np.ascontiguousarray(s['ijk'], dtype=np.int32)).to(dev)
            if w1 is not None:
                overlap = ops.OverlapStitcher(s['cube_shape'], dev, gs, pad, w1)
                vols = overlap.vols
            else:
                overlap, vols = None, ops.StitchedVolumes(s['cube_shape'], dev)

            def stitch(bb, ca, aa, ijk):
                bb, ca, aa = bb.contiguous().float(), ca.contiguous().float(), aa.contiguous().float()
                if overlap is not None:
                    overlap.accumulate(bb, ca, aa, ijk)
                else:
                    ops.postproc_stitch(bb, ca, aa, ijk, vols, gs, pad)
            step = max(self._model_batch(), 1) * 4
            for b0 in range(0, self.sample_count, step):
                b1 = min(self.sample_count, b0 + step)
                x, af, flags = self._fetch_files(b0, b1, dev)
                run_model_chunks(model, x, af, flags.cpu().numpy(), ijk_dev[b0:b1], stitch, self._model_batch(), d8)
            if overlap is not None:
                overlap.finalize()
            return vols, self._download(vols)

    def _run_on_devices(self, workers, w1=None):
        """The map's cubes dealt over ``workers`` (``deal_cubes``), one thread each.  Every worker stores its
        cores into ONE 23-channel block on workers[0] (``postproc_stitch_peer`` with a one-entry owner table) --
        or, with the window ``w1``, adds its weighted contributions into it (``ops.OverlapStitcher`` with that
        table), which workers[0] finalises after the last worker has finished; the host copies run once, after
        that.  Returns what ``run_inference_and_reconstruct`` returns."""
        s = self._source
        gs, pad = s['grid_size'], s['padding']
        primary, n, mb = workers[0], len(s['ijk']), self._model_batch()
        d8 = 'reference' if self.reference_batching else 'split'
        resident = s['kind'] == 'resident'
        slots = [sum(1 for d in workers[:w] if d == workers[w]) for w in range(len(workers))]
        streams = [worker_pipeline(d, slot)[1] for d, slot in zip(workers, slots)]
        pipes = [None] * len(workers)
        if resident:
            # the normalised map (and the atoms, or a dense AF3 volume) once per device; workers on one device
            # share them.  Worker 0 continues on the map's own pipeline when that lives on the primary device.
            m, a = s['map'], s['af3']
            inputs = {}
            for w, (dev, slot) in enumerate(zip(workers, slots)):
                if w == 0 and m['volume'].device == dev:
                    pipes[0] = self._pipeline(dev)
                    continue
                if dev not in inputs:
                    af3 = None
                    if a is not None and a.get('atoms') is None:
                        vol = a['volume']
                        af3 = (vol.get() if hasattr(vol, 'get') else vol).to(dev)
                    inputs[dev] = (m['volume'].to(dev),
                                   tuple(t.to(dev) for t in a['atoms']) if a is not None and a.get('atoms') is not None
                                   else None, af3)
                norm, atoms, af3 = inputs[dev]
                pipe = worker_pipeline(dev, slot)[0]
                pipe.configure(grid_size=gs, padding=pad, batch_cubes=max(1, min(self.super_batch, n)))
                pipe.set_normalized(norm, m['header'])
                if atoms is not None:
                    if not pipe.encode_af3(*atoms):
                        raise IndexError('atom index outside the grid')
                else:
                    pipe.af3, pipe._atoms_binned = af3, False
                pipes[w] = pipe
            order = self._reference_order() if self.reference_batching else None
            order = np.arange(n, dtype=np.int64) if order is None else np.asarray(order, dtype=np.int64)
            pipes[0].cube_index()
            cube_shape = pipes[0].cube_shape
            super_batch = max(1, min(self.super_batch, n))
            self._pipe = pipes[0]
        else:
            if primary.type != 'cuda':
                raise ops._lib.MicaError('mica_b200 has no CPU path')
            cube_shape = s['cube_shape']
            super_batch = max(mb, 1) * 4
            ijk_dev = {d: torch.from_numpy(np.ascontiguousarray(s['ijk'], dtype=np.int32)).to(d)
                       for d in dict.fromkeys(workers)}
        ranges = deal_cubes(n, super_batch, mb, len(workers))
        self.worker_cubes = [hi - lo for lo, hi in ranges]
        X, Y, Z = (int(v) for v in cube_shape)
        for d in dict.fromkeys(workers):
            check(lib.mica_peer_enable(d.index, primary.index), f'peer_enable({d} -> {primary})')
        with torch.cuda.device(primary):
            block = torch.zeros(23 * X * Y * Z, dtype=torch.float32, device=primary)
            zeroed = torch.cuda.Event()
            zeroed.record()
        vols = ops.StitchedVolumes.from_block(block, cube_shape, (0, 0, 0), (X, Y, Z))
        tables = {d: torch.tensor([block.data_ptr()], dtype=torch.int64, device=d) for d in dict.fromkeys(workers)}
        overlap = None
        if w1 is not None:
            overlap = {d: ops.OverlapStitcher(cube_shape, d, gs, pad, w1, vols=vols if d == primary else None,
                                              owners=ops.OverlapOwners(tables[d], 0, (0, X), (primary.index,)))
                       for d in dict.fromkeys(workers)}
        for dev, st in zip(workers, streams):
            st.wait_stream(torch.cuda.current_stream(dev))     # inputs copied / binned on the current streams
            st.wait_event(zeroed)
        for model in self._models.values():
            if hasattr(model, 'eval'):
                model.eval()

        def body(w):
            lo, hi = ranges[w]
            if hi <= lo:
                return
            dev, table, model = workers[w], tables[workers[w]], self._models[workers[w]]

            def stitch(bb, ca, aa, ijk, _vols=None):
                bb, ca, aa = bb.contiguous().float(), ca.contiguous().float(), aa.contiguous().float()
                if overlap is not None:
                    overlap[dev].accumulate(bb, ca, aa, ijk)
                else:
                    ops.postproc_stitch_peer(bb, ca, aa, ijk, cube_shape, table, (0, X), gs, pad)
            with torch.cuda.device(dev), torch.cuda.stream(streams[w]), torch.no_grad():
                if resident:
                    pipes[w].predict_and_stitch(model, vols, model_batch=mb, d8=d8, order=order[lo:hi],
                                                batches=worker_batches(lo, hi, super_batch), stitch_fn=stitch)
                    return
                for b0, b1 in worker_batches(lo, hi, super_batch):
                    x, af, flags = self._fetch_files(lo + b0, lo + b1, dev)
                    run_model_chunks(model, x, af, flags.cpu().numpy(), ijk_dev[dev][lo + b0:lo + b1], stitch, mb, d8)

        errors = [None] * len(workers)

        def run(w):
            try:
                body(w)
            except BaseException as e:                   # re-raised below, after every worker has stopped
                errors[w] = e

        threads = [threading.Thread(target=run, args=(w,), name=f'mica-worker-{w}') for w in range(len(workers))]
        try:
            for t in threads:
                t.start()
        finally:
            for t in threads:
                if t.ident is not None:
                    t.join()
            for st in streams:
                st.synchronize()                         # the primary reads the block only after every worker
            for w, pipe in enumerate(pipes):
                if pipe is not None and pipe is not pipes[0]:
                    pipe.release_map()                   # the per-device copies of this map's inputs
        for e in errors:
            if e is not None:
                raise e
        if overlap is not None:
            overlap[primary].finalize()
        return vols, self._download(vols)

    def _release(self):
        s = self._source or {}
        if s.get('kind') != 'resident':
            return
        for entry in (s['map'], s['af3']):
            if entry is not None and entry.get('source') is not None:
                session.drop(entry['source'])
        session.drop(self._map_dir())
        session.drop(self._af3_dir())
        pipe = getattr(self, '_pipe', None)
        if pipe is not None:
            pipe.release_map()

    # utils/predict.py:589-634
    def run_prediction(self):
        t_total = time.time()
        try:
            self._workers = self._resolve_workers()
            if not self.select_processing_strategy():
                return False, {}
            if not self.load_model():
                return False, {}
            t0 = time.time()
            vols, out_host = self.run_inference_and_reconstruct()
            self.timing_stats['inference'] = time.time() - t0
            t0 = time.time()
            dev_key = os.path.join(str(self.output_path), 'results', 'device_volumes')
            if self.keep_on_device:
                session.put(dev_key, **vols.as_dict())
            volumes = {}
            for k, v in vols.as_dict().items():
                volumes[k] = out_host[k].numpy() if k in out_host else DeviceVolume(v)
            self.timing_stats['reconstruction'] = time.time() - t0
            if self.save_output:
                t0 = time.time()
                os.makedirs(self.reconstruction_path, exist_ok=True)
                for k in MAP_TYPES:
                    np.save(f'{self.reconstruction_path}/{k}.npy', np.asarray(volumes[k]))
                self.timing_stats['saving'] = time.time() - t0
            if self.release_inputs:
                self._release()
            self.timing_stats['total'] = time.time() - t_total
            return True, volumes
        except Exception as e:                                   # reference: logged, (False, {}) (:632-634)
            self.logger.error(f'Prediction pipeline failed: {e}')
            return False, {}
