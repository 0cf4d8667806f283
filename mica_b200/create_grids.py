"""Drop-in for the reference's ``utils/create_grids.py::GridCreator``.

Same method names, arguments and result dictionaries (utils/create_grids.py:205-397).
By default no per-cube ``.npz`` file is written: the cube index (origins, window,
axis permutation) and the resident volume -- or, for the AF3 channels, just the atoms --
are registered under ``output_dir`` for CryoEMPredictor, which cuts the cubes on the GPU
straight into the model batch on the pipeline DataPreprocessor started.
``materialize=True`` also writes the reference's files (same names and keys).

``min_max`` (or the ``MICA_MIN_MAX`` environment variable): register -- and write -- only the cubes of the
normalised map whose window maximum is not below it, the rule the reference applies to its training grids
(create_grids_for_normalized_map.py:78).  CryoEMPredictor then predicts exactly those cubes; the cores of the
others stay 0, as in the reference's stitcher when a grid file is absent."""
from __future__ import annotations

import glob
import logging
import os
import time

import numpy as np
import torch

from . import mrc, ops, pdb, session
from ._lib import MicaError
from .pipeline import MapHeader


def env_min_max():
    """``MICA_MIN_MAX`` as a finite float, None when unset or empty; MicaError for anything else."""
    text = os.environ.get('MICA_MIN_MAX', '').strip()
    if not text:
        return None
    try:
        v = float(text)
    except ValueError:
        raise MicaError(f'MICA_MIN_MAX={text!r} is not a number') from None
    return ops.check_min_max(v)


class GridCreator:
    def __init__(self, quiet=False, device='cuda', materialize=False, min_max=None):
        """``min_max``: keep only the normalised map's cubes whose window maximum is not below this finite number
        (ties and windows holding a NaN are kept); None reads ``MICA_MIN_MAX`` (unset or empty: every cube).  A bad
        value is logged and the grid creation fails before any launch."""
        self.quiet = quiet
        self.device = torch.device(device)
        self.materialize = materialize
        self.min_max = min_max
        self.logger = logging.getLogger(__name__)
        self.processed_count = 0
        self.failed_count = 0
        self.failed_entries = []

    def print_clean(self, message):
        if not self.quiet:
            print(message)

    def transpose(self, numpy_image, axis_order, offset):
        """utils/create_grids.py:67-87 (kept for callers that use it directly)."""
        trans_offset, trans_order = [], []
        for i in range(3):
            for j in range(len(axis_order)):
                if axis_order[j] == i:
                    trans_offset.append(offset[j])
                    trans_order.append(j)
        return np.transpose(numpy_image, trans_order), trans_offset

    # ------------------------------------------------------------------ helpers
    def _load(self, path):
        entry = session.get(path)
        if entry is not None:
            self._pipe = entry.get('pipe')
            return entry['volume'], entry['header']
        self._pipe = None
        m = mrc.read_mrc(path)
        hdr = MapHeader(voxel_size=m.voxel_size, origin=m.origin, mapc=m.mapc, mapr=m.mapr, maps=m.maps,
                        nxstart=m.nxstart, nystart=m.nystart, nzstart=m.nzstart)
        vol = torch.from_numpy(np.array(m.data, dtype=np.float32)).to(self.device)
        return vol, hdr

    def _index(self, vol_shape, header, grid_size):
        perm, offset = header.transpose_order()
        cube_shape = ops.cube_space_shape(vol_shape, perm)
        return perm, offset, cube_shape, ops.cube_origins(cube_shape, grid_size)

    def _write_npz(self, vol, header, perm, cube_shape, ijk, output_dir, grid_size, padding, prefix, batch=16):
        """The reference's per-cube files (utils/create_grids.py:159-174), cut on the GPU."""
        os.makedirs(output_dir, exist_ok=True)
        d_ijk = torch.from_numpy(ijk).to(self.device)
        origin = np.rec.array(tuple(np.float32(v) for v in header.origin),
                              dtype=[('x', '<f4'), ('y', '<f4'), ('z', '<f4')])
        voxel = np.rec.array(tuple(np.float32(v) for v in header.voxel_size),
                             dtype=[('x', '<f4'), ('y', '<f4'), ('z', '<f4')])
        for b0 in range(0, len(ijk), batch):
            cubes = ops.extract_cubes(vol, d_ijk[b0:b0 + batch], grid_size, padding, perm).cpu().numpy()
            for n, (i, j, k) in enumerate(ijk[b0:b0 + batch]):
                di, dj, dk = (min(grid_size, int(cube_shape[a]) - int(v)) for a, v in enumerate((i, j, k)))
                np.savez(os.path.join(output_dir, f'{prefix}_i{i}_j{j}_k{k}.npz'), grid=cubes[n, 0],
                         i=int(i), j=int(j), k=int(k), di=di, dj=dj, dk=dk, orig_shape=cube_shape,
                         grid_size=grid_size, padding=padding, voxel_size=voxel, origin=origin,
                         mapc=header.mapc, mapr=header.mapr, maps=header.maps)

    # utils/create_grids.py:89-184
    def create_grids_from_mrc(self, mrc_file, output_dir, grid_size=48, padding=8, file_prefix='grid', *,
                              min_max=None):
        """``min_max``: only the cubes the keep rule keeps (``ops.select_cubes``) are registered and written."""
        try:
            min_max = ops.check_min_max(min_max)                  # refused before any launch
            vol, header = self._load(mrc_file)
            perm, offset, cube_shape, ijk = self._index(tuple(vol.shape), header, grid_size)
            if min_max is not None:
                maxima = ops.cube_window_max(vol, torch.from_numpy(ijk).to(vol.device), grid_size, padding, perm)
                ijk = np.ascontiguousarray(ijk[ops.select_cubes(maxima, min_max)])
            session.put(output_dir, kind='cubes', volume=vol, header=header, perm=perm, offset=offset,
                        cube_shape=cube_shape, ijk=ijk, grid_size=grid_size, padding=padding, prefix=file_prefix,
                        pipe=self._pipe, source=mrc_file, min_max=min_max)
            if self.materialize:
                self._write_npz(vol, header, perm, cube_shape, ijk, output_dir, grid_size, padding, file_prefix)
            return len(ijk), offset
        except Exception as e:                                   # reference: logged, (0, None) (:181-184)
            self.logger.error(f'Grid creation failed for {os.path.basename(str(mrc_file))}: {e}')
            return 0, None

    # utils/create_grids.py:205-267
    def create_normalized_map_grids(self, normalized_map_path, output_dir, grid_size=48, padding=8):
        start_time = time.time()
        if session.get(normalized_map_path) is None and not os.path.exists(normalized_map_path):
            error_msg = f'Normalized map not found: {normalized_map_path}'
            self.logger.error(error_msg)
            return {'success': False, 'error': error_msg}
        try:
            min_max = ops.check_min_max(self.min_max) if self.min_max is not None else env_min_max()
        except MicaError as e:
            self.logger.error(f'Grid creation refused: {e}')
            return {'success': False, 'error': str(e)}
        grid_count, offset = self.create_grids_from_mrc(normalized_map_path, output_dir, grid_size, padding,
                                                        'normalized_map_grid', min_max=min_max)
        return {'success': grid_count > 0, 'grid_count': grid_count, 'offset': offset,
                'output_directory': output_dir, 'processing_time': time.time() - start_time,
                'input_file': normalized_map_path}

    # utils/create_grids.py:269-397
    def create_AF3_encodings_grids(self, AF3_encodings_path, output_dir, grid_size=48, padding=8, parallel=True):
        start_time = time.time()
        entry = session.get(AF3_encodings_path)
        if entry is None and not os.path.exists(AF3_encodings_path):
            error_msg = f'AF3 encodings directory not found: {AF3_encodings_path}'
            self.logger.error(error_msg)
            return {'success': False, 'error': error_msg}
        errors, ok_channels = [], 0
        try:
            atoms, pipe = None, None
            if entry is not None:
                vol, header, names = entry['volume'], entry['header'], list(pdb.CHANNEL_NAMES)
                atoms, pipe = entry.get('atoms'), entry.get('pipe')
            else:
                files = glob.glob(os.path.join(AF3_encodings_path, '*_encoding.mrc'))
                if not files:
                    error_msg = f'No AF3 encoding files found in {AF3_encodings_path}'
                    self.logger.error(error_msg)
                    return {'success': False, 'error': error_msg}
                by_name = {os.path.basename(f).split('_encoding.mrc')[0]: f for f in files}
                names = [n for n in pdb.CHANNEL_NAMES if n in by_name]
                maps = [mrc.read_mrc(by_name[n]) for n in names]
                header = MapHeader(voxel_size=maps[0].voxel_size, origin=maps[0].origin, mapc=maps[0].mapc,
                                   mapr=maps[0].mapr, maps=maps[0].maps, nxstart=maps[0].nxstart,
                                   nystart=maps[0].nystart, nzstart=maps[0].nzstart)
                vol = torch.zeros((24,) + maps[0].data.shape, dtype=torch.float32, device=self.device)
                for n, m in zip(names, maps):
                    vol[pdb.CHANNEL_NAMES.index(n)] = torch.from_numpy(
                        np.array(m.data, dtype=np.float32)).to(self.device)
            perm, offset, cube_shape, ijk = self._index(tuple(vol.shape[1:]), header, grid_size)
            session.put(output_dir, kind='af3_cubes', volume=vol, header=header, perm=perm, offset=offset,
                        cube_shape=cube_shape, ijk=ijk, grid_size=grid_size, padding=padding, channels=names,
                        atoms=atoms, pipe=pipe, source=AF3_encodings_path)
            if self.materialize:
                dense = vol.get() if hasattr(vol, 'get') else vol      # LazyAf3Volume: rasterise now
                for name in names:
                    c = pdb.CHANNEL_NAMES.index(name)
                    self._write_npz(dense[c], header, perm, cube_shape, ijk,
                                    os.path.join(output_dir, f'{name}_grids'), grid_size, padding, f'{name}_grid')
            ok_channels = len(names)
        except Exception as e:
            errors.append(str(e))
            self.logger.error(f'AF3 grid creation failed: {e}')
        n_total = len(pdb.CHANNEL_NAMES) if entry is not None else max(ok_channels, 1)
        return {'success': ok_channels > 0, 'successful_channels': ok_channels,
                'failed_channels': 0 if ok_channels else n_total, 'total_channels': n_total,
                'total_grids': ok_channels * (len(ijk) if ok_channels else 0), 'output_directory': output_dir,
                'processing_time': time.time() - start_time, 'processing_errors': errors,
                'input_directory': AF3_encodings_path}
