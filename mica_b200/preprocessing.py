"""Drop-in for the reference's ``utils/preprocessing.py::DataPreprocessor``.

Same constructor, methods, return values and never-raise convention
(utils/preprocessing.py:42,80,225 and SURVEY.md 8b); the arithmetic runs in
libmica_b200.so on the GPU and the results stay resident (mica_b200.session) for
GridCreator / CryoEMPredictor, which continue on the SAME ``MapPipeline`` -- the one
``bench.py`` measures.  The reference's intermediate files (``resampled_normalized_map.mrc``,
24 ``*_encoding.mrc``) exist only to hand data to the next stage and are deleted by
``Solver.nnPred`` (utils/modeler.py:753-758); they are written with ``write_files=True``
(bit-identical payloads), not by default."""
from __future__ import annotations

import logging
import os

import numpy as np
import torch

from . import mrc, ops, pdb, session
from .pipeline import MapHeader, shared_pipeline


_STAGING = {}
#: integer payloads (MRC modes 0, 1, 6) go to the device as they are
_INT_UPLOAD = {np.dtype(np.int8): torch.int8, np.dtype(np.int16): torch.int16, np.dtype(np.uint16): torch.uint16}


def upload_map(data: np.ndarray, device) -> torch.Tensor:
    """Host map (typically the copy-on-write memory map ``mrc.read_mrc`` returns) -> device tensor: the
    planes are copied into a reused pinned staging buffer by a few threads (NumPy releases the GIL) and
    every finished chunk goes to the GPU at once, instead of one pageable copy of the whole map.
    int8 / int16 / uint16 maps keep their type (an int16 map crosses PCIe at half the float32 bytes);
    everything else becomes float32."""
    from concurrent.futures import ThreadPoolExecutor
    data = np.asarray(data)
    dev = torch.device(device)
    n = data.size
    tdt = _INT_UPLOAD.get(data.dtype, torch.float32)
    ndt = data.dtype if tdt is not torch.float32 else np.dtype(np.float32)
    out = torch.empty(data.shape, dtype=tdt, device=dev)
    if n < (1 << 22) or data.dtype != ndt or not data.flags.c_contiguous:
        out.copy_(torch.from_numpy(np.ascontiguousarray(data, dtype=ndt)))
        return out
    nbytes = n * ndt.itemsize
    stage = _STAGING.get('map')                          # bytes: one buffer serves maps of every type
    if stage is None or stage.numel() < nbytes:
        stage = _STAGING['map'] = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    typed = stage[:nbytes].view(tdt)
    flat_src, flat_dst, flat_out = data.reshape(-1), stage.numpy()[:nbytes].view(ndt), out.view(-1)
    chunks = 8
    bounds = [n * c // chunks for c in range(chunks + 1)]
    with torch.cuda.device(dev):
        torch.cuda.current_stream().synchronize()        # the staging buffer may still feed the previous map

        def fill(c):
            flat_dst[bounds[c]:bounds[c + 1]] = flat_src[bounds[c]:bounds[c + 1]]
            return c
        with ThreadPoolExecutor(4) as pool:
            for c in pool.map(fill, range(chunks)):
                flat_out[bounds[c]:bounds[c + 1]].copy_(typed[bounds[c]:bounds[c + 1]], non_blocking=True)
    return out


def _header_of(m, voxel_size=None):
    return MapHeader(voxel_size=m.voxel_size if voxel_size is None else voxel_size, origin=m.origin,
                     mapc=m.mapc, mapr=m.mapr, maps=m.maps, nxstart=m.nxstart, nystart=m.nystart,
                     nzstart=m.nzstart)


class LazyAf3Volume:
    """The dense [24,nz,ny,nx] AF3 volume of ``create_AF3_encodings`` -- built (10.6 GB at 480^3) only when
    somebody asks for it: the MRC writer, ``GridCreator(materialize=True)``.  The fast path rasterises
    the atoms straight into the cube batches and never needs it."""

    def __init__(self, atoms, origin, shape):
        self.atoms, self.origin, self.shape3 = atoms, origin, tuple(shape)
        self._vol = None

    @property
    def shape(self):
        return (24,) + self.shape3

    def get(self):
        if self._vol is None:
            vol, status = ops.af3_encode(*self.atoms, self.origin, self.shape3)
            if int(status.item()) != 0:
                raise IndexError('atom index out of bounds for the map axis (reference clip quirk)')
            self._vol = vol
        return self._vol


class DataPreprocessor:
    def __init__(self, map_path, AF3_results, normalized_map_path=None, quiet=True, device='cuda',
                 write_files=False, order=3):
        self.map_path = map_path
        self.AF3_results = AF3_results
        self.normalized_map_path = normalized_map_path
        self.quiet = quiet
        self.device = torch.device(device)
        self.write_files = write_files
        self.order = order
        self.logger = logging.getLogger(__name__)

    def print_clean(self, message):
        if not self.quiet:
            print(message)

    # utils/preprocessing.py:80-170
    def resample_and_normalize_map(self, target_voxel_size=1.0):
        success = False
        try:
            m = mrc.read_mrc(self.map_path)
            if m.mode not in (0, 1, 2, 6):
                # float16 (mode 12): scipy.ndimage.zoom refuses the array type, so the reference fails on it too
                raise ValueError(f'MRC mode {m.mode} maps are not supported (modes 0, 1, 2 and 6 are)')
            header = _header_of(m)
            pipe = shared_pipeline(self.device).configure(order=self.order, target_voxel_size=target_voxel_size)
            src = upload_map(m.data, pipe.device)
            if pipe.resample_and_normalize(src, header):
                out_path = os.path.join(os.path.dirname(self.AF3_results), 'resampled_normalized_map.mrc')
                out_header = _header_of(m, voxel_size=(np.float32(target_voxel_size),) * 3)
                if self.write_files:
                    os.makedirs(os.path.dirname(out_path) or '.', exist_ok=True)
                    mrc.write_mrc(out_path, mrc.MrcMap(
                        data=pipe.normalized.cpu().numpy(), voxel_size=out_header.voxel_size, origin=m.origin,
                        mapc=m.mapc, mapr=m.mapr, maps=m.maps, nxstart=m.nxstart, nystart=m.nystart,
                        nzstart=m.nzstart))
                pipe.header = out_header
                session.put(out_path, kind='normalized_map', volume=pipe.normalized, header=out_header,
                            median=pipe.median, p999=pipe.p999, pipe=pipe,
                            source_shape=tuple(int(v) for v in m.data.shape), source_header=header)
                self.normalized_map_path = out_path
                success = True
            else:
                reason = {1: 'No positive values found after thresholding',
                          2: 'Percentile value is zero - cannot normalize'}.get(pipe.norm_status, 'unknown')
                self.logger.error(f'Normalization failed: {reason}')
        except Exception as e:                                  # reference: swallowed and logged (:159-161)
            self.logger.error(f'Map processing failed: {e}')
        self.print_clean('Map successfully resampled and normalized' if success
                         else 'Map Resampling and Normalization Failed')

    def _reference_map(self):
        entry = session.get(self.normalized_map_path)
        if entry is not None:
            return tuple(entry['volume'].shape), entry['header'], entry.get('pipe')
        m = mrc.read_mrc(self.normalized_map_path)
        return m.data.shape, _header_of(m), None

    # utils/preprocessing.py:225-347
    def create_AF3_encodings(self, combined_docked_model_path):
        success = False
        try:
            shape, header, pipe = self._reference_map()
            coords, bb_ch, aa_ch, n_res = pdb.read_pdb_atoms(combined_docked_model_path)
            dev = pipe.device if pipe is not None else self.device
            atoms = tuple(torch.from_numpy(a).to(dev) for a in (coords, bb_ch, aa_ch))
            self.AF3_encodings = os.path.join(os.path.dirname(self.AF3_results), 'AF3_encodings')
            lazy = LazyAf3Volume(atoms, header.origin, shape)
            if pipe is not None and pipe.normalized is not None and tuple(pipe.normalized.shape) == tuple(shape):
                # fast path: bin the atoms per cube (the status word reports the reference's IndexError path, D7)
                if not pipe.encode_af3(*atoms):
                    raise IndexError('atom index out of bounds for the map axis (reference clip quirk)')
            else:
                lazy.get()
            if self.write_files:
                os.makedirs(self.AF3_encodings, exist_ok=True)
                host = lazy.get().cpu().numpy()
                for c, name in enumerate(pdb.CHANNEL_NAMES):
                    mrc.write_mrc(os.path.join(self.AF3_encodings, f'{name}_encoding.mrc'), mrc.MrcMap(
                        data=host[c], voxel_size=(np.float32(1),) * 3, origin=header.origin, mapc=header.mapc,
                        mapr=header.mapr, maps=header.maps, nxstart=header.nxstart, nystart=header.nystart,
                        nzstart=header.nzstart))
            session.put(self.AF3_encodings, kind='af3_encodings', volume=lazy, header=header,
                        atoms=atoms, n_atoms=len(coords), residues=n_res, pipe=pipe)
            success = True
        except Exception as e:                                  # reference: swallowed -> False (:344-347)
            self.print_clean(f'Encoding failed: AF3 encoding failed: {e}')
        return success
