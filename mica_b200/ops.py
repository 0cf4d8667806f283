"""Torch-tensor front end of the C ABI (device pointers in, device tensors out).

PyTorch is plumbing here -- it owns the HBM allocations and the stream; all the
arithmetic of the hot path happens in libmica_b200.so.  Every function raises
unless its tensors live on a CUDA device: there is no CPU path."""
from __future__ import annotations

import ctypes as C
import functools
import itertools
from typing import NamedTuple

import numpy as np
import torch

from . import _lib
from ._lib import lib, check

STANDARD_PERM = (2, 1, 0)     # trans_order for mapc,mapr,maps = 1,2,3 (utils/create_grids.py:120-122)


def _stream():
    """The caller's stream on the CURRENT device -- every entry point runs under ``device_guard``,
    which makes the device of its tensors current first (the C ABI launches on the CUDA runtime's
    current device)."""
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _cuda_device_of(a):
    if isinstance(a, torch.Tensor):
        return a.device if a.is_cuda else None
    d = getattr(a, 'device', None)
    if isinstance(d, torch.device) and d.type == 'cuda':
        return d if d.index is not None else torch.device('cuda', torch.cuda.current_device())
    return None


def device_guard(fn):
    """Run ``fn`` with the device of its CUDA arguments current: tensors, and objects that carry a
    ``.device`` (OrderStats, Af3CubeFiller, StitchedVolumes).  All of them must live on ONE
    device; a call whose tensors sit on cuda:1 while cuda:0 is current would otherwise launch on
    GPU 0, on a GPU-0 stream, against GPU-1 pointers."""
    @functools.wraps(fn)
    def wrapper(*args, **kw):
        dev = None
        for a in args + tuple(kw.values()):
            d = _cuda_device_of(a)
            if d is None:
                continue
            if dev is None:
                dev = d
            elif d != dev:
                raise _lib.MicaError(f'{fn.__name__}: arguments live on different devices ({dev} and {d})')
        if dev is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kw)
        with torch.cuda.device(dev):
            return fn(*args, **kw)
    return wrapper


def _dev(t: torch.Tensor, dtype, name: str):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.MicaError(f'{name} must be a CUDA tensor (mica_b200 has no CPU fallback)')
    if t.dtype != dtype:
        raise _lib.MicaError(f'{name} must be {dtype}, got {t.dtype}')
    if not t.is_contiguous():
        raise _lib.MicaError(f'{name} must be contiguous')
    return C.c_void_p(t.data_ptr())


#: element types of the model-facing buffers (cube batches, logits) -> MICA_DTYPE_* code; maps and volumes are float32
MODEL_DTYPES = {torch.float32: _lib.DTYPE_F32, torch.bfloat16: _lib.DTYPE_BF16}


def model_dtype(dtype) -> torch.dtype:
    """``dtype`` if it is a dtype the cube batches and logits can have (float32, bfloat16); MicaError otherwise."""
    if dtype not in MODEL_DTYPES:
        raise _lib.MicaError(f'model inputs and logits are torch.float32 or torch.bfloat16, got {dtype!r}')
    return dtype


def _logits(bb, ca, aa, B, W):
    """(pointers, MICA_DTYPE code) of one batch of logits: [B,4|4|21,W,W,W] CUDA tensors, contiguous, all float32 or
    all bfloat16."""
    for t, c, name in ((bb, 4, 'bb'), (ca, 4, 'ca'), (aa, 21, 'aa')):
        if tuple(t.shape) != (B, c, W, W, W):
            raise _lib.MicaError(f'{name} logits must be [{B},{c},{W},{W},{W}], got {tuple(t.shape)}')
    dt = bb.dtype
    if dt not in MODEL_DTYPES or ca.dtype != dt or aa.dtype != dt:
        raise _lib.MicaError(f'logits must be all float32 or all bfloat16, got {bb.dtype}, {ca.dtype}, {aa.dtype}')
    return (_dev(bb, dt, 'bb'), _dev(ca, dt, 'ca'), _dev(aa, dt, 'aa')), MODEL_DTYPES[dt]


def require_gpu():
    n = lib.mica_device_count()
    if n < 0:
        raise _lib.MicaError(f'no usable CUDA device: {_lib.last_error()}')
    return n


def launch_count() -> int:
    return int(lib.mica_launch_count())


# ------------------------------------------------------------------ R1 resample
def zoom_output_shape(in_zyx, zoom_zyx):
    """int(round(float32(n) * float32(zoom))) per axis (scipy.ndimage.zoom under NumPy 2)."""
    out = (C.c_int * 3)()
    check(lib.mica_zoom_output_shape(_lib.int3(in_zyx), _lib.float3(zoom_zyx), out), 'zoom_output_shape')
    return tuple(int(v) for v in out)


def resample_slab_source_planes(sz: int, nz: int, dst_z0: int, dst_nz_local: int):
    """Source planes [lo, hi) a rank holds so that its output planes [dst_z0, dst_z0+dst_nz_local) come out
    bit-identical to the whole map's (the z prefilter's segments and windows are those of the whole line)."""
    lo, hi = C.c_int(), C.c_int()
    check(lib.mica_resample_slab_source_planes(int(sz), int(nz), int(dst_z0), int(dst_nz_local),
                                               C.byref(lo), C.byref(hi)), 'resample_slab_source_planes')
    return int(lo.value), int(hi.value)


def resample_slab_source_planes_general(sz: int, nz: int, dst_z0: int, dst_nz_local: int):
    """The same for the general path that integer maps take (16 prefilter segments per z line, numbered on the
    whole line).  Raises MicaError unless 96 <= sz <= 800."""
    lo, hi = C.c_int(), C.c_int()
    check(lib.mica_resample_slab_source_planes_general(int(sz), int(nz), int(dst_z0), int(dst_nz_local),
                                                       C.byref(lo), C.byref(hi)), 'resample_slab_source_planes_general')
    return int(lo.value), int(hi.value)


#: sample types of the maps resample / normalize take -> MICA_DTYPE_* code
MAP_DTYPES = {torch.float32: _lib.DTYPE_F32, torch.int8: _lib.DTYPE_I8, torch.int16: _lib.DTYPE_I16,
              torch.uint16: _lib.DTYPE_U16}
#: integer maps (MRC modes 0, 1, 6): rounded resample, float64 statistics (DESIGN.md D12)
INT_DTYPES = (torch.int8, torch.int16, torch.uint16)


@device_guard
def resample(src: torch.Tensor, out_shape, order: int = 3, *, src_z0: int = 0, src_shape=None,
             dst_z0: int = 0, dst_nz_local=None, out: torch.Tensor | None = None) -> torch.Tensor:
    """Cubic B-spline (order=3) / trilinear (order=1) resample of ``src`` (sz,sy,sx) to
    the global shape ``out_shape``.  Slab form: ``src`` holds global planes
    [src_z0, src_z0+len) of a (src_shape) volume; planes [dst_z0, dst_z0+dst_nz_local)
    of the output are produced.  ``src`` is float32, int8, int16 or uint16 and the output has its
    type: an integer map is resampled in float64 and rounded as scipy.ndimage.zoom stores into an
    integer array (half away from zero, saturating; DESIGN.md D12)."""
    dt = src.dtype if isinstance(src, torch.Tensor) and src.dtype in MAP_DTYPES else torch.float32
    p_src = _dev(src, dt, 'src')
    code = MAP_DTYPES[dt]
    sz_l, sy, sx = src.shape
    sz = int(src_shape[0]) if src_shape is not None else sz_l
    nz, ny, nx = (int(v) for v in out_shape)
    nzl = nz - dst_z0 if dst_nz_local is None else int(dst_nz_local)
    if out is None:
        out = torch.empty((nzl, ny, nx), dtype=dt, device=src.device)
    p_out = _dev(out, dt, 'out')
    if tuple(out.shape) != (nzl, ny, nx):
        raise _lib.MicaError(f'out has shape {tuple(out.shape)}, expected {(nzl, ny, nx)}')
    nbytes = lib.mica_resample_workspace_bytes(sz_l, sy, sx, nz, ny, nx, order)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=src.device)
    check(lib.mica_resample(p_src, code, sz, sy, sx, src_z0, sz_l, p_out, code, nz, ny, nx, dst_z0, nzl,
                            C.c_void_p(ws.data_ptr()), nbytes, order, _stream()), 'resample')
    return out


# --------------------------------------------------------------- R2/R3 normalise
class OrderStats:
    """Device-resident state of the exact radix select (median + 99.9 percentile)."""

    def __init__(self, device, n_hint: int = 0):
        """``n_hint``: voxels per rank the workspace should hold a compact buffer for (0 = allocate it on the
        first ``run``).  The guided digit-0 pass compacts the candidate voxels there and the later digit passes
        read them instead of streaming the map four more times; without room they stream the map."""
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise _lib.MicaError(f'OrderStats needs a CUDA device, got {self.device} (mica_b200 has no CPU fallback)')
        self._n_cap = -1
        self._alloc(int(n_hint))

    def _alloc(self, n_local: int):
        with torch.cuda.device(self.device):
            nbytes = lib.mica_select_workspace_bytes_for(n_local) if n_local > 0 else lib.mica_select_workspace_bytes()
            self.ws = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
            self._p = C.c_void_p(self.ws.data_ptr())
            if n_local > 0:
                check(lib.mica_select_set_compact(self._p, nbytes, _stream()), 'select_set_compact')
            self._n_cap = n_local

    def hist_view(self) -> torch.Tensor:
        """int64 view of the histogram words a multi-GPU run all-reduces between hist and pick."""
        off = lib.mica_select_hist_ptr(self._p) - self.ws.data_ptr()
        return self.ws[off:off + 8 * _lib.SELECT_HIST_WORDS].view(torch.int64)

    @device_guard
    def run(self, x: torch.Tensor, n_total: int | None = None, all_reduce=None, peer=None):
        """Multi-GPU: the histograms of all ranks are summed between hist and pick, either by
        ``peer`` (a peer.PeerHistogram: one fused kernel over NVLink peer memory) or by
        ``all_reduce(hist_int64_tensor)`` (torch.distributed.all_reduce over NCCL), both on the
        current stream."""
        p_x = _dev(x, torch.float32, 'x')
        n_local = x.numel()
        n_total = n_local if n_total is None else int(n_total)
        if n_local > self._n_cap and n_local >= (1 << 22):     # first map, or a larger one: (re)size the compact buffer
            self._alloc(n_local)
        st = _stream()
        if all_reduce is None and peer is None:
            check(lib.mica_order_stats_f32(p_x, n_local, self._p, st), 'order_stats')
            return self
        check(lib.mica_select_init(self._p, n_total, st), 'select_init')
        hist = self.hist_view() if peer is None else None
        for r in range(_lib.SELECT_PASSES):
            check(lib.mica_select_hist(p_x, n_local, self._p, r, st), 'select_hist')
            if peer is not None:
                peer.reduce(self, r)
            else:
                all_reduce(hist)
            check(lib.mica_select_pick(self._p, r, st), 'select_pick')
        return self

    @device_guard
    def compact_info(self):
        """(in_use, floats_appended, capacity) of the compact buffer after a run -- synchronises the stream."""
        out = (C.c_int64 * 3)()
        with torch.cuda.device(self.device):
            check(lib.mica_select_compact_info(self._p, out, _stream()), 'select_compact_info')
        return bool(out[0]), int(out[1]), int(out[2])

    def result(self):
        """(median, p999, n_pos, status) -- synchronises the stream."""
        med, p, npos, status = C.c_float(), C.c_float(), C.c_int64(), C.c_int()
        check(lib.mica_select_result(self._p, C.byref(med), C.byref(p), C.byref(npos), C.byref(status),
                                     _stream()), 'select_result')
        return np.float32(med.value), np.float32(p.value), int(npos.value), int(status.value)

    @device_guard
    def result_async(self, record: torch.Tensor | None = None) -> torch.Tensor:
        """Enqueue the copy of the 32-byte result record into pinned host memory (no synchronisation);
        decode it with ``OrderStats.decode`` once the stream has passed this point."""
        if record is None:
            record = torch.zeros(32, dtype=torch.uint8).pin_memory()
        check(lib.mica_select_result_async(self._p, C.c_void_p(record.data_ptr()), _stream()), 'select_result_async')
        return record

    @staticmethod
    def decode(record: torch.Tensor):
        """(median, p999, n_pos, status) from a result record."""
        raw = record.numpy()
        n_pos = int(raw[8:16].view(np.int64)[0])
        med, p = raw[16:24].view(np.float32)
        return np.float32(med), np.float32(p), n_pos, int(raw[28:32].view(np.int32)[0])

    @device_guard
    def apply(self, x: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        p_x = _dev(x, torch.float32, 'x')
        if out is None:
            out = torch.zeros_like(x)
        p_y = _dev(out, torch.float32, 'out')
        check(lib.mica_normalize_apply_f32(p_x, p_y, x.numel(), self._p, _stream()), 'normalize_apply')
        return out


class IntOrderStats:
    """Device-resident state of the exact order statistics of an integer map (int8 / int16 / uint16, DESIGN.md
    D12): one histogram pass and one pick give the float64 median and 99.9 percentile NumPy computes on the
    integer array."""

    RESULT_BYTES = _lib.INT_STATS_RESULT_BYTES

    def __init__(self, device):
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise _lib.MicaError(f'IntOrderStats needs a CUDA device, got {self.device} (mica_b200 has no CPU fallback)')
        with torch.cuda.device(self.device):
            self.ws = torch.empty(lib.mica_int_stats_workspace_bytes(), dtype=torch.uint8, device=self.device)
        self._p = C.c_void_p(self.ws.data_ptr())

    @staticmethod
    def _int_map(x, name):
        if isinstance(x, torch.Tensor) and x.dtype not in INT_DTYPES:
            raise _lib.MicaError(f'{name} must be int8, int16 or uint16, got {x.dtype}')
        dt = x.dtype if isinstance(x, torch.Tensor) else torch.int16
        return _dev(x, dt, name), MAP_DTYPES[dt]

    def hist_view(self, dtype) -> torch.Tensor:
        """int64 view of the live histogram bins of a ``dtype`` map (2^8 or 2^16) that a multi-GPU run sums
        between hist and pick."""
        bins = 256 if dtype == torch.int8 else 65536
        off = lib.mica_int_stats_hist_ptr(self._p) - self.ws.data_ptr()
        return self.ws[off:off + 8 * bins].view(torch.int64)

    @device_guard
    def run(self, x: torch.Tensor, n_total: int | None = None, all_reduce=None, peer=None):
        """Multi-GPU (``x`` = this rank's voxels, ``n_total`` = all ranks'): the histograms of all ranks are
        summed between hist and pick, either by ``peer`` (a peer.PeerIntHistogram: over NVLink peer memory) or by
        ``all_reduce(hist_int64_tensor)`` (torch.distributed.all_reduce over NCCL), both on the current stream."""
        p_x, code = self._int_map(x, 'x')
        st = _stream()
        if all_reduce is None and peer is None:
            check(lib.mica_int_order_stats(p_x, code, x.numel(), self._p, st), 'int_order_stats')
            return self
        n_total = x.numel() if n_total is None else int(n_total)
        check(lib.mica_int_stats_init(self._p, code, n_total, st), 'int_stats_init')
        check(lib.mica_int_stats_hist(p_x, code, x.numel(), self._p, st), 'int_stats_hist')
        if peer is not None:
            peer.reduce(self, code)
        else:
            all_reduce(self.hist_view(x.dtype))
        check(lib.mica_int_stats_pick(self._p, code, st), 'int_stats_pick')
        return self

    @device_guard
    def result(self):
        """(median, p999, n_pos, status), median and p999 as Python floats (float64) -- synchronises the stream."""
        med, p, npos, status = C.c_double(), C.c_double(), C.c_int64(), C.c_int()
        check(lib.mica_int_stats_result(self._p, C.byref(med), C.byref(p), C.byref(npos), C.byref(status),
                                        _stream()), 'int_stats_result')
        return float(med.value), float(p.value), int(npos.value), int(status.value)

    @device_guard
    def result_async(self, record: torch.Tensor | None = None) -> torch.Tensor:
        """Enqueue the copy of the 32-byte result record into pinned host memory (no synchronisation);
        decode it with ``IntOrderStats.decode`` once the stream has passed this point."""
        if record is None:
            record = torch.zeros(self.RESULT_BYTES, dtype=torch.uint8).pin_memory()
        check(lib.mica_int_stats_result_async(self._p, C.c_void_p(record.data_ptr()), _stream()),
              'int_stats_result_async')
        return record

    @staticmethod
    def decode(record: torch.Tensor):
        """(median, p999, n_pos, status) from a result record."""
        raw = record.numpy()
        med, p = raw[0:16].view(np.float64)
        return float(med), float(p), int(raw[16:24].view(np.int64)[0]), int(raw[24:28].view(np.int32)[0])

    @device_guard
    def apply(self, x: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """The float32 normalised map of ``x`` (a new tensor unless ``out`` is given; left as it was when the
        status is not NORM_OK)."""
        p_x, code = self._int_map(x, 'x')
        if out is None:
            out = torch.empty(x.shape, dtype=torch.float32, device=x.device)
        p_y = _dev(out, torch.float32, 'out')
        if out.numel() != x.numel():
            raise _lib.MicaError(f'out has {out.numel()} elements, x {x.numel()}')
        check(lib.mica_normalize_apply_int(p_x, code, p_y, x.numel(), self._p, _stream()), 'normalize_apply_int')
        return out


@device_guard
def normalize(x: torch.Tensor, inplace: bool = False):
    """utils/preprocessing.py:122-133 on the device.  Returns (normalised, OrderStats).  An integer map
    (int8 / int16 / uint16) gets the float64 statistics of ``IntOrderStats`` and a new float32 volume:
    ``inplace=True`` raises for it."""
    if isinstance(x, torch.Tensor) and x.dtype in INT_DTYPES:
        if inplace:
            raise _lib.MicaError(f'normalize: a {x.dtype} map cannot be normalised in place (the result is float32)')
        st = IntOrderStats(x.device).run(x)
        return st.apply(x, torch.zeros(x.shape, dtype=torch.float32, device=x.device)), st
    st = OrderStats(x.device).run(x)
    return st.apply(x, x if inplace else None), st


# ---------------------------------------------------------------- R4 AF3 encode
@device_guard
def af3_encode(coords: torch.Tensor, bb_ch: torch.Tensor, aa_ch: torch.Tensor, origin_xyz, shape_zyx,
               clip_hi_xyz=None, *, z0: int = 0, nz_local=None, out: torch.Tensor | None = None):
    """24-channel rasteriser.  ``clip_hi_xyz`` defaults to the reference's (quirky)
    bounds (nz-1, ny-1, nx-1) applied to (x,y,z) (utils/preprocessing.py:177,294).
    Returns (vol24 [24,nz_local,ny,nx], status int32 tensor[1]; 1 == IndexError path)."""
    nz, ny, nx = (int(v) for v in shape_zyx)
    if clip_hi_xyz is None:
        clip_hi_xyz = (nz - 1, ny - 1, nx - 1)
    nzl = nz - z0 if nz_local is None else int(nz_local)
    n = coords.shape[0]
    p_xyz = _dev(coords, torch.float32, 'coords') if n else None
    p_bb = _dev(bb_ch, torch.int8, 'bb_ch') if n else None
    p_aa = _dev(aa_ch, torch.int8, 'aa_ch') if n else None
    dev = coords.device
    if out is None:
        out = torch.empty((24, nzl, ny, nx), dtype=torch.float32, device=dev)
    p_out = _dev(out, torch.float32, 'out')
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ox, oy, oz = (float(np.float32(v)) for v in origin_xyz)
    check(lib.mica_af3_encode(p_xyz, p_bb, p_aa, n, ox, oy, oz, int(clip_hi_xyz[0]), int(clip_hi_xyz[1]),
                              int(clip_hi_xyz[2]), nz, ny, nx, z0, nzl, p_out,
                              C.c_void_p(status.data_ptr()), _stream()), 'af3_encode')
    return out, status


class Af3CubeFiller:
    """Sparse AF3 path (R4 + R5 fused): keeps a [n_slots,24,W,W,W] model-input buffer equal to
    "zeros + the atoms of the cube currently in each slot" without ever building the dense
    24-channel volume.  ``bin`` once per map, ``fill`` once per batch.  ``dtype``: the buffer's element
    type, float32 or bfloat16 (1.0 and 0.0 are exact in both)."""

    def __init__(self, device, n_slots, grid_size=48, padding=8, perm=(2, 1, 0), dtype=torch.float32):
        self.dtype = model_dtype(dtype)
        self.device, self.n_slots = device, int(n_slots)
        self.grid_size, self.padding, self.perm = int(grid_size), int(padding), tuple(perm)
        self.buffer = None          # [n_slots,24,W,W,W], allocated (zeroed) by the first fill
        self.status = torch.zeros(1, dtype=torch.int32, device=device)
        self.ws = None
        self._geom = None
        self._shown = None          # the ijk tensor whose cubes the slots currently show (kept alive)
        self._shown_orient = 0      # ... and the orientation they show them in

    @device_guard
    def _fill(self, ijk, nonzero_ptr, orient=0):
        n_atoms, (nz, ny, nx) = self._geom
        prev = self._shown
        check(lib.mica_af3_fill_cubes_as(C.c_void_p(self.ws.data_ptr()), n_atoms, nz, ny, nx,
                                         _lib.int3(self.perm), self.grid_size, self.padding,
                                         C.c_void_p(prev.data_ptr()) if prev is not None else None,
                                         int(prev.shape[0]) if prev is not None else 0,
                                         C.c_void_p(ijk.data_ptr()) if ijk is not None else None,
                                         int(ijk.shape[0]) if ijk is not None else 0,
                                         C.c_void_p(self.buffer.data_ptr()), MODEL_DTYPES[self.dtype],
                                         self.buffer.stride(0), nonzero_ptr, self._shown_orient, orient, _stream()),
              'af3_fill_cubes')
        self._shown, self._shown_orient = ijk, orient

    def retype(self, dtype):
        """Give the slot buffer element type ``dtype`` (float32 or bfloat16): the buffer is dropped and the next
        ``fill`` allocates a clean one.  The atom bins stay."""
        self.dtype = model_dtype(dtype)
        self.buffer, self._shown, self._shown_orient = None, None, 0

    def clear(self):
        """Un-scatter every slot (buffer back to all zeros)."""
        if self._shown is not None and self.ws is not None and self.buffer is not None:
            self._fill(None, None)
        self._shown = None

    @device_guard
    def bin(self, coords, bb_ch, aa_ch, origin_xyz, shape_zyx, clip_hi_xyz=None):
        """Bin the atoms per cube (global cube grid of ``shape_zyx``).  Returns the device
        status word (1 == the reference's IndexError path, as af3_encode)."""
        self.clear()                                   # with the OLD bins, before they are rebuilt
        nz, ny, nx = (int(v) for v in shape_zyx)
        if clip_hi_xyz is None:
            clip_hi_xyz = (nz - 1, ny - 1, nx - 1)
        n = int(coords.shape[0])
        nbytes = lib.mica_af3_bins_workspace_bytes(n, nz, ny, nx, _lib.int3(self.perm), self.grid_size, self.padding)
        if nbytes == 0:
            raise _lib.MicaError(f'af3 bins: {_lib.last_error()}')
        if self.ws is None or self.ws.numel() < nbytes:
            self.ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        p_xyz = _dev(coords, torch.float32, 'coords') if n else None
        p_bb = _dev(bb_ch, torch.int8, 'bb_ch') if n else None
        p_aa = _dev(aa_ch, torch.int8, 'aa_ch') if n else None
        ox, oy, oz = (float(np.float32(v)) for v in origin_xyz)
        check(lib.mica_af3_bin_atoms(p_xyz, p_bb, p_aa, n, ox, oy, oz, int(clip_hi_xyz[0]), int(clip_hi_xyz[1]),
                                     int(clip_hi_xyz[2]), nz, ny, nx, _lib.int3(self.perm), self.grid_size,
                                     self.padding, C.c_void_p(self.ws.data_ptr()), self.ws.numel(),
                                     C.c_void_p(self.status.data_ptr()), _stream()), 'af3_bin_atoms')
        self._geom = (n, (nz, ny, nx))
        return self.status

    def share_bins(self, other: 'Af3CubeFiller'):
        """Use ``other``'s per-cube atom bins (one binning pass serves several slot buffers)."""
        self.clear()
        self.ws, self._geom, self.status = other.ws, other._geom, other.status

    def fill(self, ijk: torch.Tensor, nonzero: torch.Tensor | None = None, orient: int = 0) -> torch.Tensor:
        """AF3 channels of the cubes ``ijk`` (int32 [B,3], B <= n_slots) -> view [B,24,W,W,W], every cube in
        orientation ``orient`` (``orientation``; ``nonzero`` does not depend on it)."""
        orient = _orientation_arg(orient)
        B = int(ijk.shape[0])
        if B > self.n_slots:
            raise _lib.MicaError(f'batch of {B} cubes exceeds the {self.n_slots} slots')
        if self._geom is None:
            raise _lib.MicaError('Af3CubeFiller.fill before bin')
        p_nz = _dev(nonzero, torch.int32, 'nonzero') if nonzero is not None else None
        _dev(ijk, torch.int32, 'ijk')
        if self.buffer is None:
            W = self.grid_size + 2 * self.padding
            self.buffer = torch.zeros((self.n_slots, 24, W, W, W), dtype=self.dtype, device=self.device)
        self._fill(ijk, p_nz, orient)
        return self.buffer[:B]


# ------------------------------------------------- test-time augmentation: orientations of the window
#: the permutations of the window axes (0, 1, 2) in lexicographic order (the p of an orientation code)
_AXIS_PERMS = tuple(itertools.permutations(range(3)))
N_ORIENTATIONS = 48
#: the named orientation sets of ``tta_orientations``
TTA_SETS = ('flips', 'rot90', 'all')


def _orientation_arg(code) -> int:
    if isinstance(code, (bool, np.bool_)) or not isinstance(code, (int, np.integer)):
        raise _lib.MicaError(f'an orientation is an int in 0..{N_ORIENTATIONS - 1}, got {code!r}')
    if not 0 <= int(code) < N_ORIENTATIONS:
        raise _lib.MicaError(f'orientation {int(code)} is not in 0..{N_ORIENTATIONS - 1}')
    return int(code)


def orientation(code):
    """(perm, flips) of an orientation code 0..47 of the W^3 model-input window: ``code = 8 p + f``, ``perm`` the
    p-th permutation of the axes (0, 1, 2) in lexicographic order, ``flips[a]`` = bit a of f.  The oriented window is
    ``O[u0, u1, u2] = C[v]`` with ``v[perm[a]] = W-1-u_a if flips[a] else u_a``, i.e. ``np.transpose(C, perm)``
    then ``np.flip`` along every output axis a with ``flips[a]`` (``orient_array``).  Code 0 is the identity.

    The axes are those of the model input ``[B, C, u0, u1, u2]`` -- the window AFTER the D6 axis permutation of the
    map (``perm`` of ``extract_cubes``), not the map's (z, y, x)."""
    code = _orientation_arg(code)
    return _AXIS_PERMS[code >> 3], tuple(bool((code >> a) & 1) for a in range(3))


def orientation_code(perm, flips) -> int:
    """The code of (perm, flips): inverse of ``orientation``."""
    return 8 * _AXIS_PERMS.index(tuple(int(a) for a in perm)) + sum(1 << a for a in range(3) if flips[a])


def orientation_det(code) -> int:
    """+1 for a proper rotation (keeps chirality), -1 for a mirror image."""
    perm, flips = orientation(code)
    inversions = sum(1 for a in range(3) for b in range(a + 1, 3) if perm[a] > perm[b])
    return (-1) ** (inversions + sum(flips))


def orient_array(a: np.ndarray, code) -> np.ndarray:
    """The window(s) ``a`` (the last three axes) in orientation ``code`` (a view)."""
    perm, flips = orientation(code)
    lead = a.ndim - 3
    out = np.transpose(a, tuple(range(lead)) + tuple(lead + p for p in perm))
    for ax in range(3):
        if flips[ax]:
            out = np.flip(out, lead + ax)
    return out


@functools.lru_cache(maxsize=None)
def _orientation_table():
    """compose[g][h] = code of orienting by h, then by g; every orientation acts faithfully on the 8 corners."""
    probe = np.arange(8).reshape(2, 2, 2)
    key = {orient_array(probe, c).tobytes(): c for c in range(N_ORIENTATIONS)}
    return tuple(tuple(key[orient_array(orient_array(probe, h), g).tobytes()] for h in range(N_ORIENTATIONS))
                 for g in range(N_ORIENTATIONS))


def compose_orientations(g, h) -> int:
    """The code of ``orient_array(orient_array(C, h), g)``."""
    return _orientation_table()[_orientation_arg(g)][_orientation_arg(h)]


def inverse_orientation(code) -> int:
    """The code that maps ``orient_array(C, code)`` back to ``C``."""
    return _orientation_table()[_orientation_arg(code)].index(0)


def tta_orientations(tta):
    """The orientation codes of a test-time augmentation, validated: None (no augmentation) -> None;
    'flips' -> the 8 mirrorings of the axes (p = 0); 'rot90' -> the 24 proper rotations (det +1: they keep the
    chirality of a protein); 'all' -> the 48; or a non-empty sequence of distinct codes 0..47, kept in its order.
    Raises MicaError otherwise."""
    if tta is None:
        return None
    if isinstance(tta, str):
        if tta == 'flips':
            return tuple(range(8))
        if tta == 'rot90':
            return tuple(c for c in range(N_ORIENTATIONS) if orientation_det(c) == 1)
        if tta == 'all':
            return tuple(range(N_ORIENTATIONS))
        raise _lib.MicaError(f"tta must be one of {TTA_SETS}, a sequence of orientation codes or None, got {tta!r}")
    try:
        codes = tuple(_orientation_arg(c) for c in tta)
    except TypeError:
        raise _lib.MicaError(f'tta must be one of {TTA_SETS}, a sequence of orientation codes or None, '
                             f'got {tta!r}') from None
    if not codes:
        raise _lib.MicaError('tta: an empty list of orientations')
    if len(set(codes)) != len(codes):
        raise _lib.MicaError(f'tta: orientation codes must be distinct, got {list(codes)}')
    return codes


# ------------------------------------------------------------ R5/R6 cube extract
def cube_space_shape(shape_zyx, perm=STANDARD_PERM):
    return tuple(int(shape_zyx[p]) for p in perm)


def cube_origins(cube_shape, grid_size):
    """(i,j,k) in the loop order of utils/create_grids.py:143-145 -> int32 [n,3]."""
    ax = [np.arange(0, int(s), grid_size, dtype=np.int32) for s in cube_shape]
    g = np.stack(np.meshgrid(*ax, indexing='ij'), axis=-1).reshape(-1, 3)
    return np.ascontiguousarray(g)


@device_guard
def extract_cubes(vol: torch.Tensor, ijk: torch.Tensor, grid_size: int = 48, padding: int = 8,
                  perm=STANDARD_PERM, *, global_nz=None, z0: int = 0, out: torch.Tensor | None = None,
                  nonzero: torch.Tensor | None = None, cube_max: torch.Tensor | None = None, orient: int = 0):
    """vol [C,nz_local,ny,nx] (or [nz,ny,nx]) -> out [B,C,W,W,W] for the cube origins ``ijk``
    (int32 [B,3], cube space).  ``out`` may be a channel slice of a larger [B,Ctot,W,W,W]
    buffer (only the batch stride may be non-dense).  ``orient``: every window in that orientation
    (``orientation``; test-time augmentation), cut straight from the map; 0 = the windows as they are.
    ``out`` may be float32 (default) or bfloat16: every voxel is then rounded once to nearest even, and ``nonzero`` /
    ``cube_max`` are taken on the float32 values, so they are those of a float32 ``out``."""
    orient = _orientation_arg(orient)
    if vol.dim() == 3:
        vol = vol.unsqueeze(0)
    p_vol = _dev(vol, torch.float32, 'vol')
    Cn, nzl, ny, nx = vol.shape
    nz = nzl if global_nz is None else int(global_nz)
    p_ijk = _dev(ijk, torch.int32, 'ijk')
    B = ijk.shape[0]
    W = grid_size + 2 * padding
    if out is None:
        out = torch.empty((B, Cn, W, W, W), dtype=torch.float32, device=vol.device)
    if not out.is_cuda or out.dtype not in MODEL_DTYPES or tuple(out.shape) != (B, Cn, W, W, W):
        raise _lib.MicaError(f'out must be a CUDA float32 or bfloat16 [{B},{Cn},{W},{W},{W}] tensor')
    if B and out.stride()[1:] != (W ** 3, W * W, W, 1):
        raise _lib.MicaError('out must be dense in every axis but the batch')
    cube_stride = out.stride(0) if B else Cn * W ** 3
    p_nz = _dev(nonzero, torch.int32, 'nonzero') if nonzero is not None else None
    p_mx = _dev(cube_max, torch.float32, 'cube_max') if cube_max is not None else None
    check(lib.mica_extract_cubes_as(p_vol, vol.stride(0), Cn, nz, ny, nx, z0, nzl, _lib.int3(perm), grid_size,
                                    padding, p_ijk, B, C.c_void_p(out.data_ptr()), MODEL_DTYPES[out.dtype], cube_stride,
                                    p_nz, p_mx, orient, _stream()), 'extract_cubes')
    return out


def check_min_max(min_max):
    """``min_max`` as a float, or None.  A finite number is the only other thing accepted (refused before any launch)."""
    if min_max is None:
        return None
    if isinstance(min_max, (bool, np.bool_)) or not isinstance(min_max, (int, float, np.integer, np.floating)):
        raise _lib.MicaError(f'min_max must be a finite number or None, got {min_max!r}')
    v = float(min_max)
    if not np.isfinite(v):
        raise _lib.MicaError(f'min_max must be a finite number or None, got {min_max!r}')
    return v


@device_guard
def cube_window_max(vol: torch.Tensor, ijk: torch.Tensor, grid_size: int = 48, padding: int = 8,
                    perm=STANDARD_PERM, *, global_nz=None, z0: int = 0, out: torch.Tensor | None = None):
    """float32 [B] device tensor: the maximum of every cube's W^3 window (the one ``extract_cubes`` cuts from ``vol``,
    [nz_local, ny, nx] holding global planes [z0, z0 + nz_local) of ``global_nz``), zeros standing for the parts
    outside the map, NaN if the window holds a NaN -- ``np.max`` over the reference's ``np.pad``-ed window."""
    p_vol = _dev(vol, torch.float32, 'vol')
    if vol.dim() != 3:
        raise _lib.MicaError(f'vol must be [nz, ny, nx], got shape {tuple(vol.shape)}')
    nzl, ny, nx = vol.shape
    nz = nzl if global_nz is None else int(global_nz)
    p_ijk = _dev(ijk, torch.int32, 'ijk')
    B = int(ijk.shape[0])
    if out is None:
        out = torch.empty(B, dtype=torch.float32, device=vol.device)
    p_out = _dev(out, torch.float32, 'out')
    if tuple(out.shape) != (B,):
        raise _lib.MicaError(f'out must be [{B}], got {tuple(out.shape)}')
    check(lib.mica_cube_window_max(p_vol, nz, ny, nx, int(z0), nzl, _lib.int3(perm), int(grid_size), int(padding),
                                   p_ijk, B, p_out, _stream()), 'cube_window_max')
    return out


def select_cubes(maxima: torch.Tensor, min_max) -> np.ndarray:
    """The cubes the reference's training-grid rule keeps (create_grids_for_normalized_map.py:78, negated):
    ``not (window.max() < min_max)`` in float32 -- a tie and a NaN window are kept.  Returns the kept indices into
    ``maxima`` (int64, ascending) after one device-to-host copy of the maxima."""
    t = check_min_max(min_max)
    if t is None:
        raise _lib.MicaError('select_cubes needs a finite min_max')
    m = maxima.detach().to('cpu').numpy()
    if m.dtype != np.float32:
        raise _lib.MicaError(f'maxima must be float32, got {m.dtype}')
    with np.errstate(over='ignore', invalid='ignore'):      # a threshold beyond float32's range; NaN compares False
        return np.flatnonzero(~(m < np.float32(t))).astype(np.int64)


# ------------------------------------------------------ R7/R8 post-process + stitch
class StitchedVolumes:
    """The four volumes CryoEMPredictor.run_prediction returns (utils/predict.py:526-531),
    resident on the device; ``box`` = (org, ext) of this rank's part of cube space."""

    def __init__(self, cube_shape, device, org=None, ext=None):
        self.shape = tuple(int(v) for v in cube_shape)
        self.device = torch.device(device)
        self.org = tuple(org) if org is not None else (0, 0, 0)
        self.ext = tuple(ext) if ext is not None else self.shape
        e = self.ext
        self.backbone_probability = torch.zeros(e, dtype=torch.float32, device=device)
        self.carbon_alpha_probability = torch.zeros(e, dtype=torch.float32, device=device)
        self.amino_acid_prediction = torch.zeros(e, dtype=torch.float32, device=device)
        self.amino_acid_probability = torch.zeros((20,) + e, dtype=torch.float32, device=device)

    @classmethod
    def from_block(cls, block: torch.Tensor, cube_shape, org, ext):
        """Volumes that live in ONE caller-owned float32 block of 23 * prod(ext) elements, laid out
        [backbone | carbon_alpha | amino_acid_prediction | amino_acid_probability x 20] -- the layout
        ``postproc_stitch_peer`` writes into a rank's exported memory."""
        self = cls.__new__(cls)
        self.shape = tuple(int(v) for v in cube_shape)
        self.device = block.device
        self.org, self.ext = tuple(int(v) for v in org), tuple(int(v) for v in ext)
        n = self.ext[0] * self.ext[1] * self.ext[2]
        if block.dtype != torch.float32 or block.numel() < 23 * n or not block.is_contiguous():
            raise _lib.MicaError('from_block needs a contiguous float32 block of 23 * prod(ext) elements')
        flat = block.view(-1)
        self.backbone_probability = flat[0:n].view(self.ext)
        self.carbon_alpha_probability = flat[n:2 * n].view(self.ext)
        self.amino_acid_prediction = flat[2 * n:3 * n].view(self.ext)
        self.amino_acid_probability = flat[3 * n:23 * n].view((20,) + self.ext)
        self.block = block
        return self

    def as_dict(self):
        return {k: getattr(self, k) for k in ('backbone_probability', 'carbon_alpha_probability',
                                              'amino_acid_prediction', 'amino_acid_probability')}


@device_guard
def postproc_stitch(bb: torch.Tensor, ca: torch.Tensor, aa: torch.Tensor, ijk: torch.Tensor,
                    vols: StitchedVolumes, grid_size: int = 48, padding: int = 8):
    """Fused utils/predict.py:342-349 + :494-501 for one batch of cubes.  The logits are all float32 or all bfloat16
    (widened exactly on load: the volumes equal the float32 call on ``logits.float()``)."""
    B = ijk.shape[0]
    W = grid_size + 2 * padding
    ptrs, code = _logits(bb, ca, aa, B, W)
    X, Y, Z = vols.shape
    check(lib.mica_postproc_stitch_as(
        *ptrs, code, _dev(ijk, torch.int32, 'ijk'), B, X, Y, Z, _lib.int3(vols.org), _lib.int3(vols.ext), grid_size, padding,
        _dev(vols.backbone_probability, torch.float32, 'bb_vol'),
        _dev(vols.carbon_alpha_probability, torch.float32, 'ca_vol'),
        _dev(vols.amino_acid_probability, torch.float32, 'aa_prob_vol'),
        _dev(vols.amino_acid_prediction, torch.float32, 'aa_pred_vol'), _stream()), 'postproc_stitch')
    return vols


@device_guard
def zero_cores(ijk: torch.Tensor, vols: StitchedVolumes, grid_size: int = 48):
    """The cores of the cubes ``ijk`` (int32 [B,3]) set to 0 in all four volumes, clipped to their box: the cubes a
    keep rule skipped (``select_cubes``), in volumes that held an earlier map."""
    X, Y, Z = vols.shape
    check(lib.mica_zero_cores(_dev(ijk, torch.int32, 'ijk'), int(ijk.shape[0]), X, Y, Z, _lib.int3(vols.org),
                              _lib.int3(vols.ext), int(grid_size),
                              _dev(vols.backbone_probability, torch.float32, 'bb_vol'),
                              _dev(vols.carbon_alpha_probability, torch.float32, 'ca_vol'),
                              _dev(vols.amino_acid_probability, torch.float32, 'aa_prob_vol'),
                              _dev(vols.amino_acid_prediction, torch.float32, 'aa_pred_vol'), _stream()), 'zero_cores')
    return vols


@device_guard
def postproc_stitch_peer(bb: torch.Tensor, ca: torch.Tensor, aa: torch.Tensor, ijk: torch.Tensor, cube_shape,
                         owner_table: torch.Tensor, x_bounds, grid_size: int = 48, padding: int = 8):
    """``postproc_stitch`` for one map whose cubes are dealt out over several GPUs: every core plane goes to
    the volume block of the rank that owns its x range (``owner_table``: int64 device tensor of ``world``
    base pointers, ``peer.PeerVolumes.table``; ``x_bounds``: world + 1 plane bounds), local or over NVLink.  Logits as
    ``postproc_stitch``: all float32 or all bfloat16."""
    B = ijk.shape[0]
    W = grid_size + 2 * padding
    ptrs, code = _logits(bb, ca, aa, B, W)
    X, Y, Z = (int(v) for v in cube_shape)
    world = int(owner_table.numel())
    bounds = (C.c_int * (world + 1))(*[int(v) for v in x_bounds])
    check(lib.mica_postproc_stitch_peer_as(
        *ptrs, code, _dev(ijk, torch.int32, 'ijk'), B, X, Y, Z, grid_size, padding,
        _dev(owner_table, torch.int64, 'owner_table'), bounds, world, _stream()), 'postproc_stitch_peer')


def overlap_window(kind, grid_size: int, padding: int) -> np.ndarray:
    """1-D weights of the overlap-weighted stitch: 'core' (1 on the core, 0 on the halo = the reference's crop),
    'uniform' (plain average of every window covering a voxel), 'triangle' (ramp peaking at the window centre),
    or an array of W = grid_size + 2 * padding finite weights >= 0, at least one of them > 0."""
    W = int(grid_size) + 2 * int(padding)
    if not isinstance(kind, str):
        w = np.ascontiguousarray(kind, dtype=np.float32)
        if w.shape != (W,):
            raise _lib.MicaError(f'window must have {W} weights, got shape {w.shape}')
        if not (np.isfinite(w).all() and (w >= 0).all() and (w > 0).any()):
            raise _lib.MicaError('window weights must be finite and >= 0, with at least one > 0')
        return w
    u = np.arange(W, dtype=np.float64)
    if kind == 'core':
        w = ((u >= padding) & (u < padding + grid_size)).astype(np.float64)
    elif kind == 'uniform':
        w = np.ones(W)
    elif kind == 'triangle':
        w = np.minimum(u + 1, W - u) / (W / 2.0)
    else:
        raise _lib.MicaError(f"window must be 'core', 'uniform', 'triangle' or an array, got {kind!r}")
    return w.astype(np.float32)


def stitch_mode(window, tta, grid_size: int, padding: int):
    """(w1, codes) of a stitch, every argument validated before any launch.  ``w1``: the weights of the overlap-weighted
    stitch (``overlap_window``), or None for the reference's paste of the cube cores; ``codes``: the orientations of a
    test-time augmentation (``tta_orientations``), or None.  ``tta`` None or (0,) is no augmentation.  Without it,
    ``window`` None or 'core' is the paste (the 1-on-the-core weighted stitch IS the paste, and runs as one).  Under it
    the window defaults to 'core' and every window, 'core' included, runs in fixed point."""
    codes = tta_orientations(tta)
    if codes == (0,):
        codes = None
    if window is None and codes is None:
        return None, None
    w1 = overlap_window('core' if window is None else window, grid_size, padding)
    if codes is None and is_core_window(w1, grid_size, padding):
        return None, None
    return w1, codes


def is_core_window(w1, grid_size: int, padding: int) -> bool:
    """True for the 1-on-the-core window: its weighted stitch IS the reference's paste, and runs as one."""
    return np.array_equal(w1, overlap_window('core', grid_size, padding))


def overlap_norm_tables(w1, cube_shape, grid_size: int, padding: int, tta_k: int = 1):
    """Reciprocals (0 where the sum is 0) of the 1-D weight sums Wx, Wy, Wz of the full cube lattice
    (``cube_origins``): the weight sum of the overlap-weighted stitch at voxel (x, y, z) is Wx[x] Wy[y] Wz[z], with
    Wx[x] = sum over the origins i covering x of w1[x - i + padding].  float64, origins added in ascending order.
    Whatever part of the lattice a run stitches, these come from all of it.  ``tta_k``: the number of orientations
    of a test-time augmentation, every window then contributing k times; the x table holds 1 / (k Wx)."""
    w = np.asarray(w1, dtype=np.float32).astype(np.float64)
    W = len(w)
    out = []
    for axis, n in enumerate(int(v) for v in cube_shape):
        s = np.zeros(n, np.float64)
        for i in range(0, n, int(grid_size)):
            lo = i - int(padding)
            x0, x1 = max(0, lo), min(n, lo + W)
            s[x0:x1] += w[x0 - lo:x1 - lo]
        r = np.zeros(n, np.float64)
        np.divide(1.0, s * int(tta_k) if axis == 0 else s, out=r, where=s > 0)
        out.append(r)
    return out


def overlap_owner(coord: int, bounds) -> int:
    """The rank whose planes [bounds[r], bounds[r+1]) hold ``coord`` -- the lookup of the peer accumulate kernel
    (empty ranks are skipped)."""
    r = 0
    while r + 1 < len(bounds) - 1 and coord >= bounds[r + 1]:
        r += 1
    return r


def peer_atomics_supported(device: int, peer_device: int) -> bool:
    """Whether ``device`` can add into ``peer_device``'s memory with native atomics (True for the same device)."""
    rc = lib.mica_peer_atomics_supported(int(device), int(peer_device))
    if rc < 0:
        check(rc, 'peer_atomics_supported')
    return bool(rc)


class OverlapOwners(NamedTuple):
    """Where a stitch (paste or weighted) stores when the output is split over ranks: rank r owns planes
    [bounds[r], bounds[r+1]) of cube axis ``axis`` (0 = x, 2 = k) as the 23-channel block at ``table[r]`` (int64 device
    tensor of base pointers, ``peer.PeerVolumes.table``); ``devices``: the CUDA device index of each owner, whose
    memory the weighted stitch must be able to add into atomically."""
    table: torch.Tensor
    axis: int
    bounds: tuple
    devices: tuple


class Stitcher:
    """The stitch of one map's batches of logits, its mode and destination bound once (``stitch_mode``).

    The paste: the reference's softmax/argmax and paste of the disjoint cube cores (``postproc_stitch``), final batch
    by batch (``per_batch``).  The weighted stitch, the north_star's "stitch with overlap weights": every voxel of every
    window adds its probabilities times the window weight, normalised by the weight sum of the full cube lattice, in
    2^-31 fixed point (uint32), so the result does not depend on the order of the cubes, the batches or the partition;
    ``finalize`` converts in place.  NOT the reference's arithmetic (DESIGN.md D2), and several times its cost: every
    voxel of every 64^3 window is post-processed and added, not just the 32^3 (48^3) cores.  ``tta``: test-time
    augmentation; every window is stitched once per orientation (``orientations``), from the logits of the model run on
    the window in that orientation, and the result is the average over the k orientations (the 1/k is in the
    normaliser tables) -- always the weighted stitch.

    ``vols``: the volumes on ``device`` it stores into; the weighted stitch needs ``StitchedVolumes.from_block``
    volumes, zeroed.  ``owners``: a ``OverlapOwners`` table -- every core plane (paste, along cube axis 0, plain stores)
    or window contribution (weighted, along axis 0 or 2, native peer atomics required) goes to the block of the rank
    that owns its plane, locally or over NVLink; ``vols`` is then this rank's own box, if any.  Default: a zeroed
    whole-map block of its own."""

    def __init__(self, cube_shape, device, grid_size: int = 48, padding: int = 8, window=None, *, tta=None, vols=None,
                 owners: OverlapOwners | None = None):
        self.shape = tuple(int(v) for v in cube_shape)
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        self.grid_size, self.padding = int(grid_size), int(padding)
        self.w1, codes = stitch_mode(window, tta, grid_size, padding)
        #: the paste: the volumes are final batch by batch; the weighted stitch: after ``finalize``
        self.per_batch = self.w1 is None
        #: the orientations the batches come in: (0,) without test-time augmentation
        self.orientations = codes or (0,)
        if owners is not None:
            if owners.axis not in ((0,) if self.per_batch else (0, 2)):
                raise _lib.MicaError(f'owners along cube axis {owners.axis}: the weighted stitch splits along 0 or 2, '
                                     'the paste along 0')
            for d in () if self.per_batch else owners.devices:
                if not peer_atomics_supported(self.device.index, d):
                    raise _lib.MicaError(f'overlap-weighted stitching over several GPUs adds into the owners\' '
                                         f'memory atomically: cuda:{self.device.index} has no native peer atomics '
                                         f'with cuda:{d}')
        X, Y, Z = self.shape
        if vols is None and owners is None:
            with torch.cuda.device(self.device):
                vols = StitchedVolumes.from_block(torch.zeros(23 * X * Y * Z, dtype=torch.float32, device=self.device),
                                                  self.shape, (0, 0, 0), self.shape)
        if vols is not None and _cuda_device_of(vols) != self.device:
            raise _lib.MicaError(f'the volumes live on {vols.device}, the stitcher on {self.device}')
        if vols is not None and not self.per_batch and getattr(vols, 'block', None) is None:
            raise _lib.MicaError('the weighted stitch needs volumes of StitchedVolumes.from_block')
        self.vols = vols
        # the arguments that do not change from batch to batch, converted to ctypes once: the drop-in feeds the model
        # in the reference's batches of <= 8 cubes, i.e. hundreds of stitch calls per map
        gs, pad = self.grid_size, self.padding
        if owners is not None:
            table = _dev(owners.table, torch.int64, 'owner_table')
            bounds = (C.c_int * len(owners.bounds))(*[int(v) for v in owners.bounds])
            world = int(owners.table.numel())
        if self.per_batch and owners is None:
            self._fn, self._what = lib.mica_postproc_stitch_as, 'postproc_stitch'
            self._head, self._tail = (X, Y, Z, _lib.int3(vols.org), _lib.int3(vols.ext), gs, pad,
                                      _dev(vols.backbone_probability, torch.float32, 'bb_vol'),
                                      _dev(vols.carbon_alpha_probability, torch.float32, 'ca_vol'),
                                      _dev(vols.amino_acid_probability, torch.float32, 'aa_prob_vol'),
                                      _dev(vols.amino_acid_prediction, torch.float32, 'aa_pred_vol')), ()
        elif self.per_batch:
            self._fn, self._what = lib.mica_postproc_stitch_peer_as, 'postproc_stitch_peer'
            self._head, self._tail = (X, Y, Z, gs, pad, table, bounds, world), ()
        else:
            with torch.cuda.device(self.device):
                self.norm = torch.from_numpy(np.concatenate(
                    overlap_norm_tables(self.w1, self.shape, gs, pad, len(self.orientations)))).to(self.device)
            self._head = (X, Y, Z, gs, pad, self.w1.ctypes.data_as(C.POINTER(C.c_float)),
                          C.c_void_p(self.norm.data_ptr()))
            if owners is None:
                self._fn, self._what = lib.mica_overlap_accumulate_fixed_as, 'overlap_accumulate'
                self._tail = (C.c_void_p(vols.block.data_ptr()),)
            else:
                self._fn, self._what = lib.mica_overlap_accumulate_fixed_peer_as, 'overlap_accumulate_peer'
                self._tail = (table, int(owners.axis), bounds, world)
        self._checked = None            # (B, dtype) of the last checked call
        self._code = _lib.DTYPE_F32
        self._done = False

    @staticmethod
    def kernel_logits(bb, ca, aa):
        """Logits as the stitch kernels take them: contiguous, all float32 or all bfloat16.  Float32 and bfloat16 pass
        through (the kernels widen bfloat16 exactly); any other dtype, or a mix, becomes float32."""
        dt = bb.dtype
        if dt not in MODEL_DTYPES or ca.dtype != dt or aa.dtype != dt:
            bb, ca, aa = bb.float(), ca.float(), aa.float()
        return bb.contiguous(), ca.contiguous(), aa.contiguous()

    def __call__(self, bb, ca, aa, ijk, orient=0):
        """Stitch one batch of logits, those of the windows ``ijk`` (int32 [B,3]) in orientation ``orient`` (one of
        ``orientations``), as the model gives them (``kernel_logits``).  The logits and ``ijk`` are checked on the
        first call and whenever the batch size or the dtype changes."""
        if self.per_batch:
            if orient:
                raise _lib.MicaError(f'the paste stitches orientation 0 only, got {orient!r}')
        elif _orientation_arg(orient) not in self.orientations:
            raise _lib.MicaError(f'orientation {orient} is not one of this stitcher\'s {list(self.orientations)}')
        bb, ca, aa = self.kernel_logits(bb, ca, aa)
        B = ijk.shape[0]
        if (B, bb.dtype) != self._checked:
            _, self._code = _logits(bb, ca, aa, B, self.grid_size + 2 * self.padding)
            _dev(ijk, torch.int32, 'ijk')
            for t, name in ((bb, 'bb'), (ca, 'ca'), (aa, 'aa'), (ijk, 'ijk')):
                if t.device != self.device:
                    raise _lib.MicaError(f'{name} lives on {t.device}, the stitcher on {self.device}')
            self._checked = (B, bb.dtype)
        if torch.cuda.current_device() != self.device.index:
            with torch.cuda.device(self.device):
                return self(bb, ca, aa, ijk, orient)
        args = (bb.data_ptr(), ca.data_ptr(), aa.data_ptr(), self._code, ijk.data_ptr(), B, *self._head)
        if not self.per_batch:
            args += (int(orient), *self._tail)
        check(self._fn(*args, torch.cuda.current_stream().cuda_stream), self._what)

    def clear_cores(self, ijk):
        """The cubes ``ijk`` (int32 [n,3]) a keep rule skipped (``select_cubes``): the paste sets their cores to 0 in
        ``vols``, which may hold an earlier map; the weighted stitch adds nothing for them."""
        if self.per_batch and self.vols is not None and len(ijk):
            zero_cores(torch.as_tensor(ijk).to(self.device), self.vols, self.grid_size)

    def finalize(self) -> StitchedVolumes:
        """The four volumes: ``vols`` (for the weighted stitch, converted in place from fixed point).  With owners,
        call it once every rank's contributions have landed (stream sync + barrier)."""
        if self.per_batch or self._done:
            return self.vols
        if self.vols is None:
            raise _lib.MicaError('this Stitcher only adds into other ranks\' volumes')
        e = self.vols.ext
        with torch.cuda.device(self.device):
            check(lib.mica_overlap_finalize_fixed(C.c_void_p(self.vols.block.data_ptr()), e[0] * e[1] * e[2],
                                                  _stream()), 'overlap_finalize')
        self._done = True
        return self.vols


@device_guard
def stitch_cubes(cubes: torch.Tensor, ijk: torch.Tensor, cube_shape, grid_size: int = 48, padding: int = 8,
                 org=None, ext=None, out: torch.Tensor | None = None):
    """reconstruct_volume alone (utils/predict.py:494-501): cubes [B,C,W,W,W] -> [C,ext...]."""
    B, Cn = cubes.shape[:2]
    X, Y, Z = (int(v) for v in cube_shape)
    org = (0, 0, 0) if org is None else tuple(org)
    ext = (X, Y, Z) if ext is None else tuple(ext)
    if out is None:
        out = torch.zeros((Cn,) + ext, dtype=torch.float32, device=cubes.device)
    check(lib.mica_stitch_cubes(_dev(cubes, torch.float32, 'cubes'), Cn, _dev(ijk, torch.int32, 'ijk'), B,
                                X, Y, Z, _lib.int3(org), _lib.int3(ext), grid_size, padding,
                                _dev(out, torch.float32, 'out'), _stream()), 'stitch_cubes')
    return out


# ------------------------------------------------------------------ prediction maps
#: the four volumes of ``StitchedVolumes.as_dict`` / ``CryoEMPredictor.run_prediction``
VOLUME_KEYS = ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_prediction', 'amino_acid_probability')


def volumes_to_grid(vols, perm, working_shape, target_shape) -> dict:
    """The four stitched volumes resampled onto a target grid (oracle/prediction_maps_oracle.py), in its memory order.

    ``vols``: a ``StitchedVolumes`` or a mapping with the ``VOLUME_KEYS`` -- float32 CUDA tensors in cube space
    ``[X, Y, Z]`` (``[20, X, Y, Z]`` for ``amino_acid_probability``) covering the whole cube space; the stitched
    ``amino_acid_prediction`` is not read.  ``perm``: the map's ``MapHeader.transpose_order()[0]`` (cube axis a walks
    memory axis perm[a]).  ``working_shape`` / ``target_shape``: memory shapes (nz, ny, nx) of the normalised map and of
    the target grid (the input map's, or ``working_shape`` itself).  Returns float32 tensors ``[nz, ny, nx]`` (``[20,
    nz, ny, nx]`` for ``amino_acid_probability``), views of one new 23-channel block laid out as ``StitchedVolumes``;
    ``amino_acid_prediction`` is the arg-max of the 20 resampled probabilities.  One launch."""
    org = ext = None
    if isinstance(vols, StitchedVolumes):
        org, ext = vols.org, vols.ext
        cube_shape = vols.shape
        vols = vols.as_dict()
    missing = [k for k in VOLUME_KEYS if k not in vols]
    if missing:
        raise _lib.MicaError(f'volumes_to_grid: missing volumes {missing}')
    bb = vols['backbone_probability']
    if org is None:
        cube_shape = tuple(bb.shape)
    return _volumes_to_grid(bb, vols['carbon_alpha_probability'], vols['amino_acid_prediction'],
                            vols['amino_acid_probability'], cube_shape, org, ext, perm, working_shape, target_shape)


@device_guard
def _volumes_to_grid(bb, ca, pred, prob, cube_shape, org, ext, perm, working_shape, target_shape):
    ptrs = [_dev(t, torch.float32, name) for t, name in ((bb, 'backbone_probability'), (ca, 'carbon_alpha_probability'),
                                                         (pred, 'amino_acid_prediction'),
                                                         (prob, 'amino_acid_probability'))]
    if len(cube_shape) != 3:
        raise _lib.MicaError(f'volumes_to_grid: volumes must be [X, Y, Z], got {tuple(cube_shape)}')
    X, Y, Z = (int(v) for v in cube_shape)
    org = (0, 0, 0) if org is None else tuple(int(v) for v in org)
    ext = (X, Y, Z) if ext is None else tuple(int(v) for v in ext)
    for t, want, name in ((bb, ext, 'backbone_probability'), (ca, ext, 'carbon_alpha_probability'),
                          (pred, ext, 'amino_acid_prediction'), (prob, (20,) + ext, 'amino_acid_probability')):
        if tuple(t.shape) != want:
            raise _lib.MicaError(f'volumes_to_grid: {name} has shape {tuple(t.shape)}, expected {want}')
    target = tuple(int(v) for v in target_shape)
    working = tuple(int(v) for v in working_shape)
    if len(target) != 3 or min(target) < 1 or len(working) != 3:
        raise _lib.MicaError(f'volumes_to_grid: bad target shape {tuple(target_shape)}')
    n = target[0] * target[1] * target[2]
    block = torch.empty(23 * n, dtype=torch.float32, device=bb.device)
    out = StitchedVolumes.from_block(block, target, (0, 0, 0), target).as_dict()
    check(lib.mica_volumes_to_grid(*ptrs, X, Y, Z, _lib.int3(org), _lib.int3(ext), _lib.int3(perm),
                                   _lib.int3(working), _lib.int3(target),
                                   *(C.c_void_p(out[k].data_ptr()) for k in VOLUME_KEYS), _stream()), 'volumes_to_grid')
    return out
