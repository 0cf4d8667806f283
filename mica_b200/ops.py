"""Torch-tensor front end of the C ABI (device pointers in, device tensors out).

PyTorch is plumbing here -- it owns the HBM allocations and the stream; all the
arithmetic of the hot path happens in libmica_b200.so.  Every function raises
unless its tensors live on a CUDA device: there is no CPU path."""
from __future__ import annotations

import ctypes as C
import functools
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
    24-channel volume.  ``bin`` once per map, ``fill`` once per batch."""

    def __init__(self, device, n_slots, grid_size=48, padding=8, perm=(2, 1, 0)):
        self.device, self.n_slots = device, int(n_slots)
        self.grid_size, self.padding, self.perm = int(grid_size), int(padding), tuple(perm)
        self.buffer = None          # [n_slots,24,W,W,W], allocated (zeroed) by the first fill
        self.status = torch.zeros(1, dtype=torch.int32, device=device)
        self.ws = None
        self._geom = None
        self._shown = None          # the ijk tensor whose cubes the slots currently show (kept alive)

    @device_guard
    def _fill(self, ijk, nonzero_ptr):
        n_atoms, (nz, ny, nx) = self._geom
        prev = self._shown
        check(lib.mica_af3_fill_cubes(C.c_void_p(self.ws.data_ptr()), n_atoms, nz, ny, nx, _lib.int3(self.perm),
                                      self.grid_size, self.padding,
                                      C.c_void_p(prev.data_ptr()) if prev is not None else None,
                                      int(prev.shape[0]) if prev is not None else 0,
                                      C.c_void_p(ijk.data_ptr()) if ijk is not None else None,
                                      int(ijk.shape[0]) if ijk is not None else 0,
                                      C.c_void_p(self.buffer.data_ptr()), self.buffer.stride(0),
                                      nonzero_ptr, _stream()), 'af3_fill_cubes')
        self._shown = ijk

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

    def fill(self, ijk: torch.Tensor, nonzero: torch.Tensor | None = None) -> torch.Tensor:
        """AF3 channels of the cubes ``ijk`` (int32 [B,3], B <= n_slots) -> view [B,24,W,W,W]."""
        B = int(ijk.shape[0])
        if B > self.n_slots:
            raise _lib.MicaError(f'batch of {B} cubes exceeds the {self.n_slots} slots')
        if self._geom is None:
            raise _lib.MicaError('Af3CubeFiller.fill before bin')
        p_nz = _dev(nonzero, torch.int32, 'nonzero') if nonzero is not None else None
        _dev(ijk, torch.int32, 'ijk')
        if self.buffer is None:
            W = self.grid_size + 2 * self.padding
            self.buffer = torch.zeros((self.n_slots, 24, W, W, W), dtype=torch.float32, device=self.device)
        self._fill(ijk, p_nz)
        return self.buffer[:B]


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
                  nonzero: torch.Tensor | None = None, cube_max: torch.Tensor | None = None):
    """vol [C,nz_local,ny,nx] (or [nz,ny,nx]) -> out [B,C,W,W,W] for the cube origins ``ijk``
    (int32 [B,3], cube space).  ``out`` may be a channel slice of a larger [B,Ctot,W,W,W]
    buffer (only the batch stride may be non-dense)."""
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
    if not out.is_cuda or out.dtype != torch.float32 or tuple(out.shape) != (B, Cn, W, W, W):
        raise _lib.MicaError(f'out must be a CUDA float32 [{B},{Cn},{W},{W},{W}] tensor')
    if B and out.stride()[1:] != (W ** 3, W * W, W, 1):
        raise _lib.MicaError('out must be dense in every axis but the batch')
    cube_stride = out.stride(0) if B else Cn * W ** 3
    p_nz = _dev(nonzero, torch.int32, 'nonzero') if nonzero is not None else None
    p_mx = _dev(cube_max, torch.float32, 'cube_max') if cube_max is not None else None
    check(lib.mica_extract_cubes(p_vol, vol.stride(0), Cn, nz, ny, nx, z0, nzl, _lib.int3(perm), grid_size,
                                 padding, p_ijk, B, C.c_void_p(out.data_ptr()), cube_stride, p_nz, p_mx,
                                 _stream()), 'extract_cubes')
    return out


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
    """Fused utils/predict.py:342-349 + :494-501 for one batch of cubes."""
    B = ijk.shape[0]
    W = grid_size + 2 * padding
    for t, c, name in ((bb, 4, 'bb'), (ca, 4, 'ca'), (aa, 21, 'aa')):
        if tuple(t.shape) != (B, c, W, W, W):
            raise _lib.MicaError(f'{name} logits must be [{B},{c},{W},{W},{W}], got {tuple(t.shape)}')
    X, Y, Z = vols.shape
    check(lib.mica_postproc_stitch(
        _dev(bb, torch.float32, 'bb'), _dev(ca, torch.float32, 'ca'), _dev(aa, torch.float32, 'aa'),
        _dev(ijk, torch.int32, 'ijk'), B, X, Y, Z, _lib.int3(vols.org), _lib.int3(vols.ext), grid_size, padding,
        _dev(vols.backbone_probability, torch.float32, 'bb_vol'),
        _dev(vols.carbon_alpha_probability, torch.float32, 'ca_vol'),
        _dev(vols.amino_acid_probability, torch.float32, 'aa_prob_vol'),
        _dev(vols.amino_acid_prediction, torch.float32, 'aa_pred_vol'), _stream()), 'postproc_stitch')
    return vols


class StitchCall:
    """``postproc_stitch`` bound to one set of volumes and one geometry: everything that does not change from
    batch to batch (volume pointers, box, shapes) is converted to ctypes once, so the per-call host cost is a
    handful of microseconds -- the drop-in feeds the model in the reference's batches of <= 8 cubes, i.e.
    hundreds of stitch calls per map.  The caller guarantees CUDA float32 contiguous logits on the volumes'
    device (checked on the first call and whenever the batch size changes)."""

    def __init__(self, vols: 'StitchedVolumes', grid_size: int = 48, padding: int = 8):
        self.vols, self.grid_size, self.padding = vols, int(grid_size), int(padding)
        self.W = self.grid_size + 2 * self.padding
        X, Y, Z = vols.shape
        self._fixed = (X, Y, Z, _lib.int3(vols.org), _lib.int3(vols.ext), self.grid_size, self.padding,
                       _dev(vols.backbone_probability, torch.float32, 'bb_vol'),
                       _dev(vols.carbon_alpha_probability, torch.float32, 'ca_vol'),
                       _dev(vols.amino_acid_probability, torch.float32, 'aa_prob_vol'),
                       _dev(vols.amino_acid_prediction, torch.float32, 'aa_pred_vol'))
        self._checked_B = -1
        self._dev_index = vols.device.index

    def __call__(self, bb, ca, aa, ijk):
        B = ijk.shape[0]
        if B != self._checked_B:
            W = self.W
            for t, c, name in ((bb, 4, 'bb'), (ca, 4, 'ca'), (aa, 21, 'aa')):
                if tuple(t.shape) != (B, c, W, W, W):
                    raise _lib.MicaError(f'{name} logits must be [{B},{c},{W},{W},{W}], got {tuple(t.shape)}')
                _dev(t, torch.float32, name)
                if t.device != self.vols.device:
                    raise _lib.MicaError(f'{name} logits live on {t.device}, the volumes on {self.vols.device}')
            _dev(ijk, torch.int32, 'ijk')
            self._checked_B = B
        if torch.cuda.current_device() != self._dev_index:
            with torch.cuda.device(self._dev_index):
                return self(bb, ca, aa, ijk)
        X, Y, Z, org, ext, gs, pad, p_bb, p_ca, p_aap, p_aapred = self._fixed
        check(lib.mica_postproc_stitch(bb.data_ptr(), ca.data_ptr(), aa.data_ptr(), ijk.data_ptr(), B, X, Y, Z, org,
                                       ext, gs, pad, p_bb, p_ca, p_aap, p_aapred,
                                       torch.cuda.current_stream().cuda_stream), 'postproc_stitch')


@device_guard
def postproc_stitch_peer(bb: torch.Tensor, ca: torch.Tensor, aa: torch.Tensor, ijk: torch.Tensor, cube_shape,
                         owner_table: torch.Tensor, x_bounds, grid_size: int = 48, padding: int = 8):
    """``postproc_stitch`` for one map whose cubes are dealt out over several GPUs: every core plane goes to
    the volume block of the rank that owns its x range (``owner_table``: int64 device tensor of ``world``
    base pointers, ``peer.PeerVolumes.table``; ``x_bounds``: world + 1 plane bounds), local or over NVLink."""
    B = ijk.shape[0]
    W = grid_size + 2 * padding
    for t, c, name in ((bb, 4, 'bb'), (ca, 4, 'ca'), (aa, 21, 'aa')):
        if tuple(t.shape) != (B, c, W, W, W):
            raise _lib.MicaError(f'{name} logits must be [{B},{c},{W},{W},{W}], got {tuple(t.shape)}')
    X, Y, Z = (int(v) for v in cube_shape)
    world = int(owner_table.numel())
    bounds = (C.c_int * (world + 1))(*[int(v) for v in x_bounds])
    check(lib.mica_postproc_stitch_peer(
        _dev(bb, torch.float32, 'bb'), _dev(ca, torch.float32, 'ca'), _dev(aa, torch.float32, 'aa'),
        _dev(ijk, torch.int32, 'ijk'), B, X, Y, Z, grid_size, padding,
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


def is_core_window(w1, grid_size: int, padding: int) -> bool:
    """True for the 1-on-the-core window: its weighted stitch IS the reference's paste, and runs as one."""
    return np.array_equal(w1, overlap_window('core', grid_size, padding))


def overlap_norm_tables(w1, cube_shape, grid_size: int, padding: int):
    """Reciprocals (0 where the sum is 0) of the 1-D weight sums Wx, Wy, Wz of the full cube lattice
    (``cube_origins``): the weight sum of the overlap-weighted stitch at voxel (x, y, z) is Wx[x] Wy[y] Wz[z], with
    Wx[x] = sum over the origins i covering x of w1[x - i + padding].  float64, origins added in ascending order.
    Whatever part of the lattice a run stitches, these come from all of it."""
    w = np.asarray(w1, dtype=np.float32).astype(np.float64)
    W = len(w)
    out = []
    for n in (int(v) for v in cube_shape):
        s = np.zeros(n, np.float64)
        for i in range(0, n, int(grid_size)):
            lo = i - int(padding)
            x0, x1 = max(0, lo), min(n, lo + W)
            s[x0:x1] += w[x0 - lo:x1 - lo]
        r = np.zeros(n, np.float64)
        np.divide(1.0, s, out=r, where=s > 0)
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
    """Where the contributions of an overlap-weighted stitch go when the output is split over ranks: rank r owns
    planes [bounds[r], bounds[r+1]) of cube axis ``axis`` (0 = x, 2 = k) as the 23-channel block at ``table[r]``
    (int64 device tensor of base pointers, ``peer.PeerVolumes.table``); ``devices``: the CUDA device index of each
    owner, whose memory the accumulating device must be able to add into atomically."""
    table: torch.Tensor
    axis: int
    bounds: tuple
    devices: tuple


class OverlapStitcher:
    """The north_star's "stitch with overlap weights": every voxel of every window adds its probabilities times
    the window weight, normalised by the weight sum of the full cube lattice, in 2^-31 fixed point (uint32), so the
    result does not depend on the order of the cubes, the batches or the partition; ``finalize`` converts in place.
    NOT the reference's arithmetic, which pastes the disjoint cores (``postproc_stitch``; DESIGN.md D2) -- offered
    as a mode next to it; ``window='core'`` runs that paste.  Costs several times the reference mode: every voxel of
    every 64^3 window is post-processed and added, not just the 32^3 (48^3) cores.

    ``vols``: the volumes (``StitchedVolumes.from_block``, zeroed) this stitcher finalizes; default: a whole-map
    block of its own.  ``owners``: an ``OverlapOwners`` table -- contributions go to the block of the rank that
    owns their plane, locally or over NVLink (native peer atomics required); without ``vols`` such a stitcher only
    accumulates."""

    def __init__(self, cube_shape, device, grid_size: int = 48, padding: int = 8, window='uniform', *, vols=None,
                 owners: OverlapOwners | None = None):
        self.shape = tuple(int(v) for v in cube_shape)
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        self.grid_size, self.padding = int(grid_size), int(padding)
        self.w1 = overlap_window(window, grid_size, padding)
        self.core = is_core_window(self.w1, self.grid_size, self.padding)
        self.owners = owners
        if owners is not None:
            if owners.axis not in (0, 2) or (self.core and owners.axis != 0):
                raise _lib.MicaError(f'owners along cube axis {owners.axis}: the weighted stitch splits along 0 or 2, '
                                     'the core window (the paste) along 0')
            for d in owners.devices:
                if not peer_atomics_supported(self.device.index, d):
                    raise _lib.MicaError(f'overlap-weighted stitching over several GPUs adds into the owners\' '
                                         f'memory atomically: cuda:{self.device.index} has no native peer atomics '
                                         f'with cuda:{d}')
            self._bounds = (C.c_int * len(owners.bounds))(*[int(v) for v in owners.bounds])
        if vols is None and owners is None:
            X, Y, Z = self.shape
            with torch.cuda.device(self.device):
                vols = StitchedVolumes.from_block(torch.zeros(23 * X * Y * Z, dtype=torch.float32,
                                                              device=self.device), self.shape, (0, 0, 0), self.shape)
        if vols is not None and (getattr(vols, 'block', None) is None or vols.device != self.device):
            raise _lib.MicaError('OverlapStitcher needs volumes of StitchedVolumes.from_block on its own device')
        self.vols = vols
        if not self.core:
            with torch.cuda.device(self.device):
                self.norm = torch.from_numpy(np.concatenate(
                    overlap_norm_tables(self.w1, self.shape, self.grid_size, self.padding))).to(self.device)
        self._done = False

    @device_guard
    def accumulate(self, bb, ca, aa, ijk, vols=None):
        if self.core:
            if self.owners is not None:
                postproc_stitch_peer(bb, ca, aa, ijk, self.shape, self.owners.table, self.owners.bounds,
                                     self.grid_size, self.padding)
            else:
                postproc_stitch(bb, ca, aa, ijk, self.vols, self.grid_size, self.padding)
            return
        B = ijk.shape[0]
        W = self.grid_size + 2 * self.padding
        for t, c, name in ((bb, 4, 'bb'), (ca, 4, 'ca'), (aa, 21, 'aa')):
            if tuple(t.shape) != (B, c, W, W, W):
                raise _lib.MicaError(f'{name} logits must be [{B},{c},{W},{W},{W}], got {tuple(t.shape)}')
        X, Y, Z = self.shape
        args = (_dev(bb, torch.float32, 'bb'), _dev(ca, torch.float32, 'ca'), _dev(aa, torch.float32, 'aa'),
                _dev(ijk, torch.int32, 'ijk'), B, X, Y, Z, self.grid_size, self.padding,
                self.w1.ctypes.data_as(C.POINTER(C.c_float)), C.c_void_p(self.norm.data_ptr()))
        if self.owners is None:
            check(lib.mica_overlap_accumulate_fixed(*args, C.c_void_p(self.vols.block.data_ptr()), _stream()),
                  'overlap_accumulate')
        else:
            o = self.owners
            check(lib.mica_overlap_accumulate_fixed_peer(*args, _dev(o.table, torch.int64, 'owner_table'), int(o.axis),
                                                         self._bounds, int(o.table.numel()), _stream()),
                  'overlap_accumulate_peer')

    @device_guard
    def finalize(self) -> StitchedVolumes:
        """The four volumes (views of the accumulation block, laid out as ``StitchedVolumes.from_block``).  With
        owners, call it once every rank's contributions have landed (stream sync + barrier)."""
        if self.vols is None:
            raise _lib.MicaError('this OverlapStitcher only accumulates into other ranks\' volumes')
        if not self._done and not self.core:
            e = self.vols.ext
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
