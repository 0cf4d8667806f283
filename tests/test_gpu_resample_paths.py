"""Every kernel route of mica_bspline_resample_f32 against scipy.ndimage.zoom.

The resample picks its prefilter and interpolation kernels from the shape, the zoom and the environment.  Each case
here names the route it must take (mica_last_resample_path, so a moved threshold fails the case instead of silently
testing another kernel) and compares the result with SciPy at the bar of the other resample tests,
max|got - want| <= 2e-6 * max|want|, on two inputs: normal noise, and unit impulses on a zero background at samples
0, 1, n-2, n-1 of each long axis and at (and just before) the segment starts of the kernel under test, where a
finite warm-up or a wrong mirror index would show at full precision."""
import functools
import os
import re
from contextlib import contextmanager

import numpy as np
import pytest
import torch

from mica_b200 import _lib, ops
from mica_b200.slab import SlabPlan
from oracle import mica_oracle as orc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAR = 2e-6          # against SciPy, relative to max|want|
ROUTE_BAR = 3e-7    # fast route against the general route: float32 rounding flips only


def _kernel_ids():
    text = open(os.path.join(ROOT, 'include', 'mica_b200.h')).read()
    return {name: int(v) for name, v in re.findall(r'#define MICA_RS_(\w+) (\d+)', text)}


RS = _kernel_ids()
RS_NAME = {v: k for k, v in RS.items()}


def route():
    """(z prefilter, y prefilter, x pass, interpolation) kernels of the last resample call; None = pass not run."""
    return tuple(RS_NAME.get(_lib.lib.mica_last_resample_path(p)) for p in range(4))


@contextmanager
def force_generic():
    was = _lib.lib.mica_resample_force_generic(1)
    try:
        yield
    finally:
        _lib.lib.mica_resample_force_generic(was)


# ---------------------------------------------------------------- inputs
def _starts(n, n_seg):
    length = -(-n // n_seg)
    return list(range(0, n, length))


def _reg_row_starts(n, n_seg):
    """rows_reg_interp_kernel: ceil(n / n_seg) samples per segment, made odd (distinct banks) while below 26."""
    length = -(-n // n_seg)
    if length % 2 == 0 and length < 26:
        length += 1
    return list(range(0, n, length))


# segment starts of the kernel a case targets along its long axis
SEGS = {
    'rows_pipe_16_512': lambda n: _starts(n, 512 // 16),
    'rows_pipe_8_512': lambda n: _starts(n, 512 // 8),
    'rows_reg32': lambda n: _reg_row_starts(n, 32),
    'seg16': lambda n: _starts(n, 256 // 16),               # prefilter_cols_seg<16> / prefilter_rows_seg<16>
    'cols_reg': lambda n: _starts(n, -(-n // 26)),          # segments of <= kColLen = 26 samples
    'whole_line': lambda n: [],                             # one thread sweeps the whole line: edges only
}


def _impulses(shape, axes):
    """Unit impulses at 0, 1, n-2, n-1 and at every segment start s and s-1 along each axis in ``axes`` (axis ->
    SEGS key); impulse i sits on its own line, at cross position (7i + 3) mod m on the other axes."""
    src = np.zeros(shape, np.float32)
    for axis, seg in axes.items():
        n = shape[axis]
        pos = {0, 1, n - 2, n - 1}
        for s in SEGS[seg](n):
            pos.update(p for p in (s - 1, s) if p >= 0)
        for i, k in enumerate(sorted(pos)):
            idx = [(7 * i + 3 + 5 * a) % shape[a] for a in range(3)]
            idx[axis] = k
            src[tuple(idx)] = 1.0
    return src


def _source(shape, kind, axes):
    if kind == 'noise':
        return np.random.default_rng(sum(shape)).normal(size=shape).astype(np.float32)
    return _impulses(shape, axes)


@functools.lru_cache(maxsize=None)
def _reference(shape, voxel, kind, axes_key, order=3):
    """(source, SciPy result): the SciPy zooms take seconds on the long lines, so each is computed once."""
    src = _source(shape, kind, dict(axes_key))
    return src, orc.resample(src, (np.float32(voxel),) * 3, order=order)


def _resample(cuda, src, out_shape, order=3, **kw):
    got = ops.resample(torch.from_numpy(np.ascontiguousarray(src)).to(cuda), out_shape, order=order, **kw)
    return got.cpu().numpy(), route()


def _rel_err(got, want):
    return float(np.abs(got.astype(np.float64) - want).max()) / float(np.abs(want).max())


# ---------------------------------------------------------------- route cases
# id -> shape, voxel (Angstrom, all axes), route on the default path, route under mica_resample_force_generic(1)
# (None: not run), long axes with the segment scheme their impulses target, environment
CASES = {
    # a, b: x rows longer than the register row pass (832) through the pipelined row kernel, both tile heights
    'a_rows_pipe_16x512': ((96, 96, 867), 1.2, ('COLS_REG', 'COLS_REG', 'ROWS_PIPE_16_512', 'MARCH_YZ_TMA3'),
                           ('COLS32', 'COLS32', 'ROWS4', 'GATHER3'), {2: 'rows_pipe_16_512'}, {}),
    'b_rows_pipe_8x512': ((96, 96, 958), 1.2, ('COLS_REG', 'COLS_REG', 'ROWS_PIPE_8_512', 'MARCH_YZ_TMA3'),
                          ('COLS32', 'COLS32', 'ROWS4', 'GATHER3'), {2: 'rows_pipe_8_512'}, {}),
    # c: the two sides of the x bound, set by the row kernel's shared memory (rows_pipe_smem(sx, 8) <= 220 KiB)
    'c_x1759_fast': ((96, 96, 1759), 0.83, ('COLS_REG', 'COLS_REG', 'ROWS_PIPE_8_512', 'MARCH_YZ_TMA4'),
                     None, {2: 'rows_pipe_8_512'}, {}),
    'c_x1760_general': ((96, 96, 1760), 0.83, ('COLS_SEG16', 'COLS_SEG16', 'ROWS4', 'MARCH3_TMA4'),
                        None, {2: 'whole_line'}, {}),
    # d: y columns longer than 64 register segments (1664 samples)
    'd_y1700_cols_reg': ((96, 1700, 96), 1.06, ('COLS_REG', 'COLS_REG', 'ROWS_REG16', 'MARCH_YZ_TMA3'),
                         ('COLS32', 'COLS8', 'ROWS32', 'GATHER3'), {1: 'cols_reg'}, {}),
    # z lines longer than 64 register segments (1664) and than 1760 samples: the z pass follows the whole line, so
    # these maps and their z-slabs run the same kernels (test_long_z_slab_ranks_reproduce_one_gpu)
    'z1700_cols_reg': ((1700, 96, 96), 1.06, ('COLS_REG', 'COLS_REG', 'ROWS_REG16', 'MARCH_YZ_TMA3'),
                       ('COLS8', 'COLS32', 'ROWS32', 'GATHER3'), {0: 'cols_reg'}, {}),
    'z1800_cols_reg': ((1800, 96, 96), 1.06, ('COLS_REG', 'COLS_REG', 'ROWS_REG16', 'MARCH_YZ_TMA3'),
                       None, {0: 'cols_reg'}, {}),
    # f: the y span of the fast march: zoom_y 1.676 stages 16 rows, zoom_y 1.725 (> 12/7) leaves the fast path
    'f_zoom_y_1.676_fast': ((100, 120, 100), 0.6, ('COLS_REG', 'COLS_REG', 'ROWS_REG16', 'MARCH_YZ_TMA4'),
                            None, {0: 'whole_line', 1: 'whole_line', 2: 'whole_line'}, {}),
    'f_zoom_y_1.725_general': ((100, 120, 100), 0.58, ('COLS_SEG16', 'COLS_SEG16', 'ROWS_SEG16', 'GATHER3'),
                               None, {0: 'whole_line', 1: 'whole_line', 2: 'whole_line'}, {}),
    # g: MICA_NO_TMA=1 takes the general path; lines of 801-3200 samples sweep one per thread in shared memory
    'g_no_tma_z1024': ((1024, 96, 96), 0.83, ('COLS8', 'COLS_SEG16', 'ROWS_SEG16', 'MARCH3_4'),
                       ('COLS8', 'COLS32', 'ROWS32', 'GATHER3'), {0: 'whole_line'}, {'MICA_NO_TMA': '1'}),
    'g_no_tma_x1024': ((96, 96, 1024), 0.83, ('COLS_SEG16', 'COLS_SEG16', 'ROWS4', 'MARCH3_4'),
                       ('COLS32', 'COLS32', 'ROWS4', 'GATHER3'), {2: 'whole_line'}, {'MICA_NO_TMA': '1'}),
    # h: general by zoom (zoom_y 1.83): the per-voxel gather over long rows
    'h_gather3_x1024': ((100, 100, 1024), 0.55, ('COLS_SEG16', 'COLS_SEG16', 'ROWS4', 'GATHER3'),
                        None, {2: 'whole_line'}, {}),
    # i: lines longer than any shared-memory tile: z columns, and rows through the column kernel
    'i_z3300_global': ((3300, 8, 8), 1.2, ('COLS_GLOBAL', 'COLS32', 'ROWS32', 'MARCH3_TMA3'),
                       None, {0: 'whole_line'}, {}),
    'i_x7000_global': ((8, 8, 7000), 1.2, ('COLS32', 'COLS32', 'COLS_GLOBAL', 'MARCH3_TMA3'),
                       None, {2: 'whole_line'}, {}),
    # k: x rows of 417-832 samples: the register row pass with 32 segments per row
    'k_rows_reg32_x700': ((96, 96, 700), 1.2, ('COLS_REG', 'COLS_REG', 'ROWS_REG32', 'MARCH_YZ_TMA3'),
                          ('COLS32', 'COLS32', 'ROWS32', 'GATHER3'), {2: 'rows_reg32'}, {}),
    # l: MICA_NO_TMA=1 on a y span of <= 12 rows: the register-prefetch march staging 12 rows per plane
    'l_no_tma_march3_3': ((96, 96, 96), 1.2, ('COLS_SEG16', 'COLS_SEG16', 'ROWS_SEG16', 'MARCH3_3'),
                          ('COLS32', 'COLS32', 'ROWS32', 'GATHER3'), {0: 'seg16', 1: 'seg16', 2: 'seg16'},
                          {'MICA_NO_TMA': '1'}),
}
TRILINEAR_ROUTE = (None, None, None, 'GATHER1')   # order 1: no prefilter (test_resample_trilinear_long_rows)


def test_every_route_id_is_pinned():
    """Every MICA_RS_* id the header defines is the route of some test here, and every name a test expects is an id
    there: a kernel the resample can report has a case, and an id whose kernel is gone does not linger."""
    named = set(TRILINEAR_ROUTE)
    for _, _, want_route, generic_route, _, _ in CASES.values():
        named.update(want_route)
        named.update(generic_route or ())
    named.discard(None)
    assert sorted(set(RS) - named) == []
    assert sorted(named - set(RS)) == []


@pytest.mark.parametrize('kind', ['noise', 'impulses'])
@pytest.mark.parametrize('case', list(CASES))
def test_resample_route_matches_scipy(cuda, monkeypatch, case, kind):
    shape, voxel, want_route, generic_route, axes, env = CASES[case]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    src, want = _reference(shape, voxel, kind, tuple(sorted(axes.items())))
    out_shape = ops.zoom_output_shape(shape, (np.float32(voxel),) * 3)
    assert out_shape == want.shape
    got, r = _resample(cuda, src, out_shape)
    assert r == want_route
    err = _rel_err(got, want)
    assert err <= BAR, f'{case}/{kind}: {err:.3g} of max|want| against SciPy'
    if case.startswith(('a_', 'b_')):     # SciPy's all-zero last x plane (D11)
        assert not want[:, :, -1].any() and not got[:, :, -1].any()
    if kind == 'noise':                   # and no other all-zero face
        for ax in range(3):
            assert np.take(got, -1, axis=ax).any() == np.take(want, -1, axis=ax).any(), ax
    if generic_route is None:
        return
    with force_generic():
        general, r = _resample(cuda, src, out_shape)
    assert r == generic_route
    err_g = _rel_err(general, want)
    assert err_g <= BAR, f'{case}/{kind}: general route {err_g:.3g} of max|want| against SciPy'
    between = _rel_err(got, general)
    print(f'{case}/{kind}: fast {err:.3g}, general {err_g:.3g}, between {between:.3g} of max|want|')
    assert between <= ROUTE_BAR, f'{case}/{kind}: the two routes differ by {between:.3g} of max|want|'


@pytest.mark.parametrize('kind', ['noise', 'impulses'])
def test_resample_trilinear_long_rows(cuda, kind):
    """j: order 1 has no prefilter; gather1 over rows of 958 -> 1150 samples."""
    shape, voxel, axes = (96, 96, 958), 1.2, {2: 'whole_line'}
    src, want = _reference(shape, voxel, kind, tuple(sorted(axes.items())), order=1)
    got, r = _resample(cuda, src, want.shape, order=1)
    assert r == TRILINEAR_ROUTE
    assert _rel_err(got, want) <= BAR


# ---------------------------------------------------------------- slab form
def _slab_bounds(shape, out_shape, lo, hi, halo=16):
    """Source block of output planes [lo, hi): the taps plus ``halo`` planes (the SlabPlan halo_k) either side."""
    scale_z = (shape[0] - 1) / (out_shape[0] - 1)
    s_lo = max(0, int(np.floor(lo * scale_z)) - 1 - halo)
    s_hi = min(shape[0], int(np.floor((hi - 1) * scale_z)) + 2 + halo + 1)
    return s_lo, s_hi


@pytest.mark.parametrize('case,slabs,want_route', [
    # general path: blocks of > 800 planes take the one-thread-per-line shared-memory sweep
    ('g_no_tma_z1024', [(0, 700), (150, 850)], ('COLS8', 'COLS_SEG16', 'ROWS_SEG16', 'MARCH3_4')),
    # fast path: blocks of a 1700-plane line in the register z pass, first, middle and last planes
    ('z1700_cols_reg', [(0, 700), (500, 1300), (1100, 1802)], ('COLS_REG', 'COLS_REG', 'ROWS_REG16', 'MARCH_YZ_TMA3')),
])
@pytest.mark.parametrize('kind', ['noise', 'impulses'])
def test_resample_slab_on_long_lines(cuda, monkeypatch, case, slabs, want_route, kind):
    """A z-slab (a source block with 16 planes past the taps; src_z0 > 0 but for the first) equals the same planes
    of the whole-map SciPy result."""
    shape, voxel, _, _, axes, env = CASES[case]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    src, want = _reference(shape, voxel, kind, tuple(sorted(axes.items())))
    out_shape = want.shape
    for lo, hi in slabs:
        s_lo, s_hi = _slab_bounds(shape, out_shape, lo, hi)
        assert s_lo > 0 or lo == 0
        got, r = _resample(cuda, src[s_lo:s_hi], out_shape, src_z0=s_lo, src_shape=shape, dst_z0=lo,
                           dst_nz_local=hi - lo)
        assert r == want_route, (lo, hi)
        assert np.abs(got - want[lo:hi]).max() <= BAR * float(np.abs(want).max()), (lo, hi)


# ---------------------------------------------------------------- z-slab bit identity above 1664 planes
@pytest.mark.parametrize('sz', [1700, 1800])
def test_long_z_slab_ranks_reproduce_one_gpu(cuda, sz):
    """The ranks of a z-slab partition (SlabPlan blocks, emulated one after the other) resample their planes to
    the same bits as one GPU resampling the whole map, also where the z line is longer than 64 register segments
    (1664) or 1760 samples: the column kernel is chosen from the whole line."""
    shape, voxel = (sz, 96, 96), (np.float32(1.06),) * 3
    src = torch.from_numpy(np.random.default_rng(sz).normal(size=shape).astype(np.float32)).to(cuda)
    out_shape = ops.zoom_output_shape(shape, voxel)
    whole = ops.resample(src, out_shape)
    whole_route = route()
    assert whole_route[0] == 'COLS_REG'
    for world in (2, 3):
        plan = SlabPlan(shape, voxel, 48, 8, world)
        assert plan.out_shape == out_shape
        for rank, me in enumerate(plan.ranks):
            got = ops.resample(src[me.src_lo:me.src_hi].contiguous(), out_shape, src_z0=me.src_lo, src_shape=shape,
                               dst_z0=me.ext_lo, dst_nz_local=me.ext_hi - me.ext_lo)
            assert route() == whole_route, (world, rank)
            assert torch.equal(got, whole[me.ext_lo:me.ext_hi]), (world, rank)


# ---------------------------------------------------------------- launch-grid limit of the row fall-back
def test_row_fallback_grid_limit_is_reported_before_any_launch(cuda):
    """Rows too long for a shared-memory tile (> 6400 samples) are prefiltered one per CTA along grid y: more than
    65535 of them are refused up front with MICA_ERR_INVALID, not by a failed launch half way through."""
    src = torch.zeros((2, 32768, 6401), dtype=torch.float32, device=cuda)      # 65536 rows
    before = ops.launch_count()
    with pytest.raises(_lib.MicaError, match=r'MICA_ERR_INVALID.*65535'):
        ops.resample(src, (2, 4, 4))
    assert ops.launch_count() == before
    assert route() == (None, None, None, None)


def test_refused_call_launches_nothing(cuda):
    """A call the general path refuses (70000 z lines of one sample: more than the 65535 a launch grid holds)
    returns MICA_ERR_INVALID before it enqueues anything, the tap tables included."""
    sz, out_shape = 70000, (8, 8, 8)
    src = torch.zeros((sz, 1, 1), dtype=torch.float32, device=cuda)
    dst = torch.empty(out_shape, dtype=torch.float32, device=cuda)
    nbytes = _lib.lib.mica_resample_workspace_bytes(sz, 1, 1, *out_shape, 3)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=cuda)
    before = ops.launch_count()
    rc = _lib.lib.mica_resample(src.data_ptr(), _lib.DTYPE_F32, sz, 1, 1, 0, sz, dst.data_ptr(), _lib.DTYPE_F32,
                                *out_shape, 0, out_shape[0], ws.data_ptr(), nbytes, 3,
                                torch.cuda.current_stream().cuda_stream)
    assert _lib.ERR_NAMES.get(rc) == 'MICA_ERR_INVALID', rc
    assert ops.launch_count() == before
    assert route() == (None, None, None, None)
