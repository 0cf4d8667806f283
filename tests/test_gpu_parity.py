"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the
golden vectors the unmodified reference produced (tests/golden, oracle/make_golden.py).

Bars (BASELINE.json north_star): cube indexing, AF3 occupancy and the
median / percentile thresholds bit-exact; resampled and stitched float volumes
within 1e-5 max-abs on the [0,1] scale."""
import os

import numpy as np
import pytest
import torch

from mica_b200 import _lib, ops, synthetic
from mica_b200.pipeline import MapHeader, MapPipeline
from oracle import mica_oracle as orc

from _golden import load_stitch

pytestmark = pytest.mark.gpu

TOL = 1e-5


def dev(a, cuda, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.to(cuda)


# ------------------------------------------------------------------ R1 resample
@pytest.mark.parametrize('shape,voxel', [
    ((20, 23, 17), (1.06, 1.06, 1.06)),
    ((26, 30, 22), (0.97, 1.13, 1.06)),      # anisotropic (D9): zoom list [vx,vy,vz] hits axes z,y,x
    ((30, 30, 30), (0.83, 0.83, 0.83)),      # down-sampling
    ((30, 36, 33), (1.2, 1.2, 1.2)),         # 30 -> 36 overshoots on z: SciPy zero last plane (D11)
    ((64, 48, 40), (1.37, 1.21, 1.5)),
    ((5, 4, 3), (2.0, 2.5, 3.0)),            # tiny axes: general mirror formula
])
@pytest.mark.parametrize('order', [3, 1])
def test_resample_matches_scipy(cuda, shape, voxel, order):
    rng = np.random.default_rng(hash((shape, order)) % 2**32)
    src = rng.normal(size=shape).astype(np.float32)
    voxel = tuple(np.float32(v) for v in voxel)
    want = orc.resample(src, voxel, order=order)
    zf = orc.zoom_factors(voxel)
    out_shape = ops.zoom_output_shape(shape, zf)
    assert out_shape == want.shape == orc.zoom_output_shape(shape, zf)
    got = ops.resample(dev(src, cuda), out_shape, order=order).cpu().numpy()
    scale = float(np.abs(want).max())
    assert np.abs(got - want).max() <= 2e-6 * scale


@pytest.mark.parametrize('shape,voxel', [
    ((100, 104, 98), (1.2, 1.2, 1.2)),       # segment-parallel prefilter + marching gather (3 x 4 staged rows)
    ((128, 96, 112), (1.06, 1.2, 0.97)),     # anisotropic, mixed up/down-sampling
    ((150, 100, 97), (0.8, 0.8, 0.8)),       # down-sampling: wider y span (4 x 4 staged rows)
    ((128, 128, 100), (1.2, 1.2, 1.2)),      # 128 -> 154 overshoots on z and y (D11) on the fast path
    ((97, 130, 260), (1.31, 1.07, 1.13)),    # ragged tiles: nx, ny not multiples of 64 / 8
])
def test_resample_fast_path_matches_scipy_and_general_path(cuda, shape, voxel):
    rng = np.random.default_rng(hash(shape) % 2**32)
    src = rng.normal(size=shape).astype(np.float32)
    voxel = tuple(np.float32(v) for v in voxel)
    want = orc.resample(src, voxel, order=3)
    out_shape = ops.zoom_output_shape(shape, orc.zoom_factors(voxel))
    assert out_shape == want.shape
    d_src = dev(src, cuda)
    got = ops.resample(d_src, out_shape).cpu().numpy()
    was = _lib.lib.mica_resample_force_generic(1)
    try:
        general = ops.resample(d_src, out_shape).cpu().numpy()
    finally:
        _lib.lib.mica_resample_force_generic(was)
    scale = float(np.abs(want).max())
    assert np.abs(got - want).max() <= 2e-6 * scale
    assert np.abs(general - want).max() <= 2e-6 * scale
    # the two routes differ only in summation order / the 30-sample warm-up: float32 rounding flips at most
    assert np.abs(got - general).max() <= 3e-7 * scale
    if shape == (128, 128, 100):
        assert not got[-1].any() and not got[:, -1].any() and got[:-1, :-1].any()      # D11 zero faces


def test_resample_slab_fast_path(cuda):
    """A z-slab (source planes + halo in, owned output planes out) on the fast kernels equals
    the same planes of the whole-volume SciPy result."""
    shape, voxel = (330, 100, 101), (np.float32(1.2),) * 3
    src = np.random.default_rng(3).normal(size=shape).astype(np.float32)
    want = orc.resample(src, voxel, order=3)
    out_shape = want.shape
    scale_z = (shape[0] - 1) / (out_shape[0] - 1)
    scale = float(np.abs(want).max())
    for lo, hi in ((0, 140), (120, 290), (250, out_shape[0])):
        s_lo = max(0, int(np.floor(lo * scale_z)) - 1 - 16)
        s_hi = min(shape[0], int(np.floor((hi - 1) * scale_z)) + 2 + 16 + 1)
        got = ops.resample(dev(src[s_lo:s_hi], cuda), out_shape, src_z0=s_lo, src_shape=shape,
                           dst_z0=lo, dst_nz_local=hi - lo).cpu().numpy()
        assert np.abs(got - want[lo:hi]).max() <= 2e-6 * scale


def test_resample_golden_then_normalize_end_to_end(cuda, golden_dir):
    g = np.load(os.path.join(golden_dir, 'preprocess_small.npz'))
    src, voxel = g['src'], g['voxel']
    zf = orc.zoom_factors(voxel)
    res = ops.resample(dev(src, cuda), ops.zoom_output_shape(src.shape, zf))
    assert np.abs(res.cpu().numpy() - g['oracle_resampled']).max() <= 2e-6 * np.abs(g['oracle_resampled']).max()
    norm, st = ops.normalize(res)
    med, p, npos, status = st.result()
    assert status == 0
    # end to end (resample -> stats -> clip): float tolerance on the [0,1] scale
    assert np.abs(norm.cpu().numpy() - g['ref_normalized']).max() <= TOL
    assert abs(float(med) - float(g['median'])) <= 1e-6 and abs(float(p) - float(g['p999'])) <= 1e-5


# ------------------------------------------------------------- R2/R3 normalise
def _check_normalize(x, cuda):
    want, med, p = orc.normalize(x.copy())
    norm, st = ops.normalize(dev(x, cuda))
    g_med, g_p, g_npos, status = st.result()
    if want is None:
        assert status != 0
        return
    assert status == 0
    assert g_med == np.float32(med), (g_med, med)              # bit-exact thresholds
    assert g_p == np.float32(p), (g_p, p)
    got = norm.cpu().numpy()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))   # bit-exact volume
    r_med, r_p, r_npos = orc.order_stats_restated(x)
    assert g_npos == r_npos


@pytest.mark.parametrize('n', [1, 2, 3, 1000, 1001, 4099, 250_000, 1_000_003])
def test_normalize_bit_exact_sizes(cuda, n):
    rng = np.random.default_rng(n)
    x = (rng.normal(size=n) ** 3).astype(np.float32)
    _check_normalize(x.reshape(-1, 1, 1) if n < 8 else x, cuda)


def test_normalize_short_path_is_bit_identical_to_numpy_arithmetic(cuda):
    """The lean normaliser (compare / subtract / reciprocal-step division) must give the same
    float32 bits as the operation-by-operation NumPy expression, for every voxel."""
    import ctypes as C
    rng = np.random.default_rng(11)
    n = 1 << 24
    st = ops.OrderStats(cuda)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    cases = [(0.0173, 0.91), (-3.5e-3, 7.7e-4), (1.25, 33.333), (0.0, 1.0), (2.5e-5, 1.9999999),
             (1e-3, float(np.float32(1.9999999) - np.float32(1e-7))), (0.1, 3e-38), (-7.0, 1.17e-36)]
    for med, p in cases:
        med, p = np.float32(med), np.float32(p)
        x = (rng.standard_normal(n) * 3 * float(p) + float(med)).astype(np.float32)
        x[::97] = med
        x[1::193] = med + p                      # lands on / next to the clip threshold
        x[2::389] = np.nextafter(med, np.float32(np.inf))
        x[3::1021] = np.float32(3e38) * np.sign(x[3::1021])
        x[4::4099] = np.nan
        x[5::8191] = np.inf
        x[6::8191] = -np.inf
        x[7::997] = np.float32(-0.0)
        dx = dev(x, cuda)
        _lib.check(_lib.lib.mica_select_set_thresholds(st._p, float(med), float(p), stream))
        fast = st.apply(dx).cpu().numpy()
        was = _lib.lib.mica_normalize_force_reference_arith(1)
        try:
            ref = st.apply(dx).cpu().numpy()
        finally:
            _lib.lib.mica_normalize_force_reference_arith(was)
        assert np.array_equal(fast.view(np.uint32), ref.view(np.uint32)), (med, p)
        # and the operation-by-operation path is NumPy's result (utils/preprocessing.py:122-133)
        with np.errstate(all='ignore'):
            v = np.nan_to_num(x[:1 << 20])
            m = (v > med) * (v - med)
            want = ((m < p) * m + (m >= p) * p) / p
        assert np.array_equal(ref[:1 << 20].view(np.uint32), want.astype(np.float32).view(np.uint32)), (med, p)


def test_order_stats_guided_pass_fallback_and_adversarial_sample(cuda):
    """The digit-0 pass trusts a 1/64 sample only after verifying it on exact counts: a forced
    rejection and a map whose sampled voxels are decoys must both give NumPy's thresholds."""
    rng = np.random.default_rng(21)
    x = (rng.standard_normal(1 << 22) * 0.05).astype(np.float32)
    x[::37] += rng.random(x[::37].shape, dtype=np.float32)
    want = orc.normalize(x)
    was = _lib.lib.mica_select_force_fallback(1)
    try:
        norm, st = ops.normalize(dev(x, cuda))
    finally:
        _lib.lib.mica_select_force_fallback(was)
    med, p, npos, status = st.result()
    assert status == 0 and np.float32(med) == np.float32(want[1]) and np.float32(p) == np.float32(want[2])
    assert np.array_equal(norm.cpu().numpy(), want[0])
    # decoys exactly where the sample looks (every 64th float4 of the 16-byte aligned array)
    y = x.copy()
    y.reshape(-1, 256)[:, :4] = 1000.0 + rng.random((y.size // 256, 4), dtype=np.float32)
    want = orc.normalize(y)
    norm, st = ops.normalize(dev(y, cuda))
    med, p, npos, status = st.result()
    assert status == 0 and np.float32(med) == np.float32(want[1]) and np.float32(p) == np.float32(want[2])
    assert np.array_equal(norm.cpu().numpy(), want[0])
    # and the other way round: the sample sees only background, the tail is elsewhere
    z = x.copy()
    z.reshape(-1, 256)[:, :4] = 0.0
    want = orc.normalize(z)
    norm, st = ops.normalize(dev(z, cuda))
    med, p, npos, status = st.result()
    assert status == 0 and np.float32(med) == np.float32(want[1]) and np.float32(p) == np.float32(want[2])
    assert np.array_equal(norm.cpu().numpy(), want[0])


def test_order_stats_compact_buffer_paths(cuda):
    """From 4 M voxels on, the guided digit-0 pass compacts the candidate voxels and the four later digit
    passes read that buffer instead of the map.  Thresholds must stay NumPy's on every path: buffer used,
    buffer overflowing (heavy ties: the median's bin holds most of the map), guided pass rejected, an
    unaligned array (scalar head / tail), and a second, smaller map through the same workspace."""
    rng = np.random.default_rng(33)
    n = 6_000_003
    x = (rng.standard_normal(n) * 0.05).astype(np.float32)
    x[::41] += rng.random(x[::41].shape, dtype=np.float32)
    st = ops.OrderStats(cuda)

    def check(arr, expect_used):
        want = orc.normalize(arr)
        d = dev(arr, cuda) if isinstance(arr, np.ndarray) else arr
        st.run(d)
        med, p, npos, status = st.result()
        used, count, cap = st.compact_info()
        assert status == 0 and np.float32(med) == np.float32(want[1]) and np.float32(p) == np.float32(want[2]), (med, p, want[1:])
        assert np.array_equal(st.apply(d).cpu().numpy(), want[0])
        if expect_used is not None:
            assert used == expect_used, (used, count, cap)
        return used, count, cap

    used, count, cap = check(x, True)
    assert 0 < count < cap and cap >= n // 8                   # a few percent of the map
    ties = x.copy()
    ties[: int(0.6 * n)] = 0.0125                              # the median's digit-0 bin overflows the buffer
    rng.shuffle(ties)
    used, count, cap = check(ties, False)
    assert count > cap
    was = _lib.lib.mica_select_force_fallback(1)               # guided pass rejected -> full histogram, no buffer
    try:
        check(x, False)
    finally:
        _lib.lib.mica_select_force_fallback(was)
    big = dev(np.concatenate([np.zeros(1, np.float32), x]), cuda)
    want = orc.normalize(x)                                    # x[1:] of a 16-byte aligned buffer: unaligned view
    view = big[1:]
    st.run(view)
    med, p, _, status = st.result()
    assert status == 0 and np.float32(med) == np.float32(want[1]) and np.float32(p) == np.float32(want[2])
    assert st.compact_info()[0] is True
    check(x[:4_500_001].copy(), True)                          # smaller map, same workspace
    check(x[:100_000].copy(), None)                            # tiny map: everything is a candidate


def test_normalize_bit_exact_on_oracle_resampled(cuda, golden_dir):
    """Stage isolation (SURVEY 8c): feed SciPy's own float32 volume to the GPU normaliser."""
    g = np.load(os.path.join(golden_dir, 'preprocess_small.npz'))
    norm, st = ops.normalize(dev(g['oracle_resampled'], cuda))
    med, p, _, status = st.result()
    assert status == 0 and med == g['median'] and p == g['p999']
    assert np.array_equal(norm.cpu().numpy().view(np.uint32), g['ref_normalized'].view(np.uint32))


def test_normalize_heavy_ties_and_specials(cuda):
    rng = np.random.default_rng(5)
    x = rng.normal(size=(40, 50, 60)).astype(np.float32)
    x[:20] = 0.25                                   # half the volume is one constant
    x[20:25] = np.round(x[20:25], 1)                # few distinct values
    x[30, 0, :5] = [np.nan, np.inf, -np.inf, -0.0, 0.0]
    _check_normalize(x, cuda)
    y = np.zeros((16, 16, 16), np.float32)          # no positives -> failure status
    _check_normalize(y, cuda)
    y[3, 3, 3] = 1.0                                # a single positive
    _check_normalize(y, cuda)
    z = np.abs(rng.normal(size=300_001)).astype(np.float32) * 1e-42   # denormals
    _check_normalize(z, cuda)
    w = -np.abs(rng.normal(size=(31, 33, 35))).astype(np.float32)     # all negative
    _check_normalize(w, cuda)


def test_normalize_synthetic_map(cuda):
    vol = synthetic.synthetic_map((96, 80, 72), seed=4)
    _check_normalize(vol, cuda)


@pytest.mark.parametrize('n', [(1 << 24) + 12345, 40_000_000])
def test_normalize_large_float32_index_quirk(cuda, n):
    """N > 2^24: NumPy 2 computes the percentile's virtual index in float32 (D3)."""
    rng = np.random.default_rng(1)
    x = rng.standard_normal(n, dtype=np.float32)
    _check_normalize(x, cuda)


# ---------------------------------------------------------------- R4 AF3 encode
def _encode(st, origin, shape, cuda, keep=None):
    keep = ~st['hetero'] if keep is None else keep
    bb, aa = orc.channel_codes([a for a, k in zip(st['atom_names'], keep) if k],
                               [r for r, k in zip(st['res_names'], keep) if k])
    coords = st['coords'][keep]
    want, ok = orc.af3_encode(coords, bb, aa, origin, shape)
    vol, status = ops.af3_encode(dev(coords, cuda), dev(bb, cuda), dev(aa, cuda), origin, shape)
    return want, ok, vol.cpu().numpy(), int(status.item())


def test_af3_encode_golden(cuda, golden_dir):
    for name in ('af3_cubic.npz',):
        g = np.load(os.path.join(golden_dir, name))
        shape = tuple(int(v) for v in g['shape'])
        vol, status = ops.af3_encode(dev(g['coords'], cuda), dev(g['bb_ch'], cuda), dev(g['aa_ch'], cuda),
                                     g['origin'], shape)
        assert int(status.item()) == 0
        nzi = np.argwhere(vol.cpu().numpy() > 0).astype(np.int32)
        assert np.array_equal(nzi, g['af3_nonzero'])
        assert set(np.unique(vol.cpu().numpy())) <= {0.0, 1.0}
    g = np.load(os.path.join(golden_dir, 'preprocess_small.npz'))     # non-cubic: IndexError path
    shape = g['ref_normalized'].shape
    _, status = ops.af3_encode(dev(g['coords'], cuda), dev(g['bb_ch'], cuda), dev(g['aa_ch'], cuda),
                               g['origin'], shape)
    assert bool(g['af3_ok']) == (int(status.item()) == 0)


@pytest.mark.parametrize('shape', [(40, 40, 40), (64, 48, 32), (32, 48, 64), (50, 100, 70)])
def test_af3_encode_vs_oracle(cuda, shape):
    nz, ny, nx = shape
    origin = (np.float32(-12.5), np.float32(3.25), np.float32(100.0))
    st = synthetic.synthetic_structure(300, (nx, ny, nz), seed=nz, origin_xyz=origin, margin=0.0,
                                       hetero_every=11, unknown_every=6)
    st['coords'][::7] += np.float32(5.0)
    st['coords'][3::23] = np.floor(st['coords'][3::23]) + np.float32(0.5)       # ties -> half-even
    want, ok, got, status = _encode(st, origin, shape, cuda)
    assert ok == (status == 0)
    if ok:
        assert np.array_equal(got, want)


def test_af3_encode_misclamp_quirk(cuda):
    """D7 on (nz,ny,nx)=(70,100,50): x is clamped to nz-1=69 >= nx -> IndexError path;
    on (50,100,70) a valid x=65 is silently moved to 49."""
    origin = (np.float32(0), np.float32(0), np.float32(0))
    coords = np.array([[65.2, 10.0, 20.0]], np.float32)
    bb = np.array([0], np.int8)
    aa = np.array([4], np.int8)
    want, ok = orc.af3_encode(coords, bb, aa, origin, (50, 100, 70))
    vol, status = ops.af3_encode(dev(coords, cuda), dev(bb, cuda), dev(aa, cuda), origin, (50, 100, 70))
    assert ok and int(status.item()) == 0 and np.array_equal(vol.cpu().numpy(), want)
    assert want[0, 20, 10, 49] == 1.0
    want, ok = orc.af3_encode(coords, bb, aa, origin, (70, 100, 50))
    _, status = ops.af3_encode(dev(coords, cuda), dev(bb, cuda), dev(aa, cuda), origin, (70, 100, 50))
    assert (not ok) and int(status.item()) == 1


def test_af3_encode_empty(cuda):
    e = torch.zeros((0, 3), dtype=torch.float32, device=cuda)
    c = torch.zeros((0,), dtype=torch.int8, device=cuda)
    vol, status = ops.af3_encode(e, c, c, (0, 0, 0), (8, 9, 10))
    assert vol.shape == (24, 8, 9, 10) and float(vol.abs().sum()) == 0 and int(status.item()) == 0


# ------------------------------------------------- R4 + R5 fused: sparse AF3 cube fill
@pytest.mark.parametrize('shape,gs,pad,axes', [((40, 40, 40), 32, 16, (1, 2, 3)), ((50, 100, 70), 48, 8, (1, 2, 3)),
                                               ((64, 48, 32), 48, 8, (2, 3, 1)), ((21, 30, 17), 8, 2, (3, 1, 2))])
def test_sparse_af3_cube_fill_equals_dense_extract(cuda, shape, gs, pad, axes):
    """fill(bin(atoms)) == extract_cubes(af3_encode(atoms)) bit for bit, across slot reuse."""
    nz, ny, nx = shape
    origin = (np.float32(3.5), np.float32(-2.25), np.float32(0.0))
    st = synthetic.synthetic_structure(400, (min(nx, nz), ny, min(nx, nz)), seed=nx, origin_xyz=origin, margin=0.0,
                                       hetero_every=11, unknown_every=6)
    keep = ~st['hetero']
    bb, aa = orc.channel_codes([a for a, k in zip(st['atom_names'], keep) if k],
                               [r for r, k in zip(st['res_names'], keep) if k])
    coords = st['coords'][keep]
    d_atoms = (dev(coords, cuda), dev(bb, cuda), dev(aa, cuda))
    vol, status = ops.af3_encode(*d_atoms, origin, shape)
    assert int(status.item()) == 0
    perm, _ = orc.transpose_order(*axes, (0, 0, 0))
    ijk = ops.cube_origins(ops.cube_space_shape(shape, perm), gs)
    d_ijk = dev(ijk, cuda)
    filler = ops.Af3CubeFiller(cuda, 5, gs, pad, perm)
    assert int(filler.bin(*d_atoms, origin, shape).item()) == 0
    order = np.random.default_rng(1).permutation(len(ijk))          # arbitrary batch composition
    d_ijk = d_ijk[torch.from_numpy(order).to(cuda)].contiguous()
    for b0 in range(0, len(ijk), 5):
        sub = d_ijk[b0:b0 + 5].contiguous()
        nzf = torch.empty(len(sub), dtype=torch.int32, device=cuda)
        got = filler.fill(sub, nzf)
        want = ops.extract_cubes(vol, sub, gs, pad, perm)
        assert torch.equal(got, want), b0
        assert torch.equal(nzf != 0, want.reshape(len(sub), -1).abs().sum(1) > 0)
    filler.clear()
    assert float(filler.buffer.abs().sum()) == 0.0                   # un-scatter restores all zeros
    # re-bin with other atoms: the buffer must follow
    d2 = (d_atoms[0][::2].contiguous() + 1.0, d_atoms[1][::2].contiguous(), d_atoms[2][::2].contiguous())
    vol2, _ = ops.af3_encode(*d2, origin, shape)
    filler.fill(d_ijk[:3].contiguous())
    filler.bin(*d2, origin, shape)
    assert torch.equal(filler.fill(d_ijk[:4].contiguous()), ops.extract_cubes(vol2, d_ijk[:4].contiguous(), gs, pad, perm))


def test_sparse_af3_reports_the_index_error_path(cuda):
    origin = (np.float32(0), np.float32(0), np.float32(0))
    coords = dev(np.array([[65.2, 10.0, 20.0]], np.float32), cuda)
    bb, aa = dev(np.array([0], np.int8), cuda), dev(np.array([4], np.int8), cuda)
    f = ops.Af3CubeFiller(cuda, 2, 48, 8)
    assert int(f.bin(coords, bb, aa, origin, (50, 100, 70)).item()) == 0       # silently mis-clamped (D7 i)
    assert int(f.bin(coords, bb, aa, origin, (70, 100, 50)).item()) == 1       # IndexError path (D7 ii)


# ------------------------------------------------------------ R5/R6 cube extract
def _extract(vol, cuda, grid_size, padding, axes=(1, 2, 3), transpose=True):
    if transpose:
        perm, _ = orc.transpose_order(*axes, (0, 0, 0))
    else:
        perm = (0, 1, 2)
    want, meta, shp, _ = orc.extract_cubes(vol, *axes, (0, 0, 0), grid_size, padding, transpose=transpose)
    ijk = ops.cube_origins(ops.cube_space_shape(vol.shape, perm), grid_size)
    assert np.array_equal(ijk, meta[:, :3])
    got = ops.extract_cubes(dev(vol, cuda), dev(ijk, cuda), grid_size, padding, perm)
    return want, got[:, 0].cpu().numpy()


@pytest.mark.parametrize('axes', [(1, 2, 3), (2, 3, 1), (3, 1, 2), (1, 3, 2), (2, 1, 3), (3, 2, 1)])
def test_extract_all_axis_orders_small_window(cuda, axes):
    rng = np.random.default_rng(sum(axes))
    vol = rng.random((9, 21, 13), dtype=np.float32)
    want, got = _extract(vol, cuda, 8, 2, axes)
    assert np.array_equal(got, want)


def test_extract_reference_defaults_noncubic(cuda, golden_dir):
    g = np.load(os.path.join(golden_dir, 'cubes.npz'))
    rng = np.random.default_rng(2022)
    vol = rng.random((50, 100, 70), dtype=np.float32)           # same draw as make_golden
    want, got = _extract(vol, cuda, 48, 8)
    assert np.array_equal(got, want)
    assert np.array_equal(np.array([np.bitwise_xor.reduce(c.view(np.uint32).ravel()) for c in got]), g['d_xor'])
    assert np.allclose([c.astype(np.float64).sum() for c in got], g['d_sum'], rtol=0, atol=0)
    # dense small-window goldens incl. a non-standard axis order
    small = g['s_vol']
    _, got = _extract(small, cuda, 8, 2)
    assert np.array_equal(got, g['s_cubes'])
    _, got = _extract(small, cuda, 8, 2, axes=(2, 3, 1))
    assert np.array_equal(got, g['a_cubes'])


def test_extract_training_twin_no_transpose_and_max_filter(cuda, golden_dir):
    g = np.load(os.path.join(golden_dir, 'cubes.npz'))
    vol = g['t_vol']
    want, meta, _, _ = orc.extract_cubes(vol, grid_size=8, padding=2, transpose=False)
    ijk = ops.cube_origins(vol.shape, 8)
    cmax = torch.empty(len(ijk), dtype=torch.float32, device=cuda)
    got = ops.extract_cubes(dev(vol, cuda), dev(ijk, cuda), 8, 2, (0, 1, 2), cube_max=cmax)
    assert np.array_equal(got[:, 0].cpu().numpy(), want)
    keep = cmax.cpu().numpy() >= 0.01          # create_grids_for_normalized_map.py:78
    assert np.array_equal(ijk[keep], g['t_meta'][:, :3])


def test_extract_stride32_multichannel_and_flags(cuda):
    rng = np.random.default_rng(8)
    vol = (rng.random((25, 40, 70, 50)) < 0.002).astype(np.float32)    # 25 channels, sparse
    vol[0] = rng.random((40, 70, 50), dtype=np.float32)
    ijk = ops.cube_origins((50, 70, 40), 32)
    out = torch.empty((len(ijk), 25, 64, 64, 64), dtype=torch.float32, device=cuda)
    nzf = torch.empty(len(ijk), dtype=torch.int32, device=cuda)
    d = dev(vol, cuda)
    ops.extract_cubes(d[:1], dev(ijk, cuda), 32, 16, out=out[:, :1])
    ops.extract_cubes(d[1:], dev(ijk, cuda), 32, 16, out=out[:, 1:], nonzero=nzf)
    got = out.cpu().numpy()
    for c in (0, 1, 7, 24):
        want, _, _, _ = orc.extract_cubes(vol[c], grid_size=32, padding=16)
        assert np.array_equal(got[:, c], want)
    assert np.array_equal(nzf.cpu().numpy() != 0, (np.abs(got[:, 1:]).reshape(len(ijk), -1).sum(1) > 0))


@pytest.mark.parametrize('gs,pad', [(48, 8), (32, 16)])
@pytest.mark.parametrize('shape', [(44, 52, 60), (100, 36, 64), (33, 70, 128)])
def test_extract_tma_path_matches_oracle_and_fallback(cuda, shape, gs, pad, monkeypatch):
    """nx % 4 == 0 and W == 64 take the TMA box-load kernel; it must equal both the oracle
    and the shared-memory transpose kernel (forced with MICA_NO_TMA)."""
    from mica_b200._lib import lib
    rng = np.random.default_rng(shape[0])
    vol = rng.normal(size=(3,) + shape).astype(np.float32)
    vol[2] = (rng.random(shape) < 0.001)
    ijk = ops.cube_origins(ops.cube_space_shape(shape), gs)
    d_vol, d_ijk = dev(vol, cuda), dev(ijk, cuda)
    nzf = torch.empty(len(ijk), dtype=torch.int32, device=cuda)
    cmax = torch.empty(len(ijk), dtype=torch.float32, device=cuda)
    got = ops.extract_cubes(d_vol, d_ijk, gs, pad, nonzero=nzf, cube_max=cmax).cpu().numpy()
    assert lib.mica_last_extract_path() == 2
    monkeypatch.setenv('MICA_NO_TMA', '1')
    ref = ops.extract_cubes(d_vol, d_ijk, gs, pad).cpu().numpy()
    assert lib.mica_last_extract_path() == 1
    assert np.array_equal(got, ref)
    for c in range(3):
        want, _, _, _ = orc.extract_cubes(vol[c], grid_size=gs, padding=pad)
        assert np.array_equal(got[:, c], want)
    assert np.array_equal(nzf.cpu().numpy() != 0, np.abs(got).reshape(len(ijk), -1).sum(1) > 0)
    assert np.array_equal(cmax.cpu().numpy(), got[:, 0].reshape(len(ijk), -1).max(1))


# ------------------------------------------------------ R7/R8 post-process + stitch
def _stitch_case(cube_shape, grid_size, padding, cuda, seed=3):
    ijk = ops.cube_origins(cube_shape, grid_size)
    n, W = len(ijk), grid_size + 2 * padding
    bb, ca, aa = synthetic.synthetic_logits(n, W, seed=seed)
    meta = np.concatenate([ijk, np.minimum(grid_size, np.array(cube_shape)[None] - ijk)], axis=1).astype(np.int64)
    want = orc.postprocess_and_stitch(bb, ca, aa, meta, cube_shape, padding)
    vols = ops.StitchedVolumes(cube_shape, cuda)
    ops.postproc_stitch(dev(bb, cuda), dev(ca, cuda), dev(aa, cuda), dev(ijk, cuda), vols, grid_size, padding)
    return want, {k: v.cpu().numpy() for k, v in vols.as_dict().items()}, (bb, ca, aa, meta)


def _check_stitched(want, got, logits):
    for k in ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_probability'):
        assert got[k].shape == want[k].shape and got[k].dtype == np.float32
        assert np.abs(got[k] - want[k]).max() <= TOL, k
    # argmax: identical wherever the oracle's top-2 probabilities are separated by more than float noise
    p = np.sort(want['amino_acid_probability'], axis=0)
    gap = p[-1] - p[-2]
    diff = got['amino_acid_prediction'] != want['amino_acid_prediction']
    assert not (diff & (gap > 4e-6)).any()
    assert diff.mean() < 1e-4


@pytest.mark.parametrize('cube_shape,gs,pad', [((52, 20, 12), 48, 8), ((70, 33, 50), 32, 16), ((21, 13, 9), 8, 2),
                                               ((20, 24, 90), 32, 16), ((40, 31, 49), 32, 16)])
def test_postproc_stitch_vs_oracle(cuda, cube_shape, gs, pad):
    want, got, logits = _stitch_case(cube_shape, gs, pad, cuda)
    _check_stitched(want, got, logits)


@pytest.mark.parametrize('cube_shape,gs,pad', [((70, 33, 50), 32, 16), ((52, 20, 12), 48, 8)])
def test_overlap_weighted_stitch_modes(cuda, cube_shape, gs, pad):
    """The north_star's overlap-weighted stitching (NOT the reference's arithmetic; DESIGN.md D2): with the
    core-indicator window it must reproduce the reference-mode kernel bit for bit, with the uniform and the
    triangle window it must equal the NumPy statement sum(w p) / sum(w) -- float32 atomics in arbitrary
    order against float64 accumulation, so with a tolerance."""
    want_core, got_core, (bb, ca, aa, meta) = _stitch_case(cube_shape, gs, pad, cuda)
    d = [dev(a, cuda) for a in (bb, ca, aa)]
    ijk = dev(np.ascontiguousarray(meta[:, :3], dtype=np.int32), cuda)
    half = len(meta) // 2                                   # two accumulate calls: batches add up
    for window in ('core', 'uniform', 'triangle'):
        st = ops.OverlapStitcher(cube_shape, cuda, gs, pad, window)
        st.accumulate(d[0][:half], d[1][:half], d[2][:half], ijk[:half])
        st.accumulate(d[0][half:], d[1][half:], d[2][half:], ijk[half:])
        got = {k: v.cpu().numpy() for k, v in st.finalize().as_dict().items()}
        if window == 'core':
            for k in ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_probability'):
                assert np.array_equal(got[k], got_core[k]), k       # same softmax, weight 1, one contribution
            _check_stitched(want_core, got, None)
            continue
        w1 = orc.overlap_window(window, gs, pad)
        assert np.array_equal(w1, ops.overlap_window(window, gs, pad))
        want = orc.postprocess_and_stitch_overlap(bb, ca, aa, meta, cube_shape, gs, pad, w1)
        for k in ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_probability'):
            assert np.abs(got[k] - want[k]).max() <= TOL, (window, k)
        p = np.sort(want['amino_acid_probability'], axis=0)
        clear = (p[-1] - p[-2]) > 4e-6
        assert np.array_equal(got['amino_acid_prediction'][clear], want['amino_acid_prediction'][clear]), window
        # every voxel of the map is covered by at least one window: probabilities of the 20 classes sum to 1
        assert np.abs(got['amino_acid_probability'].sum(0) - 1).max() <= 1e-5
    with pytest.raises(_lib.MicaError):
        ops.OverlapStitcher(cube_shape, cuda, gs, pad, 'hamming')


def test_pipeline_overlap_window_option(cuda):
    """MapPipeline.predict_and_stitch(overlap_window=...) routes the batches through the OverlapStitcher; 'core'
    equals the default mode."""
    src = synthetic.synthetic_map((40, 44, 36), voxel=1.0, seed=9)
    hdr = MapHeader(voxel_size=(np.float32(1.0),) * 3)
    pipe = MapPipeline(cuda, 32, 16, batch_cubes=3)
    assert pipe.resample_and_normalize(dev(src, cuda), hdr)
    with torch.no_grad():
        ref = pipe.predict_and_stitch(synthetic.pointwise_model)
        core = pipe.predict_and_stitch(synthetic.pointwise_model, overlap_window='core')
        uni = pipe.predict_and_stitch(synthetic.pointwise_model, overlap_window='uniform')
    for k in ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_probability'):
        assert torch.equal(core.as_dict()[k], ref.as_dict()[k]), k
    # a pointwise model gives every window the same value at a voxel: averaging changes nothing but rounding
    for k in ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_probability'):
        assert float((uni.as_dict()[k] - ref.as_dict()[k]).abs().max()) <= 1e-6, k


def test_postproc_stitch_golden(cuda, golden_dir):
    g = load_stitch(golden_dir)
    cube_shape = tuple(int(v) for v in g['orig_shape'])
    want, got, _ = _stitch_case(cube_shape, 48, 8, cuda, seed=int(g['logits_seed']))
    ref = {k: g[k] for k in want}
    for k in want:
        assert np.array_equal(want[k], ref[k])        # oracle == unmodified reference
    _check_stitched(ref, got, None)


def test_stitch_cubes_plain_paste_and_roundtrip(cuda):
    """extract -> stitch is the identity on the volume (size-independent property)."""
    rng = np.random.default_rng(12)
    vol = rng.random((3, 60, 50, 70), dtype=np.float32)          # (C, nz, ny, nx)
    cube_shape = (70, 50, 60)
    ijk = dev(ops.cube_origins(cube_shape, 48), cuda)
    cubes = ops.extract_cubes(dev(vol, cuda), ijk, 48, 8)
    back = ops.stitch_cubes(cubes, ijk, cube_shape, 48, 8).cpu().numpy()
    assert np.array_equal(back, vol.transpose(0, 3, 2, 1))


# ------------------------------------------------------------ host-buffer API (the e2e path of bench.py)
@pytest.mark.parametrize('batch', [3, 7, 64])
def test_host_api_overlapped_drain_equals_plain_copy(cuda, batch):
    """run_map_pipeline_host streams finished x-layers of the volumes to pinned memory while later
    batches run; the result must equal copying the finished volumes afterwards."""
    from mica_b200.pdb import channel_codes
    from mica_b200.pipeline import MapHeader, MapPipeline, run_map_pipeline_host
    src = synthetic.synthetic_map((40, 36, 52), voxel=1.2, seed=3)
    hdr = MapHeader(voxel_size=(np.float32(1.2),) * 3)
    n_out = ops.zoom_output_shape(src.shape, [np.float32(1.2)] * 3)
    st = synthetic.synthetic_structure(80, n_out[::-1], seed=3)
    bb_ch, aa_ch = channel_codes(st['atom_names'], st['res_names'])
    src_h = torch.from_numpy(src).pin_memory()
    atoms_h = tuple(torch.from_numpy(a).pin_memory() for a in (st['coords'], bb_ch, aa_ch))
    pipe = MapPipeline(cuda, 16, 8, batch_cubes=batch)
    W = 32
    gen = torch.Generator(device=cuda).manual_seed(1)
    ring = tuple(torch.randn((batch, c, W, W, W), generator=gen, device=cuda) for c in (4, 4, 21))

    def model_fn(x, af):
        return tuple(t[:x.shape[0]] for t in ring)

    plain, h2d, d2h = run_map_pipeline_host(src_h, hdr, atoms_h, model_fn, pipe, None)
    shape = tuple(plain['backbone_probability'].shape)
    out_h = {k: torch.full(v.shape, -1.0).pin_memory() for k, v in plain.items()}
    got, h2d2, d2h2 = run_map_pipeline_host(src_h, hdr, atoms_h, model_fn, pipe, out_h)
    assert h2d == h2d2 and d2h == d2h2 == 23 * 4 * int(np.prod(shape))
    for k in plain:
        assert torch.equal(got[k], plain[k]), k


def test_deferred_status_check_reports_failures_from_finish(cuda):
    """run(..., defer_check=True) does not synchronise; finish() raises what run() would have raised."""
    from mica_b200._lib import MicaError
    from mica_b200.pipeline import MapHeader, MapPipeline
    hdr = MapHeader(voxel_size=(np.float32(1.0),) * 3)
    pipe = MapPipeline(cuda, 16, 8, batch_cubes=8)
    ring = tuple(torch.zeros((8, c, 32, 32, 32), device=cuda) for c in (4, 4, 21))
    model_fn = lambda x, af: tuple(t[:x.shape[0]] for t in ring)
    good = dev(synthetic.synthetic_map((24, 24, 24), voxel=1.0, seed=1), cuda)
    v1 = pipe.run(good, hdr, None, model_fn)
    v2 = pipe.run(good, hdr, None, model_fn, defer_check=True)
    pipe.finish()
    assert torch.equal(v1.backbone_probability, v2.backbone_probability) and pipe.norm_status == 0
    flat = torch.full((24, 24, 24), 2.0, device=cuda)           # no voxel above the median
    pipe.run(flat, hdr, None, model_fn, defer_check=True)        # does not raise here
    with pytest.raises(MicaError):
        pipe.finish()
    with pytest.raises(MicaError):
        pipe.run(flat, hdr, None, model_fn)
