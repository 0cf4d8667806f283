"""Host arithmetic of the order-free overlap-weighted stitch: the 1-D lattice coverage tables, the uint32 bound of
the fixed-point sums, and the owner lookup of the split accumulate (no GPU needed)."""
import numpy as np
import pytest

from mica_b200 import _lib, ops
from mica_b200.slab import SlabPlan, _split_even

GEOMETRIES = [(48, 8), (32, 16), (8, 2), (16, 0)]


def _windows(gs, pad, rng):
    W = gs + 2 * pad
    custom = rng.random(W).astype(np.float32)
    custom[rng.integers(0, W, 3)] = 0.0                       # zeros inside the window are allowed
    return [ops.overlap_window(k, gs, pad) for k in ('uniform', 'triangle', 'core')] + [custom]


def _brute_weight_sum(w1, cube_shape, gs, pad):
    """sum over every cube of the 3-D lattice of its window weight at each voxel, float64."""
    X, Y, Z = cube_shape
    W = len(w1)
    w = w1.astype(np.float64)
    w3 = w[:, None, None] * w[None, :, None] * w[None, None, :]
    tot = np.zeros(cube_shape)
    for i, j, k in ops.cube_origins(cube_shape, gs):
        lo = (i - pad, j - pad, k - pad)
        sv, sc = [], []
        for o, n in zip(lo, cube_shape):
            v0, v1 = max(0, o), min(n, o + W)
            sv.append(slice(v0, v1))
            sc.append(slice(v0 - o, v1 - o))
        tot[tuple(sv)] += w3[tuple(sc)]
    return tot


@pytest.mark.parametrize('gs,pad', GEOMETRIES)
@pytest.mark.parametrize('cube_shape', [(21, 13, 9), (50, 33, 17), (64, 20, 49)])
def test_coverage_tables_match_the_lattice(gs, pad, cube_shape):
    rng = np.random.default_rng(hash((gs, pad, cube_shape)) % 2**32)
    for w1 in _windows(gs, pad, rng):
        nx, ny, nz = ops.overlap_norm_tables(w1, cube_shape, gs, pad)
        want = _brute_weight_sum(w1, cube_shape, gs, pad)
        got = np.zeros(cube_shape)
        ok = want > 0
        prod = nx[:, None, None] * ny[None, :, None] * nz[None, None, :]
        got[ok] = 1.0 / prod[ok]
        assert np.array_equal(prod == 0, ~ok)                 # 0 exactly where no weight reaches
        assert np.allclose(got, want, rtol=1e-12, atol=0)


def _fixed(p, w1, nx, ny, nz, a, b, c, x, y, z):
    """The kernel's rounding recipe (overlap_scale / overlap_fixed in stitch.cu), in NumPy float64."""
    w = (np.float64(w1[a]) * np.float64(w1[b])) * np.float64(w1[c])
    n = (nx[x] * ny[y]) * nz[z]
    return np.rint(np.float64(p) * ((w * n) * 2.0 ** 31))


@pytest.mark.parametrize('gs,pad', GEOMETRIES)
def test_fixed_point_sums_stay_inside_uint32(gs, pad):
    """Even with p = 1 in every channel of every window the sum at a voxel is at most 2^31 + n_cover / 2."""
    cube_shape = (gs * 2 + 5, gs + 3, 2 * gs + 1)
    rng = np.random.default_rng(gs)
    W = gs + 2 * pad
    for w1 in _windows(gs, pad, rng):
        nx, ny, nz = ops.overlap_norm_tables(w1, cube_shape, gs, pad)
        X, Y, Z = cube_shape
        tot = np.zeros(cube_shape)
        cover = np.zeros(cube_shape, np.int64)
        u = np.arange(W)
        for i, j, k in ops.cube_origins(cube_shape, gs):
            gx, gy, gz = i - pad + u, j - pad + u, k - pad + u
            mx, my, mz = (gx >= 0) & (gx < X), (gy >= 0) & (gy < Y), (gz >= 0) & (gz < Z)
            A, B, Cc = np.meshgrid(u[mx], u[my], u[mz], indexing='ij')
            x, y, z = A + i - pad, B + j - pad, Cc + k - pad
            q = _fixed(np.float32(1.0), w1, nx, ny, nz, A, B, Cc, x, y, z)
            np.add.at(tot, (x, y, z), q)
            np.add.at(cover, (x, y, z), 1)
        assert tot.max() <= 2.0 ** 31 + cover.max() / 2
        assert tot.max() < 2.0 ** 32
        reached = tot > 0
        # the sum of p = 1 is one, within the rounding of n_cover contributions
        assert np.abs(tot[reached] * 2.0 ** -31 - 1).max() <= cover.max() * 2.0 ** -32 + 1e-12


@pytest.mark.parametrize('world', [2, 3, 8])
@pytest.mark.parametrize('gs,pad', [(48, 8), (32, 16)])
def test_every_contribution_goes_to_the_rank_whose_box_holds_it(world, gs, pad):
    """z-slabs (cube axis 2, SlabPlan's owned planes) and balanced cubes (cube axis 0, even x split): the owner the
    kernel's lookup picks for each voxel a window reaches is the rank whose box holds that voxel, also with empty
    ranks at the end of the line."""
    plan = SlabPlan((150, 40, 36), (np.float32(1.0),) * 3, gs, pad, world)
    k_bounds = [r.out_lo for r in plan.ranks] + [plan.ranks[-1].out_hi]
    nz = plan.out_shape[0]
    assert k_bounds[0] == 0 and k_bounds[-1] == nz
    X = 77
    x_bounds = _split_even(X, world)
    for bounds, n, boxes in ((k_bounds, nz, [(r.out_lo, r.out_hi) for r in plan.ranks]),
                             (x_bounds, X, [(x_bounds[r], x_bounds[r + 1]) for r in range(world)])):
        for o in range(0, n, gs):
            for g in range(max(0, o - pad), min(n, o + gs + pad)):
                r = ops.overlap_owner(g, bounds)
                assert boxes[r][0] <= g < boxes[r][1], (g, r, boxes)


def test_bad_windows_are_refused_on_the_host():
    W = 32 + 2 * 16
    for bad in (np.full(W, -0.5), np.r_[np.ones(W - 1), np.nan], np.ones(W - 1), np.zeros(W),
                np.r_[np.ones(W - 1), np.inf]):
        with pytest.raises(_lib.MicaError):
            ops.overlap_window(bad, 32, 16)
    with pytest.raises(_lib.MicaError):
        ops.overlap_window('hamming', 32, 16)
    assert ops.is_core_window(ops.overlap_window('core', 32, 16), 32, 16)
    assert not ops.is_core_window(ops.overlap_window('uniform', 32, 16), 32, 16)


def test_accumulate_entry_points_reject_bad_arguments_before_touching_the_device():
    import ctypes as C
    lib = _lib.lib
    W = 8 + 2 * 2
    good = (C.c_float * W)(*([1.0] * W))
    norm = C.c_void_p(8)                                      # never dereferenced: the checks come first
    blk = C.c_void_p(8)
    for w in ([-1.0] + [1.0] * (W - 1), [float('nan')] + [1.0] * (W - 1), [0.0] * W, [float('inf')] * W):
        arr = (C.c_float * W)(*w)
        assert lib.mica_overlap_accumulate_fixed(None, None, None, None, 0, 4, 4, 4, 8, 2, arr, norm, blk, None) == -1
    assert lib.mica_overlap_accumulate_fixed(None, None, None, None, 0, 4, 4, 4, 8, 2, good, None, blk, None) == -1
    assert lib.mica_overlap_accumulate_fixed(None, None, None, None, 0, 4, 4, 4, 8, 2, good, norm, blk, None) == 0
    assert lib.mica_overlap_accumulate_fixed(None, None, None, None, 0, 4, 4, 4, 100, 20, good, norm, blk, None) == -1
    bounds = (C.c_int * 3)(0, 2, 4)
    table = C.c_void_p(8)
    assert lib.mica_overlap_accumulate_fixed_peer(None, None, None, None, 0, 4, 4, 4, 8, 2, good, norm, table, 1,
                                                  bounds, 2, None) == -1          # axis 1 is not an owner axis
    assert lib.mica_overlap_accumulate_fixed_peer(None, None, None, None, 0, 4, 4, 4, 8, 2, good, norm, table, 2,
                                                  bounds, 2, None) == 0
    bad = (C.c_int * 3)(0, 3, 2)
    assert lib.mica_overlap_accumulate_fixed_peer(None, None, None, None, 0, 4, 4, 4, 8, 2, good, norm, table, 0,
                                                  bad, 2, None) == -1
    assert lib.mica_overlap_finalize_fixed(None, 10, None) == -1
    assert lib.mica_peer_atomics_supported(-1, 0) == -1
