"""Test-time augmentation without a GPU: the orientation convention of ``ops`` (codes, inverses, composition, the
named sets, refusals), the float64 statement in oracle/tta_oracle.py against a brute-force sum, and the uint32 bound
of the fixed-point accumulator with k = 48 orientations."""
import itertools

import numpy as np
import pytest

from mica_b200 import _lib, ops
from oracle import tta_oracle as tto


def _cube(W=5, lead=()):
    return np.random.default_rng(0).random(lead + (W, W, W))


@pytest.mark.parametrize('code', range(48))
def test_codes_are_transpose_then_flip(code):
    c = _cube(lead=(2,))
    p, f = divmod(code, 8)
    want = np.transpose(c, (0,) + tuple(1 + a for a in list(itertools.permutations(range(3)))[p]))
    for a in range(3):
        if (f >> a) & 1:
            want = np.flip(want, 1 + a)
    assert np.array_equal(ops.orient_array(c, code), want)
    assert np.array_equal(tto.orient(c, code), want)
    perm, flips = ops.orientation(code)
    assert ops.orientation_code(perm, flips) == code
    # the element-wise definition: O[u] = C[v], v[perm[a]] = W-1-u_a if flips[a] else u_a
    W = c.shape[-1]
    u = (1, 3, 4)
    v = [0, 0, 0]
    for a in range(3):
        v[perm[a]] = W - 1 - u[a] if flips[a] else u[a]
    assert want[(1,) + u] == c[(1,) + tuple(v)]


def test_identity_inverse_and_composition():
    c = _cube()
    assert ops.orientation(0) == ((0, 1, 2), (False, False, False))
    assert np.array_equal(ops.orient_array(c, 0), c)
    for g in range(48):
        gi = ops.inverse_orientation(g)
        assert np.array_equal(ops.orient_array(ops.orient_array(c, g), gi), c)
        assert np.array_equal(tto.unorient(ops.orient_array(c, g), g), c)
        assert ops.compose_orientations(gi, g) == 0 and ops.compose_orientations(g, gi) == 0
        for h in (0, 5, 13, 47, g):
            assert np.array_equal(ops.orient_array(ops.orient_array(c, h), g),
                                  ops.orient_array(c, ops.compose_orientations(g, h)))
    # a group: closed, every product distinct per row
    assert all(sorted(ops.compose_orientations(g, h) for h in range(48)) == list(range(48)) for g in range(48))


def test_named_sets():
    assert ops.tta_orientations(None) is None
    assert ops.tta_orientations('flips') == tuple(range(8))
    assert ops.tta_orientations('all') == tuple(range(48))
    rot = ops.tta_orientations('rot90')
    dets = {}
    for g in range(48):
        perm, flips = ops.orientation(g)
        m = np.zeros((3, 3))
        for a in range(3):
            m[a, perm[a]] = -1 if flips[a] else 1
        dets[g] = round(np.linalg.det(m))
    assert rot == tuple(g for g in range(48) if dets[g] == 1) and len(rot) == 24
    assert all(ops.orientation_det(g) == dets[g] for g in range(48))
    # the proper rotations are closed under composition (a subgroup)
    assert all(ops.compose_orientations(g, h) in rot for g in rot for h in rot)
    assert ops.tta_orientations([3, 0, np.int64(47)]) == (3, 0, 47)


@pytest.mark.parametrize('bad', ['rot', 'ALL', '', [], [0, 0], [48], [-1], [1.0], [True], 7, [None], 'flip'])
def test_refusals(bad):
    with pytest.raises(_lib.MicaError):
        ops.tta_orientations(bad)


@pytest.mark.parametrize('bad', [48, -1, 1.5, True, '3', None])
def test_single_code_refusals(bad):
    with pytest.raises(_lib.MicaError):
        ops.orientation(bad)


def _pointwise_model(Cin, seed):
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((29, Cin))
    b = rng.standard_normal(29)

    def model(x):
        y = np.einsum('oc,cxyz->oxyz', A, x) + b[:, None, None, None]
        return y[:4], y[4:8], y[8:]
    return model


def _window_model(W, seed):
    """Position-dependent logits: a different value for every orientation of a window."""
    rng = np.random.default_rng(seed)
    A, P = rng.standard_normal((29, W, W, W)), rng.standard_normal((29, W, W, W))

    def model(x):
        y = x[0][None] * A + P
        return y[:4], y[4:8], y[8:]
    return model


@pytest.mark.parametrize('window', ['uniform', 'triangle', 'core'])
def test_oracle_against_brute_force(window):
    gs, pad, shape = 3, 1, (7, 5, 4)
    W = gs + 2 * pad
    ijk = ops.cube_origins(shape, gs)
    rng = np.random.default_rng(1)
    windows = rng.standard_normal((len(ijk), 2, W, W, W))
    model = _window_model(W, 2)
    w1 = ops.overlap_window(window, gs, pad).astype(np.float64)
    codes = (0, 5, 13, 30, 47)
    got = tto.tta_stitch(windows, ijk, shape, gs, pad, w1, codes, model)
    num, den = np.zeros((22,) + shape), np.zeros(shape)
    for n, (i, j, k) in enumerate(ijk):
        for g in codes:
            bb, ca, aa = model(ops.orient_array(windows[n], g))
            p = tto.probabilities(bb, ca, aa)
            for u in itertools.product(range(W), repeat=3):
                perm, flips = ops.orientation(g)
                v = [0, 0, 0]
                for a in range(3):
                    v[perm[a]] = W - 1 - u[a] if flips[a] else u[a]
                x = (i - pad + v[0], j - pad + v[1], k - pad + v[2])
                if all(0 <= x[m] < shape[m] for m in range(3)):
                    wt = w1[v[0]] * w1[v[1]] * w1[v[2]]
                    num[(slice(None),) + x] += wt * p[(slice(None),) + u]
                    den[x] += wt
    ok = den > 0
    want = np.where(ok[None], num / np.where(ok, den, 1)[None], 0)
    assert np.allclose(got['backbone_probability'], want[0], atol=1e-12)
    assert np.allclose(got['amino_acid_probability'], want[2:], atol=1e-12)


def test_equivariant_model_gains_nothing():
    """A pointwise model commutes with every orientation: averaging over them changes nothing."""
    gs, pad, shape = 4, 2, (9, 6, 5)
    W = gs + 2 * pad
    ijk = ops.cube_origins(shape, gs)
    windows = np.random.default_rng(4).standard_normal((len(ijk), 3, W, W, W))
    model = _pointwise_model(3, 5)
    w1 = ops.overlap_window('triangle', gs, pad)
    a = tto.tta_stitch(windows, ijk, shape, gs, pad, w1, range(48), model)
    b = tto.tta_stitch(windows, ijk, shape, gs, pad, w1, (0,), model)
    for k in a:
        assert np.allclose(a[k], b[k], atol=1e-12), k


@pytest.mark.parametrize('gs,pad', [(32, 16), (16, 8), (48, 8)])
@pytest.mark.parametrize('window', ['uniform', 'triangle', 'core'])
def test_uint32_bound_with_48_orientations(gs, pad, window):
    """Every contribution is q = rint(p w N 2^31) with p <= 1 (+ float32 rounding), and the weights times the
    normaliser of one voxel sum to 1 over its k * n_cover contributions; so a voxel's uint32 sum is at most
    (1 + 2^-20) 2^31 + k n_cover / 2, far below 2^32, at stride 32 and 16 with k = 48."""
    k = 48
    shape = (5 * gs + 3, 2 * gs + 1, 3 * gs)
    w1 = ops.overlap_window(window, gs, pad)
    nx, ny, nz = ops.overlap_norm_tables(w1, shape, gs, pad, tta_k=k)
    sx, sy, sz = tto.lattice_weight_sums(w1, shape, gs, pad)
    assert np.allclose(nx[sx > 0] * k * sx[sx > 0], 1, rtol=1e-15)
    w = w1.astype(np.float64)
    W = len(w)

    # the largest per-voxel sum of w * N over every covering window, per axis (the 3-D sum is their product)
    def axis_max(n, norm):
        best = 0.0
        for x in range(n):
            s = sum(w[x - (i - pad)] for i in range(0, n, gs) if 0 <= x - (i - pad) < W)
            best = max(best, s * norm[x])
        return best
    worst = k * axis_max(shape[0], nx) * axis_max(shape[1], ny) * axis_max(shape[2], nz)
    n_cover = (-(-W // gs)) ** 3
    bound = worst * (1 + 2.0 ** -20) * 2.0 ** 31 + k * n_cover / 2
    assert worst <= 1 + 1e-12
    assert bound < 2.0 ** 32
