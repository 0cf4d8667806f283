"""Integer maps (MRC modes 0, 1, 6; DESIGN.md D12) without a GPU: the oracle's restatements of what the
reference computes on them, pinned against the installed SciPy and NumPy, and the argument checks of the
new C-ABI entry points."""
import numpy as np
import pytest
from scipy.ndimage import zoom

from oracle import int_maps_oracle as iorc
from oracle import mica_oracle as orc

INT_TYPES = (np.int8, np.int16, np.uint16)


def _noise(dtype, shape, seed):
    info = np.iinfo(dtype)
    return np.random.default_rng(seed).integers(int(info.min), int(info.max) + 1, shape).astype(dtype)


@pytest.mark.parametrize('dtype', INT_TYPES, ids=lambda d: np.dtype(d).name)
def test_zoom_stores_integers_rounding_half_away_and_saturating(dtype):
    # order 1, exact halves: 2.5 -> 3, 7.5 -> 8, and -2.5 -> -3 for the signed types
    lo = -3 if np.dtype(dtype).kind == 'i' else 2
    a = np.array([[[lo, lo + 1, 2, 3, 7, 8]]], dtype=dtype)
    zf = (1.0, 1.0, np.float32(11 / 6))
    got = zoom(a, zf, order=1)
    f64 = zoom(a.astype(np.float64), zf, order=1)
    halves = f64[np.abs(f64 - np.round(f64)) == 0.5]
    assert halves.size >= 3
    assert np.array_equal(got, iorc.int_store(f64, dtype))
    assert np.array_equal(iorc.int_store(np.array([2.5, 7.5, -2.5, 2.4999, -0.4]), np.int16), [3, 8, -3, 2, 0])
    # order 3 on full-range noise: the spline overshoots and the store saturates
    a = _noise(dtype, (12, 13, 14), seed=3)
    zf = [np.float32(1.2)] * 3
    f64 = zoom(a.astype(np.float64), zf, order=3)
    info = np.iinfo(dtype)
    assert ((f64 < info.min - 0.5) | (f64 > info.max + 0.5)).sum() > 0
    got = zoom(a, zf, order=3)
    assert got.dtype == dtype
    assert np.array_equal(got, iorc.int_store(f64, dtype))
    assert np.array_equal(got, iorc.resample_int_restated(a, zf, 3))
    # D10: all zoom factors 1 return a copy of the integer array
    assert np.array_equal(zoom(a, [1.0, 1.0, 1.0], order=3), a)
    assert np.array_equal(iorc.resample_int_restated(a, [1.0] * 3), a)


def _arrays(rng, count):
    """Random integer arrays: n from 1 up, ties, negatives, all-equal, and npos in {0, 1, 2}."""
    for i in range(count):
        dtype = INT_TYPES[i % 3]
        info = np.iinfo(dtype)
        kind = i % 7
        n = int(rng.integers(1, 40)) if i % 2 else int(rng.integers(1, 3000))
        if kind == 0:                                      # all equal
            yield np.full(n, rng.integers(int(info.min), int(info.max) + 1), dtype=dtype)
        elif kind == 1:                                    # heavy ties in a narrow range
            yield rng.integers(max(int(info.min), -3), 4, n).astype(dtype)
        elif kind in (2, 3):                               # npos = kind - 1: one or two values above a flat floor
            x = np.full(n + kind, 5, dtype=dtype)
            x[rng.choice(n + kind, kind - 1, replace=False)] = 9 - kind
            yield x
        else:
            yield rng.integers(int(info.min), int(info.max) + 1, n).astype(dtype)


def test_histogram_median_and_percentile_equal_numpy():
    rng = np.random.default_rng(7)
    seen = {'npos0': 0, 'npos1': 0, 'npos2': 0, 'half': 0, 'n1': 0}
    count = 0
    for x in _arrays(rng, 10500):
        count += 1
        med, p, npos = iorc.int_order_stats_restated(x)
        want_med = np.median(x)
        assert want_med.dtype == np.float64 and med == want_med, (x, med, want_med)
        m = (x > want_med) * (x - want_med)
        pos = m[m > 0]
        assert npos == pos.size
        if npos:
            want_p = np.percentile(pos, 99.9)
            assert want_p.dtype == np.float64 and p == want_p, (x, p, want_p)
        else:
            assert p is None
        seen['npos0'] += npos == 0
        seen['npos1'] += npos == 1
        seen['npos2'] += npos == 2
        seen['half'] += med != np.floor(med)
        seen['n1'] += x.size == 1
    assert count >= 10 ** 4 and all(v > 0 for v in seen.values()), seen


@pytest.mark.parametrize('dtype', INT_TYPES, ids=lambda d: np.dtype(d).name)
def test_float64_normalisation_equals_the_oracle(dtype):
    x = zoom(_noise(dtype, (10, 11, 12), seed=5), [np.float32(1.1)] * 3, order=3)
    want, med, p = orc.normalize(x)
    got, gmed, gp = iorc.normalize_int_restated(x)
    assert med == gmed and p == gp and want.dtype == np.float32
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    flat = np.full((4, 4, 4), 7, dtype=dtype)
    assert orc.normalize(flat)[0] is None and iorc.normalize_int_restated(flat)[0] is None


def test_float16_is_refused_by_zoom():
    with pytest.raises(RuntimeError):
        zoom(np.ones((4, 4, 4), dtype=np.float16), [1.2] * 3, order=3)


def test_int_entry_points_reject_bad_arguments_before_touching_the_device():
    from mica_b200 import _lib
    lib = _lib.lib
    ws = bytearray(64)
    buf = (np.zeros(8, dtype=np.uint8)).ctypes.data
    for bad in (3, 5, 12, -1, 99):
        assert lib.mica_resample(buf, bad, 4, 4, 4, 0, 4, buf, bad, 5, 5, 5, 0, 5, buf, 1 << 20, 3, None) == -1
        assert b'dtype' in lib.mica_last_error()
        assert lib.mica_int_order_stats(buf, bad, 8, buf, None) == -1
        assert lib.mica_normalize_apply_int(buf, bad, buf, 8, buf, None) == -1
    # float32 <-> integer and integer <-> another integer type are refused
    for a, b in ((_lib.DTYPE_F32, _lib.DTYPE_I16), (_lib.DTYPE_I16, _lib.DTYPE_F32), (_lib.DTYPE_I8, _lib.DTYPE_I16),
                 (_lib.DTYPE_U16, _lib.DTYPE_I16)):
        assert lib.mica_resample(buf, a, 4, 4, 4, 0, 4, buf, b, 5, 5, 5, 0, 5, buf, 1 << 20, 3, None) == -1
    for code in (_lib.DTYPE_I8, _lib.DTYPE_I16, _lib.DTYPE_U16, _lib.DTYPE_F32):
        assert lib.mica_resample(None, code, 4, 4, 4, 0, 4, buf, code, 5, 5, 5, 0, 5, buf, 1 << 20, 3, None) == -1
        assert b'null' in lib.mica_last_error()
        assert lib.mica_resample(buf, code, 4, 4, 4, 0, 4, buf, code, 5, 5, 5, 0, 5, buf, 1 << 20, 2, None) == -1
    assert lib.mica_int_order_stats(None, _lib.DTYPE_I16, 8, buf, None) == -1
    assert lib.mica_int_order_stats(buf, _lib.DTYPE_I16, 8, None, None) == -1
    assert lib.mica_int_order_stats(buf, _lib.DTYPE_I16, -1, buf, None) == -1
    assert lib.mica_int_order_stats(buf, _lib.DTYPE_F32, 8, buf, None) == -1      # float32 takes the radix select
    assert lib.mica_normalize_apply_int(None, _lib.DTYPE_I8, buf, 8, buf, None) == -1
    assert lib.mica_normalize_apply_int(buf, _lib.DTYPE_I8, None, 8, buf, None) == -1
    assert lib.mica_normalize_apply_int(buf, _lib.DTYPE_I8, buf, 8, None, None) == -1
    assert lib.mica_int_stats_result_async(None, buf, None) == -1
    assert lib.mica_int_stats_result_async(buf, None, None) == -1
    assert lib.mica_int_stats_result(None, None, None, None, None, None) == -1
    assert lib.mica_int_stats_workspace_bytes() > 65536 * 8
    del ws


def test_ops_refuse_integer_misuse_without_a_gpu():
    import torch
    from mica_b200 import _lib, ops
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    with pytest.raises(_lib.MicaError):
        ops.normalize(torch.zeros(8, dtype=torch.int16))
    with pytest.raises(_lib.MicaError):
        ops.IntOrderStats('cpu')
    with pytest.raises(_lib.MicaError):
        ops.resample(torch.zeros((4, 4, 4), dtype=torch.int16), (5, 5, 5))
