"""CPU restatements of what the reference computes on an integer map (MRC modes 0, 1, 6; DESIGN.md D12).

TEST INFRASTRUCTURE ONLY, like ``mica_oracle``.  The reference calls ``scipy.ndimage.zoom`` and its
normalisation on the integer array itself; ``mica_oracle.resample`` / ``mica_oracle.normalize`` call the
same installed routines, and this module spells out what they do on such arrays (probed on SciPy 1.18.1 /
NumPy 2.3.5; tests/test_int_maps_cpu.py pins every statement against the installed libraries):

1. zoom(int_array, zf, order) runs the float64 prefilter and interpolation of a float64 copy and stores into
   the input's type: ``t > 0 ? t + 0.5 : t - 0.5`` truncated toward zero, saturated at the type's range
   (``int_store``).  All zoom factors 1 return a copy of the integer array (D10).
2. np.median is float64 (the middle element or the float64 mean of the two middle ones); the positives
   (x > med) * (x - med) are float64 multiples of 0.5; np.percentile(pos, 99.9) interpolates in float64 with
   vi = (npos - 1) * (99.9 / 100) (``int_order_stats_restated``, from a histogram).
3. The normalisation is the float64 expression of ``mica_oracle.normalize`` cast to float32.
"""
from __future__ import annotations

import numpy as np

from . import mica_oracle

INT_TYPES = (np.int8, np.int16, np.uint16)


def int_store(values, dtype):
    """SciPy's store of float64 interpolated values into an integer output array."""
    info = np.iinfo(dtype)
    t = np.asarray(values, dtype=np.float64)
    t = np.where(t > 0, t + 0.5, t - 0.5)
    return np.trunc(np.clip(t, info.min, info.max)).astype(dtype)


def resample_int_restated(data, zf, order=3):
    """zoom(data, zf, order) for an integer ``data``: the float64 algorithm, then ``int_store``."""
    data = np.asarray(data)
    if all(float(z) == 1.0 for z in zf):            # D10
        return data.copy()
    return int_store(mica_oracle.resample_restated(data, zf, order), data.dtype)


def int_order_stats_restated(x):
    """(median, percentile or None, n_pos) as float64 / int, the way np.median and np.percentile(pos, 99.9)
    compute them on an integer array, found from an exact histogram of the values."""
    x = np.asarray(x).ravel()
    info = np.iinfo(x.dtype)
    hist = np.bincount((x.astype(np.int64) - info.min), minlength=int(info.max) - int(info.min) + 1)
    cum = np.cumsum(hist)
    n = int(cum[-1])

    def value_at(rank):                             # 0-based order statistic, and count(x <= it)
        k = int(np.searchsorted(cum, rank, side='right'))
        return float(k + int(info.min)), int(cum[k])

    a, cum_a = value_at((n - 1) // 2)
    b, cum_b = value_at(n // 2)
    med = b if n % 2 else (a + b) / 2.0
    n_le = cum_b if med >= b else cum_a
    npos = n - n_le
    if npos == 0:
        return med, None, 0
    q = 99.9 / 100
    vi = (npos - 1) * q
    prev = np.floor(vi)
    g = vi - prev
    if vi >= npos - 1:
        lo = hi = npos - 1
    else:
        lo, hi = int(prev), min(int(prev) + 1, npos - 1)
    pa = value_at(n_le + lo)[0] - med
    pb = value_at(n_le + hi)[0] - med
    d = pb - pa
    r = pb - d * (1.0 - g) if g >= 0.5 else pa + d * g
    return med, r, npos


def normalize_int_restated(x):
    """(normalised float32 volume or None, median, percentile) of an integer volume: the float64 expression."""
    med, p, npos = int_order_stats_restated(x)
    if npos == 0:
        return None, med, None
    if p == 0:
        return None, med, p
    m = np.asarray(x, dtype=np.float64) - med
    y = np.where(m > 0, np.minimum(m, p) / p, 0.0)
    return y.astype(np.float32), med, p
