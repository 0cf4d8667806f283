"""NumPy statement of the prediction maps (``save_maps=``): the four stitched volumes resampled onto the input map's
grid (``'input'``) or the 1 A working grid (``'working'``), in the target's memory order, for MRC files that overlay
the user's map.

  1. the stitched volumes are cube space ``[X, Y, Z]``: the normalised map's memory axes permuted by ``perm`` (cube
     axis a walks memory axis perm[a], ``MapHeader.transpose_order``); ``to_memory_order`` undoes that;
  2. the target grid has the memory shape (nz, ny, nx) of the input map or of the normalised map.  Per memory axis, with
     n_w working samples and n_s target samples, target index s reads the working coordinate

         c  = float64(s * (n_w - 1)) / float64(n_s - 1)       (the integer product, ONE rounding; c = 0 if n_s == 1)
         i0 = min(floor(c), max(n_w - 2, 0)),  i1 = min(i0 + 1, n_w - 1),  t = c - i0

     -- exact at both ends and when n_w == n_s (``s * ((n_w-1)/(n_s-1))`` misses the last sample by an ulp for some
     pairs: DESIGN.md D11's cause);
  3. each probability channel is interpolated trilinearly in float64, every product and sum rounded in this order
     (no fused multiply-add), and the result rounded to float32:

         fx(z,y) = v[z,y,i0x]*(1-tx) + v[z,y,i1x]*tx
         fy(z)   = fx(z,i0y)*(1-ty) + fx(z,i1y)*ty
         f       = fy(i0z)*(1-tz) + fy(i1z)*tz

  4. ``amino_acid_prediction`` on the target grid is the index of the largest of the 20 resampled float32
     probabilities (``np.argmax``: the first maximum wins, a NaN counts as the largest), stored as float32."""
from __future__ import annotations

import numpy as np

MAP_TYPES = ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_prediction', 'amino_acid_probability')


def inverse_perm(perm):
    inv = [0, 0, 0]
    for a, m in enumerate(perm):
        inv[int(m)] = a
    return tuple(inv)


def to_memory_order(vol, perm):
    """A cube-space volume ``[..., X, Y, Z]`` (leading channel axes allowed) as the working map's memory order."""
    v = np.asarray(vol)
    lead = v.ndim - 3
    return np.transpose(v, tuple(range(lead)) + tuple(lead + a for a in inverse_perm(perm)))


def axis_coords(n_s, n_w):
    """(i0 int64 [n_s], i1 int64 [n_s], t float64 [n_s]): the working samples target indices 0..n_s-1 read."""
    n_s, n_w = int(n_s), int(n_w)
    s = np.arange(n_s, dtype=np.int64)
    if n_s == 1:
        c = np.zeros(1, np.float64)
    else:
        c = (s * (n_w - 1)).astype(np.float64) / np.float64(n_s - 1)
    i0 = np.minimum(np.floor(c).astype(np.int64), max(n_w - 2, 0))
    i1 = np.minimum(i0 + 1, n_w - 1)
    return i0, i1, c - i0.astype(np.float64)


def resample_channel(v, target_shape, out_dtype=np.float32):
    """One working-grid channel (memory order [nz, ny, nx]) -> float32 on the target's memory shape (``out_dtype`` =
    float64: the value before that last rounding)."""
    v = np.asarray(v, np.float64)
    (z0, z1, tz), (y0, y1, ty), (x0, x1, tx) = (axis_coords(n, w) for n, w in zip(target_shape, v.shape))
    fx = v[:, :, x0] * (1.0 - tx) + v[:, :, x1] * tx                         # [nz_w, ny_w, nx_s]
    fy = fx[:, y0, :] * (1.0 - ty)[:, None] + fx[:, y1, :] * ty[:, None]     # [nz_w, ny_s, nx_s]
    f = fy[z0] * (1.0 - tz)[:, None, None] + fy[z1] * tz[:, None, None]      # [nz_s, ny_s, nx_s]
    return f.astype(out_dtype)


def volumes_to_grid(vols, perm, target_shape):
    """The four volumes (cube space, ``MAP_TYPES`` keys; the stitched ``amino_acid_prediction`` is not read) -> the
    four target-grid maps in memory order: float32 [nz, ny, nx], [20, nz, ny, nx] for ``amino_acid_probability``."""
    target_shape = tuple(int(v) for v in target_shape)
    out = {k: resample_channel(to_memory_order(vols[k], perm), target_shape)
           for k in ('backbone_probability', 'carbon_alpha_probability')}
    prob = to_memory_order(vols['amino_acid_probability'], perm)
    out['amino_acid_probability'] = np.stack([resample_channel(prob[c], target_shape) for c in range(prob.shape[0])])
    out['amino_acid_prediction'] = np.argmax(out['amino_acid_probability'], axis=0).astype(np.float32)
    return out
