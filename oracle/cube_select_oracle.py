"""NumPy statement of the inference keep rule (``min_max=``): the rule the reference applies to its training grids
(scripts_for_training_data/create_grids_for_normalized_map.py:78 writes no window whose maximum is below 0.01), applied
to the windows the reference cuts at inference (utils/create_grids.py:119-176).

  1. every window is the reference's: ``np.pad`` with zeros, then the W^3 slice at the cube origin (``extract_cubes``
     of mica_oracle); its maximum is ``np.max`` (NaN if the window holds one);
  2. a cube is kept iff ``not (max < min_max)`` in float32 -- the reference's test, negated: a tie and a NaN window are
     kept;
  3. paste: the reference's stitcher (utils/predict.py:458-501) over the kept cubes' rows only -- a skipped cube has no
     grid file, so its core stays 0 in all four volumes;
  4. overlap-weighted stitching and test-time augmentation (NOT the reference's arithmetic): a skipped window adds
     nothing, the denominator is still the weight sum of the full cube lattice."""
from __future__ import annotations

import numpy as np

from . import mica_oracle as orc
from . import tta_oracle as tto


def window_maxima(volume, mapc=1, mapr=2, maps=3, grid_size=48, padding=8):
    """(maxima float32 [n], meta int64 [n, 6], orig_shape): ``np.max`` of every window the reference cuts, in its
    loop order."""
    cubes, meta, orig_shape, _ = orc.extract_cubes(volume, mapc, mapr, maps, (0, 0, 0), grid_size, padding)
    maxima = np.array([np.max(c) for c in cubes], dtype=np.float32)
    return maxima, np.asarray(meta, np.int64), tuple(orig_shape)


def kept(maxima, min_max):
    """Boolean [n]: the cubes the rule keeps."""
    with np.errstate(invalid='ignore'):
        return ~(np.asarray(maxima, np.float32) < np.float32(min_max))


def paste(bb_logits, ca_logits, aa_logits, meta, orig_shape, keep, padding=8):
    """The four volumes of the reference's predictor when only the kept cubes' grid files exist.  Logits are those of
    every cube of ``meta`` ([n, 4 | 4 | 21, W, W, W]); only the kept rows are stitched."""
    k = np.asarray(keep, bool)
    return orc.postprocess_and_stitch(np.asarray(bb_logits)[k], np.asarray(ca_logits)[k], np.asarray(aa_logits)[k],
                                      np.asarray(meta)[k], orig_shape, padding)


def weighted(windows, ijk, cube_shape, grid_size, padding, w1, codes, model, keep):
    """Overlap-weighted / TTA volumes (``tta_oracle.tta_stitch``) with the skipped windows' probabilities set to 0:
    only the kept windows are added, the denominator is the full lattice's (``codes=(0,)``: the plain weighted
    stitch)."""
    k = np.asarray(keep, bool)
    return tto.tta_stitch(np.asarray(windows)[k], np.asarray(ijk)[k], cube_shape, grid_size, padding, w1, codes, model)
