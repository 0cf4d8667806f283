"""Readers of golden files whose arrays are stored in a packed form (oracle/make_golden.py)."""
import os

import numpy as np


def from_byte_planes(planes):
    """Inverse of make_golden.byte_planes: (4,) + shape uint8 -> float32 of that shape, bit for bit."""
    return np.ascontiguousarray(np.moveaxis(planes, 0, -1)).view(np.float32)[..., 0]


def load_stitch(golden_dir):
    """stitch.npz with its float volumes unpacked (stored as byte planes, which deflate well below 1 MB)."""
    g = np.load(os.path.join(golden_dir, 'stitch.npz'))
    out = {k: g[k] for k in g.files if not k.endswith('_planes')}
    out.update({k[:-len('_planes')]: from_byte_planes(g[k]) for k in g.files if k.endswith('_planes')})
    out['amino_acid_prediction'] = out['amino_acid_prediction'].astype(np.float32)
    return out
