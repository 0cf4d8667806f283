"""Float64 NumPy statement of test-time augmentation (TTA) over the cube's orientations -- NOT the reference's
arithmetic (it runs every window once, as it is).

For every window (the model input cut at a cube origin) and every orientation code g of the set:
  1. orient the window: ``np.transpose`` by the axis permutation of g, then ``np.flip`` along its flipped axes;
  2. run the model on it;
  3. turn the logits into probabilities (the reference's softmaxes, utils/predict.py:342-349) and inverse-orient
     them back onto the window;
  4. add them, times the separable window weight w1[a] w1[b] w1[c], at the window's voxels of the volume;
then 5. divide by k times the weight sum of the full cube lattice (the k orientations each cover a voxel as often as
the plain stitch does).  amino_acid_prediction is the arg-max of the averaged 20 probabilities.

Orientation code = 8 p + f: p indexes the permutation of the window axes (0, 1, 2) in lexicographic order, bit a of
f flips output axis a (the convention of ``mica_b200.ops.orientation``, restated here from its definition)."""
import itertools

import numpy as np

PERMS = tuple(itertools.permutations(range(3)))


def orient(c, code):
    """The window(s) ``c`` (last three axes) in orientation ``code``."""
    perm, f = PERMS[code >> 3], code & 7
    lead = c.ndim - 3
    o = np.transpose(c, tuple(range(lead)) + tuple(lead + p for p in perm))
    for a in range(3):
        if (f >> a) & 1:
            o = np.flip(o, lead + a)
    return o


def unorient(o, code):
    """Inverse of ``orient``: undo the flips, then the transpose."""
    perm, f = PERMS[code >> 3], code & 7
    lead = o.ndim - 3
    for a in range(3):
        if (f >> a) & 1:
            o = np.flip(o, lead + a)
    return np.transpose(o, tuple(range(lead)) + tuple(lead + int(np.argsort(perm)[m]) for m in range(3)))


def _softmax(x, axis=0):
    e = np.exp(x - x.max(axis=axis, keepdims=True))
    return e / e.sum(axis=axis, keepdims=True)


def probabilities(bb, ca, aa):
    """[22, W, W, W] float64: backbone, carbon_alpha, amino_acid_probability x 20 of one window's logits
    ([4 | 4 | 21, W, W, W])."""
    bb, ca, aa = (np.asarray(t, np.float64) for t in (bb, ca, aa))
    out = [_softmax(bb[[0, 2, 3]])[2], _softmax(ca[[0, 2, 3]])[2]]
    return np.concatenate([np.stack(out), _softmax(aa[1:])])


def lattice_weight_sums(w1, cube_shape, grid_size, padding):
    """The 1-D weight sums of the full cube lattice along each axis (float64)."""
    w = np.asarray(w1, np.float32).astype(np.float64)
    W = len(w)
    out = []
    for n in (int(v) for v in cube_shape):
        s = np.zeros(n)
        for i in range(0, n, grid_size):
            lo = i - padding
            x0, x1 = max(0, lo), min(n, lo + W)
            s[x0:x1] += w[x0 - lo:x1 - lo]
        out.append(s)
    return out


def tta_stitch(windows, ijk, cube_shape, grid_size, padding, w1, codes, model):
    """The four volumes of a TTA run.  ``windows``: [n, C, W, W, W] model inputs at the cube origins ``ijk``
    ([n, 3], cube space); ``model(x [C, W, W, W]) -> (bb [4, W^3], ca [4, W^3], aa [21, W^3])`` logits;
    ``codes``: the orientations; ``w1``: the W window weights."""
    X, Y, Z = (int(v) for v in cube_shape)
    W = grid_size + 2 * padding
    w = np.asarray(w1, np.float32).astype(np.float64)
    w3 = w[:, None, None] * w[None, :, None] * w[None, None, :]
    num = np.zeros((22, X, Y, Z))
    for n, (i, j, k) in enumerate(np.asarray(ijk, np.int64)):
        sv, sc = [], []
        for o, dim in zip((i - padding, j - padding, k - padding), (X, Y, Z)):
            v0, v1 = max(0, o), min(dim, o + W)
            sv.append(slice(v0, v1))
            sc.append(slice(v0 - o, v1 - o))
        sv, sc = tuple(sv), tuple(sc)
        for g in codes:
            p = unorient(probabilities(*model(np.ascontiguousarray(orient(windows[n], g)))), g)
            num[(slice(None),) + sv] += (w3 * p)[(slice(None),) + sc]
    sx, sy, sz = lattice_weight_sums(w1, cube_shape, grid_size, padding)
    den = len(codes) * sx[:, None, None] * sy[None, :, None] * sz[None, None, :]
    ok = den > 0
    out = np.where(ok[None], num / np.where(ok, den, 1.0)[None], 0.0)
    pred = np.where(ok, out[2:].argmax(axis=0), 0)
    return {'backbone_probability': out[0], 'carbon_alpha_probability': out[1],
            'amino_acid_prediction': pred.astype(np.float64), 'amino_acid_probability': out[2:]}
