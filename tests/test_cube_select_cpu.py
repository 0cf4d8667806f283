"""Host side of the inference keep rule (``min_max=``): the threshold checks, the selection on a host tensor, how the
rule combines with ``order=``, the registered-subset mapping of the drop-in and the oracle's statement.  No GPU."""
import types

import numpy as np
import pytest
import torch

from mica_b200 import _lib, ops
from mica_b200.create_grids import GridCreator, env_min_max
from mica_b200.pipeline import MapPipeline
from mica_b200.predict import CryoEMPredictor
from oracle import cube_select_oracle as cso
from oracle import mica_oracle as orc


@pytest.mark.parametrize('bad', [float('nan'), float('inf'), -float('inf'), '0.01', True, np.bool_(False), [0.01]])
def test_check_min_max_refuses(bad):
    with pytest.raises(_lib.MicaError):
        ops.check_min_max(bad)


def test_check_min_max_accepts_finite_numbers():
    assert ops.check_min_max(None) is None
    assert ops.check_min_max(0) == 0.0 and ops.check_min_max(np.float32(0.01)) == np.float32(0.01)
    assert ops.check_min_max(-3) == -3.0


def test_select_cubes_keeps_ties_and_nan():
    t = np.float32(0.01)
    m = np.array([0, t, np.nextafter(t, np.float32(0)), np.nan, 0.5, -1, np.nextafter(t, np.float32(1))], np.float32)
    got = ops.select_cubes(torch.from_numpy(m), 0.01)
    assert got.dtype == np.int64 and list(got) == [1, 3, 4, 6]
    assert np.array_equal(np.flatnonzero(cso.kept(m, 0.01)), got)
    assert list(ops.select_cubes(torch.from_numpy(m), 1e39)) == [3]       # beyond float32: only the NaN window
    with pytest.raises(_lib.MicaError):
        ops.select_cubes(torch.from_numpy(m), None)
    with pytest.raises(_lib.MicaError):
        ops.select_cubes(torch.from_numpy(m.astype(np.float64)), 0.01)


def _stub(maxima, n):
    s = types.SimpleNamespace(ijk=None, ijk_host=np.arange(3 * n, dtype=np.int32).reshape(n, 3))
    s._window_max = lambda ijk: torch.from_numpy(np.asarray(maxima, np.float32))
    return s


def test_keep_rule_follows_the_order():
    mx = [0.5, 0.0, 0.2, 0.0, 0.3]
    s = _stub(mx, 5)
    order, skipped = MapPipeline._keep_rule(s, 0.01, None)
    assert list(order) == [0, 2, 4] and np.array_equal(skipped, s.ijk_host[[1, 3]])
    order, _ = MapPipeline._keep_rule(s, 0.01, [4, 3, 1, 0, 2])
    assert list(order) == [4, 0, 2]
    order, skipped = MapPipeline._keep_rule(s, 1.0, None)
    assert len(order) == 0 and len(skipped) == 5


def test_registered_subset_maps_onto_the_lattice():
    cube_shape, gs = (40, 20, 33), 16
    full = ops.cube_origins(cube_shape, gs)
    pipe = types.SimpleNamespace(grid_size=gs, cube_shape=cube_shape, cube_index=lambda: full)
    pr = CryoEMPredictor('unused', '/nonexistent/', '/tmp/unused', save_output=False, quiet=True)
    pr._source = {'ijk': full}
    assert pr._lattice_subset(pipe) is None
    pick = np.array([1, 4, 7, len(full) - 1])
    pr._source = {'ijk': full[pick]}
    assert np.array_equal(pr._lattice_subset(pipe), pick)
    pr._source = {'ijk': full[pick] + 1}
    with pytest.raises(_lib.MicaError):
        pr._lattice_subset(pipe)


def test_env_knob(monkeypatch):
    monkeypatch.delenv('MICA_MIN_MAX', raising=False)
    assert env_min_max() is None
    monkeypatch.setenv('MICA_MIN_MAX', '  ')
    assert env_min_max() is None
    monkeypatch.setenv('MICA_MIN_MAX', '0.01')
    assert env_min_max() == 0.01
    for bad in ('nan', 'inf', 'x'):
        monkeypatch.setenv('MICA_MIN_MAX', bad)
        with pytest.raises(_lib.MicaError):
            env_min_max()


def test_grid_creator_refuses_bad_values_without_raising(tmp_path, monkeypatch):
    monkeypatch.delenv('MICA_MIN_MAX', raising=False)
    path = tmp_path / 'map.mrc'
    path.write_bytes(b'')                                  # exists: the refusal comes before it is read
    n0 = ops.launch_count()
    for bad in (float('nan'), 'x', True):
        r = GridCreator(quiet=True, min_max=bad).create_normalized_map_grids(str(path), str(tmp_path / 'g'))
        assert r['success'] is False and 'min_max' in r['error']
    monkeypatch.setenv('MICA_MIN_MAX', 'inf')
    r = GridCreator(quiet=True).create_normalized_map_grids(str(path), str(tmp_path / 'g'))
    assert r['success'] is False and 'min_max' in r['error']
    assert ops.launch_count() == n0


def test_oracle_statement():
    rng = np.random.default_rng(0)
    vol = (rng.random((20, 18, 22)) * (rng.random((20, 18, 22)) > 0.97)).astype(np.float32)
    vol[:, :, 12:] = 0                                     # a solvent half: windows there hold only zeros
    gs, pad = 8, 2
    mx, meta, shape = cso.window_maxima(vol, grid_size=gs, padding=pad)
    cubes, _, _, _ = orc.extract_cubes(vol, grid_size=gs, padding=pad)
    assert np.array_equal(mx, [c.max() for c in cubes])
    keep = cso.kept(mx, 0.01)
    assert 0 < keep.sum() < len(keep)
    W = gs + 2 * pad
    n = len(meta)
    bb, ca, aa = (rng.standard_normal((n, c, W, W, W)).astype(np.float32) for c in (4, 4, 21))
    got = cso.paste(bb, ca, aa, meta, shape, keep, pad)
    full = orc.postprocess_and_stitch(bb, ca, aa, meta, shape, pad)
    core = np.zeros(shape, bool)
    for i, j, k, di, dj, dk in meta[keep]:
        core[i:i + di, j:j + dj, k:k + dk] = True
    for k_ in full:
        assert np.allclose(got[k_][..., core], full[k_][..., core], rtol=0, atol=1e-6)     # batch-size rounding
        assert not got[k_][..., ~core].any()
    # the weighted statement: the kept windows only, the full lattice's denominator
    A = rng.standard_normal(29)

    def model(x):
        y = A[:, None, None, None] * x
        return y[:4], y[4:8], y[8:]
    windows = cubes[:, None].astype(np.float64)
    w1 = np.ones(W, np.float32)
    out = cso.weighted(windows, meta[:, :3], shape, gs, pad, w1, (0,), model, keep)
    none = cso.weighted(windows, meta[:, :3], shape, gs, pad, w1, (0,), model, np.zeros(n, bool))
    assert not none['backbone_probability'].any() and out['backbone_probability'].any()
