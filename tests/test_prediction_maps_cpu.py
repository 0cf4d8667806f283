"""Prediction maps (``save_maps=``), host side: the oracle against SciPy, the coordinate table's exact ends, the
``save_maps`` / ``MICA_SAVE_MAPS`` parsing and the predictor's refusals, the C ABI's refusals without a device, and the
MRC files' headers."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
from scipy import ndimage

from mica_b200 import _lib, mrc, ops, session
from mica_b200.pipeline import MapHeader
from mica_b200.predict import MAP_TYPES, CryoEMPredictor, map_file_names, parse_save_maps, write_map_files
from oracle import prediction_maps_oracle as pmo


def _scipy(v, target_shape):
    coords = [i0 + t for i0, _, t in (pmo.axis_coords(n, w) for n, w in zip(target_shape, v.shape))]
    grid = np.meshgrid(*coords, indexing='ij')
    return ndimage.map_coordinates(np.asarray(v, np.float64), grid, order=1, mode='nearest')


@pytest.mark.parametrize('working,target', [
    ((13, 17, 11), (13, 17, 11)),            # identity
    ((12, 15, 9), (10, 13, 8)),              # down (1.2 A input)
    ((10, 13, 8), (12, 15, 9)),              # up (0.83 A input)
    ((7, 1, 9), (5, 1, 12)),                 # a 1-sample axis
    ((1, 6, 5), (4, 6, 5)),                  # one working sample, several targets
    ((6, 5, 7), (1, 9, 3)),                  # one target sample
    ((23, 11, 5), (9, 30, 14)),              # anisotropic, odd
])
def test_oracle_equals_map_coordinates(working, target):
    v = np.random.default_rng(3).random(working)
    got = pmo.resample_channel(v, target, out_dtype=np.float64)
    want = _scipy(v, target)
    assert got.shape == tuple(target)
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)
    assert np.array_equal(pmo.resample_channel(v, target), got.astype(np.float32))


def test_identity_is_the_permuted_copy():
    rng = np.random.default_rng(4)
    for perm in ((2, 1, 0), (0, 1, 2), (1, 2, 0), (2, 0, 1), (0, 2, 1), (1, 0, 2)):
        working = (7, 9, 5)
        cube = rng.random(tuple(working[p] for p in perm)).astype(np.float32)
        vols = {'backbone_probability': cube, 'carbon_alpha_probability': cube * 0.5,
                'amino_acid_prediction': cube * 0, 'amino_acid_probability': rng.random((20,) + cube.shape).astype(np.float32)}
        out = pmo.volumes_to_grid(vols, perm, working)
        inv = pmo.inverse_perm(perm)
        assert np.array_equal(out['backbone_probability'], np.transpose(cube, inv))
        assert np.array_equal(out['amino_acid_probability'], np.transpose(vols['amino_acid_probability'], (0,) + tuple(1 + a for a in inv)))
        assert np.array_equal(out['amino_acid_prediction'], np.argmax(out['amino_acid_probability'], 0).astype(np.float32))


def test_coordinate_table_ends_are_exact():
    for n_s in range(2, 401):
        s = np.arange(n_s, dtype=np.int64)
        for n_w in range(2, 401):
            i0, i1, t = pmo.axis_coords(n_s, n_w)
            assert i0[0] == 0 and t[0] == 0.0
            assert i0[-1] + t[-1] == n_w - 1 and i1[-1] == n_w - 1, (n_s, n_w)
            assert (t >= 0).all() and (t <= 1).all() and (i1 <= n_w - 1).all()
            if n_w == n_s:
                assert np.array_equal(i0[:-1], s[:-1]) and (t[:-1] == 0).all() and t[-1] == 1.0


def test_argmax_first_maximum_and_nan():
    def label(fill):
        prob = np.zeros((20, 1, 1, 1), np.float32)
        fill(prob)
        vols = {'backbone_probability': prob[0], 'carbon_alpha_probability': prob[0], 'amino_acid_prediction': prob[0],
                'amino_acid_probability': prob}
        return float(pmo.volumes_to_grid(vols, (0, 1, 2), (1, 1, 1))['amino_acid_prediction'].item())

    def tie(p):
        p[3] = p[7] = 0.5
    assert label(tie) == 3.0                                      # a tie: the first wins

    def nan(p):
        p[5], p[9] = np.nan, 1.0
    assert label(nan) == 5.0                                      # a NaN counts as the largest
    assert label(lambda p: None) == 0.0


@pytest.mark.parametrize('spec,want', [(None, None), ('', None), ('  ', None), ('input', 'input'),
                                       (' Working ', 'working'), ('INPUT', 'input')])
def test_parse_save_maps(spec, want):
    assert parse_save_maps(spec) == want


@pytest.mark.parametrize('bad', ['mrc', 'inputs', 'true', 1, True, ['input'], b'input'])
def test_parse_save_maps_refusals(bad):
    with pytest.raises(ValueError):
        parse_save_maps(bad)


@pytest.fixture
def _env(monkeypatch):
    for k in ('MICA_DEVICES', 'MICA_MIN_MAX', 'MICA_PRECISION', 'MICA_SAVE_MAPS'):
        monkeypatch.delenv(k, raising=False)
    session.clear()
    yield monkeypatch
    session.clear()


def _predictor(tmp_path, **kw):
    pr = CryoEMPredictor('unused', str(tmp_path / 'grids') + '/', str(tmp_path / 'out'), save_output=False,
                         quiet=True, model=lambda x, af: None, **kw)
    pr.logger.disabled = True
    return pr


def test_bad_values_are_refused_before_any_launch(tmp_path, _env):
    n0 = ops.launch_count()
    for kw, env in (({'save_maps': 'mrc'}, None), ({}, 'both'), ({'save_maps': 2}, 'input')):
        if env is None:
            _env.delenv('MICA_SAVE_MAPS', raising=False)
        else:
            _env.setenv('MICA_SAVE_MAPS', env)
        assert _predictor(tmp_path, **kw).run_prediction() == (False, {})
    assert ops.launch_count() == n0


def test_explicit_save_maps_wins_over_the_environment(tmp_path, _env):
    _env.setenv('MICA_SAVE_MAPS', 'bogus')
    pr = _predictor(tmp_path, save_maps='')
    pr._source = {'kind': 'files'}
    assert pr._resolve_maps_target() is None                     # '' given: no maps, the environment is not read


def test_per_cube_files_are_refused(tmp_path, _env):
    d = tmp_path / 'grids' / 'normalized_map_grids'
    os.makedirs(d)
    np.savez(d / 'normalized_map_grid_i0_j0_k0.npz', grid=np.zeros((32, 32, 32), np.float32), i=0, j=0, k=0,
             orig_shape=np.array([16, 16, 16]), grid_size=16, padding=8)
    n0 = ops.launch_count()
    for mode in ('input', 'working'):
        pr = _predictor(tmp_path, save_maps=mode)
        assert pr.run_prediction() == (False, {})
        with pytest.raises(_lib.MicaError, match='per-cube'):
            pr._resolve_maps_target()
    assert ops.launch_count() == n0
    assert not os.path.exists(tmp_path / 'out')


def _resident(tmp_path, source=None):
    vol = torch.zeros((20, 18, 16))
    hdr = MapHeader(voxel_size=(np.float32(1),) * 3)
    session.put(os.path.join(str(tmp_path / 'grids'), 'normalized_map_grids'), kind='cubes', volume=vol, header=hdr,
                perm=(2, 1, 0), offset=[0.0] * 3, cube_shape=(16, 18, 20), ijk=ops.cube_origins((16, 18, 20), 16),
                grid_size=16, padding=8, prefix='grid', pipe=None, source=source, min_max=None)
    return vol, hdr


def test_input_needs_data_preprocessor(tmp_path, _env):
    _resident(tmp_path, source=str(tmp_path / 'resampled_normalized_map.mrc'))  # a file GridCreator read itself
    n0 = ops.launch_count()
    pr = _predictor(tmp_path, save_maps='input')
    assert pr.run_prediction() == (False, {})
    with pytest.raises(_lib.MicaError, match='DataPreprocessor'):
        pr._resolve_maps_target()
    assert ops.launch_count() == n0
    # 'working' needs only the registered map; with DataPreprocessor's entry 'input' finds the input grid
    pr = _predictor(tmp_path, save_maps='working')
    pr._resolve_source()
    mode, perm, working, target, hdr = pr._resolve_maps_target()
    assert (mode, perm, working, target) == ('working', (2, 1, 0), (20, 18, 16), (20, 18, 16))
    src_hdr = MapHeader(voxel_size=(np.float32(1.2),) * 3, mapc=3, mapr=2, maps=1)
    session.put(str(tmp_path / 'resampled_normalized_map.mrc'), kind='normalized_map', source_shape=(17, 15, 13),
                source_header=src_hdr)
    pr = _predictor(tmp_path, save_maps='input')
    pr._resolve_source()
    assert pr._resolve_maps_target() == ('input', (2, 1, 0), (20, 18, 16), (17, 15, 13), src_hdr)


def _ptr(v=16):
    return C.c_void_p(v)                                         # never dereferenced: every call below is refused


def _call(**over):
    a = dict(bb=_ptr(), ca=_ptr(), pred=_ptr(), prob=_ptr(), X=5, Y=6, Z=7, org=(0, 0, 0), ext=(5, 6, 7),
             perm=(2, 1, 0), working=(7, 6, 5), target=(8, 7, 6), obb=_ptr(), oca=_ptr(), opred=_ptr(), oprob=_ptr())
    a.update(over)
    i3 = lambda v: None if v is None else _lib.int3(v)           # noqa: E731
    return _lib.lib.mica_volumes_to_grid(a['bb'], a['ca'], a['pred'], a['prob'], a['X'], a['Y'], a['Z'], i3(a['org']),
                                         i3(a['ext']), i3(a['perm']), i3(a['working']), i3(a['target']), a['obb'],
                                         a['oca'], a['opred'], a['oprob'], None)


@pytest.mark.parametrize('over,msg', [
    ({'bb': None}, 'null input'), ({'pred': None}, 'null input'), ({'prob': None}, 'null input'),
    ({'obb': None}, 'null output'), ({'oprob': None}, 'null output'),
    ({'org': None}, 'null shape'), ({'perm': None}, 'null shape'), ({'target': None}, 'null shape'),
    ({'X': 0, 'ext': (0, 6, 7)}, 'bad cube shape'), ({'target': (8, 0, 6)}, 'bad shape'),
    ({'working': (7, -1, 5)}, 'bad shape'),
    ({'perm': (2, 2, 0)}, 'not a permutation'), ({'perm': (3, 1, 0)}, 'not a permutation'),
    ({'perm': (-1, 1, 0)}, 'not a permutation'),
    ({'org': (1, 0, 0)}, 'whole cube space'), ({'ext': (5, 6, 6)}, 'whole cube space'),
    ({'perm': (0, 1, 2)}, 'permuted by'), ({'working': (7, 6, 4)}, 'permuted by'),
])
def test_abi_refuses_bad_arguments_without_a_device(over, msg):
    assert _call(**over) == -1                                    # MICA_ERR_INVALID, before any CUDA call
    assert msg in _lib.last_error()


def test_ops_refuses_partial_boxes_and_shapes():
    vols = {k: torch.zeros((20, 5, 6, 7) if k == 'amino_acid_probability' else (5, 6, 7)) for k in MAP_TYPES}
    with pytest.raises(_lib.MicaError, match='CUDA tensor'):
        ops.volumes_to_grid(vols, (2, 1, 0), (7, 6, 5), (8, 7, 6))
    with pytest.raises(_lib.MicaError, match='missing'):
        ops.volumes_to_grid({k: v for k, v in vols.items() if k != 'amino_acid_probability'}, (2, 1, 0), (7, 6, 5),
                            (8, 7, 6))


def test_map_files_round_trip(tmp_path):
    hdr = MapHeader(voxel_size=(np.float32(1.2), np.float32(0.9), np.float32(1.35)),
                    origin=(np.float32(-12.5), np.float32(3.25), np.float32(100.0)), mapc=3, mapr=2, maps=1,
                    nxstart=-4, nystart=7, nzstart=11)
    rng = np.random.default_rng(5)
    maps = {'backbone_probability': rng.random((5, 6, 7), dtype=np.float32),
            'carbon_alpha_probability': rng.random((5, 6, 7), dtype=np.float32),
            'amino_acid_prediction': rng.integers(0, 20, (5, 6, 7)).astype(np.float32),
            'amino_acid_probability': rng.random((20, 5, 6, 7), dtype=np.float32)}
    for k, v in maps.items():
        write_map_files(str(tmp_path), k, v, hdr)
    names = sorted(n for k in MAP_TYPES for n in map_file_names(k))
    assert sorted(os.listdir(tmp_path)) == names and len(names) == 23
    for k, v in maps.items():
        planes = v if k == 'amino_acid_probability' else [v]
        for name, plane in zip(map_file_names(k), planes):
            m = mrc.read_mrc(str(tmp_path / name))
            assert m.mode == (0 if k == 'amino_acid_prediction' else 2)
            assert m.data.shape == (5, 6, 7)
            assert np.array_equal(np.asarray(m.data, np.float32), plane)
            assert m.origin == hdr.origin                         # the voxel size is cella / n: within an ulp
            np.testing.assert_allclose(np.array(m.voxel_size), np.array(hdr.voxel_size), rtol=2e-7, atol=0)
            assert (m.mapc, m.mapr, m.maps, m.nxstart, m.nystart, m.nzstart) == (3, 2, 1, -4, 7, 11)
    with pytest.raises(ValueError):
        write_map_files(str(tmp_path), 'amino_acid_probability', maps['amino_acid_probability'][:3], hdr)
