"""Prediction maps on the device (``ops.volumes_to_grid``, ``CryoEMPredictor(save_maps=)``): the kernel bit for bit
against oracle/prediction_maps_oracle.py for every axis permutation and ratio, and the drop-in's MRC files on the input
and working grids against the oracle applied to the volumes the predictor returned."""
import os

import numpy as np
import pytest
import torch

from mica_b200 import mrc, ops, session, synthetic
from mica_b200.create_grids import GridCreator
from mica_b200.predict import MAP_TYPES, CryoEMPredictor, map_file_names
from mica_b200.preprocessing import DataPreprocessor
from oracle import prediction_maps_oracle as pmo

from test_gpu_cube_select import T, _masked_map
from test_gpu_devices import _assert_same
from test_gpu_overlap_split import _int16_map
from test_gpu_tta import PointwiseModel

pytestmark = pytest.mark.gpu

PERMS = ((2, 1, 0), (0, 1, 2), (0, 2, 1), (1, 0, 2), (1, 2, 0), (2, 0, 1))


def _volumes(cube_shape, cuda, seed):
    """Stitched-like volumes: probabilities in [0, 1) with exact ties in some labels."""
    g = torch.Generator(device=cuda).manual_seed(seed)
    prob = torch.rand((20,) + tuple(cube_shape), generator=g, device=cuda)
    prob[3] = prob[5]                                             # ties: the first maximum must win
    return {'backbone_probability': torch.rand(cube_shape, generator=g, device=cuda),
            'carbon_alpha_probability': torch.rand(cube_shape, generator=g, device=cuda),
            'amino_acid_prediction': torch.full(cube_shape, 7.0, device=cuda),   # not read
            'amino_acid_probability': prob}


def _assert_oracle(got, vols, perm, target):
    want = pmo.volumes_to_grid({k: v.cpu().numpy() for k, v in vols.items()}, perm, target)
    for k in MAP_TYPES:
        g = got[k].cpu().numpy() if isinstance(got[k], torch.Tensor) else np.asarray(got[k])
        assert g.dtype == np.float32 and g.shape == want[k].shape, k
        assert np.array_equal(g, want[k]), (k, int((g != want[k]).sum()))


@pytest.mark.parametrize('perm', PERMS)
@pytest.mark.parametrize('working,target', [
    ((37, 29, 41), (31, 24, 34)),            # a 1.2 A input, clipped edge tiles on every axis
    ((31, 24, 34), (37, 29, 41)),            # a 0.83 A input
    ((23, 19, 27), (23, 19, 27)),            # identity
    ((66, 51, 60), (22, 17, 20)),            # a 3 A input
    ((17, 13, 15), (34, 26, 30)),            # a 0.5 A input
    ((9, 1, 40), (5, 1, 71)),                # a one-sample axis
    ((1, 8, 6), (3, 1, 11)),                 # one working plane, one target row
])
def test_kernel_equals_oracle(cuda, perm, working, target):
    cube = ops.cube_space_shape(working, perm)
    vols = _volumes(cube, cuda, seed=sum(working) + perm[0])
    n0 = ops.launch_count()
    got = ops.volumes_to_grid(vols, perm, working, target)
    assert ops.launch_count() - n0 == 1
    _assert_oracle(got, vols, perm, target)
    if working == target:                                         # 'working': the permuted copy, bit for bit
        inv = pmo.inverse_perm(perm)
        for k in ('backbone_probability', 'carbon_alpha_probability'):
            assert torch.equal(got[k], vols[k].permute(inv))
        assert torch.equal(got['amino_acid_probability'],
                           vols['amino_acid_probability'].permute((0,) + tuple(1 + a for a in inv)))


def test_kernel_equals_oracle_on_a_larger_map(cuda):
    working, target, perm = (131, 97, 112), (109, 81, 93), (2, 1, 0)
    vols = _volumes(ops.cube_space_shape(working, perm), cuda, seed=11)
    _assert_oracle(ops.volumes_to_grid(vols, perm, working, target), vols, perm, target)


def test_stitched_volumes_and_refusals(cuda):
    working, perm = (20, 18, 16), (2, 1, 0)
    cube = ops.cube_space_shape(working, perm)
    sv = ops.StitchedVolumes(cube, cuda)
    for k, v in _volumes(cube, cuda, 2).items():
        getattr(sv, k).copy_(v)
    _assert_oracle(ops.volumes_to_grid(sv, perm, working, (17, 15, 13)), sv.as_dict(), perm, (17, 15, 13))
    n0 = ops.launch_count()
    part = ops.StitchedVolumes(cube, cuda, org=(0, 0, 0), ext=(8, 18, 20))
    with pytest.raises(ops._lib.MicaError, match='whole cube space'):
        ops.volumes_to_grid(part, perm, working, (17, 15, 13))
    with pytest.raises(ops._lib.MicaError, match='permuted by'):
        ops.volumes_to_grid(sv, (0, 1, 2), working, (17, 15, 13))
    with pytest.raises(ops._lib.MicaError, match='not a permutation'):
        ops.volumes_to_grid(sv, (2, 2, 0), working, (17, 15, 13))
    with pytest.raises(ops._lib.MicaError, match='target shape'):
        ops.volumes_to_grid(sv, perm, working, (17, 0, 13))
    assert ops.launch_count() == n0


# ------------------------------------------------------------------------------------------------ drop-in
@pytest.fixture
def _env(monkeypatch):
    for k in ('MICA_DEVICES', 'MICA_MIN_MAX', 'MICA_PRECISION', 'MICA_SAVE_MAPS'):
        monkeypatch.delenv(k, raising=False)
    session.clear()
    yield monkeypatch
    session.clear()


def _case(tmp_path, data, voxel, mapc=1, mapr=2, maps=3, min_max=None):
    """DataPreprocessor -> GridCreator(grid_size=16, padding=8) on an MRC file holding ``data``; returns (grids path,
    input MrcMap as written)."""
    case = tmp_path / 'input' / 'ID'
    os.makedirs(case / 'AF3_results', exist_ok=True)
    map_path = str(case / 'map.mrc')
    m = mrc.MrcMap(data=data, voxel_size=tuple(np.float32(v) for v in voxel),
                   origin=(np.float32(-10.5), np.float32(4.25), np.float32(30.0)), mapc=mapc, mapr=mapr, maps=maps,
                   nxstart=3, nystart=-2, nzstart=5)
    mrc.write_mrc(map_path, m, dtype=data.dtype)
    dp = DataPreprocessor(map_path=map_path, AF3_results=str(case / 'AF3_results'), quiet=True)
    dp.resample_and_normalize_map()
    assert session.get(dp.normalized_map_path) is not None
    grids = str(case / 'grids') + '/'
    r = GridCreator(quiet=True, min_max=min_max).create_normalized_map_grids(
        dp.normalized_map_path, os.path.join(grids, 'normalized_map_grids'), 16, 8)
    assert r['success']
    return grids, mrc.read_mrc(map_path)


def _run(grids, out, **kw):
    kw.setdefault('save_output', False)
    pr = CryoEMPredictor('unused', grids, str(out), quiet=True, model=PointwiseModel().to('cuda'),
                         host_volumes=MAP_TYPES, release_inputs=False, super_batch=20, **kw)
    ok, vols = pr.run_prediction()
    assert ok
    return pr, vols


def _read_maps(pr):
    out = {}
    for k in MAP_TYPES:
        ms = [mrc.read_mrc(os.path.join(pr.reconstruction_path, n)) for n in map_file_names(k)]
        out[k] = np.stack([np.asarray(m.data, np.float32) for m in ms]) if len(ms) > 1 else np.asarray(ms[0].data,
                                                                                                       np.float32)
        out[k + '/headers'] = ms
    return out


def _check_files(pr, vols, src):
    """The files: the input's shape and header fields; data = the oracle of the returned volumes."""
    mode, perm, working, target, hdr = pr._maps_target
    files = _read_maps(pr)
    for k in MAP_TYPES:
        for m in files[k + '/headers']:
            assert m.data.shape == target and m.mode == (0 if k == 'amino_acid_prediction' else 2), k
            assert (m.mapc, m.mapr, m.maps, m.nxstart, m.nystart, m.nzstart) == \
                (hdr.mapc, hdr.mapr, hdr.maps, hdr.nxstart, hdr.nystart, hdr.nzstart)
            assert m.origin == tuple(np.float32(v) for v in hdr.origin)
            np.testing.assert_allclose(np.array(m.voxel_size), np.array(hdr.voxel_size, np.float32), rtol=2e-7)
    want = pmo.volumes_to_grid({k: np.asarray(vols[k]) for k in MAP_TYPES}, perm, target)
    for k in MAP_TYPES:
        assert np.array_equal(files[k], want[k]), k
    if mode == 'input':
        assert target == src.data.shape
        assert (hdr.mapc, hdr.mapr, hdr.maps, hdr.nxstart, hdr.nystart, hdr.nzstart) == \
            (src.mapc, src.mapr, src.maps, src.nxstart, src.nystart, src.nzstart)
        assert tuple(hdr.voxel_size) == tuple(src.voxel_size) and tuple(hdr.origin) == tuple(src.origin)
    return files


def test_dropin_input_grid_anisotropic_axis_order(cuda, tmp_path, _env):
    data = synthetic.synthetic_map((38, 44, 34), voxel=1.2, seed=3)
    grids, src = _case(tmp_path, data, (1.2, 1.1, 1.3), mapc=3, mapr=2, maps=1)
    pr, vols = _run(grids, tmp_path / 'o', save_maps='input')
    assert pr._maps_target[1] != (2, 1, 0) and pr._maps_target[3] == (38, 44, 34)
    assert set(pr.maps_timing) == {'kernel', 'download', 'write'} and pr.timing_stats['saving'] > 0
    _check_files(pr, vols, src)
    assert not any(f.endswith('.npy') for f in os.listdir(pr.reconstruction_path))   # independent of save_output

    # 'working' through the environment: the 1 A grid with the normalised map's header, the permuted copy
    _env.setenv('MICA_SAVE_MAPS', 'working')
    pw, vw = _run(grids, tmp_path / 'w')
    _assert_same(vols, vw)
    files = _check_files(pw, vw, src)
    assert pw._maps_target[3] == tuple(session.get(os.path.join(grids, 'normalized_map_grids'))['volume'].shape)
    inv = pmo.inverse_perm(pw._maps_target[1])
    assert np.array_equal(files['backbone_probability'], np.transpose(np.asarray(vw['backbone_probability']), inv))
    assert all(np.float32(v) == np.float32(1) for v in pw._maps_target[4].voxel_size)


def test_dropin_int16_map_and_one_angstrom_identity(cuda, tmp_path, _env):
    grids, src = _case(tmp_path / 'i16', _int16_map((36, 40, 44), 4), (1.2, 1.2, 1.2))
    pr, vols = _run(grids, tmp_path / 'o16', save_maps='input')
    _check_files(pr, vols, src)
    session.clear()
    # a 1.0 A map: the working grid is the input grid, and 'input' is the permuted copy bit for bit (D10)
    grids, src = _case(tmp_path / 'one', synthetic.synthetic_map((30, 34, 26), voxel=1.0, seed=5), (1.0, 1.0, 1.0),
                       mapc=2, mapr=3, maps=1)
    pr, vols = _run(grids, tmp_path / 'o1', save_maps='input')
    mode, perm, working, target, _ = pr._maps_target
    assert working == target == src.data.shape
    files = _check_files(pr, vols, src)
    inv = pmo.inverse_perm(perm)
    for k in ('backbone_probability', 'carbon_alpha_probability'):
        assert np.array_equal(files[k], np.transpose(np.asarray(vols[k]), inv)), k
    assert np.array_equal(files['amino_acid_probability'],
                          np.transpose(np.asarray(vols['amino_acid_probability']), (0,) + tuple(1 + a for a in inv)))


def test_dropin_devices_tta_bf16_min_max(cuda, tmp_path, _env):
    grids, src = _case(tmp_path, synthetic.synthetic_map((36, 40, 34), voxel=1.2, seed=6), (1.2, 1.2, 1.2))
    p1, v1 = _run(grids, tmp_path / 'a1', save_maps='input')
    p2, v2 = _run(grids, tmp_path / 'a2', save_maps='input', devices=[0, 0])
    _assert_same(v1, v2)
    _assert_same(_read_maps(p1), _read_maps(p2))
    t1, w1 = _run(grids, tmp_path / 't1', save_maps='input', tta='flips')
    t2, w2 = _run(grids, tmp_path / 't2', save_maps='input', tta='flips', devices=[0, 0])
    _assert_same(_read_maps(t1), _read_maps(t2))
    _check_files(t1, w1, src)
    pb, vb = _run(grids, tmp_path / 'bf', save_maps='input', precision='bf16')
    _check_files(pb, vb, src)
    session.clear()
    grids, src = _case(tmp_path / 'mm', _masked_map((80, 80, 80), 5), (1.0, 1.0, 1.0), min_max=T)   # corners empty
    pm, vm = _run(grids, tmp_path / 'mm_o', save_maps='input')
    assert len(pm._source['ijk']) < np.prod([-(-int(v) // 16) for v in pm._source['cube_shape']])
    _check_files(pm, vm, src)


def test_dropin_refusals_and_no_maps_by_default(cuda, tmp_path, _env):
    grids, src = _case(tmp_path, synthetic.synthetic_map((30, 32, 28), voxel=1.2, seed=7), (1.2, 1.2, 1.2))
    pr, _ = _run(grids, tmp_path / 'none', save_output=True)
    names = os.listdir(pr.reconstruction_path)
    assert sorted(names) == sorted(f'{k}.npy' for k in MAP_TYPES)      # save_maps unset: no MRC file

    n0 = ops.launch_count()
    for kw in ({'save_maps': 'inputs'}, {'save_maps': 1}):
        p = CryoEMPredictor('unused', grids, str(tmp_path / 'bad'), save_output=False, quiet=True,
                            model=PointwiseModel().to(cuda), **kw)
        p.logger.disabled = True
        assert p.run_prediction() == (False, {})
    _env.setenv('MICA_SAVE_MAPS', 'mrc')
    p = CryoEMPredictor('unused', grids, str(tmp_path / 'bad'), save_output=False, quiet=True,
                        model=PointwiseModel().to(cuda))
    p.logger.disabled = True
    assert p.run_prediction() == (False, {})
    assert ops.launch_count() == n0
    _env.delenv('MICA_SAVE_MAPS')
    # a normalised map GridCreator reads from its file did not come through DataPreprocessor: no input grid
    session.clear()
    norm = tmp_path / 'norm.mrc'
    mrc.write_mrc(str(norm), mrc.MrcMap(data=synthetic.synthetic_map((40, 36, 44), voxel=1.0, seed=8)))
    g2 = str(tmp_path / 'g2') + '/'
    GridCreator(quiet=True).create_normalized_map_grids(str(norm), os.path.join(g2, 'normalized_map_grids'), 16, 8)
    n0 = ops.launch_count()
    p = CryoEMPredictor('unused', g2, str(tmp_path / 'bad2'), save_output=False, quiet=True,
                        model=PointwiseModel().to(cuda), save_maps='input')
    p.logger.disabled = True
    assert p.run_prediction() == (False, {})
    assert ops.launch_count() == n0
    assert not os.path.exists(tmp_path / 'bad') and not os.path.exists(tmp_path / 'bad2')
    pw, vw = _run(g2, tmp_path / 'g2w', save_maps='working')                # 'working' needs only the header
    _check_files(pw, vw, None)
