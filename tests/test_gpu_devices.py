"""One map's cubes dealt over several workers in one process (``CryoEMPredictor(devices=)``): the four volumes
are bit-identical to the one-device predictor's.  Several workers on one GPU (``devices=['cuda:0'] * 3``, each
with its own stream and pipeline) exercise the dealing, the threads and the one-owner peer stitch on one B200;
``devices='all'`` runs the same comparison across real GPUs where there are at least two."""
import os
import threading

import numpy as np
import pytest
import torch

from mica_b200 import mrc, session, synthetic
from mica_b200.create_grids import GridCreator
from mica_b200.predict import CryoEMPredictor, MAP_TYPES
from mica_b200.preprocessing import DataPreprocessor
from test_gpu_dropin import BranchingModel, PointwiseModel

pytestmark = pytest.mark.gpu

EMULATED = ['cuda:0'] * 3


class BatchCoupledModel(BranchingModel):
    """MICA's whole-batch zero-AF3 branch, plus a term that depends on every cube of the batch -- as TF32
    convolutions make a cube's logits depend on its batch: any change in which cubes share a model call
    changes the volumes."""

    def forward(self, x, af):
        bb, ca, aa = super().forward(x, af)
        return bb + 0.01 * x.mean(), ca, aa


def _drop_in(tmp_path, shape_zyx=(96, 96, 96), materialize=False):
    """DataPreprocessor -> GridCreator(grid_size=16, padding=8) on a synthetic map at 1.0 A whose atoms cover
    only the low corner of the map.  Returns the grids path."""
    case = tmp_path / 'input' / 'ID'
    os.makedirs(case / 'AF3_results', exist_ok=True)
    src = synthetic.synthetic_map(shape_zyx, voxel=1.0, seed=5)
    map_path = str(case / 'map.mrc')
    mrc.write_mrc(map_path, mrc.MrcMap(data=src, voxel_size=(np.float32(1.0),) * 3))
    st = synthetic.synthetic_structure(60, (40, 40, 40), seed=5)
    pdb_path = str(case / 'ID_af3_docked.pdb')
    synthetic.write_pdb(pdb_path, st)
    dp = DataPreprocessor(map_path=map_path, AF3_results=str(case / 'AF3_results'), quiet=True)
    dp.resample_and_normalize_map()
    assert dp.create_AF3_encodings(pdb_path)
    grids = str(case / 'grids') + '/'
    # materialize: the per-cube map files only (the 24 AF3 channels would be 25 times as many files); a file
    # source without AF3 files gets zero AF3 features, as the reference's dataset does
    r = GridCreator(quiet=True, materialize=materialize).create_normalized_map_grids(
        dp.normalized_map_path, os.path.join(grids, 'normalized_map_grids'), 16, 8)
    assert r['success']
    assert GridCreator(quiet=True).create_AF3_encodings_grids(
        dp.AF3_encodings, os.path.join(grids, 'AF3_encoding_grids'), 16, 8)['success']
    return grids, r['grid_count']


def _predict(grids, out, model, **kw):
    pr = CryoEMPredictor('unused', grids, str(out), save_output=False, quiet=True, model=model, host_volumes=MAP_TYPES,
                         release_inputs=False, super_batch=20, **kw)
    ok, vols = pr.run_prediction()
    assert ok
    return pr, vols


def _assert_same(a, b):
    for k in MAP_TYPES:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k


@pytest.fixture(autouse=True)
def _no_env(monkeypatch):
    monkeypatch.delenv('MICA_DEVICES', raising=False)
    session.clear()
    yield
    session.clear()


def test_resident_d8_split_matches_one_device(cuda, tmp_path):
    grids, n = _drop_in(tmp_path)
    assert n == 216                                       # > 200 cubes: the reference's batches of <= 8
    m1, m3 = BatchCoupledModel(), BatchCoupledModel()
    p1, v1 = _predict(grids, tmp_path / 'o1', m1)
    p3, v3 = _predict(grids, tmp_path / 'o3', m3, devices=EMULATED)
    assert p1.worker_cubes is None and p3.optimal_batch_size == 8
    assert sum(p3.worker_cubes) == 216 and min(p3.worker_cubes) > 0
    assert sorted(m1.seen) == sorted(m3.seen)             # the same calls, in whatever order the threads ran
    assert {z for _, z in m1.seen} == {True, False}       # atoms cover only part of the map
    _assert_same(v1, v3)


def test_reference_batching_and_file_source_match_one_device(cuda, tmp_path):
    grids, _ = _drop_in(tmp_path, materialize=True)
    # resident volumes, cubes in the glob order of the grid files, mixed batches
    _, v1 = _predict(grids, tmp_path / 'o1', BatchCoupledModel(), reference_batching=True)
    _, v3 = _predict(grids, tmp_path / 'o3', BatchCoupledModel(), reference_batching=True, devices=EMULATED)
    _assert_same(v1, v3)
    # the reference's .npz files only (a fresh process: empty session)
    session.clear()
    p1, f1 = _predict(grids, tmp_path / 'f1', BatchCoupledModel())
    session.clear()
    p3, f3 = _predict(grids, tmp_path / 'f3', BatchCoupledModel(), devices=EMULATED)
    assert p1._source['kind'] == p3._source['kind'] == 'files' and min(p3.worker_cubes) > 0
    _assert_same(f1, f3)


def test_small_map_model_batch_one(cuda, tmp_path):
    grids, n = _drop_in(tmp_path, shape_zyx=(80, 96, 96))
    assert n == 180
    _, v1 = _predict(grids, tmp_path / 'o1', BatchCoupledModel())
    p3, v3 = _predict(grids, tmp_path / 'o3', BatchCoupledModel(), devices=EMULATED)
    assert p3.optimal_batch_size == 1 and min(p3.worker_cubes) > 0
    _assert_same(v1, v3)
    # a {device: callable} mapping serves as well
    _, vm = _predict(grids, tmp_path / 'om', {'cuda:0': BatchCoupledModel()}, devices=['cuda:0', 0])
    _assert_same(v1, vm)


def test_worker_failure_returns_false_and_stops_every_thread(cuda, tmp_path):
    grids, _ = _drop_in(tmp_path)

    class FailsOnSecondCall(PointwiseModel):
        calls = 0

        def forward(self, x, af):
            type(self).calls += 1
            if type(self).calls == 2:
                raise RuntimeError('model failure')
            return super().forward(x, af)
    before = threading.active_count()
    pr = CryoEMPredictor('unused', grids, str(tmp_path / 'o'), save_output=False, quiet=True,
                         model=FailsOnSecondCall(), super_batch=20, devices=EMULATED)
    assert pr.run_prediction() == (False, {})
    assert threading.active_count() == before
    # the inputs were not released: the same map still runs
    _, v = _predict(grids, tmp_path / 'o2', PointwiseModel(), devices=EMULATED)
    assert np.asarray(v['backbone_probability']).any()


def test_environment_variable(cuda, tmp_path, monkeypatch):
    grids, _ = _drop_in(tmp_path, shape_zyx=(80, 96, 96))
    p0, v0 = _predict(grids, tmp_path / 'o0', PointwiseModel())
    monkeypatch.setenv('MICA_DEVICES', '')
    pe, ve = _predict(grids, tmp_path / 'oe', PointwiseModel())
    assert p0.worker_cubes is None and pe.worker_cubes is None
    _assert_same(v0, ve)
    monkeypatch.setenv('MICA_DEVICES', 'all')
    pa, va = _predict(grids, tmp_path / 'oa', PointwiseModel())
    assert (pa.worker_cubes is None) == (torch.cuda.device_count() == 1)
    _assert_same(v0, va)
    for bad in ('0,0', 'garbage'):                        # repeats only through devices=
        monkeypatch.setenv('MICA_DEVICES', bad)
        pr = CryoEMPredictor('unused', grids, str(tmp_path / 'ob'), save_output=False, quiet=True,
                             model=PointwiseModel(), release_inputs=False)
        assert pr.run_prediction() == (False, {})


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs at least two GPUs')
@pytest.mark.parametrize('model_cls', [PointwiseModel, BatchCoupledModel])
def test_real_devices_match_one_device(cuda, tmp_path, model_cls):
    from mica_b200 import _lib
    assert _lib.lib.mica_peer_enable(0, 1) == 0 and _lib.lib.mica_peer_enable(0, 1) == 0    # already enabled: ok
    grids, _ = _drop_in(tmp_path)
    _, v1 = _predict(grids, tmp_path / 'o1', model_cls().to(cuda))
    pa, va = _predict(grids, tmp_path / 'oa', model_cls().to(cuda), devices='all')
    assert len(pa.worker_cubes) == torch.cuda.device_count()
    _assert_same(v1, va)
    # a plain callable cannot be copied to the other GPUs: refused
    pr = CryoEMPredictor('unused', grids, str(tmp_path / 'ob'), save_output=False, quiet=True,
                         model=lambda x, af: PointwiseModel()(x, af), devices='all', release_inputs=False)
    assert pr.run_prediction() == (False, {})
