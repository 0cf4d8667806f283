"""The reference-facing classes (DataPreprocessor / GridCreator / CryoEMPredictor
mirrors) driven the way Solver.getData / Solver.nnPred drive the originals
(utils/modeler.py:673-760), checked against the oracle."""
import os

import numpy as np
import pytest
import torch

from mica_b200 import mrc, pdb, session, synthetic
from mica_b200.create_grids import GridCreator
from mica_b200.predict import CryoEMPredictor, DeviceVolume, HostPool, MAP_TYPES, SMALL_VOLUMES
from mica_b200.preprocessing import DataPreprocessor
from oracle import mica_oracle as orc

pytestmark = pytest.mark.gpu


class PointwiseModel(torch.nn.Module):
    """Deterministic stand-in for MICA with its (exp_map, af_features) -> (bb, ca, aa)
    signature; elementwise, so the CPU oracle can evaluate it on the oracle's cubes."""

    def forward(self, x, af):
        s = af.sum(dim=1, keepdim=True)
        bb = torch.cat([x, -x, 2 * x - 0.5 + s, x * x], dim=1)
        ca = torch.cat([0.5 - x, x, x * 3 - 1, 1.5 * x + af[:, :1]], dim=1)
        aa = torch.cat([x * (0.1 * t) + af[:, t % 24:t % 24 + 1] * (t % 3) + np.sin(t) for t in range(21)], dim=1)
        return bb, ca, aa


def _inputs(tmp_path, shape=(40, 40, 40), voxel=1.1):
    case = tmp_path / 'input' / 'ID'
    os.makedirs(case / 'AF3_results', exist_ok=True)
    src = synthetic.synthetic_map(shape, voxel=voxel, seed=31)
    origin = (np.float32(12.5), np.float32(-4.0), np.float32(0.75))
    map_path = str(case / 'map.mrc')
    mrc.write_mrc(map_path, mrc.MrcMap(data=src, voxel_size=(np.float32(voxel),) * 3, origin=origin,
                                       nxstart=2, nystart=3, nzstart=5))
    n = round(shape[0] * voxel)
    st = synthetic.synthetic_structure(150, (n, n, n), seed=31, origin_xyz=origin, hetero_every=13)
    pdb_path = str(case / 'ID_af3_docked.pdb')
    synthetic.write_pdb(pdb_path, st)
    return src, origin, map_path, pdb_path, str(case / 'AF3_results'), str(case / 'grids')   # as run.py:108-112


def test_get_data_then_nn_pred_like_the_solver(cuda, tmp_path):
    session.clear()
    src, origin, map_path, pdb_path, af3_results, grids_path = _inputs(tmp_path)
    voxel = (np.float32(1.1),) * 3
    # ---- Solver.getData
    dp = DataPreprocessor(map_path=map_path, AF3_results=af3_results, quiet=True, write_files=True)
    assert dp.resample_and_normalize_map() is None
    assert dp.normalized_map_path.endswith('resampled_normalized_map.mrc')
    o_norm, _, _ = orc.normalize(orc.resample(src, voxel))
    written = mrc.read_mrc(dp.normalized_map_path)
    assert np.abs(written.data - o_norm).max() <= 1e-5
    assert written.voxel_size == (1.0, 1.0, 1.0) and written.origin == origin and written.nzstart == 5
    assert dp.create_AF3_encodings(pdb_path) is True
    coords, bb_ch, aa_ch, _ = pdb.read_pdb_atoms(pdb_path)
    o_af3, ok = orc.af3_encode(coords, bb_ch, aa_ch, origin, o_norm.shape)
    assert ok
    for c, name in enumerate(pdb.CHANNEL_NAMES):
        got = mrc.read_mrc(os.path.join(dp.AF3_encodings, f'{name}_encoding.mrc')).data
        assert np.array_equal(got, o_af3[c]), name
    gc = GridCreator(quiet=True)
    r1 = gc.create_normalized_map_grids(dp.normalized_map_path, os.path.join(grids_path, 'normalized_map_grids'))
    r2 = gc.create_AF3_encodings_grids(dp.AF3_encodings, os.path.join(grids_path, 'AF3_encoding_grids'))
    o_cubes, o_meta, o_shape, o_off = orc.extract_cubes(o_norm, nstart_zyx=(5, 3, 2))
    assert r1['success'] and r1['grid_count'] == len(o_cubes) and r1['offset'] == o_off
    assert set(r1) == {'success', 'grid_count', 'offset', 'output_directory', 'processing_time', 'input_file'}
    assert r2['success'] and r2['successful_channels'] == 24 and r2['total_grids'] == 24 * len(o_cubes)
    # ---- Solver.nnPred
    pr = CryoEMPredictor(model_path='unused', grids_path=grids_path, output_path=str(tmp_path / 'out'),
                         save_output=True, device='cuda', quiet=True, model=PointwiseModel())
    ok, vols = pr.run_prediction()
    assert ok and set(vols) == {'backbone_probability', 'carbon_alpha_probability', 'amino_acid_prediction',
                                'amino_acid_probability'}
    # default hand-over: three NumPy volumes, the 20-channel one as an array-like that stayed in HBM
    assert all(isinstance(vols[k], np.ndarray) for k in SMALL_VOLUMES)
    aap = vols['amino_acid_probability']
    assert isinstance(aap, DeviceVolume) and aap.shape == (20,) + vols['backbone_probability'].shape
    picks = (np.array([3, 7]), np.array([5, 9]), np.array([11, 2]))
    gathered = aap[:, picks[0], picks[1], picks[2]]                  # the reference's only use (modeler.py:850)
    vols = dict(vols, amino_acid_probability=np.asarray(aap))
    assert np.array_equal(gathered, vols['amino_acid_probability'][:, picks[0], picks[1], picks[2]])
    # the consumed session entries are gone (Solver.nnPred deletes the files at this point), the device volumes stay
    assert session.get(dp.normalized_map_path) is None and session.get(os.path.join(grids_path, 'normalized_map_grids')) is None
    assert session.get(os.path.join(str(tmp_path / 'out'), 'results', 'device_volumes')) is not None
    # oracle: same model on the oracle's cubes, reference post-processing + stitching
    norm_dev = torch.from_numpy(written.data)
    o_x = torch.from_numpy(orc.extract_cubes(written.data)[0][:, None])
    o_af = torch.from_numpy(np.stack([orc.extract_cubes(o_af3[c])[0] for c in range(24)], axis=1))
    with torch.no_grad():
        bb, ca, aa = PointwiseModel()(o_x, o_af)
    want = orc.postprocess_and_stitch(bb, ca, aa, o_meta, o_shape)
    for k in ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_probability'):
        assert vols[k].shape == want[k].shape and np.abs(vols[k] - want[k]).max() <= 2e-5, k
    top2 = np.sort(want['amino_acid_probability'], axis=0)[-2:]
    clear = (top2[1] - top2[0]) > 4e-6                             # equal wherever the top-2 gap is not rounding
    assert np.array_equal(vols['amino_acid_prediction'][clear], want['amino_acid_prediction'][clear])
    assert os.path.exists(os.path.join(str(tmp_path / 'out'), 'results', 'ID', 'amino_acid_probability.npy'))


def test_materialized_npz_files_and_file_fallback(cuda, tmp_path):
    """materialize=True writes the reference's per-cube files; a predictor in a fresh
    process (empty session) consumes them and gives the same volumes."""
    session.clear()
    rng = np.random.default_rng(4)
    vol = rng.random((20, 52, 30), dtype=np.float32)
    p = str(tmp_path / 'resampled_normalized_map.mrc')
    mrc.write_mrc(p, mrc.MrcMap(data=vol, nxstart=1, nystart=2, nzstart=3))
    grids = str(tmp_path / 'grids' / 'ID') + '/'
    gc = GridCreator(quiet=True, materialize=True)
    res = gc.create_normalized_map_grids(p, os.path.join(grids, 'normalized_map_grids'))
    o_cubes, o_meta, o_shape, o_off = orc.extract_cubes(vol, nstart_zyx=(3, 2, 1))
    assert res['grid_count'] == len(o_cubes)
    for c, m in zip(o_cubes, o_meta):
        d = np.load(os.path.join(grids, 'normalized_map_grids', f'normalized_map_grid_i{m[0]}_j{m[1]}_k{m[2]}.npz'))
        assert np.array_equal(d['grid'], c) and (int(d['di']), int(d['dj']), int(d['dk'])) == tuple(m[3:])
        assert tuple(d['orig_shape']) == tuple(o_shape) and int(d['padding']) == 8
    model = PointwiseModel()
    ok1, v1 = CryoEMPredictor('unused', grids, str(tmp_path / 'o1'), save_output=False, model=model,
                              quiet=True).run_prediction()
    session.clear()
    ok2, v2 = CryoEMPredictor('unused', grids, str(tmp_path / 'o2'), save_output=False, model=model,
                              quiet=True).run_prediction()
    assert ok1 and ok2
    for k in v1:
        assert np.array_equal(np.asarray(v1[k]), np.asarray(v2[k])), k


def test_failure_conventions(cuda, tmp_path):
    """Never raise at the boundary: return None / False / (False, {}) like the reference."""
    session.clear()
    dp = DataPreprocessor(map_path=str(tmp_path / 'missing.mrc'), AF3_results=str(tmp_path / 'AF3_results') + '/')
    assert dp.resample_and_normalize_map() is None and dp.normalized_map_path is None
    flat = str(tmp_path / 'flat.mrc')
    mrc.write_mrc(flat, mrc.MrcMap(data=np.zeros((8, 8, 8), np.float32)))
    dp = DataPreprocessor(map_path=flat, AF3_results=str(tmp_path / 'AF3_results') + '/')
    dp.resample_and_normalize_map()
    assert dp.normalized_map_path is None                       # no positive values -> nothing written
    gc = GridCreator(quiet=True)
    assert gc.create_normalized_map_grids(str(tmp_path / 'nope.mrc'), str(tmp_path / 'g'))['success'] is False
    assert gc.create_grids_from_mrc(str(tmp_path / 'nope.mrc'), str(tmp_path / 'g')) == (0, None)
    ok, vols = CryoEMPredictor('unused', str(tmp_path / 'empty') + '/', str(tmp_path / 'o')).run_prediction()
    assert ok is False and vols == {}


def _d8_case(tmp_path, materialize=False):
    """3 cubes along x; only the first has AF3 signal."""
    rng = np.random.default_rng(9)
    vol = rng.random((20, 20, 100), dtype=np.float32)
    af3 = np.zeros((24, 20, 20, 100), np.float32)
    af3[3, 5, 5, 10] = 1.0
    p = str(tmp_path / 'resampled_normalized_map.mrc')
    mrc.write_mrc(p, mrc.MrcMap(data=vol))
    enc = tmp_path / 'AF3_encodings'
    os.makedirs(enc)
    for c, name in enumerate(pdb.CHANNEL_NAMES):
        mrc.write_mrc(str(enc / f'{name}_encoding.mrc'), mrc.MrcMap(data=af3[c]))
    grids = str(tmp_path / 'grids' / 'ID') + '/'
    gc = GridCreator(quiet=True, materialize=materialize)
    gc.create_normalized_map_grids(p, os.path.join(grids, 'normalized_map_grids'))
    gc.create_AF3_encodings_grids(str(enc), os.path.join(grids, 'AF3_encoding_grids'))
    return grids


class BranchingModel(PointwiseModel):
    """Has MICA's whole-batch zero-AF3 branch (models/model.py:60-63)."""

    def __init__(self):
        super().__init__()
        self.seen = []

    def forward(self, x, af):
        zero = bool(af.abs().sum() < 1e-6)
        self.seen.append((x.shape[0], zero))
        bb, ca, aa = super().forward(x, af)
        return (bb + 1.0, ca - 1.0, aa * 0.5) if zero else (bb, ca, aa)


def test_zero_af3_cubes_are_batched_apart(cuda, tmp_path):
    """D8, default mode: with batching on, a cube without AF3 signal never shares a model call with one that
    has some -- every cube gets the logits of the reference's single-sample mode."""
    session.clear()
    grids = _d8_case(tmp_path)
    m8, m1 = BranchingModel(), BranchingModel()
    pr = CryoEMPredictor('unused', grids, str(tmp_path / 'o'), save_output=False, model=m8, quiet=True,
                         release_inputs=False)
    pr.batch_threshold = 1                                      # force the batched strategy
    ok, v8 = pr.run_prediction()
    assert ok and sorted(m8.seen) == [(1, False), (2, True)]
    pr1 = CryoEMPredictor('unused', grids, str(tmp_path / 'o1'), save_output=False, model=m1, quiet=True)
    ok, v1 = pr1.run_prediction()                               # 3 cubes <= 200: single-sample strategy
    assert ok and sorted(m1.seen) == [(1, False), (1, True), (1, True)]
    for k in v8:
        assert np.array_equal(np.asarray(v8[k]), np.asarray(v1[k])), k


def test_reference_batching_reproduces_the_mixed_batches(cuda, tmp_path):
    """D8, ``reference_batching=True``: cubes in the reference's glob order, mixed batches, MICA's branch taken
    on the whole batch -- compared with the oracle's statement of that batch (one model call on all three cubes,
    then the reference's stitch, pinned by stitch.npz) and, where a copy of it is present, with the UNMODIFIED
    reference predictor run on the same files and model."""
    from oracle import ref_harness
    session.clear()
    grids = _d8_case(tmp_path, materialize=True)
    model = BranchingModel()
    pr = CryoEMPredictor('unused', grids, str(tmp_path / 'o'), save_output=False, model=model, quiet=True,
                         reference_batching=True, host_volumes=MAP_TYPES)
    pr.batch_threshold = 1
    ok, got = pr.run_prediction()
    assert ok and model.seen == [(3, False)]                    # one mixed batch: nobody takes the zero branch
    norm = mrc.read_mrc(str(tmp_path / 'resampled_normalized_map.mrc')).data
    af3 = [mrc.read_mrc(str(tmp_path / 'AF3_encodings' / f'{name}_encoding.mrc')).data for name in pdb.CHANNEL_NAMES]
    o_cubes, o_meta, o_shape, _ = orc.extract_cubes(norm)
    o_af = torch.from_numpy(np.stack([orc.extract_cubes(a)[0] for a in af3], axis=1))
    o_model = BranchingModel()
    with torch.no_grad():
        logits = o_model(torch.from_numpy(o_cubes[:, None]), o_af)
    assert o_model.seen == [(3, False)]
    _check_mixed_batches(got, orc.postprocess_and_stitch(*logits, o_meta, o_shape))
    if not ref_harness.available():
        return
    ref_harness._setup_path()
    from utils.predict import CryoEMPredictor as RefPredictor
    with ref_harness._quiet():
        rp = RefPredictor(model_path='unused', grids_path=grids, output_path=str(tmp_path / 'ref'),
                          save_output=False, device='cpu', quiet=True)
        rp.logger.disabled = True
        rp.batch_threshold = 1
        assert rp.select_processing_strategy()
        rp.model = BranchingModel()
        good, loader = rp.prepare_data()
        assert good and rp.run_inference(loader)
        good, want = rp.reconstruct_and_save_volumes()
    assert good and rp.model.seen == [(3, False)]
    _check_mixed_batches(got, want)


def _check_mixed_batches(got, want):
    for k in ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_probability'):
        assert np.abs(got[k] - want[k]).max() <= 1e-5, k
    top2 = np.sort(want['amino_acid_probability'], axis=0)[-2:]
    clear = (top2[1] - top2[0]) > 4e-6                             # equal wherever the top-2 gap is not rounding
    same = got['amino_acid_prediction'] == want['amino_acid_prediction']
    assert same[clear].all() and same.mean() > 0.9999


def test_host_pool_and_all_four_volumes(cuda, tmp_path):
    """host_volumes=MAP_TYPES returns four NumPy arrays like the reference; a HostPool reuses the pinned buffers."""
    session.clear()
    grids = _d8_case(tmp_path)
    pool = HostPool()
    kw = dict(save_output=False, model=PointwiseModel(), quiet=True, host_volumes=MAP_TYPES, host_pool=pool,
              release_inputs=False)
    ok, a = CryoEMPredictor('unused', grids, str(tmp_path / 'o'), **kw).run_prediction()
    assert ok and all(isinstance(a[k], np.ndarray) for k in MAP_TYPES)
    keep = {k: v.copy() for k, v in a.items()}
    ok, b = CryoEMPredictor('unused', grids, str(tmp_path / 'o'), **kw).run_prediction()
    assert ok
    for k in MAP_TYPES:
        assert np.array_equal(b[k], keep[k]) and b[k].ctypes.data == a[k].ctypes.data      # same pinned buffer


def test_device_argument_is_honoured_when_another_gpu_is_current(cuda):
    """ops entry points run on the device of their tensors (ADVICE round 1): exercised with the only GPU a
    test box is sure to have by making sure the guard passes through, and on a second GPU when present."""
    from mica_b200 import ops
    x = torch.rand(4096, device=cuda)
    y, _ = ops.normalize(x)
    if torch.cuda.device_count() > 1:
        other = torch.device('cuda', 1)
        x1 = x.to(other)
        with torch.cuda.device(0):
            y1, _ = ops.normalize(x1)                           # current device 0, tensors on device 1
        assert y1.device == other and torch.equal(y1.cpu(), y.cpu())
        with pytest.raises(Exception):
            ops.extract_cubes(x1.view(16, 16, 16), torch.zeros((1, 3), dtype=torch.int32, device=cuda))
