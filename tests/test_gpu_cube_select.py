"""The inference keep rule (``min_max=``): the window-maximum pass equals ``np.max`` over the reference's zero-padded
windows, the selection equals oracle/cube_select_oracle.py (ties and NaN kept), skipped cores are 0 and kept ones keep
their bits, the model sees only kept cubes, and the split maps and the drop-in give the one-GPU bits."""
import glob
import os

import numpy as np
import pytest
import torch

from mica_b200 import _lib, mrc, ops, session, synthetic
from mica_b200.create_grids import GridCreator
from mica_b200.peer import PeerVolumes
from mica_b200.pipeline import MapHeader, MapPipeline, _SlabDrain
from mica_b200.predict import CryoEMPredictor, MAP_TYPES
from mica_b200.preprocessing import DataPreprocessor
from mica_b200.slab import BalancedCubePipeline, SlabPipeline, SlabPlan
from oracle import cube_select_oracle as cso

from test_gpu_devices import EMULATED, _assert_same
from test_gpu_overlap_split import _int16_map, _lockstep
from test_gpu_tta import PointwiseModel

pytestmark = pytest.mark.gpu

HDR = MapHeader(voxel_size=(np.float32(1.0),) * 3)
T = 0.01


def _dev(a, cuda):
    return torch.from_numpy(np.ascontiguousarray(a)).to(cuda)


def _ellipsoid(shape, frac=0.3):
    g = np.meshgrid(*[(np.arange(n) - (n - 1) / 2) / (frac * n) for n in shape], indexing='ij')
    return sum(v * v for v in g) <= 1.0


def _masked_map(shape, seed, frac=0.3):
    """A synthetic map, non-negative, times an ellipsoidal mask: exact zeros outside it, as in a masked map."""
    return (np.abs(synthetic.synthetic_map(shape, voxel=1.0, seed=seed)) * _ellipsoid(shape, frac)).astype(np.float32)


class CountingModel(PointwiseModel):
    """``PointwiseModel`` (batch-independent) that counts the cubes it runs and records each cube's input sum."""

    def __init__(self, seed=0):
        super().__init__(seed)
        self.cubes, self.calls, self.sums = 0, 0, []

    def forward(self, x, af):
        self.cubes += int(x.shape[0])
        self.calls += 1
        self.sums += x.double().sum(dim=(1, 2, 3, 4)).cpu().tolist()
        return super().forward(x, af)


def _np(vols):
    return {k: v.cpu().numpy() for k, v in vols.as_dict().items()}


def _core_mask(cube_shape, gs, ijk):
    m = np.zeros(cube_shape, bool)
    for i, j, k in np.asarray(ijk):
        m[i:i + gs, j:j + gs, k:k + gs] = True
    return m


# ------------------------------------------------------------------------------------------ window maxima
@pytest.mark.parametrize('case', ['tma', 'fallback', 'perm', 'slab', 'negative', 'nan'])
def test_window_max_equals_np_max(cuda, case):
    gs, pad, shape = 16, 8, (37, 41, 44)               # nx % 4 == 0, W = 32: the extract takes its TMA route
    hdr = MapHeader()
    if case == 'fallback':
        gs, pad = 12, 3
    if case == 'perm':
        hdr = MapHeader(mapc=2, mapr=3, maps=1)
    if case == 'negative':                             # every voxel < 0: a window reaching out of the map has max 0
        shape = (70, 66, 72)
    vol = synthetic.synthetic_map(shape, voxel=1.0, seed=3).astype(np.float32)
    if case == 'negative':
        vol = vol - np.float32(vol.max() + 1)
    if case == 'nan':
        rng = np.random.default_rng(4)
        for _ in range(5):
            vol[tuple(rng.integers(0, n) for n in shape)] = np.nan
    perm, _ = hdr.transpose_order()
    if case == 'perm':
        assert perm == (0, 2, 1)
    want, meta, orig_shape = cso.window_maxima(vol, hdr.mapc, hdr.mapr, hdr.maps, gs, pad)
    ijk = ops.cube_origins(ops.cube_space_shape(vol.shape, perm), gs)
    assert orig_shape == ops.cube_space_shape(vol.shape, perm) and np.array_equal(meta[:, :3], ijk)
    d_ijk = _dev(ijk, cuda)
    if case == 'slab':                                 # a z-slab rank owning planes [16, 32), halo included
        lo, hi = 16, 32
        blk = (max(0, lo - pad), min(shape[0], hi + pad))
        mine = (ijk[:, 2] >= lo) & (ijk[:, 2] < hi)
        got = ops.cube_window_max(_dev(vol[blk[0]:blk[1]], cuda), _dev(ijk[mine], cuda), gs, pad, perm,
                                  global_nz=shape[0], z0=blk[0]).cpu().numpy()
        assert np.array_equal(got, want[mine])
        return
    got = ops.cube_window_max(_dev(vol, cuda), d_ijk, gs, pad, perm).cpu().numpy()
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    assert np.array_equal(got[~nan], want[~nan])
    if case == 'nan':
        assert nan.any() and not nan.all()
        return
    if case == 'negative':                             # the zeros of every face and the interior windows
        assert (got == 0).any() and (got < 0).any()
        for a, n in enumerate(orig_shape):
            assert (got[ijk[:, a] == 0] == 0).all()                          # low face
            assert (got[ijk[:, a] + gs + pad > n] == 0).all()                # high face
    cube_max = torch.empty(len(ijk), dtype=torch.float32, device=cuda)
    ops.extract_cubes(_dev(vol, cuda), d_ijk, gs, pad, perm, cube_max=cube_max)
    assert np.array_equal(cube_max.cpu().numpy(), got)


def test_selection_ties_ulps_and_nan(cuda):
    gs, pad, n = 16, 8, 96
    t = np.float32(T)
    below = np.nextafter(t, np.float32(0))
    norm = np.zeros((n, n, n), np.float32)
    norm[8, 8, 8] = t                                   # windows reaching (x, y, z) = (8, 8, 8): a tie, kept
    norm[8, 8, 56] = below                              # one ulp below: dropped
    norm[56, 56, 56] = np.nan                           # NaN: kept
    norm[88, 40, 88] = np.float32(0.5)
    pipe = MapPipeline(cuda, gs, pad, batch_cubes=8)
    pipe.set_normalized(_dev(norm, cuda), HDR)
    ijk = pipe.cube_index()
    maxima = ops.cube_window_max(pipe.normalized, pipe.ijk, gs, pad, pipe.perm)
    got = ops.select_cubes(maxima, T)
    want_max, _, _ = cso.window_maxima(norm, grid_size=gs, padding=pad)
    want = np.flatnonzero(cso.kept(want_max, T))
    assert np.array_equal(got, want)
    m = maxima.cpu().numpy()
    assert (m == t).any() and set(np.flatnonzero(m == t)) <= set(got)
    assert (m == below).any() and not set(np.flatnonzero(m == below)) & set(got)
    assert np.isnan(m).any() and set(np.flatnonzero(np.isnan(m))) <= set(got)
    assert len(got) < len(ijk)


@pytest.mark.parametrize('bad', [float('nan'), float('inf'), -float('inf'), '0.01', True])
def test_bad_min_max_is_refused_before_any_launch(cuda, bad):
    pipe = MapPipeline(cuda, 16, 8, batch_cubes=8)
    pipe.set_normalized(_dev(_masked_map((48, 48, 48), 1), cuda), HDR)
    n0 = ops.launch_count()
    with pytest.raises(_lib.MicaError):
        pipe.predict_and_stitch(PointwiseModel().to(cuda), min_max=bad)
    with pytest.raises(_lib.MicaError):
        ops.select_cubes(torch.zeros(3, device=cuda), bad)
    assert ops.launch_count() == n0


# ------------------------------------------------------------------------------------------ paste
def _masked_pipe(cuda, batch=7, shape=(96, 96, 96), seed=11):
    pipe = MapPipeline(cuda, 16, 8, batch_cubes=batch)
    assert pipe.resample_and_normalize(_dev(_masked_map(shape, seed), cuda), HDR)
    return pipe


def test_paste_keeps_kept_cores_and_zeroes_skipped_ones(cuda):
    pipe = _masked_pipe(cuda)
    gs = pipe.grid_size
    with torch.no_grad():
        full_model, sel_model = CountingModel().to(cuda), CountingModel().to(cuda)
        full = _np(pipe.predict_and_stitch(full_model))
        none = _np(pipe.predict_and_stitch(PointwiseModel().to(cuda), min_max=None))
        sel = _np(pipe.predict_and_stitch(sel_model, min_max=T))
    ijk = pipe.cube_index()
    kept = ops.select_cubes(ops.cube_window_max(pipe.normalized, pipe.ijk, gs, pipe.padding, pipe.perm), T)
    assert 0 < len(kept) < len(ijk)
    assert full_model.cubes == len(ijk) and sel_model.cubes == len(kept)
    for k in MAP_TYPES:
        assert np.array_equal(none[k], full[k]), k
    core = _core_mask(pipe.cube_shape, gs, ijk[kept])
    for k in MAP_TYPES:
        assert np.array_equal(sel[k][..., core], full[k][..., core]), k
        assert not sel[k][..., ~core].any(), k
    # the oracle's paste: the unfiltered probabilities of the kept cores, 0 elsewhere
    m = cso.kept(cso.window_maxima(pipe.normalized.cpu().numpy(), grid_size=gs, padding=pipe.padding)[0], T)
    assert np.array_equal(np.flatnonzero(m), kept)

    # volumes that held another map: the skipped cores are cleared
    other = MapPipeline(cuda, 16, 8, batch_cubes=7)
    assert other.resample_and_normalize(_dev(synthetic.synthetic_map((96, 96, 96), voxel=1.0, seed=2), cuda), HDR)
    with torch.no_grad():
        vols = other.predict_and_stitch(PointwiseModel().to(cuda))
        assert _np(vols)['backbone_probability'][~core].any()
        reused = _np(pipe.predict_and_stitch(PointwiseModel().to(cuda), vols, min_max=T))
    for k in MAP_TYPES:
        assert np.array_equal(reused[k], sel[k]), k


def test_order_prefetch_d8_and_drain_under_the_rule(cuda):
    pipe = _masked_pipe(cuda, batch=5)
    ijk = pipe.cube_index()
    kept = ops.select_cubes(ops.cube_window_max(pipe.normalized, pipe.ijk, 16, 8, pipe.perm), T)
    with torch.no_grad():
        want = _np(pipe.predict_and_stitch(PointwiseModel().to(cuda), min_max=T))
        # a custom order: the kept cubes in its relative sequence
        order = np.random.default_rng(0).permutation(len(ijk))
        m = CountingModel().to(cuda)
        got = _np(pipe.predict_and_stitch(m, order=order, model_batch=2, d8='split', min_max=T))
        kept_set = set(kept.tolist())
        want_seq = [int(o) for o in order if int(o) in kept_set]
        x = pipe.normalized
        ref = CountingModel().to(cuda)
        for o in want_seq:
            ref(ops.extract_cubes(x, _dev(ijk[o:o + 1], cuda), 16, 8, pipe.perm),
                torch.zeros((1, 24, 32, 32, 32), device=cuda))
        assert m.cubes == len(kept) and np.allclose(m.sums, ref.sums, rtol=1e-12, atol=0)
        pipe.prefetch = False
        unfetched = _np(pipe.predict_and_stitch(PointwiseModel().to(cuda), min_max=T))
        pipe.prefetch = True
        # the drain still streams finished layers: the kept list is in loop order
        pipe.cube_index()
        vols = pipe._new_volumes()
        out = {k: torch.empty(tuple(v.shape), dtype=v.dtype).pin_memory() for k, v in vols.as_dict().items()}
        drain = _SlabDrain(pipe, out)
        seen = []

        def on_batch(v, n_done):
            drain(v, n_done)
            seen.append(drain.sent_layers)
        pipe.predict_and_stitch(PointwiseModel().to(cuda), vols, on_batch=on_batch, min_max=T)
        drain.finish()
        torch.cuda.synchronize()
    assert len(seen) > 2 and 0 < seen[len(seen) // 2] < vols.ext[0]
    for k in MAP_TYPES:
        assert np.array_equal(got[k], want[k]), k
        assert np.array_equal(unfetched[k], want[k]), k
        assert np.array_equal(out[k].numpy(), want[k]), k


def test_no_cube_kept_gives_zero_volumes_without_the_model(cuda):
    pipe = _masked_pipe(cuda)
    m = CountingModel().to(cuda)
    with torch.no_grad():
        vols = _np(pipe.predict_and_stitch(m, min_max=2.0))            # normalised maps are <= 1
        wvols = _np(pipe.predict_and_stitch(m, min_max=2.0, overlap_window='triangle', tta='flips'))
    assert m.calls == 0
    for v in (vols, wvols):
        for k in MAP_TYPES:
            assert not v[k].any(), k


# ------------------------------------------------------------------------------------------ overlap + TTA
@pytest.mark.parametrize('window,tta', [('triangle', None), ('uniform', (0, 5, 30)), ('core', 'flips')])
def test_overlap_and_tta_against_the_statement(cuda, window, tta):
    gs, pad = 16, 8
    W = gs + 2 * pad
    pipe = MapPipeline(cuda, gs, pad, batch_cubes=5)
    assert pipe.resample_and_normalize(_dev(_masked_map((64, 56, 72), 5), cuda), HDR)
    model = PointwiseModel(seed=3).to(cuda)
    with torch.no_grad():
        got = _np(pipe.predict_and_stitch(model, overlap_window=window, tta=tta, min_max=T))
        pipe.configure(batch_cubes=3)
        codes = ops.tta_orientations(tta)
        rev = None if codes is None else list(reversed(codes))
        again = _np(pipe.predict_and_stitch(model, overlap_window=window, tta=rev, min_max=T))
    for k in MAP_TYPES:
        assert np.array_equal(got[k], again[k]), k
    ijk = pipe.cube_index()
    windows = ops.extract_cubes(pipe.normalized, pipe.ijk, gs, pad, pipe.perm).cpu().numpy().astype(np.float64)
    keep = cso.kept(cso.window_maxima(pipe.normalized.cpu().numpy(), grid_size=gs, padding=pad)[0], T)
    assert 0 < keep.sum() < len(keep)
    A, b = model.A.float().double().cpu().numpy(), model.b.float().double().cpu().numpy()

    def f(x):                                          # the model on one window, no AF3 signal
        y = (A[:, :1] * x.reshape(1, -1) + b[:, None]).astype(np.float32).astype(np.float64).reshape((29,) + x.shape[1:])
        return y[:4], y[4:8], y[8:]
    want = cso.weighted(windows, ijk, pipe.cube_shape, gs, pad, ops.overlap_window(window, gs, pad),
                        codes or (0,), f, keep)
    for k in ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_probability'):
        assert np.abs(got[k] - want[k]).max() <= 1e-5, k


# ------------------------------------------------------------------------------------------ split maps
@pytest.mark.parametrize('world', [2, 3, 8])
@pytest.mark.parametrize('dtype', ['float32', 'int16'])
def test_slab_ranks_equal_one_gpu(cuda, world, dtype):
    gs, pad = 16, 8
    if dtype == 'float32':
        src_shape, voxel = (136, 24, 20), 1.0
        src = _masked_map(src_shape, 13, frac=0.25)
    else:
        src_shape, voxel = (120, 20, 18), 1.1
        src = (_int16_map(src_shape, seed=13) * _ellipsoid(src_shape, 0.25)).astype(np.int16)
    hdr = MapHeader(voxel_size=(np.float32(voxel),) * 3)
    d_src = torch.from_numpy(src).to(cuda)
    model = PointwiseModel(seed=2).to(cuda)
    single = MapPipeline(cuda, gs, pad, batch_cubes=4)
    assert single.resample_and_normalize(d_src, hdr)
    with torch.no_grad():
        want = single.predict_and_stitch(model, min_max=T).as_dict()
        full = single.predict_and_stitch(model).as_dict()
    assert not torch.equal(want['backbone_probability'], full['backbone_probability'])    # some cube was skipped

    plan = SlabPlan(src_shape, hdr.voxel_size, gs, pad, world, dtype=d_src.dtype)
    nz, ny, nx = plan.out_shape
    pipes = [SlabPipeline(cuda, r, world, gs, pad, batch_cubes=4, global_src_shape=src_shape, group=False)
             for r in range(world)]
    res, owned = [], []
    for p in pipes:
        me = plan.ranks[p.rank]
        p._exchange = lambda own, me=me: d_src[me.src_lo:me.src_hi].contiguous()
        r_, o_ = p.slab_resample(d_src[me.own_lo:me.own_hi].contiguous(), hdr)
        res.append(r_)
        owned.append(o_)
    for p, r_, s in zip(pipes, res, _lockstep(owned, nz * ny * nx)):
        p.stats = s
        p.slab_normalize(r_)
        assert p.check_status()
    with torch.no_grad():
        for p in pipes:
            vols = p.predict_and_stitch(model, min_max=T)
            (_, _, o2), (_, _, e2) = p.box
            for k, t in vols.as_dict().items():
                assert torch.equal(t, want[k][..., o2:o2 + e2]), (p.rank, k)


@pytest.mark.parametrize('world', [2, 3, 8])
def test_balanced_cube_ranks_equal_one_gpu(cuda, world):
    gs, pad = 16, 8
    d_src = _dev(_masked_map((48, 40, 96), 21, frac=0.25), cuda)
    model = PointwiseModel(seed=1).to(cuda)
    single = MapPipeline(cuda, gs, pad, batch_cubes=5)
    assert single.resample_and_normalize(d_src, HDR)
    with torch.no_grad():
        want = single.predict_and_stitch(model, min_max=T, model_batch=2, d8='split').as_dict()
    single.cube_index()
    n_kept = len(ops.select_cubes(single._window_max(single.ijk), T))
    pipes = [BalancedCubePipeline(cuda, r, world, gs, pad, batch_cubes=5, group=False) for r in range(world)]
    for p in pipes:
        assert p.resample_and_normalize(d_src, HDR)
        p.cube_index()
    assert n_kept < len(ops.cube_origins(pipes[0].cube_shape, gs))
    groups = PeerVolumes.emulate(cuda, world, pipes[0]._n_max())
    vols = []
    for p, g_ in zip(pipes, groups):
        p.peer_volumes = g_
        vols.append(p._new_volumes())
        vols[-1].block.fill_(7.0)                      # as if it held another map: the owner clears skipped cores
    with torch.no_grad():
        for p, v in zip(pipes, vols):
            p.predict_and_stitch(model, v, model_batch=2, d8='split', min_max=T)
    for p in pipes:
        p.finish_map()
        assert sum(p.cubes_per_rank) == n_kept and max(p.cubes_per_rank) - min(p.cubes_per_rank) <= 1
    for r, (p, v) in enumerate(zip(pipes, vols)):
        x0, x1 = p.x_bounds[r], p.x_bounds[r + 1]
        for k, t in v.as_dict().items():
            ref = want[k][:, x0:x1] if want[k].dim() == 4 else want[k][x0:x1]
            assert torch.equal(t, ref), (r, k)
    groups[0].close()


# ------------------------------------------------------------------------------------------ drop-in
@pytest.fixture
def _clean(monkeypatch):
    monkeypatch.delenv('MICA_DEVICES', raising=False)
    monkeypatch.delenv('MICA_MIN_MAX', raising=False)
    session.clear()
    yield monkeypatch
    session.clear()


def _grids(tmp_path, min_max=T, materialize=False, shape=(96, 96, 96)):
    """DataPreprocessor -> GridCreator(grid_size=16, padding=8, min_max=) on a masked map, without atoms (a file
    source then matches the resident one: both have zero AF3 features).  Returns (grids path, result, normalised
    map as NumPy)."""
    case = tmp_path / 'input' / 'ID'
    os.makedirs(case / 'AF3_results', exist_ok=True)
    map_path = str(case / 'map.mrc')
    mrc.write_mrc(map_path, mrc.MrcMap(data=_masked_map(shape, 5), voxel_size=(np.float32(1.0),) * 3))
    dp = DataPreprocessor(map_path=map_path, AF3_results=str(case / 'AF3_results'), quiet=True)
    dp.resample_and_normalize_map()
    grids = str(case / 'grids') + '/'
    r = GridCreator(quiet=True, materialize=materialize, min_max=min_max).create_normalized_map_grids(
        dp.normalized_map_path, os.path.join(grids, 'normalized_map_grids'), 16, 8)
    norm = session.get(dp.normalized_map_path)['volume'].cpu().numpy()
    return grids, r, norm, dp


def _run(grids, out, model, **kw):
    pr = CryoEMPredictor('unused', grids, str(out), save_output=False, quiet=True, model=model, host_volumes=MAP_TYPES,
                         release_inputs=False, super_batch=20, **kw)
    ok, vols = pr.run_prediction()
    assert ok
    return pr, vols


def test_dropin_materialize_routes_and_devices(cuda, tmp_path, _clean):
    grids, r, norm, _ = _grids(tmp_path, materialize=True)
    mx, meta, _ = cso.window_maxima(norm, grid_size=16, padding=8)
    keep = cso.kept(mx, T)
    assert r['success'] and r['grid_count'] == keep.sum() and 0 < keep.sum() < len(keep)
    names = sorted(os.path.basename(f) for f in glob.glob(os.path.join(grids, 'normalized_map_grids', '*.npz')))
    assert names == sorted(f'normalized_map_grid_i{i}_j{j}_k{k}.npz' for i, j, k, *_ in meta[keep])

    m1 = CountingModel().to(cuda)
    p1, v1 = _run(grids, tmp_path / 'o1', m1)
    assert m1.cubes == keep.sum() and p1.sample_count == keep.sum()
    assert p1.use_optimized_batching == (keep.sum() > 200)
    _, v3 = _run(grids, tmp_path / 'o3', PointwiseModel().to(cuda), devices=EMULATED)
    _assert_same(v1, v3)
    _, vt1 = _run(grids, tmp_path / 't1', PointwiseModel().to(cuda), tta='flips', overlap_window='triangle')
    _, vt3 = _run(grids, tmp_path / 't3', PointwiseModel().to(cuda), tta='flips', overlap_window='triangle',
                  devices=EMULATED)
    _assert_same(vt1, vt3)
    mr = CountingModel().to(cuda)
    _, vr = _run(grids, tmp_path / 'or', mr, reference_batching=True)
    _assert_same(v1, vr)
    files = glob.glob(os.path.join(grids, 'normalized_map_grids', '*.npz'))           # the reference's glob order
    assert np.allclose(mr.sums, [np.load(f)['grid'].astype(np.float64).sum() for f in files], rtol=1e-6, atol=1e-6)

    # the oracle's paste over the kept cubes, logits from the same model
    core = _core_mask(tuple(norm.shape[::-1]), 16, meta[keep][:, :3])
    full = {k: np.asarray(v) for k, v in v1.items()}
    for k in MAP_TYPES:
        assert not full[k][..., ~core].any(), k

    session.clear()                                    # the reference's files alone
    mf = CountingModel().to(cuda)
    _, vf = _run(grids, tmp_path / 'of', mf)
    assert mf.cubes == keep.sum()
    _assert_same(v1, vf)
    _, vf3 = _run(grids, tmp_path / 'of3', PointwiseModel().to(cuda), devices=EMULATED)
    _assert_same(v1, vf3)

    from oracle import ref_harness
    if not ref_harness.available():
        return
    ref_harness._setup_path()
    from utils.predict import CryoEMPredictor as RefPredictor
    with ref_harness._quiet():
        rp = RefPredictor(model_path='unused', grids_path=grids, output_path=str(tmp_path / 'ref'),
                          save_output=False, device='cpu', quiet=True)
        rp.logger.disabled = True
        assert rp.select_processing_strategy()
        rp.model = PointwiseModel()
        good, loader = rp.prepare_data()
        assert good and rp.run_inference(loader)
        good, want = rp.reconstruct_and_save_volumes()
    assert good
    for k in ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_probability'):
        assert np.abs(np.asarray(v1[k]) - want[k]).max() <= 1e-5, k


def test_dropin_env_knob_and_refusals(cuda, tmp_path, _clean):
    grids, r, _, dp = _grids(tmp_path / 'arg')
    want = session.get(os.path.join(grids, 'normalized_map_grids'))['ijk']
    _clean.setenv('MICA_MIN_MAX', '0.01')
    out = os.path.join(str(tmp_path), 'env', 'normalized_map_grids')
    r2 = GridCreator(quiet=True).create_normalized_map_grids(dp.normalized_map_path, out, 16, 8)
    assert r2['success'] and r2['grid_count'] == r['grid_count']
    assert np.array_equal(session.get(out)['ijk'], want)
    _clean.setenv('MICA_MIN_MAX', '')
    r3 = GridCreator(quiet=True).create_normalized_map_grids(dp.normalized_map_path, out, 16, 8)
    assert r3['grid_count'] == 216
    n0 = ops.launch_count()
    for bad in (float('nan'), float('inf'), 'x', True):
        rb = GridCreator(quiet=True, min_max=bad).create_normalized_map_grids(dp.normalized_map_path, out, 16, 8)
        assert not rb['success']
    for text in ('nan', 'inf', 'abc'):
        _clean.setenv('MICA_MIN_MAX', text)
        rb = GridCreator(quiet=True).create_normalized_map_grids(dp.normalized_map_path, out, 16, 8)
        assert not rb['success']
    assert ops.launch_count() == n0
    _clean.delenv('MICA_MIN_MAX')
    rz = GridCreator(quiet=True, min_max=2.0).create_normalized_map_grids(dp.normalized_map_path, out, 16, 8)
    assert not rz['success'] and rz['grid_count'] == 0
