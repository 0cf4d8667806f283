"""Overlap-weighted stitching (``ops.Stitcher``, NOT the reference's arithmetic; DESIGN.md D2) is order free:
the same bits whatever the batch, the cube order or the partition -- z-slabs, balanced cubes, several workers of
the drop-in -- and within TOL of the float64 NumPy statement.  The stand-in model gives every position of a window
its own logits, so a voxel covered by several windows really averages different values."""
import ctypes as C

import numpy as np
import pytest
import torch

from mica_b200 import _lib, ops, session, synthetic
from mica_b200.peer import PeerVolumes
from mica_b200.pipeline import MapHeader, MapPipeline
from mica_b200.predict import CryoEMPredictor, MAP_TYPES
from mica_b200.slab import BalancedCubePipeline, SlabPipeline, SlabPlan
from oracle import mica_oracle as orc

from test_gpu_devices import EMULATED, _assert_same, _drop_in, _predict

pytestmark = pytest.mark.gpu

TOL = 1e-5
CHANNELS = (4, 4, 21)


class WindowModel(torch.nn.Module):
    """logits = x * A + P with A, P fixed random per channel and window position: elementwise (no batch coupling),
    different at one voxel for every window that covers it."""

    def __init__(self, W, seed=0):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        for n, c in zip(('bb', 'ca', 'aa'), CHANNELS):
            self.register_buffer(f'a_{n}', torch.randn((c, W, W, W), generator=g))
            self.register_buffer(f'p_{n}', 2 * torch.randn((c, W, W, W), generator=g))

    def forward(self, x, af):
        return tuple(x * getattr(self, f'a_{n}') + getattr(self, f'p_{n}') for n in ('bb', 'ca', 'aa'))


def _dev(a, cuda):
    return torch.from_numpy(np.ascontiguousarray(a)).to(cuda)


def _lattice_logits(cube_shape, gs, pad, cuda, seed=3):
    ijk = ops.cube_origins(cube_shape, gs)
    bb, ca, aa = synthetic.synthetic_logits(len(ijk), gs + 2 * pad, seed=seed)
    return ijk, (bb, ca, aa)


def _stitch(cube_shape, gs, pad, window, cuda, logits, ijk, order, batch):
    st = ops.Stitcher(cube_shape, cuda, gs, pad, window)
    d = [_dev(a[order], cuda) for a in logits]
    ij = _dev(ijk[order].astype(np.int32), cuda)
    for b0 in range(0, len(order), batch):
        st(d[0][b0:b0 + batch], d[1][b0:b0 + batch], d[2][b0:b0 + batch], ij[b0:b0 + batch])
    return st.finalize().as_dict()


@pytest.mark.parametrize('cube_shape,gs,pad', [((70, 33, 50), 32, 16), ((21, 13, 9), 8, 2)])
@pytest.mark.parametrize('window', ['uniform', 'triangle'])
def test_stitcher_result_does_not_depend_on_batches_or_cube_order(cuda, cube_shape, gs, pad, window):
    ijk, logits = _lattice_logits(cube_shape, gs, pad, cuda)
    n = len(ijk)
    ref = _stitch(cube_shape, gs, pad, window, cuda, logits, ijk, np.arange(n), n)
    perm = np.random.default_rng(7).permutation(n)
    for order, batch in ((np.arange(n), 1), (np.arange(n), 3), (perm, n), (perm, 2)):
        got = _stitch(cube_shape, gs, pad, window, cuda, logits, ijk, order, batch)
        for k in MAP_TYPES:
            assert torch.equal(got[k], ref[k]), (k, batch)


@pytest.mark.parametrize('cube_shape,gs,pad', [((70, 33, 50), 32, 16), ((53, 21, 13), 48, 8), ((21, 13, 9), 8, 2)])
def test_stitcher_windows_against_the_float64_statement(cuda, cube_shape, gs, pad):
    ijk, (bb, ca, aa) = _lattice_logits(cube_shape, gs, pad, cuda, seed=11)
    meta = np.concatenate([ijk, np.minimum(gs, np.array(cube_shape)[None] - ijk)], axis=1).astype(np.int64)
    custom = (0.05 + np.random.default_rng(gs).random(gs + 2 * pad)).astype(np.float32)
    for window in ('uniform', 'triangle', custom):
        got = {k: v.cpu().numpy() for k, v in
               _stitch(cube_shape, gs, pad, window, cuda, (bb, ca, aa), ijk, np.arange(len(ijk)), 5).items()}
        w1 = ops.overlap_window(window, gs, pad)
        want = orc.postprocess_and_stitch_overlap(bb, ca, aa, meta, cube_shape, gs, pad, w1)
        for k in ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_probability'):
            assert np.abs(got[k] - want[k]).max() <= TOL, (k, window)
        p = np.sort(want['amino_acid_probability'], axis=0)
        clear = (p[-1] - p[-2]) > 4e-6
        assert np.array_equal(got['amino_acid_prediction'][clear], want['amino_acid_prediction'][clear])
        assert np.abs(got['amino_acid_probability'].sum(0) - 1).max() <= 1e-5


def _lockstep(owned, n_total):
    """The statistics every rank of a real group computes (histograms summed between hist and pick)."""
    lib, st = _lib.lib, C.c_void_p(torch.cuda.current_stream().cuda_stream)
    if owned[0].dtype in ops.INT_DTYPES:
        code = ops.MAP_DTYPES[owned[0].dtype]
        stats = [ops.IntOrderStats(o.device) for o in owned]
        for s, o in zip(stats, owned):
            _lib.check(lib.mica_int_stats_init(s._p, code, n_total, st))
            _lib.check(lib.mica_int_stats_hist(C.c_void_p(o.data_ptr()), code, o.numel(), s._p, st))
        total = sum(s.hist_view(owned[0].dtype).clone() for s in stats)
        for s in stats:
            s.hist_view(owned[0].dtype).copy_(total)
            _lib.check(lib.mica_int_stats_pick(s._p, code, st))
        return stats
    stats = [ops.OrderStats(o.device) for o in owned]
    for s in stats:
        _lib.check(lib.mica_select_init(s._p, n_total, st))
    for step in range(_lib.SELECT_PASSES):
        for s, o in zip(stats, owned):
            _lib.check(lib.mica_select_hist(C.c_void_p(o.data_ptr()), o.numel(), s._p, step, st))
        total = sum(s.hist_view().clone() for s in stats)
        for s in stats:
            s.hist_view().copy_(total)
            _lib.check(lib.mica_select_pick(s._p, step, st))
    return stats


def _int16_map(shape, seed):
    d = synthetic.synthetic_map(shape, seed=seed).astype(np.float64)
    d = (d - d.min()) / max(float(d.max() - d.min()), 1e-6)
    return np.round(-30000 + d * 60000).astype(np.int16)


@pytest.mark.parametrize('world', [2, 3, 8])
@pytest.mark.parametrize('dtype', ['float32', 'int16'])
def test_slab_ranks_equal_one_gpu(cuda, world, dtype):
    """Each rank adds the windows of its cubes -- reaching ``padding`` planes into its neighbours' slabs -- into
    the owners' blocks; after finish_map every rank's box equals the whole map's bit for bit."""
    gs, pad = 16, 8
    if dtype == 'float32':
        src_shape, voxel = (136, 24, 20), 1.0
        src = synthetic.synthetic_map(src_shape, voxel=voxel, seed=13)
    else:
        src_shape, voxel = (120, 20, 18), 1.1                     # a z line of 96..800 planes: the general path
        src = _int16_map(src_shape, seed=13)
    hdr = MapHeader(voxel_size=(np.float32(voxel),) * 3)
    d_src = torch.from_numpy(src).to(cuda)
    model = WindowModel(gs + 2 * pad).to(cuda)
    single = MapPipeline(cuda, gs, pad, batch_cubes=4)
    assert single.resample_and_normalize(d_src, hdr)
    with torch.no_grad():
        want = single.predict_and_stitch(model, overlap_window='triangle').as_dict()

    plan = SlabPlan(src_shape, hdr.voxel_size, gs, pad, world, dtype=d_src.dtype)
    nz, ny, nx = plan.out_shape
    assert all(r.out_hi > r.out_lo for r in plan.ranks)
    groups = PeerVolumes.emulate(cuda, world, max(r.out_hi - r.out_lo for r in plan.ranks) * nx * ny)
    pipes = [SlabPipeline(cuda, r, world, gs, pad, batch_cubes=4, global_src_shape=src_shape, group=False,
                          _peer_volumes=groups[r]) for r in range(world)]
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
    vols = []
    for p in pipes:                                           # every owner clears its block before anybody adds
        p.cube_index()
        vols.append(p._exported_volumes(p._n_max()))
    with torch.no_grad():
        for p, v in zip(pipes, vols):
            p.predict_and_stitch(model, v, overlap_window='triangle')
    for p in pipes:
        p.finish_map()
    for p, v in zip(pipes, vols):
        (_, _, o2), (_, _, e2) = p.box
        for k, t in v.as_dict().items():
            assert torch.equal(t, want[k][..., o2:o2 + e2]), (p.rank, k)
    groups[0].close()


@pytest.mark.parametrize('world', [2, 3, 8])
def test_balanced_cube_ranks_equal_one_gpu(cuda, world):
    from mica_b200.pdb import channel_codes
    gs, pad = 32, 16
    src = synthetic.synthetic_map((56, 40, 100), voxel=1.0, seed=21)
    hdr = MapHeader(voxel_size=(np.float32(1.0),) * 3)
    d_src = torch.from_numpy(src).to(cuda)
    st = synthetic.synthetic_structure(200, (100, 40, 56), seed=21)
    bb_ch, aa_ch = channel_codes(st['atom_names'], st['res_names'])
    atoms = tuple(torch.from_numpy(a).to(cuda) for a in (st['coords'], bb_ch, aa_ch))
    model = WindowModel(gs + 2 * pad, seed=1).to(cuda)
    single = MapPipeline(cuda, gs, pad, batch_cubes=5)
    with torch.no_grad():
        want = single.run(d_src, hdr, atoms, model, overlap_window='triangle').as_dict()
    _, Y, Z = single.cube_shape
    pipes = [BalancedCubePipeline(cuda, r, world, gs, pad, batch_cubes=5, group=False) for r in range(world)]
    for p in pipes:
        assert p.resample_and_normalize(d_src, hdr) and p.encode_af3(*atoms)
        p.cube_index()
    groups = PeerVolumes.emulate(cuda, world, pipes[0]._n_max())
    vols = []
    for p, g_ in zip(pipes, groups):
        p.peer_volumes = g_
        vols.append(p._new_volumes())
    with torch.no_grad():
        for p, v in zip(pipes, vols):
            p.predict_and_stitch(model, v, model_batch=2, d8='split', overlap_window='triangle')
    for p in pipes:
        p.finish_map()
    for r, (p, v) in enumerate(zip(pipes, vols)):
        x0, x1 = p.x_bounds[r], p.x_bounds[r + 1]
        for k, t in v.as_dict().items():
            ref = want[k][:, x0:x1] if want[k].dim() == 4 else want[k][x0:x1]
            assert torch.equal(t, ref), (r, k)
    groups[0].close()


@pytest.fixture
def _clean_session(monkeypatch):
    monkeypatch.delenv('MICA_DEVICES', raising=False)
    session.clear()
    yield
    session.clear()


def test_dropin_workers_and_sources_equal_one_device(cuda, tmp_path, _clean_session):
    grids, n = _drop_in(tmp_path, materialize=True)
    W = 16 + 2 * 8
    _, v1 = _predict(grids, tmp_path / 'o1', WindowModel(W).to(cuda), overlap_window='triangle')
    _, v3 = _predict(grids, tmp_path / 'o3', WindowModel(W).to(cuda), overlap_window='triangle', devices=EMULATED)
    _assert_same(v1, v3)
    _, vd = _predict(grids, tmp_path / 'od', WindowModel(W).to(cuda))
    _, vc = _predict(grids, tmp_path / 'oc', WindowModel(W).to(cuda), overlap_window='core')
    _assert_same(vd, vc)
    assert not np.array_equal(np.asarray(vd['backbone_probability']), np.asarray(v1['backbone_probability']))
    # the three small volumes on the host, amino_acid_probability left on the device: same values
    pr = CryoEMPredictor('unused', grids, str(tmp_path / 'os'), save_output=False, quiet=True,
                         model=WindowModel(W).to(cuda), release_inputs=False, super_batch=20,
                         overlap_window='triangle')
    ok, vs = pr.run_prediction()
    assert ok and not isinstance(vs['amino_acid_probability'], np.ndarray)
    _assert_same(v1, vs)
    # the reference's .npz files only: one device and three workers agree
    session.clear()
    _, f1 = _predict(grids, tmp_path / 'f1', WindowModel(W).to(cuda), overlap_window='uniform')
    session.clear()
    _, f3 = _predict(grids, tmp_path / 'f3', WindowModel(W).to(cuda), overlap_window='uniform', devices=EMULATED)
    _assert_same(f1, f3)
    assert np.abs(np.asarray(f1['amino_acid_probability']).sum(0) - 1).max() <= 1e-5


def test_stitcher_and_split_refusals(cuda, tmp_path, monkeypatch, _clean_session):
    gs, pad = 32, 16
    W = gs + 2 * pad
    bad_windows = [np.full(W, -1.0), np.r_[np.ones(W - 1), np.nan], np.ones(W + 1)]
    assert _lib.lib.mica_peer_atomics_supported(0, 0) == 1
    src = synthetic.synthetic_map((40, 44, 36), voxel=1.0, seed=9)
    pipe = MapPipeline(cuda, gs, pad, batch_cubes=3)
    assert pipe.resample_and_normalize(_dev(src, cuda), MapHeader(voxel_size=(np.float32(1.0),) * 3))
    torch.cuda.synchronize()
    for w in bad_windows:
        with pytest.raises(_lib.MicaError):
            ops.Stitcher((36, 44, 40), cuda, gs, pad, w)
        n0 = ops.launch_count()
        with pytest.raises(_lib.MicaError):
            pipe.predict_and_stitch(WindowModel(W).to(cuda), overlap_window=w)
        assert ops.launch_count() == n0                       # refused before any launch
    grids, _ = _drop_in(tmp_path)
    for w in [np.full(32, -1.0), np.r_[np.ones(31), np.nan], np.ones(5)]:
        pr = CryoEMPredictor('unused', grids, str(tmp_path / 'o'), save_output=False, quiet=True,
                             model=WindowModel(32).to(cuda), release_inputs=False, overlap_window=w)
        assert pr.run_prediction() == (False, {})
    # without native peer atomics a split run refuses, with a message that says so
    monkeypatch.setattr(ops, 'peer_atomics_supported', lambda a, b: False)
    pr = CryoEMPredictor('unused', grids, str(tmp_path / 'o'), save_output=False, quiet=True,
                         model=WindowModel(32).to(cuda), release_inputs=False, overlap_window='triangle',
                         devices=EMULATED)
    assert pr.run_prediction() == (False, {})
    p = BalancedCubePipeline(cuda, 0, 2, gs, pad, batch_cubes=3, group=False)
    assert p.resample_and_normalize(_dev(src, cuda), MapHeader(voxel_size=(np.float32(1.0),) * 3))
    p.cube_index()
    groups = PeerVolumes.emulate(cuda, 2, p._n_max())
    p.peer_volumes = groups[0]
    with pytest.raises(_lib.MicaError, match='native peer atomics'):
        p.predict_and_stitch(WindowModel(W).to(cuda), p._new_volumes(), overlap_window='triangle')
    groups[0].close()
