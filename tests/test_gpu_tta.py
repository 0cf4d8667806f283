"""Test-time augmentation over the cube's 48 orientations (NOT the reference's arithmetic): the oriented map extract
and AF3 fill equal the NumPy-oriented plain windows bit for bit, the oriented accumulate matches the float64
statement of oracle/tta_oracle.py, and a TTA run gives the same bits whatever the batches, the orientation order or
the partition -- z-slabs, balanced cubes, several workers of the drop-in."""
import numpy as np
import pytest
import torch

from mica_b200 import _lib, ops, session, synthetic
from mica_b200.pdb import channel_codes
from mica_b200.peer import PeerVolumes
from mica_b200.pipeline import MapHeader, MapPipeline
from mica_b200.predict import CryoEMPredictor, MAP_TYPES
from mica_b200.slab import BalancedCubePipeline, SlabPipeline, SlabPlan
from oracle import tta_oracle as tto

from test_gpu_devices import EMULATED, _assert_same, _drop_in, _predict
from test_gpu_overlap_split import WindowModel, _int16_map, _lockstep

pytestmark = pytest.mark.gpu

ALL = tuple(range(48))
HDR = MapHeader(voxel_size=(np.float32(1.0),) * 3)


class PointwiseModel(torch.nn.Module):
    """A 1x1x1 convolution (25 -> 29 channels, float32 on CUDA cores): it commutes with every orientation."""

    def __init__(self, seed=0):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.register_buffer('A', torch.randn((29, 25), generator=g, dtype=torch.float64))
        self.register_buffer('b', torch.randn(29, generator=g, dtype=torch.float64))

    def forward(self, x, af):
        inp = torch.cat([x, af], 1)
        y = (self.A.float()[None, :, :, None, None, None] * inp[:, None]).sum(2)
        y = y + self.b.float()[None, :, None, None, None]
        return y[:, :4], y[:, 4:8], y[:, 8:]


def _dev(a, cuda):
    return torch.from_numpy(np.ascontiguousarray(a)).to(cuda)


def _orient_t(t, g):
    return torch.from_numpy(np.ascontiguousarray(ops.orient_array(t.cpu().numpy(), g)))


# ------------------------------------------------------------------------------------------------ extract
@pytest.mark.parametrize('case', ['tma', 'fallback', 'slab', 'perm'])
def test_oriented_extract_all_codes(cuda, case):
    gs, pad, perm = 16, 8, ops.STANDARD_PERM
    vol = synthetic.synthetic_map((37, 41, 44), voxel=1.0, seed=3)       # (nz, ny, nx), nx % 4 == 0: TMA eligible
    kw = {}
    if case == 'fallback':
        gs, pad = 12, 3                                                  # W = 18: no TMA
    if case == 'perm':
        perm = (0, 2, 1)
    cube_shape = ops.cube_space_shape(vol.shape, perm)
    ijk = _dev(ops.cube_origins(cube_shape, gs), cuda)
    src = _dev(vol, cuda)
    if case == 'slab':                                                   # planes [9, 30) of the map on this rank
        src, kw = _dev(vol[9:30], cuda), dict(global_nz=vol.shape[0], z0=9)
    nz0 = torch.empty(len(ijk), dtype=torch.int32, device=cuda)
    mx0 = torch.empty(len(ijk), dtype=torch.float32, device=cuda)
    plain = ops.extract_cubes(src, ijk, gs, pad, perm, nonzero=nz0, cube_max=mx0, **kw)
    path0 = _lib.lib.mica_last_extract_path()
    if case == 'tma':
        assert path0 == 2
    for g in ALL:
        nz = torch.empty_like(nz0)
        mx = torch.empty_like(mx0)
        got = ops.extract_cubes(src, ijk, gs, pad, perm, nonzero=nz, cube_max=mx, orient=g, **kw)
        assert _lib.lib.mica_last_extract_path() == (path0 if g == 0 else 3)
        assert torch.equal(got.cpu(), _orient_t(plain, g)), g
        assert torch.equal(nz, nz0) and torch.equal(mx, mx0), g


# ------------------------------------------------------------------------------------------------ AF3 fill
def test_oriented_af3_fill_and_slot_reuse(cuda):
    gs, pad, perm = 16, 8, ops.STANDARD_PERM
    shape = (40, 36, 44)
    st = synthetic.synthetic_structure(300, shape[::-1], seed=8)
    bb_ch, aa_ch = channel_codes(st['atom_names'], st['res_names'])
    atoms = tuple(_dev(a, cuda) for a in (st['coords'], bb_ch, aa_ch))
    dense, status = ops.af3_encode(*atoms, (0, 0, 0), shape)
    assert int(status.item()) == 0
    cube_shape = ops.cube_space_shape(shape, perm)
    ijk = _dev(ops.cube_origins(cube_shape, gs), cuda)
    filler = ops.Af3CubeFiller(cuda, 8, gs, pad, perm)
    filler.bin(*atoms, (0, 0, 0), shape)
    # the same cubes in a new orientation, new cubes in the same one, fewer cubes, back to 0
    steps = [(0, 8, 0), (0, 8, 5), (0, 8, 30), (8, 16, 30), (8, 14, 47), (3, 11, 0), (0, 8, 13), (1, 3, 13)]
    for b0, b1, g in steps:
        sub = ijk[b0:b1].contiguous()
        nz = torch.empty(b1 - b0, dtype=torch.int32, device=cuda)
        want_nz = torch.empty_like(nz)
        got = filler.fill(sub, nz, orient=g)
        want = ops.extract_cubes(dense, sub, gs, pad, perm, nonzero=want_nz, orient=g)
        assert torch.equal(got, want), (b0, b1, g)
        assert torch.equal(nz, want_nz), (b0, b1, g)
        assert filler.buffer[b1 - b0:].abs().sum().item() == 0            # the other slots stay clean
    filler.clear()
    assert filler.buffer.abs().sum().item() == 0


# ------------------------------------------------------------------------------------------------ accumulate
@pytest.mark.parametrize('gs,pad,window', [(16, 8, 'triangle'), (8, 2, 'uniform'), (16, 8, 'core')])
def test_stitcher_tta_against_the_float64_statement(cuda, gs, pad, window):
    W = gs + 2 * pad
    cube_shape = (37, 21, 30)
    ijk = ops.cube_origins(cube_shape, gs)
    rng = np.random.default_rng(gs)
    windows = rng.standard_normal((len(ijk), 1, W, W, W)).astype(np.float32)
    A, P = rng.standard_normal((29, W, W, W)), 2 * rng.standard_normal((29, W, W, W))

    def model(x):                                                        # position-dependent: TTA really averages
        y = (x[0][None] * A + P).astype(np.float32).astype(np.float64)
        return y[:4], y[4:8], y[8:]
    codes = (0, 1, 5, 10, 19, 30, 47)                                    # fastest axis kept, reversed, and moved
    st = ops.Stitcher(cube_shape, cuda, gs, pad, window, tta=codes)
    ij = _dev(ijk.astype(np.int32), cuda)
    for g in codes:
        logits = np.stack([np.concatenate(model(ops.orient_array(w, g).astype(np.float64))) for w in windows])
        t = _dev(logits.astype(np.float32), cuda)
        st(t[:, :4].contiguous(), t[:, 4:8].contiguous(), t[:, 8:].contiguous(), ij, orient=g)
    got = {k: v.cpu().numpy() for k, v in st.finalize().as_dict().items()}
    want = tto.tta_stitch(windows.astype(np.float64), ijk, cube_shape, gs, pad, ops.overlap_window(window, gs, pad),
                          codes, model)
    for k in ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_probability'):
        assert np.abs(got[k] - want[k]).max() <= 1e-5, k
    p = np.sort(want['amino_acid_probability'], axis=0)
    clear = (p[-1] - p[-2]) > 4e-6
    assert np.array_equal(got['amino_acid_prediction'][clear], want['amino_acid_prediction'][clear])


# ------------------------------------------------------------------------------------------------ pipeline
def _pipe(cuda, gs=16, pad=8, batch=5, seed=21, shape=(40, 36, 44)):
    src = synthetic.synthetic_map(shape, voxel=1.0, seed=seed)
    st = synthetic.synthetic_structure(200, shape[::-1], seed=seed)
    bb_ch, aa_ch = channel_codes(st['atom_names'], st['res_names'])
    atoms = tuple(_dev(a, cuda) for a in (st['coords'], bb_ch, aa_ch))
    pipe = MapPipeline(cuda, gs, pad, batch_cubes=batch)
    assert pipe.resample_and_normalize(_dev(src, cuda), HDR) and pipe.encode_af3(*atoms)
    return pipe


def _run(pipe, model, **kw):
    with torch.no_grad():
        return {k: v.clone() for k, v in pipe.predict_and_stitch(model, **kw).as_dict().items()}


def _same(a, b):
    for k in MAP_TYPES:
        assert torch.equal(a[k], b[k]), k


def test_identity_only_is_no_tta(cuda):
    pipe = _pipe(cuda)
    model = WindowModel(32).to(cuda)
    _same(_run(pipe, model, tta=[0]), _run(pipe, model))
    _same(_run(pipe, model, tta=[0], overlap_window='triangle'), _run(pipe, model, overlap_window='triangle'))


def test_equivariant_model_all_orientations(cuda):
    pipe = _pipe(cuda)
    model = PointwiseModel().to(cuda)
    want = _run(pipe, model)
    got = _run(pipe, model, tta='all', model_batch=2, d8='split')
    for k in ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_probability'):
        assert (got[k] - want[k]).abs().max().item() <= 1e-6, k
    w = want['amino_acid_probability'].sort(0).values
    clear = (w[-1] - w[-2]) > 1e-5
    assert torch.equal(got['amino_acid_prediction'][clear], want['amino_acid_prediction'][clear])


def test_order_and_batches_do_not_matter(cuda):
    model = WindowModel(32, seed=2).to(cuda)
    pipe = _pipe(cuda, batch=5)
    want = _run(pipe, model, tta='flips', overlap_window='uniform')
    order = list(np.random.default_rng(3).permutation(8))
    _same(_run(pipe, model, tta=[int(g) for g in order], overlap_window='uniform'), want)
    pipe.prefetch = False
    _same(_run(pipe, model, tta='flips', overlap_window='uniform'), want)
    _same(_run(_pipe(cuda, batch=7), model, tta=order[::-1], overlap_window='uniform'), want)
    rot = _run(pipe, model, tta='rot90')
    assert not torch.equal(rot['backbone_probability'], want['backbone_probability'])


@pytest.mark.parametrize('world', [2, 3])
@pytest.mark.parametrize('dtype', ['float32', 'int16'])
def test_slab_ranks_equal_one_gpu(cuda, world, dtype):
    gs, pad, codes = 16, 8, (0, 3, 21, 46)
    if dtype == 'float32':
        src_shape, voxel = (136, 24, 20), 1.0
        src = synthetic.synthetic_map(src_shape, voxel=voxel, seed=13)
    else:
        src_shape, voxel = (120, 20, 18), 1.1
        src = _int16_map(src_shape, seed=13)
    hdr = MapHeader(voxel_size=(np.float32(voxel),) * 3)
    d_src = torch.from_numpy(src).to(cuda)
    model = WindowModel(gs + 2 * pad).to(cuda)
    single = MapPipeline(cuda, gs, pad, batch_cubes=4)
    assert single.resample_and_normalize(d_src, hdr)
    want = _run(single, model, tta=codes)
    plan = SlabPlan(src_shape, hdr.voxel_size, gs, pad, world, dtype=d_src.dtype)
    nz, ny, nx = plan.out_shape
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
    for p in pipes:
        p.cube_index()
        vols.append(p._exported_volumes(p._n_max()))
    with torch.no_grad():
        for p, v in zip(pipes, vols):
            p.predict_and_stitch(model, v, tta=codes)
    for p in pipes:
        p.finish_map()
    for p, v in zip(pipes, vols):
        (_, _, o2), (_, _, e2) = p.box
        for k, t in v.as_dict().items():
            assert torch.equal(t, want[k][..., o2:o2 + e2]), (p.rank, k)
    groups[0].close()


def test_balanced_cube_ranks_equal_one_gpu(cuda):
    world, gs, pad = 2, 16, 8
    single = _pipe(cuda, gs, pad, batch=5)
    model = WindowModel(gs + 2 * pad, seed=1).to(cuda)
    want = _run(single, model, tta='flips', model_batch=2, d8='split')
    src = synthetic.synthetic_map((40, 36, 44), voxel=1.0, seed=21)
    st = synthetic.synthetic_structure(200, (44, 36, 40), seed=21)
    bb_ch, aa_ch = channel_codes(st['atom_names'], st['res_names'])
    atoms = tuple(_dev(a, cuda) for a in (st['coords'], bb_ch, aa_ch))
    pipes = [BalancedCubePipeline(cuda, r, world, gs, pad, batch_cubes=5, group=False) for r in range(world)]
    for p in pipes:
        assert p.resample_and_normalize(_dev(src, cuda), HDR) and p.encode_af3(*atoms)
        p.cube_index()
    groups = PeerVolumes.emulate(cuda, world, pipes[0]._n_max())
    vols = []
    for p, g_ in zip(pipes, groups):
        p.peer_volumes = g_
        vols.append(p._new_volumes())
    with torch.no_grad():
        for p, v in zip(pipes, vols):
            p.predict_and_stitch(model, v, model_batch=2, d8='split', tta='flips')
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


def test_dropin_workers_equal_one_device(cuda, tmp_path, _clean_session):
    grids, n = _drop_in(tmp_path, materialize=True)
    W = 16 + 2 * 8
    _, v1 = _predict(grids, tmp_path / 'o1', WindowModel(W).to(cuda), tta='flips')
    _, v2 = _predict(grids, tmp_path / 'o2', WindowModel(W).to(cuda), tta='flips', devices=['cuda:0'] * 2)
    _, v3 = _predict(grids, tmp_path / 'o3', WindowModel(W).to(cuda), tta='flips', devices=EMULATED)
    _assert_same(v1, v2)
    _assert_same(v1, v3)
    _, vd = _predict(grids, tmp_path / 'od', WindowModel(W).to(cuda))
    _, v0 = _predict(grids, tmp_path / 'o0', WindowModel(W).to(cuda), tta=[0])
    _assert_same(vd, v0)
    assert not np.array_equal(np.asarray(vd['backbone_probability']), np.asarray(v1['backbone_probability']))
    # the reference's per-cube files hold no volume to cut oriented cubes from: logged, (False, {})
    session.clear()
    pr = CryoEMPredictor('unused', grids, str(tmp_path / 'of'), save_output=False, quiet=True,
                         model=WindowModel(W).to(cuda), release_inputs=False, tta='flips')
    assert pr.run_prediction() == (False, {})


def test_tta_refusals_launch_nothing(cuda, tmp_path, _clean_session):
    pipe = _pipe(cuda)
    pipe.cube_index()
    model = WindowModel(32).to(cuda)
    torch.cuda.synchronize()
    for bad in ('rot', [0, 0], [48], [], [1.5], 'ALL'):
        n0 = ops.launch_count()
        with pytest.raises(_lib.MicaError):
            pipe.predict_and_stitch(model, tta=bad)
        with pytest.raises(_lib.MicaError):
            ops.Stitcher(pipe.cube_shape, cuda, 16, 8, 'core', tta=bad)
        assert ops.launch_count() == n0
    x = torch.zeros((4, 4, 4), device=cuda)
    ijk = torch.zeros((1, 3), dtype=torch.int32, device=cuda)
    n0 = ops.launch_count()
    for g in (48, -1, True):
        with pytest.raises(_lib.MicaError):
            ops.extract_cubes(x, ijk, 2, 1, orient=g)
    st = ops.Stitcher(pipe.cube_shape, cuda, 16, 8, 'core', tta='flips')
    n1 = ops.launch_count()
    t = torch.zeros((1, 4, 32, 32, 32), device=cuda)
    with pytest.raises(_lib.MicaError):
        st(t, t, torch.zeros((1, 21, 32, 32, 32), device=cuda), ijk, orient=9)              # not one of 'flips'
    assert ops.launch_count() == n1
    grids, _ = _drop_in(tmp_path)
    n0 = ops.launch_count()
    pr = CryoEMPredictor('unused', grids, str(tmp_path / 'o'), save_output=False, quiet=True, model=model,
                         release_inputs=False, tta='mirror')
    assert pr.run_prediction() == (False, {})
    assert ops.launch_count() == n0
