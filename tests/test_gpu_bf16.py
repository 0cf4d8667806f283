"""bfloat16 inference (``cube_dtype=torch.bfloat16``, ``CryoEMPredictor(precision='bf16')``): the bf16 extract and AF3
fill equal the float32 ones rounded to bf16 (flags from the float32 values) on every kernel route, the stitches with
bf16 logits equal the float32 stitches on ``logits.float()``, a bf16 pipeline equals a float32 one whose model rounds
its inputs to bf16 -- on one GPU and on split maps -- and the drop-in runs the model under bf16 autocast."""
import numpy as np
import pytest
import torch

from mica_b200 import _lib, ops, session, synthetic
from mica_b200.pdb import channel_codes
from mica_b200.peer import PeerVolumes
from mica_b200.pipeline import MapHeader, MapPipeline
from mica_b200.predict import CryoEMPredictor, MAP_TYPES
from mica_b200.slab import BalancedCubePipeline, SlabPipeline, SlabPlan
from oracle import mica_oracle

from test_gpu_cube_select import T, _grids, _masked_map
from test_gpu_devices import _assert_same
from test_gpu_overlap_split import _int16_map, _lockstep
from test_gpu_tta import PointwiseModel

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
HDR = MapHeader(voxel_size=(np.float32(1.0),) * 3)


def _dev(a, cuda):
    return torch.from_numpy(np.ascontiguousarray(a)).to(cuda)


def _assert_rounded(got, want32):
    """``got`` (bf16) is ``want32`` rounded to nearest even, NaN where it has NaN (NaN payloads may differ)."""
    assert got.dtype == BF16
    want = want32.cpu().to(BF16)                      # c10's bit-level round-to-nearest-even, subnormals kept
    got = got.cpu()
    gn, wn = torch.isnan(got), torch.isnan(want)
    assert torch.equal(gn, wn)
    assert torch.equal(got.masked_fill(gn, 0).view(torch.int16), want.masked_fill(wn, 0).view(torch.int16))


def _special_map(shape, seed):
    """A synthetic map with values that round to a tie, underflow, overflow or are NaN / -0 in bf16."""
    vol = synthetic.synthetic_map(shape, voxel=1.0, seed=seed).astype(np.float32)
    specials = [1 + 2 ** -8, 1 + 3 * 2 ** -8, -(1 + 2 ** -8), 1e-41, -1e-41, 3e-39, 3.3995e38, np.nan, -0.0,
                2 ** -133, 1.00390625 * 2 ** -126]
    rng = np.random.default_rng(seed)
    for v in specials:
        for _ in range(6):
            vol[tuple(int(rng.integers(0, n)) for n in shape)] = np.float32(v)
    return vol


# ------------------------------------------------------------------------------------------------ extract
@pytest.mark.parametrize('case,route', [('tma', 2), ('rows', 0), ('transpose0', 1), ('transpose1', 1),
                                        ('slab', 2), ('slab_rows', 0)])
def test_extract_equals_rounded_float32(cuda, case, route):
    gs, pad, perm = 16, 8, ops.STANDARD_PERM
    if case in ('rows', 'slab_rows'):
        perm = (0, 1, 2)
    if case == 'transpose0':
        gs, pad = 12, 3                                                  # W = 18: not the TMA kernel
    if case == 'transpose1':
        perm = (0, 2, 1)
    vol = _special_map((37, 41, 44), seed=3)
    cube_shape = ops.cube_space_shape(vol.shape, perm)
    ijk = _dev(ops.cube_origins(cube_shape, gs), cuda)
    src, kw = _dev(vol, cuda), {}
    if case.startswith('slab'):
        src, kw = _dev(vol[9:30], cuda), dict(global_nz=vol.shape[0], z0=9)
    W, B = gs + 2 * pad, len(ijk)
    nz32, mx32 = (torch.empty(B, dtype=t, device=cuda) for t in (torch.int32, torch.float32))
    nz16, mx16 = torch.empty_like(nz32), torch.empty_like(mx32)
    want = ops.extract_cubes(src, ijk, gs, pad, perm, nonzero=nz32, cube_max=mx32, **kw)
    assert _lib.lib.mica_last_extract_path() == route
    out = torch.empty((B, 1, W, W, W), dtype=BF16, device=cuda)
    got = ops.extract_cubes(src, ijk, gs, pad, perm, nonzero=nz16, cube_max=mx16, out=out, **kw)
    assert _lib.lib.mica_last_extract_path() == route and got is out
    _assert_rounded(got, want)
    assert torch.equal(nz16, nz32) and torch.equal(mx16.cpu(), mx32.cpu())
    # a channel slice of a larger buffer (the batch stride is not dense)
    big = torch.full((B, 3, W, W, W), 7.0, dtype=BF16, device=cuda)
    ops.extract_cubes(src, ijk, gs, pad, perm, out=big[:, 1:2], **kw)
    _assert_rounded(big[:, 1:2], want)
    assert (big[:, 0] == 7).all() and (big[:, 2] == 7).all()


@pytest.mark.parametrize('case', ['tma', 'slab'])
def test_oriented_extract_all_codes(cuda, case):
    gs, pad, perm = 16, 8, ops.STANDARD_PERM
    vol = _special_map((37, 41, 44), seed=4)
    ijk = _dev(ops.cube_origins(ops.cube_space_shape(vol.shape, perm), gs), cuda)
    src, kw = _dev(vol, cuda), {}
    if case == 'slab':
        src, kw = _dev(vol[9:30], cuda), dict(global_nz=vol.shape[0], z0=9)
    W, B = gs + 2 * pad, len(ijk)
    out = torch.empty((B, 1, W, W, W), dtype=BF16, device=cuda)
    for g in range(48):
        nz32, nz16 = (torch.empty(B, dtype=torch.int32, device=cuda) for _ in range(2))
        mx32, mx16 = (torch.empty(B, dtype=torch.float32, device=cuda) for _ in range(2))
        want = ops.extract_cubes(src, ijk, gs, pad, perm, nonzero=nz32, cube_max=mx32, orient=g, **kw)
        ops.extract_cubes(src, ijk, gs, pad, perm, nonzero=nz16, cube_max=mx16, orient=g, out=out, **kw)
        assert _lib.lib.mica_last_extract_path() == (2 if g == 0 else 3)
        _assert_rounded(out, want)
        assert torch.equal(nz16, nz32) and torch.equal(mx16.cpu(), mx32.cpu()), g


def test_bad_dtypes_are_refused_before_any_launch(cuda):
    vol = torch.zeros((8, 8, 8), device=cuda)
    ijk = torch.zeros((1, 3), dtype=torch.int32, device=cuda)
    n0 = ops.launch_count()
    for dt in (torch.float16, torch.float64):
        with pytest.raises(_lib.MicaError):
            ops.extract_cubes(vol, ijk, 8, 0, out=torch.zeros((1, 1, 8, 8, 8), dtype=dt, device=cuda))
        lg = torch.zeros((1, 4, 8, 8, 8), dtype=dt, device=cuda)
        with pytest.raises(_lib.MicaError):
            ops.postproc_stitch(lg, lg, torch.zeros((1, 21, 8, 8, 8), dtype=dt, device=cuda), ijk,
                                ops.StitchedVolumes((8, 8, 8), cuda), 8, 0)
    lg32 = torch.zeros((1, 4, 8, 8, 8), device=cuda)
    with pytest.raises(_lib.MicaError):                                   # mixed dtypes
        ops.postproc_stitch(lg32, lg32.to(BF16), torch.zeros((1, 21, 8, 8, 8), device=cuda), ijk,
                            ops.StitchedVolumes((8, 8, 8), cuda), 8, 0)
    with pytest.raises(_lib.MicaError):
        MapPipeline(cuda, cube_dtype=torch.float16)
    pipe = MapPipeline(cuda)
    with pytest.raises(_lib.MicaError):
        pipe.configure(cube_dtype=torch.float16)
    assert pipe.cube_dtype == torch.float32
    assert ops.launch_count() == n0


# ------------------------------------------------------------------------------------------------ AF3 fill
def _atoms(shape, cuda, n=300, seed=8):
    st = synthetic.synthetic_structure(n, shape[::-1], seed=seed)
    bb_ch, aa_ch = channel_codes(st['atom_names'], st['res_names'])
    return tuple(_dev(a, cuda) for a in (st['coords'], bb_ch, aa_ch))


def test_af3_fill_through_slot_switches_and_dense_mode(cuda):
    gs, pad, perm = 16, 8, ops.STANDARD_PERM
    shape = (40, 36, 44)
    atoms = _atoms(shape, cuda)
    ijk = _dev(ops.cube_origins(ops.cube_space_shape(shape, perm), gs), cuda)
    f32 = ops.Af3CubeFiller(cuda, 8, gs, pad, perm)
    f16 = ops.Af3CubeFiller(cuda, 8, gs, pad, perm, dtype=BF16)
    f32.bin(*atoms, (0, 0, 0), shape)
    f16.share_bins(f32)
    steps = [(0, 8, 0), (0, 8, 5), (0, 8, 30), (8, 16, 30), (8, 14, 47), (3, 11, 0), (0, 8, 13), (1, 3, 13), (2, 9, 0)]
    for b0, b1, g in steps:
        sub = ijk[b0:b1].contiguous()
        n32, n16 = (torch.empty(b1 - b0, dtype=torch.int32, device=cuda) for _ in range(2))
        want = f32.fill(sub, n32, orient=g)
        got = f16.fill(sub, n16, orient=g)
        assert got.dtype == BF16
        assert torch.equal(got.float(), want) and torch.equal(n16, n32), (b0, b1, g)
        assert f16.buffer[b1 - b0:].abs().sum().item() == 0
    f16.clear()
    assert f16.buffer.abs().sum().item() == 0

    # dense mode: the 24-channel volume cut into bf16 windows; and a pipeline switching dtype keeps its atom bins
    vol = synthetic.synthetic_map(shape, voxel=1.0, seed=2)
    pipes = {}
    for mode, dt in (('dense', torch.float32), ('dense', BF16), ('sparse', BF16)):
        p = MapPipeline(cuda, gs, pad, batch_cubes=6, af3_mode=mode, cube_dtype=dt)
        assert p.resample_and_normalize(_dev(vol, cuda), HDR) and p.encode_af3(*atoms)
        p.cube_index()
        pipes[mode, dt] = p
    sw = MapPipeline(cuda, gs, pad, batch_cubes=6)
    assert sw.resample_and_normalize(_dev(vol, cuda), HDR) and sw.encode_af3(*atoms)
    sw.cube_index()
    sw.extract_batch(0, 6)
    sw.configure(cube_dtype=BF16)
    for b0, b1, g in ((0, 6, 0), (6, 12, 5), (2, 5, 0)):
        x32, af32, n32 = pipes['dense', torch.float32].extract_batch(b0, b1, want_flags=True, orient=g)
        for key in (('dense', BF16), ('sparse', BF16)):
            x16, af16, n16 = pipes[key].extract_batch(b0, b1, want_flags=True, orient=g)
            _assert_rounded(x16, x32)
            assert af16.dtype == BF16 and torch.equal(af16.float(), af32) and torch.equal(n16, n32), (key, g)
        xs, afs = sw.extract_batch(b0, b1, orient=g)
        _assert_rounded(xs, x32)
        assert afs.dtype == BF16 and torch.equal(afs.float(), af32)


# ------------------------------------------------------------------------------------------------ stitches
def _bf16_logits(B, W, cuda, seed):
    g = torch.Generator(device='cpu').manual_seed(seed)
    out = []
    for c in (4, 4, 21):
        t = (3 * torch.randn((B, c, W, W, W), generator=g)).to(BF16)
        v, m = t.view(-1), (t.numel() - 1) // 997
        v[0:997 * m:997] = v[1:997 * m:997]                             # exact ties for the arg-max
        out.append(t.to(cuda))
    return out


def _np(vols):
    return {k: v.cpu().numpy() for k, v in vols.as_dict().items()}


@pytest.mark.parametrize('gs,pad', [(32, 16), (48, 8)])
def test_stitcher_paste_with_bf16_logits_equals_float32(cuda, gs, pad):
    W = gs + 2 * pad
    cube_shape = (70, 50, 90)
    ijk = _dev(ops.cube_origins(cube_shape, gs), cuda)
    B = len(ijk)
    bb, ca, aa = _bf16_logits(B, W, cuda, seed=gs)
    v16, v32 = ops.StitchedVolumes(cube_shape, cuda), ops.StitchedVolumes(cube_shape, cuda)
    ops.postproc_stitch(bb, ca, aa, ijk, v16, gs, pad)
    ops.postproc_stitch(bb.float(), ca.float(), aa.float(), ijk, v32, gs, pad)
    a, b = _np(v16), _np(v32)
    for k in MAP_TYPES:
        assert np.array_equal(a[k], b[k]), k
    # a Stitcher, switching dtype between calls
    v = ops.StitchedVolumes(cube_shape, cuda)
    call = ops.Stitcher(cube_shape, cuda, gs, pad, vols=v)
    h = B // 2
    call(bb[:h], ca[:h], aa[:h], ijk[:h])
    call(bb[h:].float(), ca[h:].float(), aa[h:].float(), ijk[h:])
    for k, t in _np(v).items():
        assert np.array_equal(t, b[k]), k
    # the peer form, owners along x: 2 and 3 emulated ranks, each block on this device
    X, Y, Z = cube_shape
    for bounds in ((0, 33, X), (0, 20, 21, X)):
        world = len(bounds) - 1
        blocks = {dt: [torch.zeros(23 * (bounds[r + 1] - bounds[r]) * Y * Z, device=cuda) for r in range(world)]
                  for dt in ('bf16', 'f32')}
        for dt, lg in (('bf16', (bb, ca, aa)), ('f32', (bb.float(), ca.float(), aa.float()))):
            table = torch.tensor([t.data_ptr() for t in blocks[dt]], dtype=torch.int64, device=cuda)
            ops.postproc_stitch_peer(*lg, ijk, cube_shape, table, bounds, gs, pad)
        for r in range(world):
            assert torch.equal(blocks['bf16'][r], blocks['f32'][r]), (bounds, r)
            vr = ops.StitchedVolumes.from_block(blocks['bf16'][r], cube_shape, (bounds[r], 0, 0),
                                                (bounds[r + 1] - bounds[r], Y, Z))
            for k, t in _np(vr).items():
                ref = b[k][:, bounds[r]:bounds[r + 1]] if t.ndim == 4 else b[k][bounds[r]:bounds[r + 1]]
                assert np.array_equal(t, ref), (bounds, r, k)


@pytest.mark.parametrize('window,tta', [('triangle', None), ('uniform', (0, 5, 30))])
def test_stitcher_accumulate_with_bf16_logits_equals_float32(cuda, window, tta):
    gs, pad = 16, 8
    W = gs + 2 * pad
    cube_shape = (37, 21, 30)
    ijk = _dev(ops.cube_origins(cube_shape, gs), cuda)
    codes = ops.tta_orientations(tta) or (0,)
    logits = {g: _bf16_logits(len(ijk), W, cuda, seed=g + 1) for g in codes}
    res = {}
    for dt in ('bf16', 'f32'):
        st = ops.Stitcher(cube_shape, cuda, gs, pad, window, tta=tta)
        for g in codes:
            lg = logits[g] if dt == 'bf16' else [t.float() for t in logits[g]]
            st(*lg, ijk, orient=g)
        res[dt] = _np(st.finalize())
    for k in MAP_TYPES:
        assert np.array_equal(res['bf16'][k], res['f32'][k]), k
    # peer: the raw fixed-point sums in the owners' blocks, along x and along k, 2 and 3 emulated ranks
    X, Y, Z = cube_shape
    for axis, bounds in ((0, (0, 17, X)), (2, (0, 9, 10, Z))):
        world = len(bounds) - 1
        n = [(bounds[r + 1] - bounds[r]) * (Y * Z if axis == 0 else X * Y) for r in range(world)]
        blocks = {}
        for dt in ('bf16', 'f32'):
            blocks[dt] = [torch.zeros(23 * m, dtype=torch.float32, device=cuda) for m in n]
            table = torch.tensor([t.data_ptr() for t in blocks[dt]], dtype=torch.int64, device=cuda)
            owners = ops.OverlapOwners(table, axis, bounds, (cuda.index if cuda.index is not None else 0,) * world)
            st = ops.Stitcher(cube_shape, cuda, gs, pad, window, owners=owners, tta=tta)
            for g in codes:
                lg = logits[g] if dt == 'bf16' else [t.float() for t in logits[g]]
                st(*lg, ijk, orient=g)
        for r in range(world):
            assert torch.equal(blocks['bf16'][r].view(torch.int32), blocks['f32'][r].view(torch.int32)), (axis, r)


# ------------------------------------------------------------------------------------------------ pipelines
class Bf16Model(PointwiseModel):
    """A deterministic, batch-independent stand-in with bf16 logits (``PointwiseModel`` in float32, rounded)."""

    def forward(self, x, af):
        return tuple(t.to(BF16) for t in super().forward(x.float(), af.float()))


def _rounding(model):
    """The float32 reference: ``model`` given its inputs rounded to bf16."""
    return lambda x, af: model(x.to(BF16), af.to(BF16))


@pytest.mark.parametrize('variant', ['prefetch', 'flips', 'min_max', 'triangle'])
def test_pipeline_equals_float32_with_rounded_inputs(cuda, variant):
    gs, pad = 16, 8
    shape = (64, 56, 72)
    vol = _masked_map(shape, 5) if variant == 'min_max' else synthetic.synthetic_map(shape, voxel=1.0, seed=5)
    atoms = _atoms(shape, cuda, n=400, seed=3)
    kw = {'prefetch': dict(model_batch=2, d8='split'), 'flips': dict(tta='flips', model_batch=3),
          'min_max': dict(min_max=T, model_batch=2, d8='split'), 'triangle': dict(overlap_window='triangle')}[variant]
    model = Bf16Model(seed=4).to(cuda)
    seen = []

    def probe(x, af):
        seen.append((x.dtype, af.dtype))
        return model(x, af)
    out = {}
    for dt in (torch.float32, BF16):
        p = MapPipeline(cuda, gs, pad, batch_cubes=5, cube_dtype=dt)
        assert p.prefetch
        assert p.resample_and_normalize(_dev(vol, cuda), HDR) and p.encode_af3(*atoms)
        with torch.no_grad():
            out[dt] = _np(p.predict_and_stitch(probe if dt == BF16 else _rounding(model), **kw))
    assert seen and all(s == (BF16, BF16) for s in seen)
    for k in MAP_TYPES:
        assert np.array_equal(out[BF16][k], out[torch.float32][k]), k


def _one_gpu(cuda, src, hdr, dt, model, gs, pad, **kw):
    single = MapPipeline(cuda, gs, pad, batch_cubes=4, cube_dtype=dt)
    assert single.resample_and_normalize(src, hdr)
    with torch.no_grad():
        return single.predict_and_stitch(model if dt == BF16 else _rounding(model), **kw).as_dict()


@pytest.mark.parametrize('world', [2, 3])
@pytest.mark.parametrize('dtype', ['float32', 'int16'])
@pytest.mark.parametrize('window', [None, 'triangle'])
def test_slab_ranks_equal_one_gpu(cuda, world, dtype, window):
    gs, pad = 16, 8
    if dtype == 'float32':
        src_shape, voxel = (136, 24, 20), 1.0
        src = synthetic.synthetic_map(src_shape, voxel=1.0, seed=13)
    else:
        src_shape, voxel = (120, 20, 18), 1.1
        src = _int16_map(src_shape, seed=13)
    hdr = MapHeader(voxel_size=(np.float32(voxel),) * 3)
    d_src = torch.from_numpy(src).to(cuda)
    model = Bf16Model(seed=2).to(cuda)
    kw = {} if window is None else dict(overlap_window=window)
    want = _one_gpu(cuda, d_src, hdr, BF16, model, gs, pad, **kw)
    ref = _one_gpu(cuda, d_src, hdr, torch.float32, model, gs, pad, **kw)
    for k in MAP_TYPES:
        assert torch.equal(want[k], ref[k]), k
    plan = SlabPlan(src_shape, hdr.voxel_size, gs, pad, world, dtype=d_src.dtype)
    nz, ny, nx = plan.out_shape
    pipes = [SlabPipeline(cuda, r, world, gs, pad, batch_cubes=4, global_src_shape=src_shape, group=False)
             for r in range(world)]
    res, owned = [], []
    for p in pipes:
        p.configure(cube_dtype=BF16)
        me = plan.ranks[p.rank]
        p._exchange = lambda own, me=me: d_src[me.src_lo:me.src_hi].contiguous()
        r_, o_ = p.slab_resample(d_src[me.own_lo:me.own_hi].contiguous(), hdr)
        res.append(r_)
        owned.append(o_)
    for p, r_, s in zip(pipes, res, _lockstep(owned, nz * ny * nx)):
        p.stats = s
        p.slab_normalize(r_)
        assert p.check_status()
    groups, vols = None, [None] * world
    if window is not None:                             # every owner clears its block before anybody adds
        groups = PeerVolumes.emulate(cuda, world, max(r.out_hi - r.out_lo for r in plan.ranks) * nx * ny)
        for r, (p, g_) in enumerate(zip(pipes, groups)):
            p.peer_volumes = g_
            p.cube_index()
            vols[r] = p._exported_volumes(p._n_max())
    with torch.no_grad():
        got = [p.predict_and_stitch(model, v, **kw) for p, v in zip(pipes, vols)]
    for p in pipes:
        p.finish_map()
    for p, vols in zip(pipes, got):
        (_, _, o2), (_, _, e2) = p.box
        for k, t in vols.as_dict().items():
            assert torch.equal(t, want[k][..., o2:o2 + e2]), (p.rank, k)
    if groups is not None:
        groups[0].close()


@pytest.mark.parametrize('world', [2, 3])
def test_balanced_cube_ranks_equal_one_gpu(cuda, world):
    gs, pad = 16, 8
    d_src = _dev(synthetic.synthetic_map((48, 40, 96), voxel=1.0, seed=21), cuda)
    model = Bf16Model(seed=1).to(cuda)
    want = _one_gpu(cuda, d_src, HDR, BF16, model, gs, pad, model_batch=2, d8='split')
    ref = _one_gpu(cuda, d_src, HDR, torch.float32, model, gs, pad, model_batch=2, d8='split')
    for k in MAP_TYPES:
        assert torch.equal(want[k], ref[k]), k
    pipes = [BalancedCubePipeline(cuda, r, world, gs, pad, batch_cubes=4, group=False) for r in range(world)]
    for p in pipes:
        p.configure(cube_dtype=BF16)
        assert p.resample_and_normalize(d_src, HDR)
        p.cube_index()
    groups = PeerVolumes.emulate(cuda, world, pipes[0]._n_max())
    vols = []
    for p, g_ in zip(pipes, groups):
        p.peer_volumes = g_
        vols.append(p._new_volumes())
    with torch.no_grad():
        for p, v in zip(pipes, vols):
            p.predict_and_stitch(model, v, model_batch=2, d8='split')
    for p in pipes:
        p.finish_map()
    for r, (p, v) in enumerate(zip(pipes, vols)):
        x0, x1 = p.x_bounds[r], p.x_bounds[r + 1]
        for k, t in v.as_dict().items():
            assert torch.equal(t, want[k][:, x0:x1] if want[k].dim() == 4 else want[k][x0:x1]), (r, k)
    groups[0].close()


# ------------------------------------------------------------------------------------------------ drop-in
class ProbeModel(PointwiseModel):
    """``PointwiseModel`` (batch-independent) returning logits of its input's dtype, as a convolution under autocast
    would; it records what it is given, whether autocast is on, and what it returns."""

    def __init__(self, seed=0):
        super().__init__(seed)
        self.seen, self.outs = [], []

    def forward(self, x, af):
        self.seen.append((x.dtype, af.dtype, torch.is_autocast_enabled('cuda')))
        out = tuple(t.to(x.dtype) for t in super().forward(x.float(), af.float()))
        self.outs.append(tuple(t.float().cpu() for t in out))
        return out


@pytest.fixture
def _env(monkeypatch):
    for k in ('MICA_DEVICES', 'MICA_MIN_MAX', 'MICA_PRECISION'):
        monkeypatch.delenv(k, raising=False)
    session.clear()
    yield monkeypatch
    session.clear()


def _run(grids, out, model, **kw):
    pr = CryoEMPredictor('unused', grids, str(out), save_output=False, quiet=True, model=model, host_volumes=MAP_TYPES,
                         release_inputs=False, super_batch=20, **kw)
    ok, vols = pr.run_prediction()
    return pr, ok, vols


def test_dropin_precision(cuda, tmp_path, _env):
    grids, r, norm, _ = _grids(tmp_path, min_max=None, shape=(64, 64, 80))
    m32 = ProbeModel().to(cuda)
    pr, ok, v32 = _run(grids, tmp_path / 'o32', m32)
    assert ok and all(s == (torch.float32, torch.float32, False) for s in m32.seen)

    m16 = ProbeModel().to(cuda)
    pr, ok, v16 = _run(grids, tmp_path / 'o16', m16, precision='bf16')
    assert ok and m16.seen and all(s == (BF16, BF16, True) for s in m16.seen)
    assert all(np.asarray(v16[k]).dtype == np.float32 for k in MAP_TYPES)
    # the oracle's paste of the module's own logits, in the loop order the cubes were fed
    ijk = np.asarray(pr._source['ijk'])
    shape = tuple(pr._source['cube_shape'])
    meta = [(i, j, k, min(16, shape[0] - i), min(16, shape[1] - j), min(16, shape[2] - k)) for i, j, k in ijk]
    bb, ca, aa = (torch.cat([o[c] for o in m16.outs]) for c in range(3))
    assert len(bb) == len(ijk)
    want = mica_oracle.postprocess_and_stitch(bb, ca, aa, meta, shape, padding=8)
    for k in MAP_TYPES:
        assert np.abs(np.asarray(v16[k]) - want[k]).max() <= 1e-5, k
    assert any(not np.array_equal(np.asarray(v16[k]), np.asarray(v32[k])) for k in MAP_TYPES)

    # the environment knob; two workers on one device give the one-device bits, also with TTA
    _env.setenv('MICA_PRECISION', 'bf16')
    me = ProbeModel().to(cuda)
    _, ok, ve = _run(grids, tmp_path / 'env', me)
    assert ok and all(s == (BF16, BF16, True) for s in me.seen)
    _assert_same(v16, ve)
    _, ok, vd = _run(grids, tmp_path / 'dev', ProbeModel().to(cuda), devices=[0, 0])
    assert ok
    _assert_same(v16, vd)
    _, ok, vt1 = _run(grids, tmp_path / 't1', ProbeModel().to(cuda), tta='flips', overlap_window='triangle')
    _, ok3, vt3 = _run(grids, tmp_path / 't3', ProbeModel().to(cuda), tta='flips', overlap_window='triangle',
                       devices=[0, 0])
    assert ok and ok3
    _assert_same(vt1, vt3)
    _env.setenv('MICA_PRECISION', 'fp32')
    _, ok, vf = _run(grids, tmp_path / 'f32', ProbeModel().to(cuda))
    assert ok
    _assert_same(v32, vf)
    _env.delenv('MICA_PRECISION')

    # the reference's per-cube files: the cubes are uploaded and cast to bf16
    session.clear()
    grids_f, _, _, _ = _grids(tmp_path / 'files', min_max=None, materialize=True, shape=(64, 64, 80))
    session.clear()
    mf = ProbeModel().to(cuda)
    _, ok, vfile = _run(grids_f, tmp_path / 'of', mf, precision='bf16')
    assert ok and mf.seen and all(s == (BF16, BF16, True) for s in mf.seen)
    _assert_same(v16, vfile)

    # refusals: logged, (False, {}), nothing launched
    n0 = ops.launch_count()
    for bad in ('fp16', 'BF17', 16, torch.bfloat16):
        _, ok, v = _run(grids, tmp_path / 'bad', ProbeModel().to(cuda), precision=bad)
        assert not ok and v == {}
    _env.setenv('MICA_PRECISION', 'half')
    _, ok, v = _run(grids, tmp_path / 'bad', ProbeModel().to(cuda))
    assert not ok and v == {}
    assert ops.launch_count() == n0
