"""Integer maps (int8 / int16 / uint16, DESIGN.md D12) split over ranks in z-slabs, the ranks emulated on ONE GPU as
in test_gpu_slab.py: every rank's resampled planes, the thresholds, the normalised owned planes and the stitched
volumes equal the one-GPU integer pipeline bit for bit.  Also the integer histogram sum over peer memory, the byte-wise
halo exchange, the halo prefetch of an integer map and the refusal of z lines the general path cannot cut."""
import ctypes as C

import numpy as np
import pytest
import torch
from scipy.ndimage import zoom

from mica_b200 import _lib, ops, synthetic
from mica_b200.pdb import channel_codes
from mica_b200.peer import PeerHalo, PeerIntHistogram
from mica_b200.pipeline import MapHeader, MapPipeline, zoom_factors
from mica_b200.slab import SlabPipeline, SlabPlan

pytestmark = pytest.mark.gpu

INT_TYPES = (torch.int8, torch.int16, torch.uint16)


def _int_map(shape, dtype, seed):
    """A density-like map scaled to most of the type's range, with full-range noise on a few planes (the cubic
    spline overshoots there: saturating stores)."""
    info = torch.iinfo(dtype)
    d = synthetic.synthetic_map(shape, seed=seed).astype(np.float64)
    d = (d - d.min()) / max(float(d.max() - d.min()), 1e-6)
    a = np.round(info.min + d * (float(info.max) - info.min) * 0.9)
    rng = np.random.default_rng(seed)
    a[shape[0] // 3] = rng.integers(info.min, info.max + 1, shape[1:])
    np_dtype = {torch.int8: np.int8, torch.int16: np.int16, torch.uint16: np.uint16}[dtype]
    return a.astype(np_dtype)


def _lockstep_int_stats(owned, n_total):
    """What ops.IntOrderStats.run(all_reduce=...) does on every rank of a real group."""
    lib = _lib.lib
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
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


# (id, source shape, voxel size (x, y, z), order).  gs = 12: every rank of 8 owns planes.
CASES = [
    ('isotropic', (120, 30, 34), (1.2, 1.2, 1.2), 3),
    ('anisotropic', (110, 26, 30), (1.1, 0.9, 1.2), 3),
    ('line_800', (800, 12, 14), (0.9, 0.9, 0.9), 3),
    ('end_init_97', (97, 20, 22), (1.06, 1.06, 1.06), 3),       # a block's warm-up starts from the end initialisation
    ('d10_copy', (100, 20, 22), (1.0, 1.0, 1.0), 3),
    ('order1', (80, 20, 22), (1.2, 1.2, 1.2), 1),
]


@pytest.mark.parametrize('world', [2, 3, 8])
@pytest.mark.parametrize('dtype', INT_TYPES, ids=str)
@pytest.mark.parametrize('case', CASES, ids=[c[0] for c in CASES])
def test_emulated_integer_slab_ranks_match_single_gpu(cuda, world, dtype, case):
    name, shape, voxel, order = case
    gs, pad = 12, 6
    src = _int_map(shape, dtype, seed=len(name) + world)
    hdr = MapHeader(voxel_size=tuple(np.float32(v) for v in voxel))
    d_src = torch.from_numpy(src).to(cuda)
    single = MapPipeline(cuda, gs, pad, order=order, batch_cubes=4)
    assert single.resample_and_normalize(d_src, hdr)
    zf = zoom_factors(hdr.voxel_size, 1.0)
    out_shape = ops.zoom_output_shape(shape, zf)
    want_res = d_src.clone() if all(float(z) == 1.0 for z in zf) else ops.resample(d_src, out_shape, order=order)
    n_out = tuple(single.normalized.shape)
    st = synthetic.synthetic_structure(120, n_out[::-1], seed=7)
    bb_ch, aa_ch = channel_codes(st['atom_names'], st['res_names'])
    atoms = tuple(torch.from_numpy(a).to(cuda) for a in (st['coords'], bb_ch, aa_ch))
    assert single.encode_af3(*atoms)
    with torch.no_grad():
        want = single.predict_and_stitch(synthetic.pointwise_model)

    pipes = [SlabPipeline(cuda, r, world, gs, pad, order=order, batch_cubes=4, global_src_shape=shape, group=False)
             for r in range(world)]
    plan = SlabPlan(shape, hdr.voxel_size, gs, pad, world, order=order, dtype=dtype)
    res, owned = [], []
    for p in pipes:
        p._exchange = lambda own, p=p: d_src[p.plan.ranks[p.rank].src_lo:p.plan.ranks[p.rank].src_hi].contiguous()
        me = plan.ranks[p.rank]
        assert me.out_hi > me.out_lo
        r_, o_ = p.slab_resample(d_src[me.own_lo:me.own_hi].contiguous(), hdr)
        assert r_.dtype == dtype and torch.equal(r_, want_res[me.ext_lo:me.ext_hi]), p.rank
        res.append(r_)
        owned.append(o_)
    stats = _lockstep_int_stats(owned, int(np.prod(n_out)))
    vols = {k: torch.zeros_like(v) for k, v in want.as_dict().items()}
    got_res = torch.empty_like(want_res)
    for p, r_, s in zip(pipes, res, stats):
        p.stats = s
        p.slab_normalize(r_)
        assert p.check_status()
        assert isinstance(p.median, float) and p.median == single.median and p.p999 == single.p999
        me = p.plan.ranks[p.rank]
        got_res[me.out_lo:me.out_hi] = r_[me.out_lo - me.ext_lo:me.out_hi - me.ext_lo]
        assert torch.equal(p.normalized[me.out_lo - me.ext_lo:me.out_hi - me.ext_lo],
                           single.normalized[me.out_lo:me.out_hi]), p.rank
        assert p.encode_af3(*atoms)
        with torch.no_grad():
            v = p.predict_and_stitch(synthetic.pointwise_model)
        (_, _, o2), (_, _, e2) = p.box
        for k, t in v.as_dict().items():
            vols[k][..., o2:o2 + e2] = t
    for k, t in want.as_dict().items():
        assert torch.equal(vols[k], t), k
    if name == 'isotropic' and dtype == torch.int16 and world == 3:
        # scipy.ndimage.zoom on the integer array, up to voxels whose float64 value lies at a k + 1/2 boundary
        got = got_res.cpu().numpy()
        ref = zoom(src, [float(z) for z in zf], order=order)
        diff = got != ref
        if diff.any():
            f64 = zoom(src.astype(np.float64), [float(z) for z in zf], order=order)
            near = np.abs(np.abs(f64) - np.floor(np.abs(f64)) - 0.5) < 1e-9
            assert not (diff & ~near).any()


@pytest.mark.parametrize('dtype', [torch.int8, torch.uint16], ids=str)
@pytest.mark.parametrize('world', [2, 3, 8])
def test_peer_memory_integer_histogram_sum_equals_single_gpu(cuda, world, dtype):
    """PeerIntHistogram (publish kernel + sum kernel over peer-mapped buffers) with `world` emulated ranks on their
    own streams, over several epochs (slot parity) with a new map each time: the thresholds equal the whole-array
    IntOrderStats.  On one GPU every rank publishes before any rank sums (a spinning sum grid could otherwise hold
    the SMs another rank's histogram needs); two ranks also go through IntOrderStats.run(peer=)."""
    lib = _lib.lib
    code = ops.MAP_DTYPES[dtype]
    groups = PeerIntHistogram.emulate(cuda, world)
    streams = [torch.cuda.Stream(cuda) for _ in range(world)]
    stats = [ops.IntOrderStats(cuda) for _ in range(world)]
    rng = np.random.default_rng(world)
    np_dtype = np.int8 if dtype == torch.int8 else np.uint16
    info = np.iinfo(np_dtype)
    for epoch in range(3):
        x = torch.from_numpy(rng.integers(info.min // 4, info.max // 2, 2_000_003).astype(np_dtype)).to(cuda)
        want = ops.IntOrderStats(cuda).run(x).result()
        b = [0] + sorted(int(v) for v in rng.integers(1, x.numel() - 1, world - 1)) + [x.numel()]
        torch.cuda.synchronize()
        if world == 2:
            for r in range(world):
                with torch.cuda.stream(streams[r]):
                    stats[r].run(x[b[r]:b[r + 1]], n_total=x.numel(), peer=groups[r])
        else:
            for r in range(world):
                with torch.cuda.stream(streams[r]):
                    st = C.c_void_p(streams[r].cuda_stream)
                    part = x[b[r]:b[r + 1]]
                    _lib.check(lib.mica_int_stats_init(stats[r]._p, code, x.numel(), st))
                    _lib.check(lib.mica_int_stats_hist(C.c_void_p(part.data_ptr()), code, part.numel(), stats[r]._p,
                                                       st))
                    groups[r].publish(stats[r], code, streams[r].cuda_stream)
            for r in range(world):
                with torch.cuda.stream(streams[r]):
                    groups[r].sum(stats[r], code, streams[r].cuda_stream)
                    _lib.check(lib.mica_int_stats_pick(stats[r]._p, code, C.c_void_p(streams[r].cuda_stream)))
        torch.cuda.synchronize()
        for r in range(world):
            got = stats[r].result()
            assert got == want, (epoch, r, got, want)
    groups[0].close()


def test_byte_halo_exchange_assembles_odd_int8_planes(cuda):
    """mica_halo_publish_bytes / mica_halo_pull_bytes on int8 planes of 7 x 9 bytes (no 4- or 16-byte alignment
    anywhere), three emulated ranks on their own streams, three epochs."""
    world, src_shape = 3, (96 * 3, 7, 9)
    plan = SlabPlan(src_shape, (np.float32(1.1),) * 3, 32, 16, world)
    need = max(b - a for r in range(world) for rng in PeerHalo.neighbour_plan(plan, r) if rng is not None
               for a, b in [rng])
    groups = PeerHalo.emulate(cuda, world, PeerHalo.slot_words(plan, need, 1))
    assert all(g_.fits(plan, g_.rank, 1) for g_ in groups)
    streams = [torch.cuda.Stream(cuda) for _ in range(world)]
    g = torch.Generator(device=cuda).manual_seed(5)
    for epoch in range(3):
        full = torch.randint(-128, 128, src_shape, generator=g, device=cuda).to(torch.int8)
        torch.cuda.synchronize()
        owns, bufs = [], []
        for r in range(world):
            me = plan.ranks[r]
            owns.append(full[me.own_lo:me.own_hi].contiguous())
            with torch.cuda.stream(streams[r]):
                groups[r].publish(owns[r], plan, streams[r].cuda_stream)
        for r in range(world):
            me = plan.ranks[r]
            with torch.cuda.stream(streams[r]):
                buf = torch.full((me.src_hi - me.src_lo,) + src_shape[1:], -1, dtype=torch.int8, device=cuda)
                lo, hi = max(me.src_lo, me.own_lo), min(me.src_hi, me.own_hi)
                buf[lo - me.src_lo:hi - me.src_lo].copy_(owns[r][lo - me.own_lo:hi - me.own_lo])
                groups[r].pull(buf, plan, streams[r].cuda_stream)
            bufs.append(buf)
        torch.cuda.synchronize()
        for r in range(world):
            me = plan.ranks[r]
            assert not groups[r].timed_out()
            assert torch.equal(bufs[r], full[me.src_lo:me.src_hi]), (epoch, r)
    groups[0].close()


def test_integer_halo_prefetch_is_consumed_and_bit_identical(cuda):
    """SlabPipeline.prefetch_source with int16 maps: the next map's halo is exchanged into int16 buffers on a side
    stream, the next slab_resample takes it (no second exchange) and its planes equal the whole map's."""
    world, src_shape, voxel = 2, (208, 30, 34), 1.1
    hdr = MapHeader(voxel_size=(np.float32(voxel),) * 3)
    plan = SlabPlan(src_shape, hdr.voxel_size, 48, 8, world, dtype=torch.int16)
    pipes = [SlabPipeline(cuda, r, world, 48, 8, global_src_shape=src_shape, group=False) for r in range(world)]
    groups = PeerHalo.emulate(cuda, world, pipes[0]._halo_slot_elems(plan))
    calls = [0] * world
    for r, p in enumerate(pipes):
        p.peer_halo = groups[r]
        real = groups[r].exchange

        def counted(own, plan_, buf=None, *, real=real, r=r):
            calls[r] += 1
            return real(own, plan_, buf)
        groups[r].exchange = counted
    streams = [torch.cuda.Stream(cuda) for _ in range(world)]
    maps = [torch.from_numpy(_int_map(src_shape, torch.int16, seed=s)).to(cuda) for s in range(3)]
    owns = [[m[me.own_lo:me.own_hi].contiguous() for me in plan.ranks] for m in maps]
    want = [ops.resample(m, plan.out_shape) for m in maps]
    torch.cuda.synchronize()
    got = {}
    for k, nxt in ((0, 1), (1, 2), (2, None)):
        for r, p in enumerate(pipes):
            with torch.cuda.stream(streams[r]):
                got[k, r], _ = p.slab_resample(owns[k][r], hdr)
                if nxt is not None:
                    p.prefetch_source(owns[nxt][r], hdr)
    torch.cuda.synchronize()
    assert calls == [3, 3]
    assert all(b.dtype == torch.int16 for p in pipes for b in p._halo_bufs)
    for (k, r), t in got.items():
        me = plan.ranks[r]
        assert not groups[r].timed_out()
        assert t.dtype == torch.int16 and torch.equal(t, want[k][me.ext_lo:me.ext_hi]), (k, r)
    groups[0].close()


def test_integer_slab_refuses_an_801_plane_line_before_any_launch(cuda):
    p = SlabPipeline(cuda, 0, 2, 48, 8, global_src_shape=(801, 16, 16), group=False)
    own = torch.zeros((400, 16, 16), dtype=torch.int16, device=cuda)
    torch.cuda.synchronize()
    before = ops.launch_count()
    with pytest.raises(_lib.MicaError, match='int16.*800'):
        p.resample_and_normalize(own, MapHeader(voxel_size=(np.float32(1.2),) * 3))
    assert ops.launch_count() == before
