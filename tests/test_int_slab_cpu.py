"""Integer maps in z-slabs, host side on CPU: the general path's prefilter segment scheme (oracle/general_segment_scheme.py)
gives every rank's block the whole line's float64 coefficients bit for bit, the library's block planes match that
statement, and integer SlabPlans partition the map with halos from direct neighbours only."""
import numpy as np
import pytest
import torch

from mica_b200 import _lib, ops
from mica_b200.peer import PeerHalo
from mica_b200.slab import SlabPlan
from oracle import general_segment_scheme as gs

INT_TORCH = (torch.int8, torch.int16, torch.uint16)


def _needed(sz, nz, dst_z0, dst_n):
    """needed_planes (resample.cu) on the whole line: source planes the z taps of the output planes read."""
    zoom = (sz - 1) / (nz - 1) if nz > 1 else 1.0
    lo = int(np.floor(dst_z0 * zoom)) - 2
    hi = int(np.floor((dst_z0 + dst_n - 1) * zoom)) + 3
    lo, hi = max(lo, 0), min(hi, sz - 1)
    if dst_z0 + dst_n >= nz:
        hi = sz - 1
    return lo, hi


def _slabs(nz, world):
    b = [round(nz * r / world) for r in range(world + 1)]
    return [(b[r], b[r + 1] - b[r]) for r in range(world) if b[r + 1] > b[r]]


@pytest.mark.parametrize('ng', [96, 97, 400, 679, 800])
def test_general_segment_blocks_are_bit_identical_to_the_whole_line(ng):
    rng = np.random.default_rng(ng)
    line = rng.integers(-32768, 32768, (3, ng)).astype(np.int16)
    whole = gs.prefilter(line, 0, ng)
    nz = int(round(ng * 1.06))
    reached_end = own_differs = 0
    for world in (2, 3, 4, 8):
        for r, (dst_z0, dst_n) in enumerate(_slabs(nz, world)):
            need_lo, need_hi = _needed(ng, nz, dst_z0, dst_n)
            seg_lo, seg_c, seg_o, c_end, raw_lo, raw_hi = gs.plan(ng, need_lo, need_hi)
            assert ops.resample_slab_source_planes_general(ng, nz, dst_z0, dst_n) == (raw_lo, raw_hi)
            got = gs.prefilter(line[:, raw_lo:raw_hi], raw_lo, ng, seg_lo, seg_c, seg_o, c_end)
            sl = slice(need_lo, need_hi + 1)
            assert np.array_equal(got[:, need_lo - raw_lo:need_hi + 1 - raw_lo].view(np.uint64),
                                  whole[:, sl].view(np.uint64)), (world, r)
            ln = gs.seg_len(ng)
            k1 = min(ng, (seg_o + 1) * ln)
            if k1 < ng and k1 + gs.HORIZON >= ng:
                reached_end += 1              # the warm-up starts from the exact end initialisation
            if raw_hi - raw_lo < ng:
                own = gs.prefilter(line[:, raw_lo:raw_hi], 0, raw_hi - raw_lo)
                own_differs += not np.array_equal(own[:, need_lo - raw_lo:need_hi + 1 - raw_lo], whole[:, sl])
    ln = gs.seg_len(ng)
    last_seg_start = (ng - 1) // ln * ln
    assert own_differs > 0
    assert reached_end > 0 or ng - last_seg_start > gs.HORIZON     # 679, 800: the last segment outlasts the horizon


def test_general_segment_block_reads_stay_in_the_named_planes():
    """Sweep of slabs: the oracle raises on any read outside [raw_lo, raw_hi)."""
    rng = np.random.default_rng(1)
    for ng in (96, 106, 121, 255, 513, 800):          # 106, 121: a last segment of one sample
        line = rng.integers(-128, 128, (1, ng)).astype(np.int8)
        whole = gs.prefilter(line, 0, ng)
        for lo in range(0, ng, 7):
            for hi in (lo, min(ng - 1, lo + 11), ng - 1):
                p = gs.plan(ng, lo, hi)
                got = gs.prefilter(line[:, p[4]:p[5]], p[4], ng, *p[:4])
                assert np.array_equal(got[:, lo - p[4]:hi + 1 - p[4]], whole[:, lo:hi + 1]), (ng, lo, hi)


def test_general_plane_function_refuses_lines_outside_96_to_800():
    for sz in (95, 801):
        with pytest.raises(_lib.MicaError, match='96..800'):
            ops.resample_slab_source_planes_general(sz, sz, 0, sz // 2)
    assert ops.resample_slab_source_planes_general(96, 100, 0, 100) == (0, 96)
    assert ops.resample_slab_source_planes_general(800, 800, 0, 400)[0] == 0


@pytest.mark.parametrize('dtype', INT_TORCH, ids=str)
def test_integer_plan_refusal_names_the_type_and_the_bound(dtype):
    for sz in (40, 95, 801):
        with pytest.raises(_lib.MicaError, match=f'{str(dtype).split(".")[1]}.*96..800'):
            SlabPlan((sz, 8, 8), (np.float32(1.2),) * 3, 48, 8, 2, dtype=dtype)
    # the D10 copy and order=1 read taps only: no bound
    SlabPlan((40, 8, 8), (np.float32(1.0),) * 3, 48, 8, 2, dtype=dtype)
    SlabPlan((40, 8, 8), (np.float32(1.2),) * 3, 48, 8, 2, order=1, dtype=dtype)


# (source shape, voxel size, grid size, padding, order, largest world whose halos all come from direct neighbours).
# The general path's z prefilter reaches a whole segment (ceil(sz / 16) planes) plus 30 planes of horizon beyond the
# taps on either side: slabs thinner than that on small maps need planes of a farther rank, which SlabPipeline then
# exchanges over NCCL.
PLANS = [((400, 40, 40), 1.2, 32, 16, 3, 4), ((720, 16, 16), 1.0, 48, 8, 3, 8), ((679, 16, 16), 1.06, 48, 8, 3, 8),
         ((96, 8, 8), 0.83, 32, 16, 3, 2), ((800, 8, 8), 0.9, 48, 8, 3, 8), ((120, 8, 8), 1.2, 32, 8, 1, 8)]


@pytest.mark.parametrize('world', [1, 2, 3, 4, 8])
@pytest.mark.parametrize('src,voxel,gs_,pad,order,neighbours_up_to', PLANS)
def test_integer_plans_own_every_plane_once_with_neighbour_halos(world, src, voxel, gs_, pad, order, neighbours_up_to):
    plan = SlabPlan(src, (np.float32(voxel),) * 3, gs_, pad, world, order=order, dtype=torch.int16)
    nz, sz = plan.out_shape[0], src[0]
    owned, have = np.zeros(nz, int), np.zeros(sz, int)
    for r, me in enumerate(plan.ranks):
        owned[me.out_lo:me.out_hi] += 1
        have[me.own_lo:me.own_hi] += 1
        if me.out_hi > me.out_lo and order == 3 and not plan.identity:
            lo, hi = ops.resample_slab_source_planes_general(sz, nz, me.ext_lo, me.ext_hi - me.ext_lo)
            assert me.src_lo <= lo and me.src_hi >= hi
        if world <= neighbours_up_to:
            assert PeerHalo.neighbour_plan(plan, r) is not None, r
        for p, a, b in plan.transfers(r)[1]:         # what r receives from p is what p sends to r
            assert (r, a, b) in plan.transfers(p)[0]
    assert (owned == 1).all() and (have == 1).all()
    if world > neighbours_up_to:
        assert any(PeerHalo.neighbour_plan(plan, r) is None for r in range(world))
