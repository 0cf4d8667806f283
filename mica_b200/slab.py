"""z-slab partition of the map pipeline over the GPUs of one box (SURVEY.md 8e).

The working grid is cut along memory axis 0 (z; cube axis k under the standard MRC
axis order) at multiples of ``grid_size`` so that every cube core -- and therefore
every stitched voxel -- has exactly one owner.  Per stage:

  resample      each rank resamples its owned output planes plus ``padding`` halo planes
                (the cube windows reach that far) from its source planes plus the
                interpolation taps plus the prefilter windows of the segments that hold them
                (>= ``halo_k`` planes of horizon; whole segments, so that the result is
                bit-identical to the one-GPU map); the source halo comes from the two
                neighbouring ranks over NVLink peer memory (peer.PeerHalo).
  order stats   local histograms over OWNED planes only, all-reduced (int64 sum) between
                the hist and pick kernels of each of the 5 radix rounds: exact.  An integer map
                (int8 / int16 / uint16, DESIGN.md D12) has one exact histogram, summed once.
  AF3 encode    atoms are replicated (a few MB); each rank rasterises its slab + halo.
  extract       a rank's cubes are those whose core lies in its slab; no exchange (the halo
                planes were resampled and normalised locally).
  stitch        cores are slab-aligned: each rank writes only its own [X, Y, z-range] box.

There is no reference counterpart (the reference is single-process); results are checked
against the single-GPU path and the CPU oracle."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from . import ops
from ._lib import MicaError, NORM_OK
from .pipeline import MapHeader, MapPipeline, zoom_factors, _on_device


def _split_even(n_items: int, parts: int):
    base, rem = divmod(n_items, parts)
    bounds = [0]
    for r in range(parts):
        bounds.append(bounds[-1] + base + (1 if r < rem else 0))
    return bounds


@dataclass
class RankSlab:
    out_lo: int          # owned output planes [out_lo, out_hi)
    out_hi: int
    ext_lo: int          # resampled planes incl. the cube halo [ext_lo, ext_hi)
    ext_hi: int
    src_lo: int          # source planes needed [src_lo, src_hi)
    src_hi: int
    own_lo: int          # source planes this rank holds before the exchange [own_lo, own_hi)
    own_hi: int


class SlabPlan:
    """Pure host arithmetic of the partition (unit-tested on CPU).  ``dtype``: the map's sample type.  An integer
    map resampled at order 3 takes the general path, whose z prefilter gives a block the whole line's bits only for
    lines of 96..800 planes (``ops.resample_slab_source_planes_general``): other lengths raise MicaError."""

    def __init__(self, src_shape, voxel_size_xyz, grid_size, padding, world, target_voxel_size=1.0,
                 halo_k=16, order=3, aligned=True, dtype=torch.float32):
        self.src_shape = tuple(int(v) for v in src_shape)
        self.world = int(world)
        self.grid_size, self.padding, self.halo_k, self.order = int(grid_size), int(padding), int(halo_k), order
        self.dtype = dtype
        zf = zoom_factors(voxel_size_xyz, target_voxel_size)
        self.identity = all(float(z) == 1.0 for z in zf)
        self.out_shape = ops.zoom_output_shape(self.src_shape, zf)
        sz, nz = self.src_shape[0], self.out_shape[0]
        general = dtype in ops.INT_DTYPES and order == 3 and not self.identity
        if general:
            try:                                # the library knows which lines the general path can cut
                ops.resample_slab_source_planes_general(sz, nz, 0, nz)
            except MicaError as e:
                raise MicaError(f'a {dtype} map cannot be resampled in z-slabs (run it on one GPU, MapPipeline): '
                                f'{e}') from None
        layers = -(-nz // self.grid_size)
        lb = _split_even(layers, self.world)
        scale = (sz - 1) / (nz - 1) if nz > 1 else 1.0
        # a rank HOLDS the source planes under its output slab (not an even split of the source): what it
        # still needs from others is then only the taps + prefilter horizon + cube halo just beyond its
        # block, i.e. planes of its two direct neighbours (the peer-memory halo exchange relies on that)
        ob = [0]
        for r in range(1, self.world):
            o = min(nz, lb[r] * self.grid_size)
            ob.append(sz if o >= nz else max(ob[-1], min(sz, int(round(o * scale)))))
        ob.append(sz)
        taps_lo, taps_hi = (1, 2) if order == 3 else (0, 1)
        k = self.halo_k if (order == 3 and not self.identity and not general) else 0
        self.ranks = []
        for r in range(self.world):
            out_lo, out_hi = min(nz, lb[r] * self.grid_size), min(nz, lb[r + 1] * self.grid_size)
            ext_lo, ext_hi = max(0, out_lo - self.padding), min(nz, out_hi + self.padding)
            if out_hi <= out_lo:
                ext_lo = ext_hi = out_lo
                src_lo = src_hi = 0
            elif self.identity:
                src_lo, src_hi = ext_lo, ext_hi
            else:
                src_lo = max(0, int(np.floor(ext_lo * scale)) - taps_lo - k)
                src_hi = min(sz, int(np.floor((ext_hi - 1) * scale)) + taps_hi + k + 1)
                if general:
                    # the segments of the general path's z prefilter that the slab computes, and their windows
                    a_lo, a_hi = ops.resample_slab_source_planes_general(sz, nz, ext_lo, ext_hi - ext_lo)
                    src_lo, src_hi = min(src_lo, a_lo), max(src_hi, a_hi)
                elif order == 3 and aligned:
                    # whole prefilter segments + their windows: the slab's coefficients are then computed
                    # from the same windows as on one GPU, i.e. the N-rank map is bit-identical to it
                    a_lo, a_hi = ops.resample_slab_source_planes(sz, nz, ext_lo, ext_hi - ext_lo)
                    src_lo, src_hi = min(src_lo, a_lo), max(src_hi, a_hi)
            self.ranks.append(RankSlab(out_lo, out_hi, ext_lo, ext_hi, src_lo, src_hi, ob[r], ob[r + 1]))

    def transfers(self, rank):
        """(sends, recvs) for ``rank``: lists of (peer, plane_lo, plane_hi) in global source planes."""
        me = self.ranks[rank]
        sends, recvs = [], []
        for p, other in enumerate(self.ranks):
            if p == rank:
                continue
            lo, hi = max(me.src_lo, other.own_lo), min(me.src_hi, other.own_hi)
            if hi > lo:
                recvs.append((p, lo, hi))
            lo, hi = max(other.src_lo, me.own_lo), min(other.src_hi, me.own_hi)
            if hi > lo:
                sends.append((p, lo, hi))
        return sends, recvs


def exchange_source_halo(own: torch.Tensor, plan: SlabPlan, rank: int, group=None) -> torch.Tensor:
    """Assemble the source planes [src_lo, src_hi) this rank needs from its own block
    ``own`` (= global planes [own_lo, own_hi)) and its neighbours' (send/recv).  The planes travel as bytes
    (uint8 views): NCCL has no int16 / uint16 type."""
    import torch.distributed as dist
    me = plan.ranks[rank]
    n = max(0, me.src_hi - me.src_lo)
    buf = torch.empty((n,) + tuple(own.shape[1:]), dtype=own.dtype, device=own.device)
    lo, hi = max(me.src_lo, me.own_lo), min(me.src_hi, me.own_hi)
    if hi > lo:
        buf[lo - me.src_lo:hi - me.src_lo].copy_(own[lo - me.own_lo:hi - me.own_lo])
    sends, recvs = plan.transfers(rank)
    own_b, buf_b = own.contiguous().view(torch.uint8), buf.view(torch.uint8)
    ops_ = []
    keep = []
    for p, a, b in sends:
        t = own_b[a - me.own_lo:b - me.own_lo].contiguous()
        keep.append(t)
        ops_.append(dist.P2POp(dist.isend, t, p, group))
    for p, a, b in recvs:
        ops_.append(dist.P2POp(dist.irecv, buf_b[a - me.src_lo:b - me.src_lo], p, group))
    if ops_:
        for req in dist.batch_isend_irecv(ops_):
            req.wait()
    return buf


class _SplitMap:
    """What the pipelines of one map split over ranks share: meeting the other ranks, the exported volume block
    (peer.PeerVolumes) the other ranks store into, and the weighted stitch, whose contributions are added into the
    block of the rank that owns their plane and finalised by ``finish_map``."""

    peer_volumes = None
    _pending = None

    def sync_ranks(self):
        torch.cuda.synchronize(self.device)
        if self.world > 1 and self.group is not False:
            import torch.distributed as dist
            dist.barrier(group=self.group)

    def finish_map(self):
        """All ranks' contributions have landed: after this every rank may read its own volume block (an
        overlap-weighted map is finalised here, each owner its own block)."""
        self.sync_ranks()
        pending, self._pending = self._pending, None
        if pending is not None:
            with torch.cuda.device(self.device):
                MapPipeline._stitch_done(self, *pending)

    def _exported_volumes(self, n_max):
        """This rank's box as volumes in its exported block (zeroed): the block other ranks store into."""
        from .peer import PeerVolumes
        if self.peer_volumes is None or self.peer_volumes.n_voxels < n_max:
            if self.peer_volumes is not None:
                self.peer_volumes.close()
            if self.world == 1:                   # nothing to map: one local block
                self.peer_volumes = PeerVolumes.emulate(self.device, 1, n_max)[0]
            elif self.group is False:
                raise MicaError('in-process emulation of several ranks: pass _peer_volumes (PeerVolumes.emulate)')
            else:
                self.peer_volumes = PeerVolumes(self.device, self.rank, self.world, n_max, self.group)
        org, ext = self.box
        n = ext[0] * ext[1] * ext[2]
        vols = ops.StitchedVolumes.from_block(self.peer_volumes.block(n_elems=23 * n), self.cube_shape, org, ext)
        vols.block.zero_()
        return vols

    def _owner_bounds(self):
        """(cube axis, world + 1 plane bounds) of the output partition."""
        raise NotImplementedError

    def _make_stitcher(self, w1, codes, vols):
        """A stitcher into the owners' exported blocks; ``vols`` (default: this rank's exported volumes, zeroed
        before the ranks meet, so nobody stores into a block before its owner has cleared it) is this rank's box."""
        if vols is None:
            vols = self._exported_volumes(self._n_max())
            self.sync_ranks()
        axis, bounds = self._owner_bounds()
        pv = self.peer_volumes
        return ops.Stitcher(self.cube_shape, self.device, self.grid_size, self.padding, w1, tta=codes, vols=vols,
                            owners=ops.OverlapOwners(pv.table, axis, tuple(bounds), tuple(pv.devices)))

    def _stitch_done(self, st, on_batch, n):
        if not st.per_batch:
            self._pending = (st, on_batch, n)         # finalised by finish_map, once every rank has added
        return st.vols


class SlabPipeline(_SplitMap, MapPipeline):
    """One rank's share of a z-slab partitioned map.  ``run`` takes this rank's OWN block
    of source planes (global planes [own_lo, own_hi) of ``global_src_shape``).

    ``predict_and_stitch`` runs this rank's cubes.  The paste stores their cores into this rank's box.  With
    ``overlap_window`` (or ``tta``) the windows reach ``padding`` planes into the neighbouring slabs: those
    contributions are added into the neighbours' exported blocks, and the volumes are final after ``finish_map()`` on
    every rank.  ``min_max``: each rank measures its own cubes on its normalised block (halo included), so the
    decisions are the one-GPU map's."""

    def __init__(self, device, rank, world, grid_size=48, padding=8, order=3, batch_cubes=16,
                 target_voxel_size=1.0, halo_k=16, global_src_shape=None, group=None, af3_mode='sparse',
                 hist_exchange='peer', halo_exchange='peer', _peer_volumes=None):
        super().__init__(device, grid_size, padding, order, batch_cubes, target_voxel_size, af3_mode)
        self.rank, self.world, self.halo_k, self.group = int(rank), int(world), halo_k, group
        self.global_src_shape = global_src_shape
        self.plan = None
        #: 'peer' = publish / pull kernels over NVLink peer memory (peer.PeerHalo, built on first use; plans
        #: that reach beyond the direct neighbours fall back to NCCL); 'nccl' = batch_isend_irecv
        if halo_exchange not in ('peer', 'nccl'):
            raise MicaError(f'halo_exchange must be peer or nccl, got {halo_exchange!r}')
        self.halo_exchange = halo_exchange
        self.peer_halo = None
        self._halo_stream = None
        self._halo_bufs, self._halo_turn = None, 0
        self._prefetched = None
        self._plan_key = None
        #: 'peer' = one fused publish/signal/wait/sum kernel over NVLink peer memory per radix round
        #: (peer.PeerHistogram, built on first use); 'nccl' = torch.distributed.all_reduce
        if hist_exchange not in ('peer', 'nccl'):
            raise MicaError(f'hist_exchange must be peer or nccl, got {hist_exchange!r}')
        self.hist_exchange = hist_exchange
        self.peer = None
        self.int_peer = None
        self.peer_volumes = _peer_volumes         # built on first use by an overlap-weighted map

    def _peer_group(self):
        if self.peer is None:
            from .peer import PeerHistogram
            self.peer = PeerHistogram(self.device, self.rank, self.world, self.group)
        return self.peer

    def _int_peer_group(self):
        if self.int_peer is None:
            from .peer import PeerIntHistogram
            self.int_peer = PeerIntHistogram(self.device, self.rank, self.world, self.group)
        return self.int_peer

    # -- collectives (torch.distributed over NCCL; injectable for single-process emulation)
    def _all_reduce_hist(self, hist):
        import torch.distributed as dist
        dist.all_reduce(hist, op=dist.ReduceOp.SUM, group=self.group)

    def _halo_slot_elems(self, plan):
        """Largest halo (in 4-byte words, of planes of the plan's sample type) any rank receives from one
        neighbour, or None when some rank needs planes from beyond its direct neighbours.  Global: the same
        answer on every rank."""
        from .peer import PeerHalo
        planes = 0
        for r in range(self.world):
            np_ = PeerHalo.neighbour_plan(plan, r)
            if np_ is None:
                return None
            planes = max([planes] + [rng[1] - rng[0] for rng in np_ if rng is not None])
        itemsize = torch.empty((), dtype=plan.dtype).element_size()
        return PeerHalo.slot_words(plan, planes, itemsize)

    def prefetch_source(self, next_own, header=None):
        """Exchange the source halo of the NEXT map now, on a side stream, so that it runs under this map's
        cube loop instead of at the head of the next step (publish never waits; the pull's wait for the
        neighbour then costs nothing on the main stream).  Call it after this map's pre-phase has been
        enqueued -- ``run(..., next_src=)`` does -- on EVERY rank, with the block the next ``run`` /
        ``slab_resample`` will be given; the block must stay untouched until then.  A next call with another
        block simply exchanges again.  No-op for plans the peer-memory exchange does not serve and for a next
        map of another geometry (shape, voxel size) than the current one."""
        if self.world == 1 or self.halo_exchange != 'peer' or self.peer_halo is None:
            return                                    # the first map builds the exchange group (a collective)
        header = self.header if header is None else header
        if self.plan is None or self._plan_key_of(tuple(next_own.shape), header, next_own.dtype) != self._plan_key:
            return                                    # another geometry: this map's plan must stay; exchanged in line
        plan = self.plan
        need = self._halo_slot_elems(plan)
        if need is None or self.peer_halo.slot_elems < need:
            return
        if self._halo_stream is None:
            self._halo_stream = torch.cuda.Stream(self.device)
        main = torch.cuda.current_stream(self.device)
        # two assembled-source buffers owned by the pipeline, used in turn: the one map k is being resampled
        # from is next written by the prefetch of map k+2, which this stream wait orders behind map k+1's
        # pre-phase (no allocator traffic between streams, no record_stream)
        me = plan.ranks[self.rank]
        shape = (max(0, me.src_hi - me.src_lo),) + tuple(next_own.shape[1:])
        if self._halo_bufs is None or tuple(self._halo_bufs[0].shape) != shape or \
                self._halo_bufs[0].dtype != next_own.dtype:
            main.wait_stream(self._halo_stream)        # a dropped prefetch may still be writing the old pair
            self._halo_bufs = [torch.empty(shape, dtype=next_own.dtype, device=self.device) for _ in range(2)]
        self._halo_turn ^= 1
        buf = self._halo_bufs[self._halo_turn]
        self._halo_stream.wait_stream(main)
        with torch.cuda.stream(self._halo_stream):
            self.peer_halo.exchange(next_own, plan, buf)
            ev = torch.cuda.Event()
            ev.record(self._halo_stream)
        self._prefetched = ((next_own.data_ptr(), tuple(next_own.shape), next_own._version, self._plan_key), buf, ev)

    def _exchange(self, own):
        pf, self._prefetched = self._prefetched, None
        if pf is not None and pf[0] == (own.data_ptr(), tuple(own.shape), own._version, self._plan_key):
            torch.cuda.current_stream(self.device).wait_event(pf[2])
            return pf[1]
        if self.halo_exchange == 'peer' and self.world > 1:
            need = self._halo_slot_elems(self.plan)      # the same on every rank (the plan is global)
            if need is not None:
                from .peer import PeerHalo
                if self.peer_halo is None or self.peer_halo.slot_elems < need:
                    if self.peer_halo is not None:
                        # a neighbour may still be pulling from the old buffers (an exchange prefetched for a map
                        # that never came): every rank takes this branch together, so wait for all of them
                        torch.cuda.synchronize(self.device)
                        if self.group is not False:
                            import torch.distributed as dist
                            if dist.is_available() and dist.is_initialized():
                                dist.barrier(group=self.group)
                        self.peer_halo.close()
                    self.peer_halo = self._make_peer_halo(need)
                return self.peer_halo.exchange(own, self.plan)
        return exchange_source_halo(own, self.plan, self.rank, self.group)

    def _make_peer_halo(self, slot_elems):
        from .peer import PeerHalo
        return PeerHalo(self.device, self.rank, self.world, slot_elems, self.group)

    def _plan_key_of(self, own_shape, header, dtype=torch.float32):
        gshape = self.global_src_shape
        if gshape is None:                      # weak-scaling default: equal blocks stacked along z
            gshape = (own_shape[0] * self.world, own_shape[1], own_shape[2])
        return (tuple(gshape), tuple(float(v) for v in header.voxel_size), self.grid_size, self.padding, self.world,
                float(self.target_voxel_size), self.halo_k, self.order, dtype)

    def make_plan(self, own_shape, header, dtype=torch.float32):
        key = self._plan_key_of(own_shape, header, dtype)
        gshape = key[0]
        if key != self._plan_key:               # host arithmetic only, but it runs once per map otherwise
            self.plan = SlabPlan(gshape, header.voxel_size, self.grid_size, self.padding, self.world,
                                 self.target_voxel_size, self.halo_k, self.order, dtype=dtype)
            self._plan_key = key
        return self.plan

    @_on_device
    def slab_resample(self, own_src, header=None):
        """Halo exchange + resample of this rank's planes.  Returns (res, owned): the local
        resampled planes [ext_lo, ext_hi) and the view of the owned ones [out_lo, out_hi).  float32, int8,
        int16 and uint16 maps; the resampled planes have the map's type (D12)."""
        dtype = getattr(own_src, 'dtype', None)
        if dtype not in ops.MAP_DTYPES:
            raise MicaError(f'SlabPipeline takes float32, int8, int16 or uint16 maps, got {dtype or type(own_src)}')
        if header is not None:
            self.header = header
        plan = self.make_plan(tuple(own_src.shape), self.header, dtype)
        me = plan.ranks[self.rank]
        nz, ny, nx = plan.out_shape
        with self.timer('halo_exchange'):
            src = self._exchange(own_src)
        with self.timer('resample'):
            if plan.identity:
                res = src.clone()
            else:
                res = ops.resample(src, plan.out_shape, order=self.order, src_z0=me.src_lo,
                                   src_shape=plan.src_shape, dst_z0=me.ext_lo, dst_nz_local=me.ext_hi - me.ext_lo)
        self.z0, self.global_nz = me.ext_lo, nz
        self.owned_voxels = (me.out_hi - me.out_lo) * ny * nx
        return res, res[me.out_lo - me.ext_lo:me.out_hi - me.ext_lo]

    def slab_normalize(self, res):
        """Apply the (globally agreed) thresholds to the local planes, halo included: in place for a float32
        map, into a new float32 volume for an integer one."""
        with self.timer('normalize_apply'):
            self.normalized = self.stats.apply(res) if res.dtype in ops.INT_DTYPES else self.stats.apply(res, res)
        self.norm_status = None

    @_on_device
    def resample_and_normalize(self, own_src, header=None, defer_status=False):
        """As ``MapPipeline.resample_and_normalize`` for this rank's planes; ``median`` and ``p999`` are Python
        floats for an integer map."""
        res, owned = self.slab_resample(own_src, header)
        nz, ny, nx = self.plan.out_shape
        integer = res.dtype in ops.INT_DTYPES
        stats = self._int_order_stats() if integer else self._order_stats()
        with self.timer('order_stats'):
            if self.hist_exchange == 'peer' and self.world > 1:
                peer = self._int_peer_group() if integer else self._peer_group()
                self.stats = stats.run(owned, n_total=nz * ny * nx, peer=peer)
            else:
                self.stats = stats.run(owned, n_total=nz * ny * nx, all_reduce=self._all_reduce_hist)
        self.slab_normalize(res)
        return True if defer_status else self.check_status()

    def _global_shape(self):
        return tuple(self.plan.out_shape)

    def _check_halo(self):
        if self.peer_halo is not None and self.peer_halo.timed_out():
            raise MicaError('halo exchange timed out: a neighbouring rank never published its source planes')

    def check_status(self):
        ok = super().check_status()
        self._check_halo()
        return ok

    def finish(self):
        super().finish()
        self._check_halo()

    @_on_device
    def encode_af3(self, coords, bb_ch, aa_ch, defer_status=False):
        if self.af3_mode == 'sparse':            # atoms are binned on the global cube grid
            return super().encode_af3(coords, bb_ch, aa_ch, defer_status)
        nz, ny, nx = self.plan.out_shape
        with self.timer('af3_encode'):
            vol, status = ops.af3_encode(coords, bb_ch, aa_ch, self.header.origin, (nz, ny, nx),
                                         clip_hi_xyz=self.af3_clip, z0=self.z0, nz_local=self.normalized.shape[0])
        self.af3, self._af3_status, self._atoms_binned = vol, status, False
        if defer_status:
            return True
        ok = int(status.item()) == 0
        self.af3 = vol if ok else None
        return ok

    def cube_index(self):
        perm, offset = self.header.transpose_order()
        if perm[2] != 0:
            raise MicaError('slab partition needs memory axis 0 to be cube axis k (standard MRC axis order)')
        self.perm, self.offset = perm, offset
        me = self.plan.ranks[self.rank]
        self.cube_shape = ops.cube_space_shape(self.plan.out_shape, perm)
        ijk = ops.cube_origins(self.cube_shape, self.grid_size)
        mine = (ijk[:, 2] >= me.out_lo) & (ijk[:, 2] < me.out_hi)
        self._set_cube_origins(ijk[mine], (self.cube_shape, self.grid_size, me.out_lo, me.out_hi))
        self.box = ((0, 0, me.out_lo), (self.cube_shape[0], self.cube_shape[1], me.out_hi - me.out_lo))
        return self.ijk_host

    def _extract_map(self, ijk, x, orient=0):
        ops.extract_cubes(self.normalized, ijk, self.grid_size, self.padding, self.perm, out=x,
                          global_nz=self.global_nz, z0=self.z0, orient=orient)

    def _extract_af3(self, ijk, af, nonzero, orient=0):
        ops.extract_cubes(self.af3, ijk, self.grid_size, self.padding, self.perm, out=af,
                          global_nz=self.global_nz, z0=self.z0, nonzero=nonzero, orient=orient)

    def _window_max(self, ijk):
        # this rank's cubes on its block, halo included: the planes are the whole map's bits, so are the decisions
        return ops.cube_window_max(self.normalized, ijk, self.grid_size, self.padding, self.perm,
                                   global_nz=self.global_nz, z0=self.z0)

    def _new_volumes(self):
        org, ext = self.box
        return ops.StitchedVolumes(self.cube_shape, self.device, org=org, ext=ext)

    def _owner_bounds(self):
        return 2, [r.out_lo for r in self.plan.ranks] + [self.plan.ranks[-1].out_hi]

    def _n_max(self):
        X, Y, _ = self.cube_shape
        return max(r.out_hi - r.out_lo for r in self.plan.ranks) * X * Y

    def _make_stitcher(self, w1, codes, vols):
        if w1 is None:                            # the paste: this rank's cores, into its own box
            return MapPipeline._make_stitcher(self, w1, codes, vols)
        return super()._make_stitcher(w1, codes, vols)


class BalancedCubePipeline(_SplitMap, MapPipeline):
    """One map, its cubes dealt out EVENLY over the ranks (BASELINE configs[4]: the model-bound inference
    loop, where whole cube layers per rank would leave 11 layers / 8 GPUs = 69 % balance).

    Every rank runs the cheap pre-phase on the whole map (resample, normalise, atom bins: ~2 ms against
    seconds of convolutions -- replicating it needs no exchange at all), cuts and feeds only ITS cubes
    (a contiguous range of the loop order), and stores every core straight into the volume block of the
    rank that owns that x range: local memory or a peer's over NVLink (``ops.postproc_stitch_peer`` --
    softmax/argmax + stitch fused with its exchange, no NCCL call).  The output is thus partitioned
    along cube axis 0, ``x_bounds[r] .. x_bounds[r+1]`` on rank r; ``finish_map()`` (stream sync +
    barrier) makes every rank's block final.  No reference counterpart (the reference is single-GPU).

    With ``overlap_window`` (or ``tta``) every window contribution is added into the block of the rank that owns its x
    plane; the normaliser comes from the full cube lattice, also under ``cube_subset``.  ``min_max``: every rank
    measures the whole map and deals the kept cubes as ``cube_subset`` (``cubes_per_rank``)."""

    def __init__(self, device, rank, world, grid_size=48, padding=8, order=3, batch_cubes=16,
                 target_voxel_size=1.0, group=None, af3_mode='sparse', cube_subset=None, _peer_volumes=None):
        super().__init__(device, grid_size, padding, order, batch_cubes, target_voxel_size, af3_mode)
        self.rank, self.world, self.group = int(rank), int(world), group
        self.cube_subset = cube_subset            # optional indices into the loop-order cube list (bounded runs)
        self.peer_volumes = _peer_volumes
        self.x_bounds = None

    def cube_index(self, subset=None):
        """Deal ``subset`` (indices into the loop-order cube list; default ``cube_subset``, None = all) over the ranks."""
        perm, offset = self.header.transpose_order()
        self.perm, self.offset = perm, offset
        self.cube_shape = ops.cube_space_shape(self.normalized.shape, perm)
        ijk = ops.cube_origins(self.cube_shape, self.grid_size)
        if subset is None:
            subset = self.cube_subset
        if subset is not None:
            subset = np.asarray(subset, dtype=np.int64)
            ijk = ijk[subset]
        b = _split_even(len(ijk), self.world)
        self.cube_range = (b[self.rank], b[self.rank + 1])
        self.cubes_per_rank = [b[r + 1] - b[r] for r in range(self.world)]
        self._set_cube_origins(ijk[b[self.rank]:b[self.rank + 1]],
                               (self.cube_shape, self.grid_size, self.rank, self.world, len(ijk),
                                None if subset is None else hash(subset.tobytes())))
        self.x_bounds = _split_even(self.cube_shape[0], self.world)
        self.box = ((self.x_bounds[self.rank], 0, 0),
                    (self.x_bounds[self.rank + 1] - self.x_bounds[self.rank], self.cube_shape[1], self.cube_shape[2]))
        return self.ijk_host

    def _keep_rule(self, min_max, order):
        """Every rank measures the whole map (``cube_subset``, if set, in its order) and deals the kept cubes -- the
        same list on every rank; every owner clears the skipped cores in its own box (nobody stores there)."""
        if order is not None:
            raise MicaError('BalancedCubePipeline deals the cubes itself: pass cube_subset, not order, with min_max')
        idx = np.arange(len(ops.cube_origins(self.cube_shape, self.grid_size)), dtype=np.int64) \
            if self.cube_subset is None else np.asarray(self.cube_subset, dtype=np.int64)
        cand = ops.cube_origins(self.cube_shape, self.grid_size)[idx]
        kept = ops.select_cubes(self._window_max(torch.from_numpy(cand).to(self.device)), min_max)
        mask = np.zeros(len(idx), dtype=bool)
        mask[kept] = True
        self.cube_index(idx[kept])
        return None, np.ascontiguousarray(cand[~mask])

    def _n_max(self):
        _, Y, Z = self.cube_shape
        return max(self.x_bounds[r + 1] - self.x_bounds[r] for r in range(self.world)) * Y * Z

    def _new_volumes(self):
        return self._exported_volumes(self._n_max())

    def _owner_bounds(self):
        return 0, self.x_bounds
