"""Peer-memory groups for the multi-GPU exchanges (SURVEY.md 8e).

One buffer per rank, mapped by the other ranks of the box through CUDA IPC, so that the exchange
kernels can publish / signal / wait / read over NVLink inside a kernel instead of an NCCL call:

  PeerHistogram   ``mica_select_peer_reduce``: the histogram all-reduce of every radix round;
  PeerIntHistogram ``mica_int_stats_peer_publish`` / ``_sum``: the histogram sum of an integer map's statistics;
  PeerHalo        ``mica_halo_publish_bytes`` / ``mica_halo_pull_bytes``: the z-halo planes of the source map;
  PeerVolumes     the stitched output volumes of every rank, so that ``postproc_stitch`` can store a
                  core straight into the volumes of the rank that owns it (config 5: cubes dealt out
                  evenly, softmax/argmax + stitch fused with its exchange).

``torch.distributed`` is only used once per group, to hand the 64-byte IPC handles around.
``emulate`` builds the same structures for several "ranks" inside one process (plain pointers, no
IPC) for the single-GPU tests."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import lib, check


class _IpcGroup:
    """``world`` device buffers of ``nbytes`` each, one per rank, every one mapped in this process."""

    def __init__(self, device, rank, world, nbytes, group=None, _emulated=None, fixed_hist=False):
        self.device, self.rank, self.world = torch.device(device), int(rank), int(world)
        self.nbytes = int(nbytes)
        self._opened, self._own, self._owned_all = [], None, []
        if _emulated is not None:                       # in-process emulation: pointers are shared directly
            ptrs = _emulated
            idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
            self.devices = [idx] * self.world
        else:
            import torch.distributed as dist
            torch.cuda.set_device(self.device)
            own = C.c_void_p()
            handle = (C.c_ubyte * 64)()
            if fixed_hist:
                check(lib.mica_peer_alloc(C.byref(own), handle), 'peer_alloc')
            else:
                check(lib.mica_ipc_alloc(self.nbytes, C.byref(own), handle), 'ipc_alloc')
            self._own = own.value
            gathered = [None] * self.world
            dist.all_gather_object(gathered, (bytes(handle), self.device.index), group=group)
            self.devices = [d for _, d in gathered]       # each rank's CUDA device index
            ptrs = []
            for r, (h, _) in enumerate(gathered):
                if r == self.rank:
                    ptrs.append(self._own)
                    continue
                p = C.c_void_p()
                buf = (C.c_ubyte * 64).from_buffer_copy(h)
                check(lib.mica_peer_open(buf, C.byref(p)), f'peer_open(rank {r})')
                self._opened.append(p.value)
                ptrs.append(p.value)
        self.ptrs = list(ptrs)
        self.table = torch.tensor(ptrs, dtype=torch.int64, device=self.device)

    @classmethod
    def _emulate_ptrs(cls, device, world, nbytes, fixed_hist=False):
        device = torch.device(device)
        torch.cuda.set_device(device)
        ptrs = []
        for _ in range(world):
            p = C.c_void_p()
            if fixed_hist:
                check(lib.mica_peer_alloc(C.byref(p), None), 'peer_alloc')
            else:
                check(lib.mica_ipc_alloc(int(nbytes), C.byref(p), None), 'ipc_alloc')
            ptrs.append(p.value)
        return ptrs

    def _stream(self, stream=None):
        return C.c_void_p(stream if stream is not None else torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        torch.cuda.synchronize(self.device)
        for p in self._opened:
            lib.mica_peer_close(C.c_void_p(p))
        self._opened = []
        for p in self._owned_all + ([self._own] if self._own else []):
            lib.mica_peer_free(C.c_void_p(p))
        self._own, self._owned_all = None, []


class PeerHistogram(_IpcGroup):
    def __init__(self, device, rank: int, world: int, group=None, _emulated=None):
        super().__init__(device, rank, world, lib.mica_peer_buffer_bytes(), group, _emulated, fixed_hist=True)
        self.epoch = 0

    @classmethod
    def emulate(cls, device, world: int):
        """``world`` groups for ranks 0..world-1 living in this process (tests)."""
        ptrs = cls._emulate_ptrs(device, world, 0, fixed_hist=True)
        groups = [cls(device, r, world, _emulated=ptrs) for r in range(world)]
        groups[0]._owned_all = ptrs                     # freed with the first group
        return groups

    def reduce(self, stats, round_index: int, stream=None):
        """Sum every rank's histogram of this round into ``stats`` (an ops.OrderStats), in stream order."""
        # the slot alternates with the EPOCH (not the select step): a map has an odd number of steps, so the
        # last exchange of one map and the first of the next would otherwise share a slot back to back
        self.epoch += 1
        with torch.cuda.device(self.device):
            check(lib.mica_select_peer_reduce(stats._p, C.c_void_p(self.table.data_ptr()), self.rank, self.world,
                                              self.epoch & 1, self.epoch, int(round_index), self._stream(stream)),
                  'select_peer_reduce')


class PeerIntHistogram(_IpcGroup):
    """The histogram sum of ``ops.IntOrderStats`` over peer memory: a publish kernel and a sum kernel per map."""

    def __init__(self, device, rank: int, world: int, group=None, _emulated=None):
        super().__init__(device, rank, world, lib.mica_int_peer_buffer_bytes(), group, _emulated)
        self.epoch = 0

    @classmethod
    def emulate(cls, device, world: int):
        """``world`` groups for ranks 0..world-1 living in this process (tests)."""
        ptrs = cls._emulate_ptrs(device, world, lib.mica_int_peer_buffer_bytes())
        groups = [cls(device, r, world, _emulated=ptrs) for r in range(world)]
        groups[0]._owned_all = ptrs                     # freed with the first group
        return groups

    def publish(self, stats, dtype_code: int, stream=None):
        """Step 1 (never waits): make this rank's histogram (``stats``, an ops.IntOrderStats after its hist)
        available to the peers, for the next epoch."""
        self.epoch += 1
        with torch.cuda.device(self.device):
            check(lib.mica_int_stats_peer_publish(stats._p, int(dtype_code), C.c_void_p(self.table.data_ptr()),
                                                  self.rank, self.world, self.epoch & 1, self.epoch,
                                                  self._stream(stream)), 'int_stats_peer_publish')

    def sum(self, stats, dtype_code: int, stream=None):
        """Step 2: wait for every peer's histogram of the current epoch and sum them into ``stats``."""
        with torch.cuda.device(self.device):
            check(lib.mica_int_stats_peer_sum(stats._p, int(dtype_code), C.c_void_p(self.table.data_ptr()),
                                              self.rank, self.world, self.epoch & 1, self.epoch,
                                              self._stream(stream)), 'int_stats_peer_sum')

    def reduce(self, stats, dtype_code: int, stream=None):
        """Both steps, in stream order: one rank per process (the ranks of one GPU must publish first, all of them)."""
        self.publish(stats, dtype_code, stream)
        self.sum(stats, dtype_code, stream)


class PeerHalo(_IpcGroup):
    """Source-halo exchange with the two z-neighbours over peer memory.  ``slot_elems``: capacity of one
    direction's halo in 4-byte words (float32 elements; planes of a narrower type fill it byte by byte); a plan
    that needs more (or planes from a rank that is not a neighbour) falls back to ``slab.exchange_source_halo``
    (NCCL send/recv)."""

    def __init__(self, device, rank: int, world: int, slot_elems: int, group=None, _emulated=None):
        self.slot_elems = int(slot_elems)
        super().__init__(device, rank, world, lib.mica_halo_buffer_bytes(self.slot_elems), group, _emulated)
        self.epoch = 0
        self.status = torch.zeros(1, dtype=torch.int32, device=self.device)

    @classmethod
    def emulate(cls, device, world: int, slot_elems: int):
        ptrs = cls._emulate_ptrs(device, world, lib.mica_halo_buffer_bytes(int(slot_elems)))
        groups = [cls(device, r, world, slot_elems, _emulated=ptrs) for r in range(world)]
        groups[0]._owned_all = ptrs
        return groups

    @staticmethod
    def neighbour_plan(plan, rank):
        """(send_lo, send_hi, recv_lo, recv_hi) as (plane_lo, plane_hi) global source-plane ranges (or None),
        or None when the plan involves a rank that is not a direct neighbour."""
        sends, recvs = plan.transfers(rank)
        out = {'send': {}, 'recv': {}}
        for kind, lst in (('send', sends), ('recv', recvs)):
            for p, a, b in lst:
                if abs(p - rank) != 1 or p in out[kind]:
                    return None
                out[kind][p] = (a, b)
        return (out['send'].get(rank - 1), out['send'].get(rank + 1), out['recv'].get(rank - 1),
                out['recv'].get(rank + 1))

    @staticmethod
    def slot_words(plan, rank_range_planes: int, itemsize: int = 4) -> int:
        """4-byte words a slot needs for ``rank_range_planes`` source planes of ``itemsize``-byte samples."""
        return -(-rank_range_planes * plan.src_shape[1] * plan.src_shape[2] * int(itemsize) // 4)

    def fits(self, plan, rank, itemsize: int = 4):
        np_ = self.neighbour_plan(plan, rank)
        if np_ is None:
            return False
        return all(r is None or self.slot_words(plan, r[1] - r[0], itemsize) <= self.slot_elems for r in np_)

    def publish(self, own: torch.Tensor, plan, stream=None):
        """Step 1 (never waits): make the boundary planes of ``own`` (this rank's block) available."""
        me = plan.ranks[self.rank]
        s_lo, s_hi, _, _ = self.neighbour_plan(plan, self.rank)
        plane = plan.src_shape[1] * plan.src_shape[2] * own.element_size()       # bytes
        self.epoch += 1
        off_lo, n_lo = ((s_lo[0] - me.own_lo) * plane, (s_lo[1] - s_lo[0]) * plane) if s_lo else (0, 0)
        off_hi, n_hi = ((s_hi[0] - me.own_lo) * plane, (s_hi[1] - s_hi[0]) * plane) if s_hi else (0, 0)
        with torch.cuda.device(self.device):
            check(lib.mica_halo_publish_bytes(C.c_void_p(own.data_ptr()), off_lo, n_lo, off_hi, n_hi,
                                              C.c_void_p(self.table.data_ptr()), self.rank, self.world,
                                              self.epoch & 1, self.epoch, 4 * self.slot_elems, self._stream(stream)),
                  'halo_publish')

    def pull(self, buf: torch.Tensor, plan, stream=None):
        """Step 2: wait for the neighbours' planes of the current epoch and copy them into ``buf``
        (global source planes [src_lo, src_hi) of this rank)."""
        me = plan.ranks[self.rank]
        _, _, r_lo, r_hi = self.neighbour_plan(plan, self.rank)
        plane = plan.src_shape[1] * plan.src_shape[2] * buf.element_size()       # bytes
        flat = buf.view(-1).view(torch.uint8)
        d_lo = flat[(r_lo[0] - me.src_lo) * plane:] if r_lo else None
        d_hi = flat[(r_hi[0] - me.src_lo) * plane:] if r_hi else None
        with torch.cuda.device(self.device):
            check(lib.mica_halo_pull_bytes(C.c_void_p(d_lo.data_ptr()) if r_lo else None,
                                           (r_lo[1] - r_lo[0]) * plane if r_lo else 0,
                                           C.c_void_p(d_hi.data_ptr()) if r_hi else None,
                                           (r_hi[1] - r_hi[0]) * plane if r_hi else 0,
                                           C.c_void_p(self.table.data_ptr()), self.rank, self.world, self.epoch & 1,
                                           self.epoch, 4 * self.slot_elems, C.c_void_p(self.status.data_ptr()),
                                           self._stream(stream)), 'halo_pull')

    def exchange(self, own: torch.Tensor, plan, buf: torch.Tensor | None = None) -> torch.Tensor:
        """Assemble source planes [src_lo, src_hi): own part by a device copy, the rest from the neighbours.
        ``buf``: a caller-owned buffer of that shape (a new one otherwise)."""
        me = plan.ranks[self.rank]
        n = max(0, me.src_hi - me.src_lo)
        self.publish(own, plan)
        shape = (n,) + tuple(own.shape[1:])
        if buf is None:
            buf = torch.empty(shape, dtype=own.dtype, device=own.device)
        elif tuple(buf.shape) != shape or buf.dtype != own.dtype or not buf.is_contiguous():
            raise _lib.MicaError(f'halo buffer has shape {tuple(buf.shape)}, expected {shape}')
        lo, hi = max(me.src_lo, me.own_lo), min(me.src_hi, me.own_hi)
        if hi > lo:
            buf[lo - me.src_lo:hi - me.src_lo].copy_(own[lo - me.own_lo:hi - me.own_lo])
        self.pull(buf, plan)
        return buf

    def timed_out(self) -> bool:
        return bool(int(self.status.item()))


class PeerVolumes(_IpcGroup):
    """Every rank's stitched volumes (23 float32 channels of one [X,Y,Z] box each) in exported memory:
    ``table`` holds the base pointer of each rank's block, laid out as
    [backbone | carbon_alpha | amino_acid_prediction | amino_acid_probability x 20] x (X*Y*Z) floats."""

    CHANNELS = 23

    def __init__(self, device, rank: int, world: int, n_voxels: int, group=None, _emulated=None):
        self.n_voxels = int(n_voxels)
        super().__init__(device, rank, world, self.CHANNELS * self.n_voxels * 4, group, _emulated)

    @classmethod
    def emulate(cls, device, world: int, n_voxels: int):
        ptrs = cls._emulate_ptrs(device, world, cls.CHANNELS * int(n_voxels) * 4)
        groups = [cls(device, r, world, n_voxels, _emulated=ptrs) for r in range(world)]
        groups[0]._owned_all = ptrs
        return groups

    def block(self, rank=None, n_elems=None) -> torch.Tensor:
        """A float32 tensor aliasing a rank's exported block (default: this rank's own)."""
        r = self.rank if rank is None else int(rank)
        n = self.CHANNELS * self.n_voxels if n_elems is None else int(n_elems)
        return torch.as_tensor(_RawCuda(self.ptrs[r], n), device=self.device)


class _RawCuda:
    """Exposes raw device memory through ``__cuda_array_interface__`` so that torch can alias it."""

    def __init__(self, ptr, n_floats):
        self.__cuda_array_interface__ = {'shape': (int(n_floats),), 'typestr': '<f4', 'data': (int(ptr), False),
                                         'version': 2, 'strides': None}
