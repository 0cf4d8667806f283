"""The voxel-parallel map pipeline, resident in HBM end to end.

    source map --resample--> 1 A grid --median/p99.9--> normalised map ---+
    docked atoms --rasterise--> 24-channel AF3 volume --------------------+--> 64^3 cube batches
        --> [model: models/model.py MICA, unchanged PyTorch] --> logits --softmax/argmax+stitch--> 4 volumes

This is the dataflow of Solver.getData + Solver.nnPred (utils/modeler.py:673-760 in the
reference) with every .mrc / .npz round trip removed: the stages hand device tensors to
each other and the cubes are cut straight into the model's input batch.  The reference
entry points (DataPreprocessor / GridCreator / CryoEMPredictor mirrors in
preprocessing.py, create_grids.py, predict.py) are thin shells over this class.
"""
from __future__ import annotations

import bisect
import functools
import time
from contextlib import contextmanager
from dataclasses import dataclass

import numpy as np
import torch

from . import ops
from ._lib import MicaError, NORM_OK


@dataclass
class MapHeader:
    """The MRC header fields the reference carries through (utils/preprocessing.py:99-107)."""
    voxel_size: tuple = (1.0, 1.0, 1.0)       # (x, y, z)
    origin: tuple = (0.0, 0.0, 0.0)           # (x, y, z)
    mapc: int = 1
    mapr: int = 2
    maps: int = 3
    nxstart: int = 0
    nystart: int = 0
    nzstart: int = 0

    def transpose_order(self):
        """GridCreator.transpose bookkeeping (utils/create_grids.py:67-87,120-122):
        returns (perm, offset) with perm[m] = memory axis walked by cube axis m."""
        axis_order = [int(self.maps) - 1, int(self.mapr) - 1, int(self.mapc) - 1]
        start = [float(self.nzstart), float(self.nystart), float(self.nxstart)]
        perm, offset = [], []
        for i in range(3):
            for j in range(3):
                if axis_order[j] == i:
                    offset.append(start[j])
                    perm.append(j)
        return tuple(perm), offset


def zoom_factors(voxel_size_xyz, target_voxel_size=1.0):
    """[vx, vy, vz] / target, float32 as under NumPy 2, applied to axes (z,y,x) in that
    order -- the reference's own (anisotropy-swapping) convention, utils/preprocessing.py:112-117."""
    return [np.float32(v) / target_voxel_size for v in voxel_size_xyz]


class StageTimer:
    """CUDA-event timing of the pipeline's stages on the launching stream.  Events are
    recorded around every stage call; ``summary()`` (after a synchronize) returns
    {stage: (calls, total_ms)}."""

    def __init__(self, only=None):
        self.spans = []
        self.only = set(only) if only is not None else None     # time just these stages (events are not free)

    @contextmanager
    def __call__(self, name):
        if self.only is not None and name not in self.only:
            yield
            return
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        try:
            yield
        finally:
            b.record()
            self.spans.append((name, a, b))

    def summary(self):
        out = {}
        for name, a, b in self.spans:
            c, t = out.get(name, (0, 0.0))
            out[name] = (c + 1, t + a.elapsed_time(b))
        return out

    def reset(self):
        self.spans = []


@contextmanager
def _no_timer(name):
    yield


def _on_device(method):
    """Run a pipeline method with the pipeline's GPU current (events, side streams and the C ABI all
    act on the CUDA runtime's current device)."""
    @functools.wraps(method)
    def wrapper(self, *args, **kw):
        if self.device.index is None or self.device.index == torch.cuda.current_device():
            return method(self, *args, **kw)
        with torch.cuda.device(self.device):
            return method(self, *args, **kw)
    return wrapper


D8_MODES = ('none', 'split', 'reference')

#: the logits hand-off of the stitch (``ops.Stitcher.kernel_logits``), importable from here as before
_f32c = ops.Stitcher.kernel_logits


def run_model_chunks(model_fn, x, af, flags_host, ijk, stitch, model_batch=None, d8='none'):
    """Feed one super-batch of cubes to ``model_fn`` the way the reference feeds MICA.forward, and hand
    every result to ``stitch(bb, ca, aa, ijk_chunk)`` (an ``ops.Stitcher``, or a function calling one).

    ``model_batch``: cubes per model call (the reference: 1 up to 200 cubes, else <= 8,
    utils/predict.py:156-215); None = the whole super-batch in one call.
    ``d8``: MICA.forward decides ``is_af_zero = af_features.abs().sum() < 1e-6`` over the WHOLE batch
    (models/model.py:60-63), so a cube without AF3 signal gets different logits when it shares a batch
    with one that has some.
      'split'      every model call sees either only zero-AF3 cubes or only non-zero ones
                   (``flags_host[b] != 0`` = cube b has AF3 signal): each cube gets what the reference's
                   single-sample mode gives it, whatever it is batched with;
      'reference'  consecutive cubes are batched as they come, mixed -- the reference's batched mode;
      'none'       same as 'reference' (for stand-in models without that branch)."""
    if d8 not in D8_MODES:
        raise MicaError(f'd8 must be one of {D8_MODES}, got {d8!r}')
    B = int(x.shape[0])
    mb = B if model_batch is None else max(1, int(model_batch))
    # all chunk views at once (three C++ calls instead of three Python slicings per chunk: the loop below runs
    # hundreds of times per map when the model takes 8 cubes at a time)
    xs, afs, ijks = x.split(mb), af.split(mb), ijk.split(mb)
    split = d8 == 'split' and mb > 1
    if split:
        nz = np.asarray(flags_host) != 0
    for n_chunk, c0 in enumerate(range(0, B, mb)):
        c1 = min(B, c0 + mb)
        groups = [None]
        if split and c1 - c0 > 1:
            f = nz[c0:c1]
            if f.any() and not f.all():
                groups = [np.flatnonzero(f), np.flatnonzero(~f)]
        for g in groups:
            if g is None:
                gx, gaf, gijk = xs[n_chunk], afs[n_chunk], ijks[n_chunk]
            else:
                idx = torch.as_tensor(g + c0, device=x.device)
                gx, gaf, gijk = x[idx], af[idx], ijk[idx].contiguous()
            bb, ca, aa = model_fn(gx, gaf)
            stitch(bb, ca, aa, gijk)


def _chunk_starts(n_cubes, super_batch, model_batch):
    """Where the model calls of a one-device run start: the visiting order is cut into super-batches of
    ``super_batch`` cubes and each of them into chunks of ``model_batch`` (``run_model_chunks``)."""
    sb, mb = max(1, int(super_batch)), max(1, int(model_batch))
    return [c for s in range(0, n_cubes, sb) for c in range(s, min(n_cubes, s + sb), mb)]


def deal_cubes(n_cubes, super_batch, model_batch, n_workers):
    """Deal a map's cubes over ``n_workers`` devices without changing any model call.

    Returns one contiguous range (lo, hi) of the visiting order per worker.  Every bound is where a
    model call of the one-device run starts (or the end), so the calls the workers make -- with
    ``worker_batches`` -- are exactly the one-device calls: with TF32 convolutions a cube's logits depend on
    the batch it is convolved in, and MICA's zero-AF3 branch is taken per batch (D8).  Each bound is the
    chunk start nearest to an even split, so every worker's count is within one chunk (``model_batch``
    cubes) of ``n_cubes / n_workers``; with fewer chunks than workers some ranges are empty."""
    n, w = int(n_cubes), int(n_workers)
    if w < 1:
        raise MicaError(f'n_workers must be >= 1, got {n_workers}')
    cuts = _chunk_starts(n, super_batch, model_batch) + [n]
    bounds = [0]
    for r in range(1, w):
        target = n * r / w
        i = bisect.bisect_left(cuts, target)
        if i == len(cuts) or (i > 0 and target - cuts[i - 1] <= cuts[i] - target):
            i -= 1
        bounds.append(max(bounds[-1], cuts[i]))
    bounds.append(n)
    return [(bounds[r], bounds[r + 1]) for r in range(w)]


def worker_batches(lo, hi, super_batch):
    """A worker's range cut at the one-device super-batch boundaries inside it, as (b0, b1) relative to ``lo``:
    the super-batches ``MapPipeline.predict_and_stitch(batches=)`` then feeds to ``run_model_chunks``."""
    sb = max(1, int(super_batch))
    cuts = [lo] + list(range((lo // sb + 1) * sb, hi, sb)) + [hi]
    return [(a - lo, b - lo) for a, b in zip(cuts[:-1], cuts[1:]) if b > a]


class MapPipeline:
    """One GPU's share of the hot path.  With ``slab`` left None it owns the whole map."""

    def __init__(self, device, grid_size: int = 48, padding: int = 8, order: int = 3,
                 batch_cubes: int = 16, target_voxel_size: float = 1.0, af3_mode: str = 'sparse',
                 cube_dtype=torch.float32):
        #: element type of the cube batches handed to ``model_fn`` (map and AF3 channels): torch.float32 or
        #: torch.bfloat16 (each voxel rounded once to nearest even; the AF3 channels' 1 / 0 are exact).  Running the
        #: model in a matching precision is the caller's job; the stitch takes float32 or bfloat16 logits.
        self.cube_dtype = ops.model_dtype(cube_dtype)
        ops.require_gpu()
        self.device = torch.device(device)
        self.grid_size, self.padding, self.order = int(grid_size), int(padding), int(order)
        self.window = self.grid_size + 2 * self.padding
        self.batch_cubes = int(batch_cubes)
        self.target_voxel_size = target_voxel_size
        self.header = MapHeader()
        self.normalized = None          # [nz,ny,nx] float32, device
        self.af3 = None                 # [24,nz,ny,nx] float32, device (None -> zero AF3 features)
        self.stats = None               # OrderStats, or IntOrderStats for an integer map
        self._stats = None
        self._int_stats = None
        self.norm_status = None
        self._x, self._af, self._nz = [None, None], [None, None], [None, None]
        self.timer = _no_timer      # bench.py swaps in a StageTimer
        #: upper clip bounds for the (x,y,z) atom indices; None = the reference's (nz-1,ny-1,nx-1) quirk (D7)
        self.af3_clip = None
        #: 'sparse' = AF3 channels of each batch written straight from binned atoms (no dense volume);
        #: 'dense'  = the reference's dataflow: dense 24-channel volume, then window extraction
        if af3_mode not in ('sparse', 'dense'):
            raise MicaError(f'af3_mode must be sparse or dense, got {af3_mode!r}')
        self.af3_mode = af3_mode
        self._fillers = [None, None]    # one per prefetch buffer
        self._bins = None               # the filler that holds the per-cube atom bins of the current map
        self._atoms_binned = False
        #: cut batch n+1 on a side stream while the model and the stitch of batch n run on the
        #: caller's stream (two input buffers).  False = everything on the caller's stream.
        self.prefetch = True
        self._deferred = []
        self._pinned_free = []          # (order-stats record, AF3 status word) pairs in pinned memory, reused:
        self._pre_stream = None         # cudaHostAlloc synchronises the device, so never allocate per step

    def configure(self, grid_size=None, padding=None, batch_cubes=None, order=None, target_voxel_size=None,
                  cube_dtype=None):
        """Change the cube geometry / batch size / ``cube_dtype`` of a live pipeline (the drop-in classes learn them
        stage by stage: ``GridCreator`` is told grid_size and padding after ``DataPreprocessor`` has already
        normalised the map).  Buffers that depend on what changed are dropped and rebuilt on demand (a new
        ``cube_dtype`` drops the slot buffers of the cubes and of the AF3 fillers; the atom bins stay)."""
        if cube_dtype is not None and ops.model_dtype(cube_dtype) != self.cube_dtype:
            self.cube_dtype = cube_dtype
            self._x, self._af, self._nz = [None, None], [None, None], [None, None]
            for f in self._fillers:
                if f is not None:
                    f.retype(cube_dtype)
        gs = self.grid_size if grid_size is None else int(grid_size)
        pad = self.padding if padding is None else int(padding)
        bc = self.batch_cubes if batch_cubes is None else int(batch_cubes)
        if order is not None:
            self.order = int(order)
        if target_voxel_size is not None:
            self.target_voxel_size = target_voxel_size
        if (gs, pad, bc) != (self.grid_size, self.padding, self.batch_cubes):
            if gs + 2 * pad != self.window or bc > self.batch_cubes:
                self._x, self._af, self._nz = [None, None], [None, None], [None, None]
            if (gs, pad) != (self.grid_size, self.padding) or bc > self.batch_cubes:
                self._fillers, self._bins, self._atoms_binned = [None, None], None, False
            self.grid_size, self.padding, self.batch_cubes = gs, pad, bc
            self.window = gs + 2 * pad
            self._ijk_key = None
        return self

    def release_map(self):
        """Forget the current map (normalised volume, dense AF3 volume, atom bins stay allocated but
        unused): lets the caller's session drop its HBM."""
        self.normalized, self.af3 = None, None
        self._atoms_binned = False

    # ------------------------------------------------------------------ stage 1+2
    @_on_device
    def resample_and_normalize(self, src: torch.Tensor, header: MapHeader | None = None, defer_status=False):
        """utils/preprocessing.py:98-133 on the device.  Returns True on success; on the
        reference's two failure modes (:152-157) returns False and leaves ``normalized`` None.
        ``defer_status=True`` skips the host read-back (one stream sync) -- the caller then
        calls ``check_status()`` once everything is enqueued.  An int8 / int16 / uint16 ``src`` is
        resampled into its own type and normalised in float64 into a new float32 volume (D12); ``median``
        and ``p999`` are then Python floats."""
        if header is not None:
            self.header = header
        zf = zoom_factors(self.header.voxel_size, self.target_voxel_size)
        out_shape = ops.zoom_output_shape(src.shape, zf)
        with self.timer('resample'):
            if all(float(z) == 1.0 for z in zf):              # SciPy early exit (D10): plain copy
                res = src.clone()
            else:
                res = ops.resample(src, out_shape, order=self.order)
        if res.dtype in ops.INT_DTYPES:                       # integer map: float64 statistics (D12)
            with self.timer('order_stats'):
                self.stats = self._int_order_stats().run(res)
            with self.timer('normalize_apply'):
                self.normalized = self.stats.apply(res)        # a new float32 volume
        else:
            with self.timer('order_stats'):
                self.stats = self._order_stats().run(res)
            with self.timer('normalize_apply'):
                self.normalized = self.stats.apply(res, res)   # in place: the resampled map is not kept
        self.norm_status = None
        return True if defer_status else self.check_status()

    def _order_stats(self):
        """The select workspace lives as long as the pipeline (allocating and zero-filling it per map
        cost a cudaMalloc-class call on the B <= 8 drop-in path); every run re-initialises it in
        stream order."""
        if self._stats is None:
            self._stats = ops.OrderStats(self.device)
        return self._stats

    def _int_order_stats(self):
        if self._int_stats is None:
            self._int_stats = ops.IntOrderStats(self.device)
        return self._int_stats

    @_on_device
    def check_status(self):
        med, p, npos, status = self.stats.result()
        self.norm_status = status
        self.median, self.p999, self.n_pos = med, p, npos
        if status != NORM_OK:
            self.normalized = None
        return status == NORM_OK

    def set_normalized(self, norm: torch.Tensor, header: MapHeader | None = None):
        if header is not None:
            self.header = header
        self.normalized = norm

    # -------------------------------------------------------------------- stage 3
    @_on_device
    def encode_af3(self, coords: torch.Tensor, bb_ch: torch.Tensor, aa_ch: torch.Tensor, defer_status=False):
        """utils/preprocessing.py:268-298.  Returns True iff the reference would have
        succeeded (no IndexError from the mis-ordered clip, D7)."""
        if self.normalized is None:
            raise MicaError('encode_af3 needs the normalised map (its shape and origin)')
        if self.af3_mode == 'sparse':
            perm, _ = self.header.transpose_order()
            for i in range(2):
                f = self._fillers[i]
                if f is None or f.perm != tuple(perm) or f.n_slots < self.batch_cubes:
                    self._fillers[i] = ops.Af3CubeFiller(self.device, self.batch_cubes, self.grid_size,
                                                         self.padding, perm, dtype=self.cube_dtype)
                else:
                    f.clear()                         # with the OLD bins, before they are rebuilt
            f = self._fillers[0]
            with self.timer('af3_bin_atoms'):
                status = f.bin(coords, bb_ch, aa_ch, self.header.origin, self._global_shape(), self.af3_clip)
            self._fillers[1].share_bins(f)
            self.af3, self._af3_status, self._atoms_binned = None, status, True
            if defer_status:
                return True
            self._atoms_binned = int(status.item()) == 0
            return self._atoms_binned
        with self.timer('af3_encode'):
            vol, status = ops.af3_encode(coords, bb_ch, aa_ch, self.header.origin, tuple(self.normalized.shape),
                                         clip_hi_xyz=self.af3_clip)
        self.af3, self._af3_status, self._atoms_binned = vol, status, False
        if defer_status:
            return True
        ok = int(status.item()) == 0
        self.af3 = vol if ok else None
        return ok

    def _global_shape(self):
        return tuple(self.normalized.shape)

    # -------------------------------------------------------------------- stage 4
    def cube_index(self):
        perm, offset = self.header.transpose_order()
        self.perm, self.offset = perm, offset
        self.cube_shape = ops.cube_space_shape(self.normalized.shape, perm)
        self._set_cube_origins(ops.cube_origins(self.cube_shape, self.grid_size), (self.cube_shape, self.grid_size))
        return self.ijk_host

    def _set_cube_origins(self, ijk_host, key):
        """Upload the cube origins once per geometry: a pageable host->device copy blocks the host until
        all earlier work of the stream has run, i.e. it would serialise consecutive maps."""
        if getattr(self, '_ijk_key', None) != key:
            self.ijk_host = np.ascontiguousarray(ijk_host)
            self.ijk = torch.from_numpy(self.ijk_host).to(self.device)
            self._ijk_key = key

    def _buffers(self, B, slot=0):
        W = self.window
        if self._x[slot] is None or self._x[slot].shape[0] < B:
            self._x[slot] = torch.empty((B, 1, W, W, W), dtype=self.cube_dtype, device=self.device)
            self._nz[slot] = torch.empty(B, dtype=torch.int32, device=self.device)
        return self._x[slot][:B], self._nz[slot][:B]

    def _af_buffer(self, B, slot=0):
        W = self.window
        if self._af[slot] is None or self._af[slot].shape[0] < B:
            self._af[slot] = torch.empty((B, 24, W, W, W), dtype=self.cube_dtype, device=self.device)
        return self._af[slot][:B]

    def _extract_map(self, ijk, x, orient=0):
        ops.extract_cubes(self.normalized, ijk, self.grid_size, self.padding, self.perm, out=x, orient=orient)

    def _extract_af3(self, ijk, af, nonzero, orient=0):
        ops.extract_cubes(self.af3, ijk, self.grid_size, self.padding, self.perm, out=af, nonzero=nonzero,
                          orient=orient)

    @_on_device
    def extract_batch(self, b0: int, b1: int, want_flags: bool = False, slot: int = 0, orient: int = 0):
        """Cubes [b0,b1) -> (exp_map [B,1,W,W,W], af_features [B,24,W,W,W][, nonzero flags]), both of
        ``cube_dtype`` -- the two tensors MICA.forward takes (models/model.py:331).  ``slot`` picks one of
        the two input buffers (the prefetch of batch n+1 must not overwrite batch n).  ``orient``: both
        tensors in that orientation (``ops.orientation``; the flags do not depend on it)."""
        x, nzf = self._buffers(b1 - b0, slot)
        ijk = self.ijk[b0:b1]
        with self.timer('extract_map'):
            self._extract_map(ijk, x, orient)
        if self._atoms_binned:
            with self.timer('af3_fill_cubes'):
                af = self._fillers[slot].fill(ijk, nzf if want_flags else None, orient)
        elif self.af3 is not None:
            af = self._af_buffer(b1 - b0, slot)
            with self.timer('extract_af3'):
                self._extract_af3(ijk, af, nzf if want_flags else None, orient)
        else:
            af = self._af_buffer(b1 - b0, slot)
            af.zero_()                                         # dataset/dataset.py:218-219
            if want_flags:
                nzf.zero_()
        return (x, af, nzf) if want_flags else (x, af)

    def _new_volumes(self):
        return ops.StitchedVolumes(self.cube_shape, self.device)

    # ---------------------------------------------------------------- stage 5 (+model)
    @_on_device
    def predict_and_stitch(self, model_fn, vols: ops.StitchedVolumes | None = None, on_batch=None, *,
                           model_batch=None, d8='none', order=None, overlap_window=None, batches=None, tta=None,
                           min_max=None, stitcher: ops.Stitcher | None = None):
        """run_inference + reconstruct_volume (utils/predict.py:307-587) without the
        per-cube files.  ``model_fn(exp_map, af_features) -> (bb, ca, aa)`` logits, enqueued
        on the current stream.  With ``prefetch`` the cubes of batch n+1 are cut on a side
        stream while the model and the softmax/argmax + stitch of batch n run.
        ``on_batch(vols, n_done)`` is called after the stitch of each batch has been enqueued
        (``n_done`` cubes of ``ijk_host`` are then final in ``vols``, in stream order).

        Cubes are cut ``batch_cubes`` at a time (one launch per stage); ``model_batch`` / ``d8`` say how
        such a super-batch is fed to the model (``run_model_chunks``: the reference's batches of <= 8 and
        its whole-batch zero-AF3 test, D8).  ``order``: a permutation of the cube indices (the reference
        visits cubes in ``glob`` order, utils/predict.py:269); default = the i-major loop order of
        utils/create_grids.py:143-145.  ``overlap_window`` ('uniform' | 'triangle' | 'core' | W weights): the
        north_star's overlap-weighted stitching instead of the reference's centre-crop paste (``ops.Stitcher``; NOT
        the reference's arithmetic, see DESIGN.md D2; 'core' is the paste).  Nothing is final before the last batch, so
        ``on_batch`` is then called once, with the finished volumes.  A split map (subclasses) supplies the owners
        of the output; its volumes are final after ``finish_map()``.  ``batches``: the super-batches as
        (b0, b1) ranges of the (ordered) cube list, each at most ``batch_cubes`` long, instead of the even cut
        (``worker_batches``: a worker's share of a map dealt over several devices).

        ``tta`` ('flips' | 'rot90' | 'all' | orientation codes, ``ops.tta_orientations``): test-time augmentation.
        Every super-batch is cut, run through the model and accumulated once per orientation, and the volumes are
        the average of the k orientations' probabilities (window weights ``overlap_window``, default 'core'), always
        in the order-free fixed point of ``ops.Stitcher`` -- NOT the reference's arithmetic.  The work list is
        the (super-batch, orientation) pairs, fed through the same two-slot prefetch.  ``on_batch`` is called once,
        with the finished volumes.  ``tta=[0]`` is ``tta=None``.

        ``stitcher``: an ``ops.Stitcher`` whose destination the caller owns (several workers adding into one map),
        instead of ``vols`` / ``overlap_window`` / ``tta``; the caller finalizes it, and ``on_batch`` runs only for the
        paste.  Returns its ``vols``.

        ``min_max`` (a finite number; None = every cube): the keep rule of the reference's training grids
        (create_grids_for_normalized_map.py:78) at inference -- only cubes whose window maximum is not below it
        (``ops.cube_window_max`` / ``ops.select_cubes``: ties and NaN windows are kept) reach the model, in the
        relative order they have in ``order`` (or the loop order).  A skipped cube's core is 0 in all four volumes
        (the reference's stitcher where a grid file is absent): caller-given ``vols`` get those cores cleared.  With
        ``overlap_window`` / ``tta`` a skipped window adds nothing and the normaliser stays the full lattice's.  No
        cube kept: zero volumes, the model is not called."""
        if self.normalized is None:
            raise MicaError('no normalised map')
        if stitcher is not None and (vols is not None or overlap_window is not None or tta is not None):
            raise MicaError('a stitcher brings its own volumes, window and orientations: pass it alone')
        w1, codes = ops.stitch_mode(overlap_window, tta, self.grid_size, self.padding)   # refused before any launch
        min_max = ops.check_min_max(min_max)
        self.cube_index()
        # an ascending order is a subsequence of the loop order: finished layers can still be drained (_SlabDrain)
        self._custom_order = order is not None and not bool(np.all(np.diff(np.asarray(order, dtype=np.int64)) > 0))
        skipped = None
        if min_max is not None:
            order, skipped = self._keep_rule(min_max, order)
        st = self._make_stitcher(w1, codes, vols) if stitcher is None else stitcher
        if skipped is not None and vols is not None:      # new volumes are zero: skipped cores need nothing
            st.clear_cores(skipped)
        vols = st.vols
        if order is not None:
            order = np.asarray(order, dtype=np.int64)
            self._set_cube_origins(self.ijk_host[order], ('ordered', id(order), len(order)))
            self._ijk_key = None                          # the next map starts from the loop order again
        n = len(self.ijk_host)
        if batches is None:
            batches = [(b0, min(n, b0 + self.batch_cubes)) for b0 in range(0, n, self.batch_cubes)]
        else:
            batches = [(int(b0), int(b1)) for b0, b1 in batches]
            if any(not 0 <= b0 < b1 <= n or b1 - b0 > self.batch_cubes for b0, b1 in batches):
                raise MicaError(f'batches must be non-empty ranges of the {n} cubes, at most {self.batch_cubes} long')
        work = [(b0, b1, g) for b0, b1 in batches for g in st.orientations]
        per_batch = on_batch if st.per_batch else None
        want_flags = d8 == 'split' and (model_batch is None or int(model_batch) > 1)
        timed = self.timer is not _no_timer

        def consume(cur, b0, b1, g):
            def stitch(bb, ca, aa, ijk):
                if timed:
                    with self.timer('postproc_stitch'):
                        st(bb, ca, aa, ijk, g)
                else:
                    st(bb, ca, aa, ijk, g)
            flags = None
            if want_flags:
                x, af, nzf = cur
                flags = nzf.cpu().numpy()                 # waits for the cut of this batch (it has to be there anyway)
            else:
                x, af = cur[0], cur[1]
            run_model_chunks(model_fn, x, af, flags, self.ijk[b0:b1], stitch, model_batch, d8)

        if not work:                                      # no cube kept (min_max)
            if per_batch is not None:
                per_batch(vols, n)
        elif not self.prefetch or len(work) == 1:
            for b0, b1, g in work:
                consume(self.extract_batch(b0, b1, want_flags=want_flags, orient=g), b0, b1, g)
                if per_batch is not None:
                    per_batch(vols, b1)
        else:
            t_enqueue = time.perf_counter()
            main = torch.cuda.current_stream(self.device)
            if self._pre_stream is None:
                self._pre_stream = torch.cuda.Stream(self.device)
            pre = self._pre_stream
            pre.wait_stream(main)                    # normalised map, atom bins, ijk are produced on `main`
            ready, consumed = [None, None], [None, None]

            def cut(i):
                slot = i & 1
                with torch.cuda.stream(pre):
                    if consumed[slot] is not None:
                        pre.wait_event(consumed[slot])           # the model has read this buffer's last batch
                    b0, b1, g = work[i]
                    out = self.extract_batch(b0, b1, want_flags=want_flags, slot=slot, orient=g)
                    ready[slot] = torch.cuda.Event()
                    ready[slot].record(pre)
                return out

            cur = cut(0)
            for i, (b0, b1, g) in enumerate(work):
                nxt = cut(i + 1) if i + 1 < len(work) else None
                main.wait_event(ready[i & 1])
                consume(cur, b0, b1, g)
                consumed[i & 1] = torch.cuda.Event()
                consumed[i & 1].record(main)
                if per_batch is not None:
                    per_batch(vols, b1)
                cur = nxt
            self.last_loop_enqueue_ms = (time.perf_counter() - t_enqueue) * 1e3     # host side of the batch loop
        return vols if stitcher is not None else self._stitch_done(st, on_batch, n)

    def _window_max(self, ijk):
        """Window maxima of the cubes ``ijk`` (device int32 [B,3]) on this pipeline's normalised map."""
        return ops.cube_window_max(self.normalized, ijk, self.grid_size, self.padding, self.perm)

    def _keep_rule(self, min_max, order):
        """(order, skipped) under the keep rule: ``order`` = the kept indices of ``ijk_host`` in ``order``'s relative
        sequence (ascending = the loop order when ``order`` is None); ``skipped`` = origins (int32 [n,3]) of the cubes
        whose cores this pipeline's volumes must show as 0."""
        kept = ops.select_cubes(self._window_max(self.ijk), min_max)
        mask = np.zeros(len(self.ijk_host), dtype=bool)
        mask[kept] = True
        skipped = np.ascontiguousarray(self.ijk_host[~mask])
        if order is None:
            return kept, skipped
        order = np.asarray(order, dtype=np.int64)
        return order[mask[order]], skipped

    def _make_stitcher(self, w1, codes, vols):
        """The ``ops.Stitcher`` of this map (``ops.stitch_mode``'s ``w1`` / ``codes``): the whole map on this GPU, into
        ``vols`` -- for the weighted stitch ``StitchedVolumes.from_block`` volumes of the whole map, zeroed.  Default:
        new zeroed volumes (the weighted stitch: a block of its own)."""
        if vols is None and w1 is None:
            vols = self._new_volumes()
        return ops.Stitcher(self.cube_shape, self.device, self.grid_size, self.padding, w1, tta=codes, vols=vols)

    def _stitch_done(self, st, on_batch, n):
        """The volumes once every batch has been stitched; ``on_batch`` once if they were not final batch by batch."""
        vols = st.finalize()
        if on_batch is not None and not st.per_batch:
            on_batch(vols, n)
        return vols

    @_on_device
    def finish(self):
        """Wait for every ``run(..., defer_check=True)`` issued so far and raise if one of them failed."""
        pending, self._deferred = self._deferred, []
        for rec, af, ev, decode in pending:
            ev.synchronize()
            self._pinned_free.append((rec, af))
            med, p, npos, status = decode(rec)
            self.norm_status, self.median, self.p999, self.n_pos = status, med, p, npos
            if status != NORM_OK:
                raise MicaError(f'normalisation failed (status {status})')
            if af[1] and int(af[0]) != 0:
                raise MicaError('AF3 encoding failed: atom index outside the grid (reference IndexError path, D7)')

    # ------------------------------------------------------------------ whole path
    def prefetch_source(self, next_src, header=None):
        """Hint: ``next_src`` is the map the next ``run`` will be given.  One GPU has nothing to fetch; a
        z-slab rank exchanges the next map's source halo under this map's cube loop (SlabPipeline)."""

    @_on_device
    def run(self, src, header, atoms, model_fn, vols=None, on_batch=None, defer_check=False, next_src=None,
            **predict_kw):
        """map + atoms -> four stitched volumes (device).  ``atoms`` = (coords, bb_ch, aa_ch)
        device tensors or None.  Raises on the reference's normalisation failures -- at once, or,
        with ``defer_check``, from ``finish()``: the status words are copied to pinned memory in
        stream order and the host does not wait, so the next map can be enqueued while this one
        still runs (a stream of maps; per-step host synchronisation also re-aligns the ranks of
        a multi-GPU run at the cost of their host jitter).  ``next_src``: the source of the map that
        follows (same header), already resident -- see ``prefetch_source``."""
        self.resample_and_normalize(src, header, defer_status=True)
        if atoms is not None:
            self.encode_af3(*atoms, defer_status=True)
        else:
            self.af3, self._atoms_binned = None, False
        if next_src is not None:
            self.prefetch_source(next_src, header)
        vols = self.predict_and_stitch(model_fn, vols, on_batch, **predict_kw)       # model_batch / d8 / order
        if defer_check:
            if self._pinned_free:
                rec, af = self._pinned_free.pop()
            else:
                rec, af = torch.zeros(32, dtype=torch.uint8).pin_memory(), torch.zeros(2, dtype=torch.int32).pin_memory()
            rec = self.stats.result_async(rec)
            af[1] = 1 if atoms is not None else 0           # host-side flag: is af[0] meaningful for this step
            if atoms is not None:
                af[:1].copy_(self._af3_status, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.device))
            self._deferred.append((rec, af, ev, self.stats.decode))
            return vols
        # one host read-back for the whole path (the reference reports these per stage)
        if not self.check_status():
            raise MicaError(f'normalisation failed (status {self.norm_status})')
        if atoms is not None and int(self._af3_status.item()) != 0:
            raise MicaError('AF3 encoding failed: atom index outside the grid (reference IndexError path, D7)')
        return vols


class _SlabDrain:
    """Streams finished parts of the stitched volumes to pinned host memory while later cube
    batches are still being processed.  Cubes are visited i-major (utils/create_grids.py:143-145),
    so once every cube of an i-layer is stitched the planes [i, i + grid_size) of the [x,y,z]
    volumes are final and contiguous: they go out on side streams behind an event."""

    def __init__(self, pipe, out_host, n_streams=2):
        self.pipe, self.out = pipe, out_host
        self.streams = [torch.cuda.Stream(pipe.device) for _ in range(n_streams)]
        self.sent_layers = 0
        self.bytes = 0
        self.turn = 0

    def __call__(self, vols, n_done):
        ijk = self.pipe.ijk_host
        n = len(ijk)
        if getattr(self.pipe, '_custom_order', False) and n_done < n:
            return                                 # cubes not in loop order: nothing is known final before the end
        # i-layers whose last cube has been stitched
        if n_done >= n:
            layer_end = vols.ext[0]
        else:
            layer_end = int(ijk[n_done][0]) - vols.org[0]      # cubes [0, n_done) cover x < i of the next cube
        x0 = self.sent_layers
        if layer_end <= x0:
            return
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.pipe.device))
        for k, v in vols.as_dict().items():
            if k not in self.out:                  # a volume the caller keeps on the device (e.g. the 20-channel
                continue                           # amino_acid_probability when candidates.py consumes it there)
            dst = self.out[k]
            parts = [(dst[x0:layer_end], v[x0:layer_end])] if v.dim() == 3 else \
                    [(dst[c, x0:layer_end], v[c, x0:layer_end]) for c in range(v.shape[0])]
            for d, s_ in parts:
                st = self.streams[self.turn % len(self.streams)]
                self.turn += 1
                st.wait_event(ev)
                with torch.cuda.stream(st):
                    d.copy_(s_, non_blocking=True)
                self.bytes += s_.numel() * s_.element_size()
        self.sent_layers = layer_end

    def finish(self):
        for st in self.streams:
            st.synchronize()


def run_map_pipeline_host(src_host: torch.Tensor, header: MapHeader, atoms_host, model_fn, pipe: MapPipeline,
                          out_host: dict | None = None, vols=None, overlap_d2h: bool = True):
    """The call a user of the reference makes, with HOST buffers on both sides: pinned
    source map (+ atom arrays) in, the four stitched volumes out in pinned host memory.
    With ``overlap_d2h`` finished x-layers of the volumes are copied out while the remaining
    cube batches run.  Returns (volumes dict of host tensors, h2d_bytes, d2h_bytes)."""
    dev = pipe.device
    src = src_host.to(dev, non_blocking=True)
    h2d = src_host.numel() * src_host.element_size()
    atoms = None
    if atoms_host is not None:
        atoms = tuple(t.to(dev, non_blocking=True) for t in atoms_host)
        h2d += sum(t.numel() * t.element_size() for t in atoms_host)
    if out_host is not None and overlap_d2h:
        drain = _SlabDrain(pipe, out_host)
        vols = pipe.run(src, header, atoms, model_fn, vols, on_batch=drain)
        drain.finish()
        torch.cuda.current_stream().synchronize()
        return dict(out_host), h2d, drain.bytes
    vols = pipe.run(src, header, atoms, model_fn, vols)
    d2h = 0
    out = {}
    for k, v in vols.as_dict().items():
        if out_host is not None and k in out_host:
            out[k] = out_host[k]
            out[k].copy_(v, non_blocking=True)
        else:
            out[k] = v.to('cpu', non_blocking=False)
        d2h += v.numel() * v.element_size()
    torch.cuda.current_stream().synchronize()
    return out, h2d, d2h


_SHARED: dict = {}


def shared_pipeline(device) -> MapPipeline:
    """One long-lived MapPipeline per GPU and process: the drop-in classes (DataPreprocessor ->
    GridCreator -> CryoEMPredictor) run consecutive maps through it, so the cube buffers, the select
    workspace, the atom bins and the side stream are allocated once, not per map."""
    dev = torch.device(device)
    if dev.type != 'cuda':
        raise MicaError(f'mica_b200 needs a CUDA device, got {device!r} (there is no CPU fallback)')
    if dev.index is None:
        ops.require_gpu()
        dev = torch.device('cuda', torch.cuda.current_device())
    pipe = _SHARED.get(dev.index)
    if pipe is None:
        pipe = _SHARED[dev.index] = MapPipeline(dev)
    return pipe


_WORKERS: dict = {}


def worker_pipeline(device, slot: int):
    """(MapPipeline, stream) of one worker of a map dealt over several devices in one process
    (``CryoEMPredictor(devices=)``), kept per (GPU, slot) across maps like ``shared_pipeline``: ``slot`` n is
    the n-th worker on that GPU, each with its own cube buffers and stream."""
    dev = torch.device(device)
    if dev.type != 'cuda' or dev.index is None:
        raise MicaError(f'worker_pipeline needs an indexed CUDA device, got {device!r}')
    key = (dev.index, int(slot))
    w = _WORKERS.get(key)
    if w is None:
        w = _WORKERS[key] = (MapPipeline(dev), torch.cuda.Stream(dev))
    return w
