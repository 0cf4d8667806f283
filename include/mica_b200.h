/* mica_b200 -- C ABI of the B200-native voxel-parallel map pipeline.
 *
 * The reference (jianlin-cheng/MICA) has no FFI: its seam is three Python classes
 * (SURVEY.md section 8b).  This header is the boundary our host-side mirrors of
 * those classes bind through ctypes (mica_b200/_lib.py); each entry point cites the
 * reference lines whose arithmetic it replaces (paths relative to the reference
 * root).  Conventions: plain pointers and sizes only; every pointer documented
 * "device" is CUDA device memory owned by the caller; the caller owns the stream
 * (a cudaStream_t passed as void*); no hidden allocations (workspaces are sized
 * by the *_workspace_bytes queries); functions return 0 or a negative MICA_ERR_*
 * and never throw; launches are asynchronous unless stated otherwise; one host
 * thread per GPU.  There is no CPU fallback.
 *
 * Index conventions: map volumes are (nz,ny,nx) C-order float32 exactly as
 * mrcfile exposes them; "cube space" is the reference's transposed view
 * (utils/create_grids.py:119-122) in which stitched volumes are indexed [x,y,z].
 * Slab arguments (z0, nz_local) describe the contiguous range of memory-axis-0
 * planes a rank holds when the volume is z-slab partitioned (SURVEY.md 8e); a
 * single GPU passes z0=0, nz_local=nz.
 */
#ifndef MICA_B200_H
#define MICA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* mica_stream_t; /* cudaStream_t */

#define MICA_OK 0
#define MICA_ERR_INVALID (-1)   /* bad argument */
#define MICA_ERR_CUDA (-2)      /* CUDA runtime error, see mica_last_error() */
#define MICA_ERR_WORKSPACE (-3) /* workspace too small */
#define MICA_ERR_NO_DEVICE (-4) /* no CUDA device / driver: the library never falls back to the CPU */

/* status word of the normaliser (mica_select_result) */
#define MICA_NORM_OK 0
#define MICA_NORM_NO_POSITIVE 1 /* utils/preprocessing.py:155-157 */
#define MICA_NORM_ZERO_PCTL 2   /* utils/preprocessing.py:152-154 */
#define MICA_NORM_PENDING 3     /* selection not finished */
#define MICA_NORM_PEER_TIMEOUT 4 /* multi-GPU: a peer rank never published its histogram */

#define MICA_SELECT_HIST_WORDS 4096 /* int64 words the histogram all-reduce covers */
#define MICA_SELECT_PASSES 7        /* hist/pick steps: sample, guided digit 0, fallback digit 0, 4 digit rounds */

int mica_version(void);
const char* mica_last_error(void);
/* number of CUDA devices visible, or MICA_ERR_NO_DEVICE */
int mica_device_count(void);
/* kernels launched by this library in this process since load (for bench.py's gpu_launches) */
int64_t mica_launch_count(void);

/* ---------------------------------------------------------------- R1 resample
 * Replaces scipy.ndimage.zoom(data, [vx,vy,vz], order=3) at
 * utils/preprocessing.py:117 and scripts_for_training_data/create_normalized_map.py:43
 * (mode='constant', cval=0, prefilter=True, grid_mode=False): cubic B-spline
 * prefilter with mirror boundaries in float64, align-corners coordinate map,
 * 64-tap gather, float32 result.  order=1 is the north-star trilinear variant
 * (no prefilter).  zoom == (1,1,1) is SciPy's early-exit copy.
 */
/* host: out[a] = int(round(float32(in[a]) * zoom[a])), banker's rounding */
int mica_zoom_output_shape(const int in_zyx[3], const float zoom_zyx[3], int out_zyx[3]);

/* workspace for a source slab of src_nz_local planes */
size_t mica_resample_workspace_bytes(int src_nz_local, int sy, int sx, int nz, int ny, int nx, int order);

/* test hook: on != 0 routes every shape through the general kernels (one thread per line /
 * per output voxel) instead of the segment-parallel prefilter and the marching gather.
 * Returns the previous setting.  Both routes implement the same arithmetic. */
int mica_resample_force_generic(int on);

/* host: the block of source planes [*src_lo, *src_hi) a rank should hold to resample output planes
 * [dst_z0, dst_z0+dst_nz_local) of a map with sz source / nz output planes (no reference counterpart:
 * the z-slab partition of SURVEY 8e).  The z prefilter cuts a line into the same segments whichever
 * block of it is in memory; with this block every coefficient the slab needs is computed from the same
 * window as on the whole map, so the slab's planes are BIT-IDENTICAL to the whole map's. */
int mica_resample_slab_source_planes(int sz, int nz, int dst_z0, int dst_nz_local, int* src_lo, int* src_hi);
/* host: the same for the general path, which integer maps take: the block that holds every raw sample that the z
 * prefilter segments (16 per line, numbered on the whole line) computed for output planes [dst_z0,
 * dst_z0+dst_nz_local) read, mirrored reads near plane 0 included.  With that block an integer map's slab is
 * BIT-IDENTICAL to the whole map.  MICA_ERR_INVALID unless 96 <= sz <= 800: lines outside that range are
 * prefiltered by one recursion over the whole line, which no block can reproduce bit for bit. */
int mica_resample_slab_source_planes_general(int sz, int nz, int dst_z0, int dst_nz_local, int* src_lo, int* src_hi);

/* src: device float32 [src_nz_local, sy, sx] = global source planes [src_z0, src_z0+src_nz_local)
 * dst: device float32 [dst_nz_local, ny, nx] = global output planes [dst_z0, dst_z0+dst_nz_local)
 * (sz,sy,sx) / (nz,ny,nx) are the GLOBAL source / output shapes.  With a partial slab the z prefilter
 * runs on the block alone: bit-identical to the whole map when the block is the one
 * mica_resample_slab_source_planes names; with any block that holds >= 16 planes beyond the taps the
 * output needs, a window that leaves the block is reflected at its end (error < 1e-9, SURVEY 8e).
 */
int mica_bspline_resample_f32(const float* src, int sz, int sy, int sx, int src_z0, int src_nz_local,
                              float* dst, int nz, int ny, int nx, int dst_z0, int dst_nz_local,
                              void* workspace, size_t workspace_bytes, int order, mica_stream_t stream);

/* Sample types of a map, numbered as the MRC2014 modes that carry them. */
#define MICA_DTYPE_I8 0  /* int8, MRC mode 0 */
#define MICA_DTYPE_I16 1 /* int16, MRC mode 1 */
#define MICA_DTYPE_F32 2 /* float32, MRC mode 2 */
#define MICA_DTYPE_U16 6 /* uint16, MRC mode 6 */

/* mica_bspline_resample_f32 for any of these types: src and dst hold samples of src_dtype / dst_dtype.  The pairs
 * accepted are float32 -> float32 (the same call as mica_bspline_resample_f32) and an integer type -> the same
 * integer type: scipy.ndimage.zoom on an integer array, which interpolates in float64 and stores into the input's
 * type rounding half away from zero and saturating at the type's range (DESIGN.md D12).  Integer maps always run
 * the float64 general path; zoom == (1,1,1) is again the caller's copy.  Any other pair is MICA_ERR_INVALID.
 * An integer block of a longer z line (order 3) must hold the planes mica_resample_slab_source_planes_general
 * names, and the line must have 96..800 planes; the result is then bit-identical to the whole map's planes. */
int mica_resample(const void* src, int src_dtype, int sz, int sy, int sx, int src_z0, int src_nz_local,
                  void* dst, int dst_dtype, int nz, int ny, int nx, int dst_z0, int dst_nz_local,
                  void* workspace, size_t workspace_bytes, int order, mica_stream_t stream);

/* diagnostic: the kernel the last mica_bspline_resample_f32 call on this thread launched for one pass
 * (pass 0 = z prefilter, 1 = y prefilter, 2 = x pass, 3 = interpolation), one of the MICA_RS_* ids below;
 * -1 when that pass did not run (order 1 has no prefilter; a call that failed its argument checks ran none).
 * The fast path's x pass prefilters and interpolates x in one kernel; its pass 3 then interpolates y and z.
 * An id keeps its number for good: the gaps are kernels that no longer exist. */
int mica_last_resample_path(int pass);
#define MICA_RS_COLS_SEG16 1          /* prefilter_cols_seg<16>: 16 lines x 16 segments in shared memory */
#define MICA_RS_COLS32 3              /* prefilter_cols<32>: one thread per line */
#define MICA_RS_COLS8 4               /* prefilter_cols<8>: one thread per line, long lines */
#define MICA_RS_COLS_GLOBAL 5         /* prefilter_cols_global: one thread per line, in global memory */
#define MICA_RS_ROWS_SEG16 6          /* prefilter_rows_seg<16> */
#define MICA_RS_ROWS32 8              /* prefilter_rows<32>: one thread per row */
#define MICA_RS_ROWS4 9               /* prefilter_rows<4>: one thread per row, long rows */
#define MICA_RS_COLS_REG 10           /* cols_reg_kernel: register segments numbered on the whole line */
#define MICA_RS_ROWS_REG16 14         /* rows_reg_interp_kernel<16> */
#define MICA_RS_ROWS_REG32 15         /* rows_reg_interp_kernel<32> */
#define MICA_RS_ROWS_PIPE_16_512 17   /* rows_pipe_interp_kernel<16, 512> */
#define MICA_RS_ROWS_PIPE_8_512 18    /* rows_pipe_interp_kernel<8, 512> */
#define MICA_RS_MARCH_YZ_TMA3 20      /* march_yz_tma_kernel<3>: 12 staged rows */
#define MICA_RS_MARCH_YZ_TMA4 21      /* march_yz_tma_kernel<4>: 16 staged rows */
#define MICA_RS_MARCH3_TMA3 22        /* march3_tma_kernel<3> */
#define MICA_RS_MARCH3_TMA4 23        /* march3_tma_kernel<4> */
#define MICA_RS_MARCH3_3 24           /* march3_kernel<3>: register prefetch, no TMA */
#define MICA_RS_MARCH3_4 25           /* march3_kernel<4> */
#define MICA_RS_GATHER3 26            /* gather3_kernel: one thread per output voxel */
#define MICA_RS_GATHER1 27            /* gather1_kernel: trilinear */

/* ------------------------------------------------------- R2/R3 normalisation
 * Replaces np.nan_to_num / np.median / np.percentile(pos, 99.9) / clip / divide
 * at utils/preprocessing.py:122-133 (twin: create_normalized_map.py:48-79) with
 * an exact 3-pass (11/11/10-bit) radix select over order-preserving uint32 keys,
 * following the installed NumPy 2.x float32 semantics (SURVEY.md 8a R3).
 * State lives in a device workspace so that multi-GPU runs can all-reduce the
 * histogram (MICA_SELECT_HIST_WORDS int64 at mica_select_hist_ptr) between
 * mica_select_hist and mica_select_pick without a host round trip.
 * Protocol: init; for step = 0 .. MICA_SELECT_PASSES-1 { hist(step); [all-reduce]; pick(step) }.
 * Steps: 0 = 1/64 sample histogram -> candidate bins; 1 = guided digit-0 pass (only voxels in
 * the candidate bins are histogrammed, the others counted) + verification on the exact counts;
 * 2 = full digit-0 histogram, a no-op unless the verification failed; 3..6 = median digits 1,2
 * and percentile digits 1,2.  Every kernel checks the device-side state, so the host never
 * branches on results.
 */
size_t mica_select_workspace_bytes(void);
/* With room for the COMPACT BUFFER: the guided digit-0 pass appends every voxel of the candidate bins (a few
 * percent of the map) to it, and the four later digit passes read that buffer instead of streaming the map
 * again (order statistics: 6 map reads -> 2).  mica_select_workspace_bytes_for(n) sizes a workspace for n
 * voxels per rank; after allocating (and zero-filling) it call mica_select_set_compact once.  A workspace
 * of the plain size, or an overflowing buffer (heavy ties), falls back to streaming the map: same results. */
size_t mica_select_workspace_bytes_for(int64_t n_local);
int mica_select_set_compact(void* workspace, size_t workspace_bytes, mica_stream_t stream);
/* diagnostics: out = {compact buffer in use (0|1), floats appended, capacity}; synchronises the stream */
int mica_select_compact_info(const void* workspace, int64_t out[3], mica_stream_t stream);
int mica_select_init(void* workspace, int64_t n_total, mica_stream_t stream);
int mica_select_hist(const float* x, int64_t n_local, void* workspace, int step, mica_stream_t stream);
int64_t* mica_select_hist_ptr(void* workspace);
int mica_select_pick(void* workspace, int step, mica_stream_t stream);
/* every step on one GPU */
int mica_order_stats_f32(const float* x, int64_t n, void* workspace, mica_stream_t stream);
/* synchronises the stream; any out pointer may be NULL */
int mica_select_result(const void* workspace, float* median, float* p999, int64_t* n_pos, int* norm_status,
                       mica_stream_t stream);
/* the same without the synchronisation: the 32-byte record {int64 n_le_med, int64 n_pos, float median,
 * float p999, float g, int32 status} is copied into host_record (pinned memory) in stream order */
#define MICA_SELECT_RESULT_BYTES 32
int mica_select_result_async(const void* workspace, void* host_record, mica_stream_t stream);
/* y = min(m, p)/p with m = (x > med) * (x - med), written exactly as
 * utils/preprocessing.py:124,131-133 evaluates it in float32; x == y allowed.
 * Reads median / percentile from the workspace on the device; leaves y untouched
 * when the status is not MICA_NORM_OK. */
int mica_normalize_apply_f32(const float* x, float* y, int64_t n, const void* workspace, mica_stream_t stream);

/* ------------------------------------------------- R2/R3 normalisation of integer maps (DESIGN.md D12)
 * The reference normalises an int8 / int16 / uint16 map as the integer array zoom returned: np.median is
 * float64 (the middle element, or the mean of the two middle ones), the positives (x > med) * (x - med) are
 * float64, np.percentile(pos, 99.9) interpolates in float64 and the normalised map is the float64 expression
 * cast to float32.  Values have at most 16 bits, so one exact histogram of 2^8 / 2^16 bins gives every rank:
 * mica_int_order_stats is one pass over x plus one single-CTA pick that finds the median, count(x <= med),
 * n_pos, the percentile and the status word (MICA_NORM_*) on the device.
 * Several GPUs: init(n_total = voxels of all ranks); hist(this rank's voxels); sum the histograms of all ranks
 * (2^8 int64 words for int8, 2^16 for int16 / uint16, at mica_int_stats_hist_ptr, or
 * mica_int_stats_peer_publish + mica_int_stats_peer_sum); pick. */
size_t mica_int_stats_workspace_bytes(void);
/* x: device samples of `dtype` (MICA_DTYPE_I8 / I16 / U16), n of them; workspace of the size above.  The same
 * launches as init + hist + pick. */
int mica_int_order_stats(const void* x, int dtype, int64_t n, void* workspace, mica_stream_t stream);
int mica_int_stats_init(void* workspace, int dtype, int64_t n_total, mica_stream_t stream);
int mica_int_stats_hist(const void* x, int dtype, int64_t n_local, void* workspace, mica_stream_t stream);
int64_t* mica_int_stats_hist_ptr(void* workspace);
/* leaves a state whose status is already final (MICA_NORM_PEER_TIMEOUT) as it is */
int mica_int_stats_pick(void* workspace, int dtype, mica_stream_t stream);
/* The histogram sum over NVLink peer memory, on the caller's stream: every rank allocates one buffer of
 * mica_int_peer_buffer_bytes with mica_ipc_alloc, the ranks open each other's (mica_peer_open) and upload the
 * table of `world` device pointers.  Per map, after hist:
 *   mica_int_stats_peer_publish  copies the local histogram into the rank's slot `parity` and raises its flag of
 *                                `epoch` in every peer's buffer -- it never waits;
 *   mica_int_stats_peer_sum      waits (bounded: on timeout the status becomes MICA_NORM_PEER_TIMEOUT, which pick
 *                                leaves alone) for every peer's flag and sums their slots into the local state.
 * `epoch` = a counter every rank increments once per map (>= 1), `parity` = epoch & 1, as for
 * mica_select_peer_reduce.  Several ranks driven on ONE GPU must enqueue every publish before any sum. */
size_t mica_int_peer_buffer_bytes(void);
int mica_int_stats_peer_publish(const void* workspace, int dtype, void* const* peer_bufs, int rank, int world,
                                int parity, int epoch, mica_stream_t stream);
int mica_int_stats_peer_sum(void* workspace, int dtype, void* const* peer_bufs, int rank, int world, int parity,
                            int epoch, mica_stream_t stream);
/* synchronises the stream; any out pointer may be NULL */
int mica_int_stats_result(const void* workspace, double* median, double* p999, int64_t* n_pos, int* norm_status,
                          mica_stream_t stream);
/* the same without the synchronisation: the 32-byte record {double median, double p999, int64 n_pos,
 * int32 status, int32 0} is copied into host_record (pinned memory) in stream order */
#define MICA_INT_STATS_RESULT_BYTES 32
int mica_int_stats_result_async(const void* workspace, void* host_record, mica_stream_t stream);
/* y (float32) = float32(min(m, p) / p), m = (x > med) * (x - med), evaluated in float64 exactly as NumPy does
 * on the integer array: +0.0 at or below the median.  Leaves y untouched when the status is not MICA_NORM_OK. */
int mica_normalize_apply_int(const void* x, int dtype, float* y, int64_t n, const void* workspace,
                             mica_stream_t stream);

/* ------------------------------------------- multi-GPU: histogram exchange over peer memory
 * No reference counterpart (the reference is single-process); replaces the NCCL all-reduce
 * between mica_select_hist and mica_select_pick.  Every rank allocates one peer buffer
 * (mica_peer_alloc; cudaMalloc + a 64-byte CUDA IPC handle), the ranks exchange the handles
 * (any channel), open each other's (mica_peer_open) and upload the table of `world` device
 * pointers (own buffer at [rank]).  mica_select_peer_reduce then does, in ONE single-CTA
 * kernel on the caller's stream: publish the local histogram, signal every peer, wait for
 * every peer's signal (bounded spin: on timeout the normalisation status becomes
 * MICA_NORM_PEER_TIMEOUT), sum the peers' histograms over NVLink into the local state.
 * `epoch` = a counter every rank increments once per call (>= 1), `parity` = epoch & 1: a slot is
 * rewritten two calls later, which a rank can only reach after every peer has signalled the call in
 * between, i.e. has finished reading it.
 */
size_t mica_peer_buffer_bytes(void);
int mica_peer_alloc(void** dev_ptr, void* ipc_handle_out /* 64 bytes, nullable */);
int mica_peer_open(const void* ipc_handle, void** dev_ptr);
int mica_peer_close(void* dev_ptr);
int mica_peer_free(void* dev_ptr);
/* Inside ONE process: lets kernels running on `device` load from and store to memory allocated on
 * `peer_device` (cudaDeviceEnablePeerAccess).  device == peer_device is a no-op; a pair already enabled (by
 * this library or by PyTorch) counts as success; a pair without a peer path is MICA_ERR_INVALID.  The caller's
 * current device is restored.  (CUDA IPC handles cannot be opened by the process that made them, so
 * mica_peer_open does not serve several GPUs driven from one process.) */
int mica_peer_enable(int device, int peer_device);
int mica_select_peer_reduce(void* workspace, void* const* peer_bufs, int rank, int world, int parity, int epoch,
                            int step /* host step 0..MICA_SELECT_PASSES-1; a step that is not due on the device
                                        (the fallback after an accepted guided pass) skips the handshake */,
                            mica_stream_t stream);

/* ------------------------------------------- multi-GPU: z-halo exchange of the source map over peer memory
 * No reference counterpart.  A rank of the z-slab partition (mica_b200/slab.py) needs a few source planes
 * of each neighbour (interpolation taps + prefilter horizon).  Every rank owns one exported buffer
 * (mica_ipc_alloc of mica_halo_buffer_bytes(slot_elems); handles exchanged once; peers opened with
 * mica_peer_open) and a table of `world` device pointers as above.  Per map, on the caller's stream:
 *   mica_halo_publish  copies `n_lo` / `n_hi` elements starting at element offsets `off_lo` / `off_hi` of the
 *                      rank's own block into its buffer (slot `parity`), then raises a flag in each neighbour's
 *                      buffer (st.release.sys) -- it never waits;
 *   mica_halo_pull     waits (ld.acquire.sys, bounded: *status becomes 1 on timeout) for the neighbours' flags
 *                      of `epoch` and copies the `n_lo` elements the LOWER neighbour published for this rank
 *                      to dst_lo and the `n_hi` elements of the UPPER neighbour to dst_hi, over NVLink.
 * `epoch` increases by one per exchange, `parity` = epoch & 1 (slot reuse is safe because the order-statistics
 * exchange of the map in between synchronises all ranks).  The _bytes forms count offsets, sizes and the slot
 * capacity in bytes (planes of any sample type); the float32 forms count float32 elements and forward x 4.
 * A buffer of mica_halo_buffer_bytes(slot_elems) holds slots of 4 * slot_elems bytes. */
size_t mica_halo_buffer_bytes(int64_t slot_elems);
int mica_ipc_alloc(size_t bytes, void** dev_ptr, void* ipc_handle_out /* 64 bytes, nullable */);
int mica_halo_publish(const float* own, int64_t off_lo, int64_t n_lo, int64_t off_hi, int64_t n_hi,
                      void* const* peer_bufs, int rank, int world, int parity, int epoch, int64_t slot_elems,
                      mica_stream_t stream);
int mica_halo_pull(float* dst_lo, int64_t n_lo, float* dst_hi, int64_t n_hi, void* const* peer_bufs, int rank,
                   int world, int parity, int epoch, int64_t slot_elems, int* status, mica_stream_t stream);
int mica_halo_publish_bytes(const void* own, int64_t off_lo, int64_t n_lo, int64_t off_hi, int64_t n_hi,
                            void* const* peer_bufs, int rank, int world, int parity, int epoch, int64_t slot_bytes,
                            mica_stream_t stream);
int mica_halo_pull_bytes(void* dst_lo, int64_t n_lo, void* dst_hi, int64_t n_hi, void* const* peer_bufs, int rank,
                         int world, int parity, int epoch, int64_t slot_bytes, int* status, mica_stream_t stream);

/* test hooks for the normaliser: (1) evaluate the NumPy expression operation by operation for
 * every voxel instead of the short equivalent path (returns the previous setting); (2) put
 * given thresholds into a select workspace as if mica_order_stats_f32 had found them. */
int mica_normalize_force_reference_arith(int on);
/* test hook: on != 0 makes the guided digit-0 pass fail its verification (exercises the fallback step) */
int mica_select_force_fallback(int on);
int mica_select_set_thresholds(void* workspace, float median, float p, mica_stream_t stream);

/* ------------------------------------------------------------ R4 AF3 encoder
 * Replaces transform_coordinates + the per-atom loop at
 * utils/preprocessing.py:172-178,275-298 (twin: create_AF3_encodings.py:52-106).
 * idx = clip(rint(coord - origin), 0, clip_hi) per (x,y,z); the reference passes
 * clip_hi = (nz-1, ny-1, nx-1) -- i.e. in (z,y,x) order against (x,y,z) indices
 * (quirk D7) -- so the three bounds are explicit.  vol24[ch, z, y, x] = 1.0 for the
 * backbone channel (bb_ch 0..3 or -1) and the residue channel (aa_ch 4..23 or -1).
 * vol24: device float32 [24, nz_local, ny, nx], zero-filled here.  *status_oob
 * (device int) is set to 1 if any clipped index still exceeds its real axis (the
 * reference then raises IndexError and returns False, :344-347); atoms whose z
 * falls outside the slab are skipped silently.
 */
int mica_af3_encode(const float* xyz, const int8_t* bb_ch, const int8_t* aa_ch, int64_t n_atoms,
                    float ox, float oy, float oz, int clip_x, int clip_y, int clip_z,
                    int nz, int ny, int nx, int z0, int nz_local,
                    float* vol24, int* status_oob, mica_stream_t stream);

/* ------------------------------------------ R4 + R5 fused: sparse AF3 cube fill
 * The AF3 channels of a cube batch written straight from the atoms, without the dense
 * 24-channel volume (utils/preprocessing.py:268-298 + utils/create_grids.py:269-352 +
 * dataset/dataset.py:209-219 in one step).  mica_af3_bin_atoms bins the atoms per cube
 * once per map (same index arithmetic and clip quirk as mica_af3_encode; status_oob as
 * there); mica_af3_fill_cubes keeps `out` ([slots, 24, W^3] at out_cube_stride, which the
 * caller zero-fills ONCE and never writes) equal to "zeros + the atoms of the cube shown in
 * each slot": slot b currently shows cube ijk_prev[b] (b < n_prev; clean otherwise) and is
 * switched to cube ijk_next[b] (b < n_next; left clean otherwise) by clearing the voxels
 * of the old cube and setting those of the new one.  Stateless: the caller passes what it
 * passed as ijk_next last time (n_prev = 0 for a fresh buffer; n_next = 0 clears).
 * nonzero (nullable, int32 [n_next]): 1 iff the cube has any atom voxel.
 * The result is bit-identical to mica_extract_cubes(mica_af3_encode(atoms)).
 */
size_t mica_af3_bins_workspace_bytes(int64_t n_atoms, int nz, int ny, int nx, const int perm[3],
                                     int grid_size, int padding);
int mica_af3_bin_atoms(const float* xyz, const int8_t* bb_ch, const int8_t* aa_ch, int64_t n_atoms,
                       float ox, float oy, float oz, int clip_x, int clip_y, int clip_z,
                       int nz, int ny, int nx, const int perm[3], int grid_size, int padding,
                       void* workspace, size_t workspace_bytes, int* status_oob, mica_stream_t stream);
int mica_af3_fill_cubes(const void* workspace, int64_t n_atoms, int nz, int ny, int nx, const int perm[3],
                        int grid_size, int padding, const int32_t* ijk_prev, int n_prev,
                        const int32_t* ijk_next, int n_next, float* out, int64_t out_cube_stride,
                        int32_t* nonzero, mica_stream_t stream);

/* --------------------------------------------------------- R5/R6 cube extract
 * Replaces GridCreator.transpose + create_grids_from_mrc (utils/create_grids.py:67-176),
 * its training twins (scripts_for_training_data/create_grids_for_*.py) and the
 * per-cube re-assembly of CryoEMTestDataset.__getitem__ (dataset/dataset.py:194-224):
 * out[b, c, u0,u1,u2] = T_c[i_b-pad+u0, j_b-pad+u1, k_b-pad+u2] (0 outside T),
 * T_c = transpose(vol_c, perm).  W = grid_size + 2*padding.
 * vol: device float32, channel c at vol + c*chan_stride, each [nz_local, ny, nx]
 * holding global planes [z0, z0+nz_local).  ijk: device int32 [B,3] cube origins
 * in cube space.  out: device, cube b / channel c at out + b*out_cube_stride + c*W^3.
 * nonzero (device int32 [B], nullable): OR-ed with 1 if cube b has any non-zero
 * voxel in these channels (D8 routing; also the training twin's max >= 0.01 test
 * is served by cube_max).  cube_max (device float32 [B], nullable, channel 0 only).
 */
int mica_extract_cubes(const float* vol, int64_t chan_stride, int n_channels,
                       int nz, int ny, int nx, int z0, int nz_local, const int perm[3],
                       int grid_size, int padding, const int32_t* ijk, int n_cubes,
                       float* out, int64_t out_cube_stride, int32_t* nonzero, float* cube_max,
                       mica_stream_t stream);

/* diagnostic: which kernel the last mica_extract_cubes call on this thread used
 * (0 = row copy, 1 = shared-memory tiled transpose, 2 = TMA box loads; -1 = none yet) */
int mica_last_extract_path(void);

/* ------------------------------------------------ R7/R8 post-process + stitch
 * Replaces the softmax/argmax block of run_inference (utils/predict.py:342-349)
 * and reconstruct_volume (utils/predict.py:439-512) in one pass over the cube
 * cores: bb = softmax(bb[{0,2,3}])[2]; ca likewise; aa_prob = softmax(aa[1:21]);
 * aa_pred = argmax(aa_prob) stored as float32 (:462).  Cores are disjoint, so no
 * atomics.  bb, ca: device [B,4,W^3]; aa: device [B,21,W^3]; ijk device int32
 * [B,3].  Volumes are cube-space boxes: global shape (X,Y,Z), this rank holding
 * [org0,org0+ext0) x [org1,..) x [org2,..) in C order; cores are clipped to it.
 * aa_prob_vol: [20, ext0, ext1, ext2].
 */
int mica_postproc_stitch(const float* bb, const float* ca, const float* aa,
                         const int32_t* ijk, int n_cubes, int X, int Y, int Z,
                         const int org[3], const int ext[3], int grid_size, int padding,
                         float* bb_vol, float* ca_vol, float* aa_prob_vol, float* aa_pred_vol,
                         mica_stream_t stream);

/* plain centre-crop paste of already post-processed cubes (reconstruct_volume on
 * its own, utils/predict.py:494-501): cubes device [B, n_ch, W^3] -> vol [n_ch, ext...] */
int mica_stitch_cubes(const float* cubes, int n_ch, const int32_t* ijk, int n_cubes,
                      int X, int Y, int Z, const int org[3], const int ext[3],
                      int grid_size, int padding, float* vol, mica_stream_t stream);

/* Multi-GPU form of mica_postproc_stitch (config 5: the cubes of ONE map dealt out evenly over the ranks,
 * no reference counterpart): the output is partitioned along cube axis 0, rank r owning planes
 * [x_bounds[r], x_bounds[r+1]) as 23 float32 channels of [x_bounds[r+1]-x_bounds[r], Y, Z] at owner_base[r]
 * ([backbone | carbon_alpha | amino_acid_prediction | amino_acid_probability x 20]); owner_base is a DEVICE
 * array of `world` pointers into peer-mapped memory (mica_ipc_alloc / mica_peer_open).  Every core plane is
 * stored straight into its owner's block over NVLink -- softmax/argmax + stitch fused with the exchange.
 * The caller synchronises all ranks (stream sync + barrier) before an owner reads its block. */
int mica_postproc_stitch_peer(const float* bb, const float* ca, const float* aa, const int32_t* ijk, int n_cubes,
                              int X, int Y, int Z, int grid_size, int padding, void* const* owner_base,
                              const int* x_bounds, int world, mica_stream_t stream);

/* ===================================================================================
 * SURVEY.md section 8(f) "next" rows, built to the same bar as R1-R8.
 * =================================================================================== */

/* ------------------------------------------------ N1: C-alpha candidates (Solver.clustering head)
 * Replaces utils/modeler.py:767-860: threshold -> DBSCAN -> cluster score filter -> greedy NMS ->
 * 3x3x3 weighted refinement, on the stitched volumes where they lie in HBM (cube space [X,Y,Z],
 * C order), so that only the picks cross PCIe.  Index work is bit-exact; see candidates.cu for the
 * two float paths.  "lin" is the C-order linear voxel index x*Y*Z + y*Z + z (int64).
 */
/* :767 np.where(vol > thr), two steps because the caller allocates the outputs:
 * count (device int64 *count_dev; read it after synchronising), then write (ascending lin =
 * np.where order; xyz_out device int32 [cap,3], nullable).  vol must not change in between. */
size_t mica_cand_threshold_workspace_bytes(int64_t n_vox);
int mica_cand_threshold_count(const float* vol, int64_t n_vox, float thr, void* workspace, size_t workspace_bytes,
                              int64_t* count_dev, mica_stream_t stream);
int mica_cand_threshold_write(const float* vol, int X, int Y, int Z, float thr, const void* workspace,
                              int64_t* lin_out, int32_t* xyz_out, int64_t cap, mica_stream_t stream);
/* out[i] = vol[lin[i]]  (BBProb[pcd[:,0],pcd[:,1],pcd[:,2]], :779) */
int mica_gather_f32(const float* vol, const int64_t* lin, int64_t n, float* out, mica_stream_t stream);
/* :768-770 Open3D cluster_dbscan(eps, min_points) on lattice points (closed ball, self included, clusters
 * numbered by first core point, border point -> first cluster reaching it, noise -1).  eps_sq = floor(eps^2).
 * lin ascending and distinct.  labels: device int32 [n]; n_clusters_dev: device int64. */
size_t mica_dbscan_workspace_bytes(int X, int Y, int Z, int64_t n_points);
int mica_dbscan_lattice(const int64_t* lin, int64_t n, int X, int Y, int Z, int eps_sq, int min_points,
                        void* workspace, size_t workspace_bytes, int32_t* labels, int64_t* n_clusters_dev,
                        mica_stream_t stream);
/* :775-786 per-label sum (float64) and count of vals; labels outside [0,n_labels) are skipped */
int mica_cand_cluster_scores(const float* vals, const int32_t* labels, int64_t n, int n_labels, double* sums,
                             int64_t* counts, mica_stream_t stream);
/* :789-797 valid[i] = label_ok[labels[i]] (0 for noise) */
int mica_cand_valid_points(const int32_t* labels, const uint8_t* label_ok, int64_t n, int n_labels, uint8_t* valid,
                           mica_stream_t stream);
/* :800-802 CAProb_clusted: out = 0 everywhere, ca at the valid points */
int mica_cand_clustered_volume(const float* ca, int64_t n_vox, const int64_t* lin, const uint8_t* valid, int64_t n,
                               float* out, mica_stream_t stream);
/* :805-832 greedy NMS over the valid points (squared distance <= nms_radius_sq suppresses; the reference
 * compares the squared distance with its `nms_radius` argument).  work: device float32 [X*Y*Z] scratch, holds
 * -p at the picks afterwards.  flag_dev: device int32.  Synchronises the stream every 8 rounds. */
int mica_cand_nms(const float* ca, int X, int Y, int Z, const int64_t* lin, const uint8_t* valid, int64_t n,
                  int nms_radius_sq, float* work, int32_t* flag_dev, int* rounds_out, mica_stream_t stream);
/* the picks in the reference's order (best probability first, ties by np.where order): sorted_lin device int64
 * [cap], sorted_xyz device int32 [cap,3]; *n_picks_dev device int64 (the call synchronises to read it and fails
 * with MICA_ERR_WORKSPACE if it exceeds cap).  Ordering is a bucketed rank count, not an m^2 comparison. */
size_t mica_cand_picks_workspace_bytes(int64_t cap);
int mica_cand_nms_picks(const float* work, int Y, int Z, const int64_t* lin, const uint8_t* valid, int64_t n,
                        int64_t cap, void* workspace, size_t workspace_bytes, int64_t* n_picks_dev,
                        int64_t* sorted_lin, int32_t* sorted_xyz, mica_stream_t stream);
/* :837-860 per pick: CA_cands (float64 [m,3]), CA_cands_AAProb rows (float32 [m,20]), CA_cands_AA
 * (float32 [m]) and ok (uint8 [m]; 0 = pick on the volume border, skipped by the reference's try/except). */
int mica_cand_refine(const float* ca, const float* aa_prob, const float* aa_pred, int X, int Y, int Z,
                     const int64_t* pick_lin, int64_t m, double* out_xyz, float* out_aaprob, float* out_aa,
                     uint8_t* out_ok, mica_stream_t stream);

/* utils/modeler.py:862-886 -- the rest of Solver.clustering: dis_out[a,b] = |c_a - c_b| (float64 [m,m], calc_dis
 * :174-181) and neigh_out[a,b] = ((distance score) + (mean backbone probability at the four interior fifths of
 * the segment)) / 2 for 2 <= dis <= 6, else 0 (float64 [m,m]); reproduces the reference's mixed float32 /
 * float64 arithmetic (python float 1.0 + np.float32 stays float32).  xyz: device float64 [m,3]; m <= 65535. */
int mica_cand_neighbor_graph(const double* xyz, int64_t m, const float* bb, int X, int Y, int Z, double* dis_out,
                             double* neigh_out, mica_stream_t stream);
/* :889-897 best[a] = (first, second): the two largest entries of row a of neigh (device int32 [m,2]; -1 where
 * the entry is 0; equal scores: the higher index counts as larger, i.e. a stable ascending sort) */
int mica_cand_best_neighbors(const double* neigh, int64_t m, int32_t* best, mica_stream_t stream);
/* :866-873 per row of dis the ascending indices with dis <= max_dis: idx device int32 [m,cap], count device
 * int32 [m] (count may exceed cap: call again with a larger cap) */
int mica_cand_neighbor_lists(const double* dis, int64_t m, double max_dis, int cap, int32_t* idx, int32_t* count,
                             mica_stream_t stream);

/* ------------------------------------------------ N3: training label masks
 * scripts_for_training_data/create_backbone_mask.py:136-172, create_carbon_alpha_mask.py:136-173:
 * xyz device float32 [A,3] of ALL atoms in file order, is_class device uint8 [A]; mask device int32 [nz,ny,nx]
 * = 3 (class atom) / 2 (other atom; the LAST atom on a voxel wins) / 1 (26-neighbour of an atom voxel) / 0.
 * clip_* as in mica_af3_encode (the reference clips (x,y,z) with (nz,ny,nx): pass nz-1, ny-1, nx-1);
 * *status_oob = 1 where numpy would raise IndexError. */
int mica_label_class_mask(const float* xyz, const uint8_t* is_class, int64_t n_atoms, float ox, float oy, float oz,
                          int clip_x, int clip_y, int clip_z, int nz, int ny, int nx, int32_t* mask,
                          int* status_oob, mica_stream_t stream);
/* scripts_for_training_data/create_amino_acid_mask.py:151-177: xyz device float32 [R,3] C-alpha coordinates in
 * file order, label device int32 [R] (1..20): lowest label on the 26 neighbours, C-alpha voxels zeroed in order. */
size_t mica_label_aa_mask_workspace_bytes(int nz, int ny, int nx);
int mica_label_aa_mask(const float* xyz, const int32_t* label, int64_t n_ca, float ox, float oy, float oz,
                       int clip_x, int clip_y, int clip_z, int nz, int ny, int nx, void* workspace,
                       size_t workspace_bytes, int32_t* mask, int* status_oob, mica_stream_t stream);

/* ------------------------------------------------ N4: docking masks
 * utils/dock_in_map.py:269: out = where(in < level, 0, in) (in == out allowed) */
int mica_contour_threshold_f32(const float* in, float* out, int64_t n, float level, mica_stream_t stream);
/* utils/dock_in_map.py:330-352: zero map (device float32 [nz,ny,nx], in place) wherever
 * distance_transform_edt(~seeds, sampling=voxel_size) <= radius; seeds = int((xyz - origin) / voxel) of the atoms
 * (device float32 [A,3]) that pass the reference's bounds test.  *status_oob = 1 where numpy would raise. */
int mica_zero_around_atoms(const float* xyz, int64_t n_atoms, const float origin_xyz[3], const float voxel_xyz[3],
                           double radius, int nz, int ny, int nx, float* map, int* status_oob, mica_stream_t stream);

/* ------------------------------------------- overlap-weighted stitching (BASELINE.json north_star variant)
 * NOT the reference's arithmetic (it pastes disjoint cores, utils/predict.py:494-501): every voxel of every window
 * adds its post-processed probabilities times a separable window weight w1[a] w1[b] w1[c] (window_w1: W = grid_size
 * + 2 padding floats on the HOST, finite, >= 0, at least one > 0), normalised by the weight sum of the full cube
 * lattice: norm is a DEVICE float64 array [X | Y | Z] of the reciprocals of the three 1-D lattice sums (0 where a
 * sum is 0).  The contributions are 2^-31 fixed point, added as uint32 into a zero-initialised 23-channel block
 * laid out [backbone | carbon_alpha | amino_acid_prediction | amino_acid_probability x 20] (the layout of
 * mica_postproc_stitch_peer), over any number of calls: the sums, and so the result, do not depend on the order,
 * the batch or the partition.  mica_overlap_finalize_fixed turns a block of n_voxels voxels into the four float32
 * volumes in place (prediction = arg-max of the 20 sums, first maximum wins).
 * _peer: the output is owned along cube axis `axis` (0 = x, 2 = k): rank r holds planes [bounds[r], bounds[r+1])
 * of that axis as such a block at owner_base[r] (a DEVICE array of `world` pointers, local or peer-mapped memory,
 * which needs native peer atomics: mica_peer_atomics_supported).  Every contribution is added into its owner's
 * block.  The caller zeroes every block, synchronises all ranks before the first accumulate and after the last,
 * then each owner finalizes its own block. */
int mica_overlap_accumulate_fixed(const float* bb, const float* ca, const float* aa, const int32_t* ijk, int n_cubes,
                                  int X, int Y, int Z, int grid_size, int padding, const float* window_w1,
                                  const double* norm, void* block, mica_stream_t stream);
int mica_overlap_accumulate_fixed_peer(const float* bb, const float* ca, const float* aa, const int32_t* ijk,
                                       int n_cubes, int X, int Y, int Z, int grid_size, int padding,
                                       const float* window_w1, const double* norm, void* const* owner_base, int axis,
                                       const int* bounds, int world, mica_stream_t stream);
int mica_overlap_finalize_fixed(void* block, int64_t n_voxels, mica_stream_t stream);
/* 1 when `device` can add into the memory of `peer_device` with native atomics over the peer path
 * (cudaDevP2PAttrNativeAtomicSupported; 1 for device == peer_device), 0 when not, negative MICA_ERR_* on error. */
int mica_peer_atomics_supported(int device, int peer_device);

/* ------------------------------------------- host I/O helper (SURVEY 8f N2; no device work)
 * Fixed-column PDB reader standing where Bio.PDB.PDBParser stands (utils/preprocessing.py:269,275-298).
 * Per ATOM (and optionally HETATM) record: xyz [n,3] float32 (float(text) rounded to float32),
 * fields [n,16] uint8 (0-3 atom name cols 13-16, 4 altloc, 5-7 residue name, 8 chain, 9-13 resSeq+iCode,
 * 14 = HETATM flag), occupancy [n], model [n] (MODEL records seen before), bb_ch / aa_ch [n] (channel codes of
 * utils/preprocessing.py:254-263, -1 = none), info[2] = {residues, 1 if an atom identity occurs twice: altlocs}.
 * Every output but xyz / fields is nullable.  Returns the record count (only
 * the first `capacity` are written; capacity 0 counts), negative MICA_ERR_* on an unparsable coordinate. */
int64_t mica_parse_pdb(const char* text, int64_t nbytes, int with_hetatm, int64_t capacity, float* xyz,
                       uint8_t* fields, float* occupancy, int32_t* model, int8_t* bb_ch, int8_t* aa_ch,
                       int64_t* info);

#ifdef __cplusplus
}
#endif
#endif /* MICA_B200_H */
