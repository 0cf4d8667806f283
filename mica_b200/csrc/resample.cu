// R1: cubic B-spline (and trilinear) resampling of the cryo-EM map.
//
// Replaces scipy.ndimage.zoom(data, zoom, order=3) as called at
// utils/preprocessing.py:117 (reference root) -- SciPy's algorithm restated in
// SURVEY.md Appendix A: float64 IIR prefilter with mirror boundaries along each
// axis, align-corners coordinate map, 4x4x4 tap gather with mirrored edge taps,
// float32 result.  SciPy quirk kept on purpose (DESIGN.md D11): an output index
// whose coordinate k*(n_in-1)/(n_out-1) overshoots n_in-1 by rounding is treated
// as outside the map (mode='constant') and yields 0.
//
// Kernels (all HBM-bound, see DESIGN.md for the byte counts):
//   taps_kernel, zwin_kernel  per-axis tap index / weight tables; the z taps folded into 4-plane windows (tiny)
// Fast path (order 3, the conditions are in fast_path_ok):
//   cols_reg_kernel      z and y prefilter, float32 in and out: a thread owns <= 26 samples of one column and
//                        runs both recursions over them and 16 samples either side in registers (no shared
//                        memory, no barrier); segments are numbered on the whole line, so a z-slab of a map
//                        gets the whole map's bits
//   rows_reg_interp_kernel   x pass, rows of <= 832 samples: cp.async-staged rows, swept by the same register
//                        segments, interpolated along x into the x-resampled float64 volume
//   rows_pipe_interp_kernel  x pass, rows of 833-1759 samples: the same, swept in a float64 shared-memory tile
//   march_yz_tma_kernel  y and z interpolation: TMA boxes of the x-resampled volume in an mbarrier ring, a
//                        4-plane register window marched along z
// General path (float64 throughout; short or very long lines, strong down-sampling, MICA_NO_TMA):
//   prefilter_cols_seg   IIR along a strided axis (z or y): a [n x 16] float64 tile of 16
//   prefilter_rows_seg   neighbouring lines (rows: [16 x n], contiguous axis) is staged in
//                        shared memory with coalesced loads; every line is cut into 16 segments
//                        swept concurrently, each warmed up over the kHorizon samples before
//                        (causal) / after (anticausal) it -- the pole's impulse response has
//                        decayed below double rounding by then -- so all 256 threads recurse
//   prefilter_cols / prefilter_rows   one thread per line in shared memory (short or long lines)
//   prefilter_cols_global             one thread per line in global memory (lines that fit no tile)
//   march3_tma_kernel    separable 4x4x4 gather: a CTA owns an [8 y x 64 x] output column and
//                        marches along z; each source plane arrives as a TMA box, is
//                        x-interpolated into shared memory, y-interpolated into a 4-plane
//                        register window, and every output plane is 4 FMAs from that window
//   march3_kernel        the same march fed by register prefetch (odd sx, wide x spans, MICA_NO_TMA)
//   gather3_kernel       one thread per output voxel (axes under 4 samples, strong down-sampling,
//                        mica_resample_force_generic)
// Order 1: gather1_kernel, trilinear, one thread per output voxel, no prefilter.
// Host side: resample_impl checks what every route shares, then hands over to resample_fast or resample_general (or
// launches gather1_kernel); each path checks its own arguments and encodes its tensor map before the first launch.
//
// Integer maps (int8 / int16 / uint16, DESIGN.md D12) always take the general path: its z prefilter reads the
// map's own type, and its interpolation kernels store with SciPy's integer rule (store_out).  The fast path's
// float32 coefficients are not exact enough to round to the reference's integers.  Given a block of a longer z line
// (a z-slab), an integer map's z prefilter numbers its segments on the whole line (seg16_plan), so the slab gets the
// whole map's bits; float32 blocks on the general path are prefiltered as lines of their own.
#include <cuda.h>
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"

namespace mica {

struct Tap {
  int idx[4];
  double w[4];
};

template <typename T>
struct IntRange;
template <>
struct IntRange<int8_t> {
  static constexpr double lo = -128.0, hi = 127.0;
};
template <>
struct IntRange<int16_t> {
  static constexpr double lo = -32768.0, hi = 32767.0;
};
template <>
struct IntRange<uint16_t> {
  static constexpr double lo = 0.0, hi = 65535.0;
};

// SciPy's store of an interpolated float64 value into the output array: float32 rounds to nearest; an integer
// type rounds half away from zero (t > 0 ? t + 0.5 : t - 0.5, truncated toward zero) and saturates at the
// type's range -- the cubic spline overshoots the input range on noisy maps
template <typename T>
__device__ __forceinline__ void store_out(T* p, double v) {
  if constexpr (std::is_same<T, float>::value) {
    st_stream(p, (float)v);
  } else {
    double t = v > 0.0 ? v + 0.5 : v - 0.5;
    t = t < IntRange<T>::lo ? IntRange<T>::lo : (t > IntRange<T>::hi ? IntRange<T>::hi : t);
    *p = (T)(int)t;
  }
}

__device__ __forceinline__ int mirror_index(long idx, int len) {
  // SciPy ni_interpolation.c edge handling for NI_EXTEND_MIRROR-like taps
  if (len <= 1) return 0;
  long s2 = 2L * len - 2;
  if (idx < 0) {
    idx = s2 * (long)(-idx / s2) + idx;
    idx = (idx <= 1 - len) ? idx + s2 : -idx;
  } else if (idx >= len) {
    idx -= s2 * (long)(idx / s2);
    if (idx >= len) idx = s2 - idx;
  }
  return (int)idx;
}

__global__ void taps_kernel(Tap* __restrict__ taps, int n_local, int k0, int n_in, int n_out, int order,
                            int in_off, int in_local) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_local) return;
  int k = k0 + i;
  double zoom = (n_out > 1) ? (double)(n_in - 1) / (double)(n_out - 1) : 1.0;
  double cc = (double)k * zoom;
  Tap t;
  if (cc < 0.0 || cc > (double)(n_in - 1)) {  // SciPy map_coordinate(NI_EXTEND_CONSTANT) -> cval
    for (int l = 0; l < 4; ++l) {
      t.idx[l] = 0;
      t.w[l] = 0.0;
    }
  } else {
    double fl = floor(cc);
    double x = cc - fl;
    long start;
    int ntap;
    if (order == 3) {
      start = (long)fl - 1;
      ntap = 4;
      double y = x, z = 1.0 - x;
      t.w[1] = (y * y * (y - 2.0) * 3.0 + 4.0) / 6.0;
      t.w[2] = (z * z * (z - 2.0) * 3.0 + 4.0) / 6.0;
      t.w[0] = z * z * z / 6.0;
      t.w[3] = 1.0 - t.w[0] - t.w[1] - t.w[2];
    } else {
      start = (long)fl;
      ntap = 2;
      t.w[0] = 1.0 - x;
      t.w[1] = x;
      t.w[2] = t.w[3] = 0.0;
    }
    for (int l = 0; l < 4; ++l) {
      int g = (l < ntap) ? mirror_index(start + l, n_in) : 0;
      int loc = g - in_off;
      loc = loc < 0 ? 0 : (loc >= in_local ? in_local - 1 : loc);
      t.idx[l] = (l < ntap) ? loc : 0;
    }
  }
  taps[i] = t;
}

// ---------------------------------------------------------------- prefilter
constexpr double kPole = -0.26794919243112270647;  // sqrt(3) - 2
constexpr int kInitHorizon = 56;                    // |pole|^56 ~ 1e-32: below double rounding

// One thread filters one line in place; `stride` is the distance (in doubles) between
// successive samples of the line (int inside a shared-memory tile, int64_t in global memory).
template <typename Stride>
__device__ __forceinline__ void iir_line(double* line, int n, Stride stride) {
  if (n < 2) return;
  const double z = kPole;
  // causal initialisation, mirror boundary, SciPy's pairing of k and n-1-k
  double z_n_1 = pow(z, (double)(n - 1));
  double c0 = line[0] + z_n_1 * line[(n - 1) * stride];
  double z_i = z;
  int lim = min(n - 1, kInitHorizon);
  for (int k = 1; k < lim; ++k) {
    c0 += z_i * (line[k * stride] + z_n_1 * line[(n - 1 - k) * stride]);
    z_i *= z;
  }
  c0 /= (1.0 - z_n_1 * z_n_1);
  line[0] = c0;
  double prev = c0;
#pragma unroll 4
  for (int k = 1; k < n; ++k) {
    prev = fma(z, prev, line[k * stride]);
    line[k * stride] = prev;
  }
  // anticausal
  double last = (z / (z * z - 1.0)) * (prev + z * line[(n - 2) * stride]);
  line[(n - 1) * stride] = last;
  prev = last;
#pragma unroll 4
  for (int k = n - 2; k >= 0; --k) {
    prev = z * (prev - line[k * stride]);
    line[k * stride] = prev;
  }
}

constexpr double kGain = (1.0 - kPole) * (1.0 - 1.0 / kPole);  // = 6

// lines along a strided axis.  grid = (ceil(n_cols / CW), n_outer)
// Strides of a column pass: sample k of column j of outer index o sits at
//   in [o * outer_in  + k * line_in  + j]     out[o * outer_out + k * line_out + j]
// (in and out differ when the output volume has a padded row pitch).
struct ColStrides {
  int64_t line_in, line_out, outer_in, outer_out;
};

template <typename TIn, int CW>
__global__ void __launch_bounds__(256)
prefilter_cols(const TIn* __restrict__ in, double* __restrict__ out, int n, int n_cols, ColStrides S) {
  extern __shared__ double tile[];  // [n][CW]
  const int col0 = blockIdx.x * CW;
  const int64_t base_in = (int64_t)blockIdx.y * S.outer_in + col0, base_out = (int64_t)blockIdx.y * S.outer_out + col0;
  const int ncol = min(CW, n_cols - col0);
  const double gain = (n >= 2) ? kGain : 1.0;  // SciPy leaves length-1 axes unfiltered
  for (int e = threadIdx.x; e < n * CW; e += blockDim.x) {
    int k = e / CW, j = e % CW;
    if (j < ncol) tile[e] = (double)in[base_in + (int64_t)k * S.line_in + j] * gain;
  }
  __syncthreads();
  if (threadIdx.x < ncol) iir_line(tile + threadIdx.x, n, CW);
  __syncthreads();
  for (int e = threadIdx.x; e < n * CW; e += blockDim.x) {
    int k = e / CW, j = e % CW;
    if (j < ncol) out[base_out + (int64_t)k * S.line_out + j] = tile[e];
  }
}

// lines along the contiguous axis.  grid = ceil(n_rows / R); tile [R][n + 1]
template <int R>
__global__ void __launch_bounds__(256)
prefilter_rows(double* __restrict__ data, int n, int64_t n_rows) {
  extern __shared__ double tile[];
  const int pitch = n | 1;  // odd pitch: rows start in different banks
  const int64_t row0 = (int64_t)blockIdx.x * R;
  const int nrow = (int)min((int64_t)R, n_rows - row0);
  double* g = data + row0 * n;
  const double gain = (n >= 2) ? kGain : 1.0;
  for (int e = threadIdx.x; e < nrow * n; e += blockDim.x) {
    int r = e / n, k = e - r * n;
    tile[r * pitch + k] = g[e] * gain;
  }
  __syncthreads();
  if (threadIdx.x < nrow) iir_line(tile + threadIdx.x * pitch, n, 1);
  __syncthreads();
  for (int e = threadIdx.x; e < nrow * n; e += blockDim.x) {
    int r = e / n, k = e - r * n;
    g[e] = tile[r * pitch + k];
  }
}


// ------------------------------------------------- segment-parallel prefilter
// |pole|^30 = 7e-18: a recursion started kHorizon samples early from a zero state (the samples
// before index 0 / after n-1 being the mirror images SciPy's boundary rule implies) has
// forgotten its start to below double rounding when it reaches the segment.
constexpr int kHorizon = 30;
constexpr int kMinSegLine = 96;     // shorter lines take the one-thread-per-line kernels

// Filters samples [k0, k1) of one line of n samples in place; all threads of the block call this together (three
// block-wide barriers inside).  `line` points at sample g0 (a block of a longer line holds samples [g0, ...); g0 = 0
// for a whole line), `stride` in doubles, k0 / k1 are numbers on the whole line.  `causal` runs the warm-up and the
// causal sweep (up to sample causal_end, exclusive), `anti` (which implies causal, and causal_end >= k1) the
// anticausal ones as well: a segment whose causal values another segment's anticausal warm-up reads, but whose own
// coefficients nobody needs, runs the causal half only, and only as far as those values go.
__device__ __forceinline__ void iir_segment(double* line, int g0, int n, int stride, int k0, int k1, int causal_end,
                                            bool causal, bool anti) {
  const double z = kPole;
  double st = 0.0;
  if (causal) {   // causal state entering the segment: sum_j z^j s[k0-1-j], mirrored below 0
    for (int m = kHorizon - 1; m >= 0; --m) {
      int idx = k0 - 1 - m;
      idx = idx < 0 ? -idx : idx;
      st = fma(z, st, line[(idx - g0) * stride]);
    }
  }
  __syncthreads();   // every warm-up read of raw samples is done before anyone overwrites them
  if (causal) {
    const int kc = min(k1, causal_end);
#pragma unroll 4
    for (int k = k0; k < kc; ++k) {
      st = fma(z, st, line[(k - g0) * stride]);
      line[(k - g0) * stride] = st;
    }
  }
  __syncthreads();
  bool at_end = false;
  if (anti) {   // anticausal state just above the segment
    if (k1 >= n) {   // the end initialisation, read here: sample n - 2 may belong to the segment below
      at_end = true;
      st = (z / (z * z - 1.0)) * (line[(n - 1 - g0) * stride] + z * line[(n - 2 - g0) * stride]);
    } else {
      int kk = k1 + kHorizon;
      int k = kk - 1;
      st = 0.0;
      if (kk >= n) {  // the exact end initialisation is within reach: start from it
        st = (z / (z * z - 1.0)) * (line[(n - 1 - g0) * stride] + z * line[(n - 2 - g0) * stride]);
        k = n - 2;
      }
      for (; k >= k1; --k) st = fma(z, st, -z * line[(k - g0) * stride]);   // z (st - c): one FMA on the chain
    }
  }
  __syncthreads();
  if (anti) {
    int k = k1 - 1;
    if (at_end) {
      line[(n - 1 - g0) * stride] = st;
      k = n - 2;
    }
#pragma unroll 4
    for (; k >= k0; --k) {
      st = fma(z, st, -z * line[(k - g0) * stride]);
      line[(k - g0) * stride] = st;
    }
  }
}

// Register-blocked variant for the pipelined row pass.  iir_segment walks shared memory inside the
// dependent chain (load -> FMA -> store per sample: ncu shows the warps waiting on the shared-memory
// scoreboard 5 cycles per issued instruction).  Here a thread first pulls its segment (<= LMAX samples) and
// its warm-up samples into registers with independent loads, runs both recursions register to register and
// writes the segment back once per sweep.  H = warm-up horizon: |pole|^20 = 4e-12, four orders below the
// float32 rounding of what these passes produce.  STRIDE is the (compile-time) distance between samples.
template <int LMAX, int H, int STRIDE>
__device__ __forceinline__ void iir_segment_reg(double* line, int n, int k0, int k1, bool active) {
  const double z = kPole;
  double s[LMAX];
  double st = 0.0;
  if (active) {
    double w[H];
#pragma unroll
    for (int m = 0; m < H; ++m) {      // samples k0-1-m, mirrored below 0
      int idx = k0 - 1 - m;
      idx = idx < 0 ? -idx : idx;
      w[m] = line[idx * STRIDE];
    }
#pragma unroll
    for (int i = 0; i < LMAX; ++i) s[i] = (k0 + i < k1) ? line[(k0 + i) * STRIDE] : 0.0;
#pragma unroll
    for (int m = H - 1; m >= 0; --m) st = fma(z, st, w[m]);
  }
  __syncthreads();   // every read of raw samples is done before anyone overwrites them
  if (active) {
#pragma unroll
    for (int i = 0; i < LMAX; ++i)
      if (k0 + i < k1) {
        st = fma(z, st, s[i]);
        s[i] = st;
        line[(k0 + i) * STRIDE] = st;   // the causal result: neighbours warm up on it
      }
  }
  __syncthreads();
  bool at_end = false;
  if (active) {      // anticausal state just above the segment
    if (k1 >= n) {
      at_end = true;
    } else if (k1 + H >= n) {   // the exact end initialisation is within reach: start from it
      st = (z / (z * z - 1.0)) * (line[(n - 1) * STRIDE] + z * line[(n - 2) * STRIDE]);
      for (int k = n - 2; k >= k1; --k) st = fma(z, st, -z * line[k * STRIDE]);
    } else {
      double w[H];
#pragma unroll
      for (int m = 0; m < H; ++m) w[m] = line[(k1 + m) * STRIDE];
      st = 0.0;
#pragma unroll
      for (int m = H - 1; m >= 0; --m) st = fma(z, st, -z * w[m]);
    }
  }
  __syncthreads();   // every warm-up read of causal results is done
  if (active) {
    const int last = k1 - 1 - k0;     // index of the segment's last sample in s[]
#pragma unroll
    for (int i = LMAX - 1; i >= 0; --i)
      if (i <= last) {
        if (at_end && i == last) {
          const double below = (i >= 1) ? s[i >= 1 ? i - 1 : 0] : line[(n - 2) * STRIDE];   // still the causal value
          st = (z / (z * z - 1.0)) * (s[i] + z * below);
        } else {
          st = fma(z, st, -z * s[i]);
        }
        line[(k0 + i) * STRIDE] = st;
      }
  }
}

// lines along a strided axis.  grid = (ceil(n_cols / L), n_outer), block = 256, tile [n][L], 256 / L segments per
// line.  The tile holds samples [g0, g0 + n) of lines of ng samples (g0 = 0, ng = n for whole lines); the segments are
// those of the WHOLE line, seg_lo .. seg_causal_hi run the causal sweep up to causal_end, seg_lo .. seg_out_hi both
// (seg16_plan).
template <typename TIn, int L>
__global__ void __launch_bounds__(256)
prefilter_cols_seg(const TIn* __restrict__ in, double* __restrict__ out, int n, int n_cols, ColStrides S, int g0,
                   int ng, int seg_lo, int seg_causal_hi, int seg_out_hi, int causal_end) {
  extern __shared__ double tile[];
  constexpr int kSegs = 256 / L;
  const int col0 = blockIdx.x * L;
  const int64_t base_in = (int64_t)blockIdx.y * S.outer_in + col0, base_out = (int64_t)blockIdx.y * S.outer_out + col0;
  const int ncol = min(L, n_cols - col0);
  const int j = threadIdx.x & (L - 1), seg = threadIdx.x / L;
  if (j < ncol) {
    const TIn* p = in + base_in + j;
#pragma unroll 8
    for (int k = seg; k < n; k += kSegs) tile[k * L + j] = (double)p[(int64_t)k * S.line_in] * kGain;
  }
  __syncthreads();
  const int len = (ng + kSegs - 1) / kSegs;
  const int k0 = seg * len, k1 = min(ng, k0 + len);
  const bool on = j < ncol && k0 < k1 && seg >= seg_lo;
  iir_segment(tile + j, g0, ng, L, k0, k1, causal_end, on && seg <= seg_causal_hi, on && seg <= seg_out_hi);
  __syncthreads();
  if (j < ncol) {
    double* q = out + base_out + j;
#pragma unroll 8
    for (int k = seg; k < n; k += kSegs) q[(int64_t)k * S.line_out] = tile[k * L + j];
  }
}

// lines along the contiguous axis.  grid = ceil(n_rows / L), block = 256, tile [L][n | 1]
template <int L>
__global__ void __launch_bounds__(256)
prefilter_rows_seg(double* __restrict__ data, int n, int64_t n_rows) {
  extern __shared__ double tile[];
  constexpr int kSegs = 256 / L;
  const int pitch = n | 1;
  const int64_t row0 = (int64_t)blockIdx.x * L;
  const int nrow = (int)min((int64_t)L, n_rows - row0);
  double* g = data + row0 * n;
  for (int r = threadIdx.x >> 5; r < nrow; r += 8)
    for (int k = threadIdx.x & 31; k < n; k += 32) tile[r * pitch + k] = g[(int64_t)r * n + k] * kGain;
  __syncthreads();
  const int r = threadIdx.x & (L - 1), seg = threadIdx.x / L;
  const int len = (n + kSegs - 1) / kSegs;
  const int k0 = seg * len, k1 = min(n, k0 + len);
  iir_segment(tile + r * pitch, 0, n, 1, k0, k1, n, r < nrow && k0 < k1, r < nrow && k0 < k1);
  __syncthreads();
  for (int rr = threadIdx.x >> 5; rr < nrow; rr += 8)
    for (int k = threadIdx.x & 31; k < n; k += 32) g[(int64_t)rr * n + k] = tile[rr * pitch + k];
}

// fallback for lines too long for shared memory: sweep in global memory
// (double output only: the sweep runs in place in global memory)
template <typename TIn>
__global__ void prefilter_cols_global(const TIn* __restrict__ in, double* __restrict__ out, int n,
                                      int64_t line_stride, int n_cols, int64_t outer_stride) {
  int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= n_cols) return;
  const int64_t base = (int64_t)blockIdx.y * outer_stride + col;
  const double gain = (n >= 2) ? kGain : 1.0;
  for (int k = 0; k < n; ++k) out[base + k * line_stride] = (double)in[base + k * line_stride] * gain;
  iir_line(out + base, n, line_stride);
}

// ------------------------------------------------------------------- gather
// grid = (ceil(nx/128), ny, nz_local); one output voxel per thread
template <typename TOut>
__global__ void __launch_bounds__(128)
gather3_kernel(const double* __restrict__ c, int sy, int sx, const Tap* __restrict__ tz,
               const Tap* __restrict__ ty, const Tap* __restrict__ tx, TOut* __restrict__ dst, int ny,
               int nx) {
  int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= nx) return;
  const int y = blockIdx.y, z = blockIdx.z;
  const Tap Tx = tx[x];
  const Tap Ty = ty[y];
  const Tap Tz = tz[z];
  const int64_t plane = (int64_t)sy * sx;
  double acc = 0.0;
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    const double* pz = c + (int64_t)Tz.idx[l] * plane;
    double accy = 0.0;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const double* row = pz + (int64_t)Ty.idx[m] * sx;
      double r = Tx.w[0] * row[Tx.idx[0]] + Tx.w[1] * row[Tx.idx[1]] + Tx.w[2] * row[Tx.idx[2]] +
                 Tx.w[3] * row[Tx.idx[3]];
      accy += Ty.w[m] * r;
    }
    acc += Tz.w[l] * accy;
  }
  store_out(dst + ((int64_t)z * ny + y) * nx + x, acc);
}


// ---------------------------------------------------------- marching gather
// Per output plane: the four (mirrored) z taps folded into one contiguous 4-plane window
// [base, base+3] of local source planes, weights of coinciding planes merged.
struct ZWin {
  int base;
  int pad;
  double w[4];
};

__global__ void zwin_kernel(const Tap* __restrict__ tz, ZWin* __restrict__ zw, int n, int in_local) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Tap t = tz[i];
  int base = 0x7fffffff;
  for (int l = 0; l < 4; ++l)
    if (t.w[l] != 0.0) base = min(base, t.idx[l]);
  // all-zero taps (D11) only occur past the end of the map: park the window at the last planes so
  // that `base` stays non-decreasing along z (the march emits a plane when its window is loaded)
  if (base == 0x7fffffff) base = in_local - 4;
  base = max(0, min(base, in_local - 4));
  ZWin z;
  z.base = base;
  z.pad = 0;
  for (int j = 0; j < 4; ++j) z.w[j] = 0.0;
  for (int l = 0; l < 4; ++l) {
    if (t.w[l] == 0.0) continue;
    const int j = min(3, max(0, t.idx[l] - base));
    z.w[j] += t.w[l];
  }
  zw[i] = z;
}

// grid = (ceil(nx / 64), ceil(ny / 8), z chunks), block = 256.  NI * 4 = source rows staged per plane.
template <int NI, typename TOut>
__global__ void __launch_bounds__(256)
march3_kernel(const double* __restrict__ c, int sy, int sx, const ZWin* __restrict__ zw,
              const Tap* __restrict__ ty, const Tap* __restrict__ tx, TOut* __restrict__ dst, int ny, int nx,
              int nz_local, int zchunk) {
  constexpr int TX = 64, TY = 8, ROWS = NI * 4;
  __shared__ double A[2][ROWS][TX];
  __shared__ int s_lo;
  const int t = threadIdx.x;
  const int lx = t & (TX - 1), lr = t >> 6;
  const int x = blockIdx.x * TX + lx;
  const int y0 = blockIdx.y * TY;
  const int z_begin = blockIdx.z * zchunk, z_end = min(nz_local, z_begin + zchunk);
  if (z_begin >= z_end) return;

  // lowest source row any output row of this tile taps (zero-weight rows, D11, excluded)
  if (t == 0) s_lo = 0x7fffffff;
  __syncthreads();
  if (t < TY * 4) {
    const int r = min(y0 + (t >> 2), ny - 1);
    if (ty[r].w[t & 3] != 0.0) atomicMin(&s_lo, ty[r].idx[t & 3]);
  }
  __syncthreads();
  const int lo_y = (s_lo == 0x7fffffff) ? 0 : s_lo;

  const Tap Tx = tx[min(x, nx - 1)];
  int iy[2][4];
  double wy[2][4];
#pragma unroll
  for (int o = 0; o < 2; ++o) {
    const Tap T = ty[min(y0 + lr + 4 * o, ny - 1)];
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      wy[o][m] = T.w[m];
      iy[o][m] = (T.w[m] != 0.0) ? min(ROWS - 1, T.idx[m] - lo_y) : 0;
    }
  }
  // source rows this thread x-interpolates: lo_y + lr + 4 i (clamped: rows past sy-1 are never tapped)
  const int64_t plane = (int64_t)sy * sx;
  const double* rowp[NI];
#pragma unroll
  for (int i = 0; i < NI; ++i) rowp[i] = c + (int64_t)min(lo_y + lr + 4 * i, sy - 1) * sx;

  double v[2][4];
#pragma unroll
  for (int o = 0; o < 2; ++o)
#pragma unroll
    for (int m = 0; m < 4; ++m) v[o][m] = 0.0;

  const int p_start = zw[z_begin].base, p_last = zw[z_end - 1].base + 3;
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const double* r = rowp[i] + (int64_t)p_start * plane;
    A[0][lr + 4 * i][lx] = Tx.w[0] * r[Tx.idx[0]] + Tx.w[1] * r[Tx.idx[1]] + Tx.w[2] * r[Tx.idx[2]] +
                           Tx.w[3] * r[Tx.idx[3]];
  }
  __syncthreads();

  int zc = z_begin;
  int next_emit = zw[zc].base + 3;
  for (int p = p_start; p <= p_last; ++p) {
    const int cur = (p - p_start) & 1;
    const bool more = p < p_last;
    double raw[NI][4];
    if (more) {   // issue the next plane's loads before touching shared memory
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const double* r = rowp[i] + (int64_t)(p + 1) * plane;
#pragma unroll
        for (int l = 0; l < 4; ++l) raw[i][l] = r[Tx.idx[l]];
      }
    }
#pragma unroll
    for (int o = 0; o < 2; ++o) {
      const double vn = wy[o][0] * A[cur][iy[o][0]][lx] + wy[o][1] * A[cur][iy[o][1]][lx] +
                        wy[o][2] * A[cur][iy[o][2]][lx] + wy[o][3] * A[cur][iy[o][3]][lx];
      v[o][0] = v[o][1];
      v[o][1] = v[o][2];
      v[o][2] = v[o][3];
      v[o][3] = vn;
    }
    while (zc < z_end && next_emit <= p) {
      const ZWin Wz = zw[zc];
#pragma unroll
      for (int o = 0; o < 2; ++o) {
        const int y = y0 + lr + 4 * o;
        const double acc = Wz.w[0] * v[o][0] + Wz.w[1] * v[o][1] + Wz.w[2] * v[o][2] + Wz.w[3] * v[o][3];
        if (x < nx && y < ny) store_out(dst + ((int64_t)zc * ny + y) * nx + x, acc);
      }
      ++zc;
      if (zc < z_end) next_emit = zw[zc].base + 3;
    }
    if (more) {
#pragma unroll
      for (int i = 0; i < NI; ++i)
        A[cur ^ 1][lr + 4 * i][lx] = Tx.w[0] * raw[i][0] + Tx.w[1] * raw[i][1] + Tx.w[2] * raw[i][2] +
                                     Tx.w[3] * raw[i][3];
    }
    __syncthreads();
  }
}

// ------------------------------------------------- marching gather, TMA-fed
// Same march as march3_kernel, but the source rows of each plane arrive as one
// cp.async.bulk.tensor box ([ROWS y] x [XB x] float64 of the coefficient volume, tensor map
// dims (x, y, z)) in a kStages-deep shared-memory ring filled by one elected thread: the loads
// of planes p+1..p+3 are in flight while plane p is interpolated, and no register is spent on
// staging.  Rows / columns past the map edge are zero-filled by the TMA unit and never tapped.
constexpr int kMarchStages = 6;

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  }
}

// ------------------------------------------------- register-only column pass (fast path, z and y axes)
// ncu on the tile kernels above: the warps wait on shared memory inside the recursion and on the four
// block-wide barriers per tile; 25-30 % of the HBM bandwidth.  This variant has NO shared memory and NO
// barrier: a thread owns `len` consecutive samples of one column and computes everything it needs itself --
// it reads its samples plus H before and H after straight from global memory (128-byte runs per row across
// the warp; the overlap with the neighbouring segments is served by L1), runs the causal recursion over
// all of them and the anticausal one back down, register to register.  Both recursions are one FMA per
// sample: with d[k] = c[k] / (-z) the anticausal step c[k] = z (c[k+1] - c+[k]) becomes
// d[k] = c+[k] + z d[k+1], the same form as the causal one; gain and -z are applied once per output.
// H = 16: |pole|^16 = 7e-10 relative, two orders below the float32 rounding of the output.
constexpr int kColH = 16;
constexpr int kColLen = 26;      // longest segment (registers: kColLen + kColH causal values)

// One segment: samples [k0, k0 + kColLen) of a line, window [k0 - H, k0 + kColLen + H).  `load(idx)` returns
// sample idx as float, `store(k, value)` takes the finished coefficient of sample k.  EDGE = the window leaves
// [0, n): indices are mirrored (SciPy's boundary rule; running the recursions over the mirror image replaces the
// closed-form end initialisation up to |pole|^H).
// Only the kColLen samples a thread OWNS and kNear samples either side of them go through float64.  The far
// part of the H-sample run-in of the causal recursion, the causal values of the far look-ahead samples and the far
// part of the run-in of the anticausal recursion are float32: an error e in such a state reaches the first owned
// sample as |pole|^(kNear+1) e = 1.4e-3 e and decays by 0.27 per sample, i.e. <= 2e-10 relative -- below the
// 7e-10 the finite horizon costs anyway, so a line cut into different segments (a z-slab of a map against the
// whole map) still rounds to the same float32 coefficients.  That shortens the dependent float64 chain from
// 100 to 68 DFMA per segment (the float32 FMAs issue at twice the rate and half the latency) and saves 24 of
// the 58 f32 -> f64 conversions.
constexpr int kNear = 4;

template <bool EDGE, typename Load, typename Store>
__device__ __forceinline__ void reg_segment(Load load, Store store, int n, int k0, int k1) {
  constexpr int H = kColH, W = kColLen + 2 * kColH, F = kColH - kNear;   // F far samples on either side
  const double z = kPole;
  const float zf = (float)kPole;
  float x[W];
#pragma unroll
  for (int i = 0; i < W; ++i) {
    int idx = k0 - H + i;
    if (EDGE) {
      idx = idx < 0 ? -idx : idx;
      idx = idx > n - 1 ? 2 * (n - 1) - idx : idx;
      idx = idx < 0 ? 0 : idx;                    // (only for lines shorter than the window)
    }
    x[i] = load(idx);
  }
  float run = 0.f;                                // causal run-in, far part: samples k0 - H .. k0 - kNear - 1
#pragma unroll
  for (int i = 0; i < F; ++i) run = fmaf(zf, run, x[i]);
  double st = (double)run;
#pragma unroll
  for (int i = F; i < H; ++i) st = fma(z, st, (double)x[i]);
  double cp[kColLen + kNear];                     // causal values of the owned samples and the kNear after them
#pragma unroll
  for (int i = 0; i < kColLen + kNear; ++i) {
    st = fma(z, st, (double)x[H + i]);
    cp[i] = st;
  }
  float ahead[F];                                 // causal values of the far look-ahead samples
  run = (float)st;
#pragma unroll
  for (int i = 0; i < F; ++i) {
    run = fmaf(zf, run, x[H + kColLen + kNear + i]);
    ahead[i] = run;
  }
  const double scale = -z * kGain;                // output = gain * c = gain * (-z) * d
  float back = 0.f;                               // anticausal run-in, downwards: far part, then the near samples
#pragma unroll
  for (int i = F - 1; i >= 0; --i) back = fmaf(zf, back, ahead[i]);
  double d = (double)back;
#pragma unroll
  for (int i = kColLen + kNear - 1; i >= kColLen; --i) d = fma(z, d, cp[i]);
#pragma unroll
  for (int i = kColLen - 1; i >= 0; --i) {     // store is called for every i, downwards (it may walk a pointer)
    d = fma(z, d, cp[i]);
    store(k0 + i, d * scale, k0 + i < k1);
  }
}

// `n` samples of the line are in memory, samples [g0, g0 + n) of a line of `ng` (a z-slab of a map holds a block
// of every z line; g0 = 0, ng = n otherwise).  k0, k1 and the window are GLOBAL sample numbers: the segments of a
// block are the segments the whole line would be cut into, so a coefficient is computed from the same window by
// the same operations whichever rank holds it -- bit-identical, as long as the block contains the window
// (SlabPlan sizes the halo for that).  A window that leaves the block without leaving the line (a halo shorter
// than that) is reflected at the block end: >= kColH real samples away from every coefficient the caller
// needs, the accuracy of the finite horizon, no longer the identical bits.
template <bool EDGE>
__device__ __forceinline__ void cols_reg_segment(const float* __restrict__ p, float* __restrict__ q, int64_t line_in,
                                                 int64_t line_out, int n, int g0, int ng, int k0, int k1) {
  float* o = q + (int64_t)(k0 - g0 + kColLen - 1) * line_out;
  if (EDGE) {
    auto store = [&](int k, double v, bool on) {
      if (on && k >= g0 && k < g0 + n) *o = (float)v;
      o -= line_out;
    };
    reg_segment<true>([&](int idx) {
      int l = idx - g0;
      l = l < 0 ? -l : l;
      l = l > n - 1 ? 2 * (n - 1) - l : l;
      l = l < 0 ? 0 : l;
      return __ldg(p + (int64_t)l * line_in);
    }, store, ng, k0, k1);
  } else {   // interior windows are read in increasing order: walk the column with pointer increments only
    auto store = [&](int, double v, bool on) {
      if (on) *o = (float)v;
      o -= line_out;
    };
    const float* r = p + (int64_t)(k0 - g0 - kColH) * line_in;
    reg_segment<false>([&](int) {
      const float v = __ldg(r);
      r += line_in;
      return v;
    }, store, ng, k0, k1);
  }
}

// grid = (ceil(n_cols / 32), ceil(n_seg / 8), n_outer), block = 256: a WARP is 32 neighbouring columns of ONE
// segment (128-byte runs per row; every lane takes the same interior / mirrored path -- with two segments per
// warp a quarter of the warps ran both), the 8 warps of a CTA are 8 consecutive segments of those columns, so
// the windows that overlap meet in the same L1.  Segments seg0 .. seg0 + n_seg - 1 of the global line are run.
__global__ void __launch_bounds__(256, 2)
cols_reg_kernel(const float* __restrict__ in, float* __restrict__ out, int n, int n_cols, ColStrides S, int len,
                int n_seg, int g0, int ng, int seg0) {
  const int j = threadIdx.x & 31, seg = blockIdx.y * 8 + (threadIdx.x >> 5);
  const int col = blockIdx.x * 32 + j;
  const int k0 = (seg0 + seg) * len, k1 = min(ng, k0 + len);
  if (col >= n_cols || seg >= n_seg || k0 >= k1) return;
  const float* p = in + (int64_t)blockIdx.z * S.outer_in + col;
  float* q = out + (int64_t)blockIdx.z * S.outer_out + col;
  if (k0 - kColH >= g0 && k0 + kColLen + kColH <= g0 + n)
    cols_reg_segment<false>(p, q, S.line_in, S.line_out, n, g0, ng, k0, k1);
  else
    cols_reg_segment<true>(p, q, S.line_in, S.line_out, n, g0, ng, k0, k1);
}

// ------------------------------------------------- x pass of the fast path: prefilter + interpolation
// A persistent CTA walks over its tiles of rows with the float32 input of the NEXT tile already in flight
// (cp.async into a small staging ring: no registers), sweeps the staged tile and interpolates it along x.
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

constexpr int kPipeStages = 2;
constexpr int kRegSeg = 32;    // longest segment a thread of rows_pipe_interp_kernel keeps in registers
constexpr int kRegHorizon = 20;

// x axis, register form (rows of <= 32 x kColLen samples): as rows_pipe_interp_kernel below, but the sweep is the
// register-only segment of the column pass -- a thread pulls the 58-sample window of its segment out of the
// staged float32 row (lanes = the 16 or 32 segments of a row: odd segment lengths keep the banks distinct), runs
// both recursions in registers and writes its <= 26 coefficients to the float64 work tile once: one barrier
// before the interpolation instead of five.  dynamic smem = L * (n | 1) * 8 + kPipeStages * L * in_pitch * 4.
template <int SEGS>
__global__ void __launch_bounds__(16 * SEGS, 512 / (16 * SEGS))
rows_reg_interp_kernel(const float* __restrict__ in, int64_t in_pitch, double* __restrict__ out, int64_t out_pitch,
                       int n, int nx, int64_t n_rows, const Tap* __restrict__ tx, int len) {
  extern __shared__ __align__(16) uint8_t pipe_smem[];
  constexpr int L = 16, THREADS = 16 * SEGS;
  const int pitch = n | 1;
  const int sp = (int)in_pitch;
  double* work = reinterpret_cast<double*>(pipe_smem);
  float* stage0 = reinterpret_cast<float*>(pipe_smem + (((size_t)L * pitch * 8 + 15) & ~(size_t)15));
  const uint32_t stage_a = smem_addr(stage0);
  const long long n_tiles = (n_rows + L - 1) / L;
  const int chunks = sp / 4;
  auto prefetch = [&](long long tile, int sidx) {
    if (tile < n_tiles) {
      const int64_t row0 = tile * L;
      const int nrow = (int)min((int64_t)L, n_rows - row0);
      const float* g = in + row0 * in_pitch;
      const uint32_t dst = stage_a + (uint32_t)sidx * (uint32_t)(L * sp * 4);
      for (int e = threadIdx.x; e < nrow * chunks; e += THREADS) cp_async16(dst + (uint32_t)(e * 16), g + (int64_t)e * 4);
    }
    cp_async_commit();
  };
  long long tile = blockIdx.x;
  for (int i = 0; i < kPipeStages - 1; ++i) prefetch(tile + (long long)i * gridDim.x, i);
  int sidx = 0;
  const int seg = threadIdx.x % SEGS, r = threadIdx.x / SEGS;
  const int k0 = seg * len, k1 = min(n, k0 + len);
  const bool interior = k0 - kColH >= 0 && k0 + kColLen + kColH <= n;
  for (; tile < n_tiles; tile += gridDim.x) {
    prefetch(tile + (long long)(kPipeStages - 1) * gridDim.x, (sidx + kPipeStages - 1) % kPipeStages);
    cp_async_wait<kPipeStages - 1>();
    __syncthreads();                                   // staged rows visible; the work tile of the last tile is consumed
    const int64_t row0 = tile * L;
    const int nrow = (int)min((int64_t)L, n_rows - row0);
    if (r < nrow && k0 < k1) {
      const float* srow = stage0 + (size_t)sidx * L * sp + (size_t)r * sp;
      double* wrow = work + (size_t)r * pitch;
      auto load = [&](int idx) { return srow[idx]; };
      auto store = [&](int k, double v, bool on) {
        if (on) wrow[k] = v;
      };
      if (interior)
        reg_segment<false>(load, store, n, k0, k1);
      else
        reg_segment<true>(load, store, n, k0, k1);
    }
    __syncthreads();
    for (int x = threadIdx.x; x < nx; x += THREADS) {
      const Tap T = tx[x];
      double* o = out + row0 * out_pitch + x;
#pragma unroll 4
      for (int rr = 0; rr < nrow; ++rr) {
        const double* row = work + rr * pitch;
        o[(int64_t)rr * out_pitch] = T.w[0] * row[T.idx[0]] + T.w[1] * row[T.idx[1]] + T.w[2] * row[T.idx[2]] +
                                     T.w[3] * row[T.idx[3]];
      }
    }
    sidx = (sidx + 1) % kPipeStages;
  }
  cp_async_wait<0>();
}

// x axis, rows too long for the register form: rows of the (z,y)-filtered float32 volume (row pitch in_pitch, a
// multiple of 4) are staged by cp.async, prefiltered in a float64 work tile and interpolated to the nx output
// columns at once: what leaves the SM is the x-RESAMPLED float64 volume [rows][out_pitch], so the march that
// follows only interpolates along y and z.  dynamic smem = L * (n | 1) * 8 + kPipeStages * L * in_pitch * 4 bytes.
template <int L, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
rows_pipe_interp_kernel(const float* __restrict__ in, int64_t in_pitch, double* __restrict__ out, int64_t out_pitch,
                        int n, int nx, int64_t n_rows, const Tap* __restrict__ tx) {
  extern __shared__ __align__(16) uint8_t pipe_smem[];
  constexpr int kSegs = THREADS / L;
  const int pitch = n | 1;
  const int sp = (int)in_pitch;                                             // staging row pitch (floats)
  double* work = reinterpret_cast<double*>(pipe_smem);                      // [L][pitch]
  float* stage0 = reinterpret_cast<float*>(pipe_smem + (((size_t)L * pitch * 8 + 15) & ~(size_t)15));
  const uint32_t stage_a = smem_addr(stage0);
  const long long n_tiles = (n_rows + L - 1) / L;
  const int chunks = sp / 4;                                                // 16-byte chunks per row

  auto prefetch = [&](long long tile, int sidx) {
    if (tile < n_tiles) {
      const int64_t row0 = tile * L;
      const int nrow = (int)min((int64_t)L, n_rows - row0);
      const float* g = in + row0 * in_pitch;
      const uint32_t dst = stage_a + (uint32_t)sidx * (uint32_t)(L * sp * 4);
      for (int e = threadIdx.x; e < nrow * chunks; e += THREADS)             // rows are contiguous: one flat copy
        cp_async16(dst + (uint32_t)(e * 16), g + (int64_t)e * 4);
    }
    cp_async_commit();
  };

  long long tile = blockIdx.x;
  for (int i = 0; i < kPipeStages - 1; ++i) prefetch(tile + (long long)i * gridDim.x, i);
  int sidx = 0;
  const int r_seg = threadIdx.x & (L - 1), seg = threadIdx.x / L;
  const int len = (n + kSegs - 1) / kSegs;
  const int k0 = seg * len, k1 = min(n, k0 + len);
  for (; tile < n_tiles; tile += gridDim.x) {
    prefetch(tile + (long long)(kPipeStages - 1) * gridDim.x, (sidx + kPipeStages - 1) % kPipeStages);
    cp_async_wait<kPipeStages - 1>();
    __syncthreads();
    const int64_t row0 = tile * L;
    const int nrow = (int)min((int64_t)L, n_rows - row0);
    const float* st = stage0 + (size_t)sidx * L * sp;
    for (int r = threadIdx.x >> 5; r < nrow; r += THREADS / 32)
      for (int k = threadIdx.x & 31; k < n; k += 32) work[r * pitch + k] = (double)st[r * sp + k] * kGain;
    __syncthreads();
    iir_segment_reg<kRegSeg, kRegHorizon, 1>(work + r_seg * pitch, n, k0, k1, r_seg < nrow && k0 < k1);
    __syncthreads();
    // a thread owns output columns x, x + THREADS, ...: its taps stay in registers while it walks the rows
    for (int x = threadIdx.x; x < nx; x += THREADS) {
      const Tap T = tx[x];
      double* o = out + row0 * out_pitch + x;
#pragma unroll 4
      for (int r = 0; r < nrow; ++r) {
        const double* row = work + r * pitch;
        o[(int64_t)r * out_pitch] = T.w[0] * row[T.idx[0]] + T.w[1] * row[T.idx[1]] + T.w[2] * row[T.idx[2]] +
                                    T.w[3] * row[T.idx[3]];
      }
    }
    __syncthreads();
    sidx = (sidx + 1) % kPipeStages;
  }
  cp_async_wait<0>();
}

// grid = (ceil(nx / 64), ceil(ny / 8), z chunks), block = 256; dynamic smem = ring + 1 KB alignment slack
// Integer outputs: 2 CTAs per SM, so that the saturating store fits the register budget without spilling.
template <int NI, typename TOut>
__global__ void __launch_bounds__(256, std::is_same<TOut, float>::value ? 3 : 2)
march3_tma_kernel(const __grid_constant__ CUtensorMap tmap, int xb, const ZWin* __restrict__ zw,
                  const Tap* __restrict__ ty, const Tap* __restrict__ tx, TOut* __restrict__ dst, int ny, int nx,
                  int nz_local, int zchunk) {
  constexpr int TX = 64, TY = 8, ROWS = NI * 4;
  extern __shared__ uint8_t march_smem[];
  __shared__ double A[2][ROWS][TX];
  __shared__ __align__(8) uint64_t full[kMarchStages];
  __shared__ int s_lo[2];
  double* ring = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(march_smem) + 127) & ~(uintptr_t)127);
  const int t = threadIdx.x;
  const int lx = t & (TX - 1), lr = t >> 6;
  const int x0 = blockIdx.x * TX, x = x0 + lx;
  const int y0 = blockIdx.y * TY;
  const int z_begin = blockIdx.z * zchunk, z_end = min(nz_local, z_begin + zchunk);
  if (z_begin >= z_end) return;
  const int stage_elems = ROWS * xb;
  const int stage_stride = (stage_elems + 15) & ~15;   // ring stages stay 128-byte aligned (TMA destination)

  if (t == 0) {
    s_lo[0] = s_lo[1] = 0x7fffffff;
    for (int i = 0; i < kMarchStages; ++i)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(&full[i])));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  // lowest source row / column any output of this tile taps (zero-weight taps, D11, excluded)
  if (t < TY * 4) {
    const int r = min(y0 + (t >> 2), ny - 1);
    if (ty[r].w[t & 3] != 0.0) atomicMin(&s_lo[0], ty[r].idx[t & 3]);
  }
  {
    const int xx = min(x, nx - 1);
#pragma unroll
    for (int l = 0; l < 4; ++l)
      if (tx[xx].w[l] != 0.0) atomicMin(&s_lo[1], tx[xx].idx[l]);
  }
  __syncthreads();
  const int lo_y = (s_lo[0] == 0x7fffffff) ? 0 : s_lo[0];
  // even: the box must start on a 16-byte boundary of the float64 rows (odd starts fault on B200)
  const int lo_x = ((s_lo[1] == 0x7fffffff) ? 0 : s_lo[1]) & ~1;

  // everything below addresses shared memory with precomputed 32-bit byte offsets (one add per
  // access): the inner loop is issue-bound, and generic 64-bit index arithmetic had tripled it
  double wx[4];
  uint32_t r_off[NI][4];   // byte offset of tap l of staged row lr + 4 i inside a ring stage
  {
    const Tap T = tx[min(x, nx - 1)];
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      wx[l] = T.w[l];
      const int ixl = (T.w[l] != 0.0) ? min(xb - 1, T.idx[l] - lo_x) : 0;
#pragma unroll
      for (int i = 0; i < NI; ++i) r_off[i][l] = (uint32_t)(((lr + 4 * i) * xb + ixl) * 8);
    }
  }
  double wy[2][4];
  uint32_t a_rd[2][4];     // byte offset of y tap m of output o inside A[0]
#pragma unroll
  for (int o = 0; o < 2; ++o) {
    const Tap T = ty[min(y0 + lr + 4 * o, ny - 1)];
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      wy[o][m] = T.w[m];
      const int iym = (T.w[m] != 0.0) ? min(ROWS - 1, T.idx[m] - lo_y) : 0;
      a_rd[o][m] = (uint32_t)((iym * TX + lx) * 8);
    }
  }
  const uint32_t a_base = smem_addr(&A[0][0][0]), ring_base = smem_addr(ring);
  const uint32_t a_wr = a_base + (uint32_t)((lr * TX + lx) * 8);      // + i * 4 rows, + buffer
  constexpr uint32_t kABuf = ROWS * TX * 8, kARow4 = 4 * TX * 8;
  double v[2][4];
#pragma unroll
  for (int o = 0; o < 2; ++o)
#pragma unroll
    for (int m = 0; m < 4; ++m) v[o][m] = 0.0;

  const int p_start = zw[z_begin].base, p_last = zw[z_end - 1].base + 3;
  const uint32_t stage_bytes = (uint32_t)stage_elems * 8u;
  auto issue = [&](int p, int sidx) {
    const uint32_t bar = smem_addr(&full[sidx]);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(stage_bytes) : "memory");
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(ring_base + (uint32_t)sidx * (uint32_t)stage_stride * 8u), "l"(&tmap), "r"(lo_x), "r"(lo_y), "r"(p), "r"(bar)
        : "memory");
  };
  if (t == 0)
    for (int i = 0; i < kMarchStages && p_start + i <= p_last; ++i) issue(p_start + i, i);

  auto lds = [](uint32_t addr) {
    double d;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(d) : "r"(addr));
    return d;
  };
  // running output pointers (advance one plane per emitted z)
  const int64_t out_plane = (int64_t)ny * nx;
  TOut* outp[2];
  bool outok[2];
#pragma unroll
  for (int o = 0; o < 2; ++o) {
    const int y = y0 + lr + 4 * o;
    outok[o] = x < nx && y < ny;
    outp[o] = dst + ((int64_t)z_begin * ny + min(y, ny - 1)) * nx + min(x, nx - 1);
  }

  int zc = z_begin;
  int next_emit = zw[zc].base + 3;
  int sidx = 0;
  uint32_t phase = 0, abuf = 0;
  for (int p = p_start; p <= p_last; ++p) {
    mbar_wait(smem_addr(&full[sidx]), phase);
    const uint32_t raw = ring_base + (uint32_t)sidx * (uint32_t)stage_stride * 8u;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const double xi = wx[0] * lds(raw + r_off[i][0]) + wx[1] * lds(raw + r_off[i][1]) +
                        wx[2] * lds(raw + r_off[i][2]) + wx[3] * lds(raw + r_off[i][3]);
      asm volatile("st.shared.f64 [%0], %1;" ::"r"(a_wr + abuf + i * kARow4), "d"(xi) : "memory");
    }
    __syncthreads();   // A[abuf] complete; every thread is done with ring stage sidx
    if (t == 0 && p + kMarchStages <= p_last) issue(p + kMarchStages, sidx);
#pragma unroll
    for (int o = 0; o < 2; ++o) {
      const uint32_t ab = a_base + abuf;
      const double vn = wy[o][0] * lds(ab + a_rd[o][0]) + wy[o][1] * lds(ab + a_rd[o][1]) +
                        wy[o][2] * lds(ab + a_rd[o][2]) + wy[o][3] * lds(ab + a_rd[o][3]);
      v[o][0] = v[o][1];
      v[o][1] = v[o][2];
      v[o][2] = v[o][3];
      v[o][3] = vn;
    }
    while (zc < z_end && next_emit <= p) {
      const ZWin Wz = zw[zc];
#pragma unroll
      for (int o = 0; o < 2; ++o) {
        const double acc = Wz.w[0] * v[o][0] + Wz.w[1] * v[o][1] + Wz.w[2] * v[o][2] + Wz.w[3] * v[o][3];
        if (outok[o]) store_out(outp[o], acc);
        outp[o] += out_plane;
      }
      ++zc;
      if (zc < z_end) next_emit = zw[zc].base + 3;
    }
    abuf ^= kABuf;
    if (++sidx == kMarchStages) {
      sidx = 0;
      phase ^= 1u;
    }
  }
}

// ------------------------------------------------- marching y/z interpolation, TMA-fed
// Input: the x-resampled float64 volume [sz_l][sy][nxp] of the x pass.  A CTA owns an
// [8 y x 64 x] output column and marches along z: each source plane's rows arrive as ONE
// cp.async.bulk.tensor box ([ROWS y] x [64 x]) in a kYzStages-deep mbarrier ring issued by one elected
// thread; y-interpolation reads the box in place into a 4-plane register window and every output plane
// is 4 FMAs from that window.  ~4 shared loads and ~10 FMAs per output voxel.
constexpr int kYzStages = 8;

template <int NI>
__global__ void __launch_bounds__(256, 4)
march_yz_tma_kernel(const __grid_constant__ CUtensorMap tmap, const ZWin* __restrict__ zw,
                    const Tap* __restrict__ ty, float* __restrict__ dst, int ny, int nx, int nz_local, int zchunk) {
  constexpr int TX = 64, TY = 8, ROWS = NI * 4;
  constexpr uint32_t kStageBytes = ROWS * TX * 8;
  extern __shared__ uint8_t march_smem[];
  __shared__ __align__(8) uint64_t full[kYzStages];
  __shared__ int s_lo;
  const uint32_t ring_base = (smem_addr(march_smem) + 127u) & ~127u;
  const int t = threadIdx.x;
  const int lx = t & (TX - 1), lr = t >> 6;
  const int x0 = blockIdx.x * TX, x = x0 + lx;
  const int y0 = blockIdx.y * TY;
  const int z_begin = blockIdx.z * zchunk, z_end = min(nz_local, z_begin + zchunk);
  if (z_begin >= z_end) return;
  if (t == 0) {
    s_lo = 0x7fffffff;
    for (int i = 0; i < kYzStages; ++i)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(&full[i])));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (t < TY * 4) {   // lowest source row any output row of this tile taps (zero-weight taps, D11, excluded)
    const int r = min(y0 + (t >> 2), ny - 1);
    if (ty[r].w[t & 3] != 0.0) atomicMin(&s_lo, ty[r].idx[t & 3]);
  }
  __syncthreads();
  const int lo_y = (s_lo == 0x7fffffff) ? 0 : s_lo;
  double wy[2][4];
  uint32_t a_rd[2][4];     // byte offset of y tap m of output o inside a ring stage
#pragma unroll
  for (int o = 0; o < 2; ++o) {
    const Tap T = ty[min(y0 + lr + 4 * o, ny - 1)];
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      wy[o][m] = T.w[m];
      const int iym = (T.w[m] != 0.0) ? min(ROWS - 1, T.idx[m] - lo_y) : 0;
      a_rd[o][m] = (uint32_t)((iym * TX + lx) * 8);
    }
  }
  double v[2][4];
#pragma unroll
  for (int o = 0; o < 2; ++o)
#pragma unroll
    for (int m = 0; m < 4; ++m) v[o][m] = 0.0;
  const int p_start = zw[z_begin].base, p_last = zw[z_end - 1].base + 3;
  auto issue = [&](int p, int sidx) {
    const uint32_t bar = smem_addr(&full[sidx]);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(kStageBytes) : "memory");
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(ring_base + (uint32_t)sidx * kStageBytes), "l"(&tmap), "r"(x0), "r"(lo_y), "r"(p), "r"(bar)
        : "memory");
  };
  if (t == 0)
    for (int i = 0; i < kYzStages && p_start + i <= p_last; ++i) issue(p_start + i, i);
  auto lds = [](uint32_t addr) {
    double d;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(d) : "r"(addr));
    return d;
  };
  const int64_t out_plane = (int64_t)ny * nx;
  float* outp[2];
  bool outok[2];
#pragma unroll
  for (int o = 0; o < 2; ++o) {
    const int y = y0 + lr + 4 * o;
    outok[o] = x < nx && y < ny;
    outp[o] = dst + ((int64_t)z_begin * ny + min(y, ny - 1)) * nx + min(x, nx - 1);
  }
  int zc = z_begin;
  int next_emit = zw[zc].base + 3;
  int sidx = 0;
  uint32_t phase = 0;
  // The 4-plane window is a ring of registers whose head is a COMPILE-TIME index (the plane loop is unrolled
  // by four), so a new plane overwrites the oldest slot instead of shifting the window: no register moves.
  auto step = [&](auto hc, int p) {
    constexpr int h = decltype(hc)::value;        // slot of plane p; the window, oldest first: h+1, h+2, h+3, h
    mbar_wait(smem_addr(&full[sidx]), phase);
    const uint32_t raw = ring_base + (uint32_t)sidx * kStageBytes;
#pragma unroll
    for (int o = 0; o < 2; ++o)
      v[o][h] = wy[o][0] * lds(raw + a_rd[o][0]) + wy[o][1] * lds(raw + a_rd[o][1]) +
                wy[o][2] * lds(raw + a_rd[o][2]) + wy[o][3] * lds(raw + a_rd[o][3]);
    __syncthreads();   // every thread has read ring stage sidx: it may be refilled
    if (t == 0 && p + kYzStages <= p_last) issue(p + kYzStages, sidx);
    while (zc < z_end && next_emit <= p) {
      const ZWin Wz = zw[zc];
#pragma unroll
      for (int o = 0; o < 2; ++o) {
        const double acc = Wz.w[0] * v[o][(h + 1) & 3] + Wz.w[1] * v[o][(h + 2) & 3] + Wz.w[2] * v[o][(h + 3) & 3] +
                           Wz.w[3] * v[o][h];
        if (outok[o]) st_stream(outp[o], (float)acc);
        outp[o] += out_plane;
      }
      ++zc;
      if (zc < z_end) next_emit = zw[zc].base + 3;
    }
    if (++sidx == kYzStages) {
      sidx = 0;
      phase ^= 1u;
    }
  };
  using I0 = std::integral_constant<int, 0>;
  using I1 = std::integral_constant<int, 1>;
  using I2 = std::integral_constant<int, 2>;
  using I3 = std::integral_constant<int, 3>;
  int p = p_start;
  for (; p + 3 <= p_last; p += 4) {
    step(I0(), p);
    step(I1(), p + 1);
    step(I2(), p + 2);
    step(I3(), p + 3);
  }
  if (p <= p_last) step(I0(), p);
  if (p + 1 <= p_last) step(I1(), p + 1);
  if (p + 2 <= p_last) step(I2(), p + 2);
}

template <typename TIn, typename TOut>
__global__ void __launch_bounds__(128)
gather1_kernel(const TIn* __restrict__ src, int sy, int sx, const Tap* __restrict__ tz,
               const Tap* __restrict__ ty, const Tap* __restrict__ tx, TOut* __restrict__ dst, int ny,
               int nx) {
  int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= nx) return;
  const int y = blockIdx.y, z = blockIdx.z;
  const Tap Tx = tx[x];
  const Tap Ty = ty[y];
  const Tap Tz = tz[z];
  const int64_t plane = (int64_t)sy * sx;
  double acc = 0.0;
#pragma unroll
  for (int l = 0; l < 2; ++l) {
    const TIn* pz = src + (int64_t)Tz.idx[l] * plane;
    double accy = 0.0;
#pragma unroll
    for (int m = 0; m < 2; ++m) {
      const TIn* row = pz + (int64_t)Ty.idx[m] * sx;
      double r = Tx.w[0] * (double)row[Tx.idx[0]] + Tx.w[1] * (double)row[Tx.idx[1]];
      accy += Ty.w[m] * r;
    }
    acc += Tz.w[l] * accy;
  }
  store_out(dst + ((int64_t)z * ny + y) * nx + x, acc);
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static int g_force_generic = 0;   // tests: run the general kernels on shapes the fast ones would take

// mica_last_resample_path: the MICA_RS_* kernel each pass of this thread's last resample launched (-1 = none)
enum { kPassZ = 0, kPassY = 1, kPassX = 2, kPassInterp = 3 };
static thread_local int g_resample_path[4] = {-1, -1, -1, -1};

// Shared-memory budgets the kernel choices are made against (a B200 block may take up to 227 KiB)
constexpr size_t kMaxTileBytes = 200 * 1024;  // general path: one prefilter tile of lines (prefilter_cols*, _rows*)
constexpr size_t kPipeSmemMax = 220 * 1024;   // fast path: the x pass's tile of staged rows (rows_pipe_smem)
constexpr size_t kSmemPerSm = 225 * 1024;     // fast path: an SM's share for x-pass CTAs, tile + 1 KiB each (rows_grid)

// Launches the kernel of one resample pass and records it for mica_last_resample_path.  A kernel that takes dynamic
// shared memory has its limit raised on every call: the attribute belongs to the current device.
template <typename... P, typename... A>
static int launch_pass(int pass, int path, const char* name, void (*kernel)(P...), dim3 grid, int threads,
                       size_t smem, cudaStream_t st, A... args) {
  if (smem) MICA_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<grid, threads, smem, st>>>(args...);
  g_resample_path[pass] = path;
  MICA_LAUNCH_CHECK(name);
  return MICA_OK;
}

// general path, z and y axes: the map's type (z) or float64 (y, in place) in, float64 out; lines that fit no tile are
// swept in global memory
template <typename TIn>
static int launch_cols_f64(const TIn* in, double* out, int n, int64_t line_stride, int n_cols,
                           int64_t outer_stride, int n_outer, cudaStream_t st, int pass) {
  const ColStrides S{line_stride, line_stride, outer_stride, outer_stride};
  const size_t per_col = (size_t)n * sizeof(double);
  if (!g_force_generic && n >= kMinSegLine && per_col * 32 <= kMaxTileBytes)
    return launch_pass(pass, MICA_RS_COLS_SEG16, "prefilter_cols", prefilter_cols_seg<TIn, 16>,
                       dim3((n_cols + 15) / 16, n_outer), 256, per_col * 16, st, in, out, n, n_cols, S, 0, n, 0, 15,
                       15, n);
  if (per_col * 32 <= kMaxTileBytes)
    return launch_pass(pass, MICA_RS_COLS32, "prefilter_cols", prefilter_cols<TIn, 32>,
                       dim3((n_cols + 31) / 32, n_outer), 256, per_col * 32, st, in, out, n, n_cols, S);
  if (per_col * 8 <= kMaxTileBytes)
    return launch_pass(pass, MICA_RS_COLS8, "prefilter_cols", prefilter_cols<TIn, 8>,
                       dim3((n_cols + 7) / 8, n_outer), 256, per_col * 8, st, in, out, n, n_cols, S);
  return launch_pass(pass, MICA_RS_COLS_GLOBAL, "prefilter_cols", prefilter_cols_global<TIn>,
                     dim3((n_cols + 127) / 128, n_outer), 128, 0, st, in, out, n, line_stride, n_cols, outer_stride);
}

// Lines prefilter_cols_seg<., 16> takes on one GPU (launch_cols_f64): kMinSegLine .. kMaxSeg16Line samples.  Only
// these can be cut into blocks with the whole line's bits: the kernels of shorter and longer lines (iir_line) run
// one causal recursion from sample 0 to the end.
constexpr int kMaxSeg16Line = (int)(kMaxTileBytes / (32 * sizeof(double)));   // 800

// The segments of prefilter_cols_seg<., 16> (16 per line of ng samples, numbered on the whole line) that a block must
// run so that global samples [need_lo, need_hi] get the whole line's coefficients, and the raw samples
// [raw_lo, raw_hi) they read.  The segments that hold the needed samples run both sweeps.  The anticausal warm-up of
// the last of them reads the CAUSAL values of the kHorizon samples above it, or of everything up to the line's end
// when the exact end initialisation is within reach: the segments that hold those run the causal sweep, up to the
// last such sample (causal_end).  The last
// segment's end initialisation reads sample ng - 2, which may lie in the segment below.  Every causal sweep reads
// the kHorizon raw samples below its segment, mirrored at sample 0.
struct Seg16Plan {
  int seg_lo, seg_causal_hi, seg_out_hi, causal_end, raw_lo, raw_hi;
};

static Seg16Plan seg16_plan(int ng, int need_lo, int need_hi) {
  const int len = (ng + 15) / 16;
  Seg16Plan p;
  p.seg_lo = need_lo / len;
  p.seg_out_hi = need_hi / len;
  const int k1 = min(ng, (p.seg_out_hi + 1) * len);
  int last = k1 - 1;                                   // last sample whose causal value is read
  if (k1 < ng) last = k1 + kHorizon >= ng ? ng - 1 : k1 + kHorizon - 1;
  if (k1 >= ng && ng >= 2 && (ng - 2) / len < p.seg_lo) p.seg_lo = (ng - 2) / len;
  p.seg_causal_hi = last / len;
  p.causal_end = last + 1;
  const int k0 = p.seg_lo * len;
  p.raw_lo = max(0, k0 - kHorizon);
  p.raw_hi = min(ng, max(p.causal_end, k0 < kHorizon ? kHorizon - k0 + 1 : 0));
  return p;
}

// z pass of the general path on a block [g0, g0 + n) of lines of ng samples (an integer map in a z-slab): always
// prefilter_cols_seg<., 16>, the kernel the whole line takes, with its segments numbered on the whole line
template <typename TIn>
static int launch_cols_seg_block(const TIn* in, double* out, int n, int64_t plane, int g0, int ng, const Seg16Plan& p,
                                 cudaStream_t st) {
  const ColStrides S{plane, plane, 0, 0};
  return launch_pass(kPassZ, MICA_RS_COLS_SEG16, "prefilter_cols", prefilter_cols_seg<TIn, 16>,
                     dim3((unsigned)((plane + 15) / 16), 1), 256, (size_t)n * sizeof(double) * 16, st, in, out, n,
                     (int)plane, S, g0, ng, p.seg_lo, p.seg_causal_hi, p.seg_out_hi, p.causal_end);
}

// a row that fits no 4-row shared-memory tile is swept in global memory, one row per CTA along grid y
static bool row_fits_smem(int n) { return (size_t)(n | 1) * sizeof(double) * 4 <= kMaxTileBytes; }

// general path, x axis: contiguous rows, in place
static int launch_rows(double* data, int n, int64_t n_rows, cudaStream_t st) {
  const size_t per_row = (size_t)(n | 1) * sizeof(double);
  if (!g_force_generic && n >= kMinSegLine && per_row * 32 <= kMaxTileBytes)
    return launch_pass(kPassX, MICA_RS_ROWS_SEG16, "prefilter_rows", prefilter_rows_seg<16>,
                       (unsigned)ceil_div64(n_rows, 16), 256, per_row * 16, st, data, n, n_rows);
  if (per_row * 32 <= kMaxTileBytes)
    return launch_pass(kPassX, MICA_RS_ROWS32, "prefilter_rows", prefilter_rows<32>, (unsigned)ceil_div64(n_rows, 32),
                       256, per_row * 32, st, data, n, n_rows);
  if (row_fits_smem(n))
    return launch_pass(kPassX, MICA_RS_ROWS4, "prefilter_rows", prefilter_rows<4>, (unsigned)ceil_div64(n_rows, 4),
                       256, per_row * 4, st, data, n, n_rows);
  // a row is a column of a [n_rows x n] matrix with unit line stride
  return launch_pass(kPassX, MICA_RS_COLS_GLOBAL, "prefilter_rows", prefilter_cols_global<double>,
                     dim3(1, (unsigned)n_rows), 1, 0, st, data, data, n, 1, 1, n);
}

}  // namespace mica

using namespace mica;

extern "C" int mica_zoom_output_shape(const int in_zyx[3], const float zoom_zyx[3], int out_zyx[3]) {
  MICA_REQUIRE(in_zyx && zoom_zyx && out_zyx, "null argument");
  for (int a = 0; a < 3; ++a) {
    volatile float prod = (float)in_zyx[a] * zoom_zyx[a];  // float32 product (NumPy 2 weak-scalar promotion)
    out_zyx[a] = (int)nearbyint((double)prod);              // round-half-even, as python round()
  }
  return MICA_OK;
}

extern "C" int mica_resample_force_generic(int on) {
  const int was = g_force_generic;
  g_force_generic = on ? 1 : 0;
  return was;
}

// The fast order-3 path: z and y prefilters write float32 coefficients (padded row pitch), the x pass
// prefilters and interpolates rows into a float64 volume [sz_l][sy][nxp], the march interpolates y and z.
static int64_t pitch_f32(int sx) { return ((int64_t)sx + 3) / 4 * 4; }
static int64_t pitch_f64(int nx) { return ((int64_t)nx + 1) / 2 * 2; }
static size_t rows_pipe_smem(int n, int L) {
  return (((size_t)L * (n | 1) * 8 + 15) & ~(size_t)15) + (size_t)kPipeStages * L * pitch_f32(n) * 4;
}

// source rows that the y taps of an 8-row output tile span: a march stages 12 or 16 rows per source plane
static int y_span(int sy, int ny) {
  const double zoom_y = ny > 1 ? (double)(sy - 1) / (double)(ny - 1) : 1.0;
  return (int)floor(7.0 * zoom_y) + 5;
}

// Source planes [*c_lo, *c_hi] (global) that hold a z tap of output planes [dst_z0, dst_z0 + dst_nz_local), with
// one plane of margin on either side, clipped to the block [src_z0, src_z0 + src_nz_local).
static void needed_planes(int sz, int nz, int dst_z0, int dst_nz_local, int src_z0, int src_nz_local, int* c_lo,
                          int* c_hi) {
  const double zoom = nz > 1 ? (double)(sz - 1) / (double)(nz - 1) : 1.0;
  int lo = (int)floor((double)dst_z0 * zoom) - 2, hi = (int)floor((double)(dst_z0 + dst_nz_local - 1) * zoom) + 3;
  lo = lo < src_z0 ? src_z0 : lo;
  hi = hi > src_z0 + src_nz_local - 1 ? src_z0 + src_nz_local - 1 : hi;
  if (dst_z0 + dst_nz_local >= nz) hi = src_z0 + src_nz_local - 1;   // the parked window of an all-zero last plane (D11)
  if (hi < lo) lo = src_z0, hi = src_z0 + src_nz_local - 1;
  *c_lo = lo;
  *c_hi = hi;
}

// segment length of cols_reg_kernel on a line of ng samples: the line cut into the fewest segments of <= kColLen
static int cols_reg_seg_len(int ng) {
  const int n_seg = (ng + kColLen - 1) / kColLen;
  return (ng + n_seg - 1) / n_seg;
}

// Block of source planes [*src_lo, *src_hi) a rank must hold so that the z prefilter of output planes
// [dst_z0, dst_z0 + dst_nz_local) sees the windows the whole map would give it (bit-identical coefficients).
extern "C" int mica_resample_slab_source_planes(int sz, int nz, int dst_z0, int dst_nz_local, int* src_lo, int* src_hi) {
  MICA_REQUIRE(src_lo && src_hi, "null pointer");
  MICA_REQUIRE(sz > 0 && nz > 0 && dst_z0 >= 0 && dst_nz_local > 0 && dst_z0 + dst_nz_local <= nz, "bad slab");
  int c_lo, c_hi;
  needed_planes(sz, nz, dst_z0, dst_nz_local, 0, sz, &c_lo, &c_hi);
  const int len = cols_reg_seg_len(sz);
  const int lo = c_lo / len * len - kColH, hi = c_hi / len * len + kColLen + kColH;
  *src_lo = lo < 0 ? 0 : lo;
  *src_hi = hi > sz ? sz : hi;
  return MICA_OK;
}

// The general path's counterpart (integer maps): the block that holds every raw sample the segments of
// prefilter_cols_seg<., 16> that output planes [dst_z0, dst_z0 + dst_nz_local) need read (seg16_plan).
extern "C" int mica_resample_slab_source_planes_general(int sz, int nz, int dst_z0, int dst_nz_local, int* src_lo,
                                                        int* src_hi) {
  MICA_REQUIRE(src_lo && src_hi, "null pointer");
  MICA_REQUIRE(sz >= kMinSegLine && sz <= kMaxSeg16Line,
               "a z line of %d samples is prefiltered in one piece on the general path: only lines of %d..%d "
               "samples can be cut into blocks with the whole line's bits", sz, kMinSegLine, kMaxSeg16Line);
  MICA_REQUIRE(nz > 0 && dst_z0 >= 0 && dst_nz_local > 0 && dst_z0 + dst_nz_local <= nz, "bad slab");
  int c_lo, c_hi;
  needed_planes(sz, nz, dst_z0, dst_nz_local, 0, sz, &c_lo, &c_hi);
  const Seg16Plan p = seg16_plan(sz, c_lo, c_hi);
  *src_lo = p.raw_lo;
  *src_hi = p.raw_hi;
  return MICA_OK;
}

// sz = planes of the whole map, src_nz_local = planes of the block in memory.  The choice follows the WHOLE line,
// so that every block of a z-slab partition runs the same kernels as the whole map (the z pass numbers its segments
// on the whole line: the same bits): no bound but the register pass's 8-plane minimum looks at the block.
static bool fast_path_ok(int sz, int src_nz_local, int sy, int sx, int ny) {
  if (g_force_generic || getenv("MICA_NO_TMA")) return false;
  // No kernel needs this bound (the y pass, cols_reg_kernel, takes lines of any length): it only keeps maps with y
  // lines of more than 1760 samples on the general path they have always taken.
  if (sy > 1760) return false;
  if (sz < kMinSegLine || sy < kMinSegLine || sx < kMinSegLine) return false;             // segment-parallel sweeps
  if (src_nz_local < 8) return false;
  if (rows_pipe_smem(sx, 8) > kPipeSmemMax) return false;            // 8 rows in the x pass's tile: sx <= 1759
  if (y_span(sy, ny) > 16) return false;
  return tensor_map_encode_fn() != nullptr;
}

// register-only column pass: 32 columns x 8 segments per CTA, segments of <= kColLen samples.  The line in memory
// is samples [g0, g0 + n) of a line of ng; the segments of the GLOBAL line that hold samples [need_lo, need_hi]
// (global numbers) are computed.
static int launch_cols_reg(const float* in, float* out, int n, int n_cols, int n_outer, ColStrides S, cudaStream_t st,
                           int pass, int g0, int ng, int need_lo, int need_hi) {
  const int len = cols_reg_seg_len(ng);
  const int seg0 = need_lo / len, n_seg = need_hi / len - seg0 + 1;
  return launch_pass(pass, MICA_RS_COLS_REG, "cols_reg_kernel", cols_reg_kernel,
                     dim3((n_cols + 31) / 32, (n_seg + 7) / 8, n_outer), 256, 0, st, in, out, n, n_cols, S, len,
                     n_seg, g0, ng, seg0);
}

// persistent grid of the x pass: as many CTAs as fit an SM's shared memory (at most max_per_sm), no more than there
// are tiles of L rows; the tiles are dealt round-robin
static unsigned rows_grid(size_t smem, int max_per_sm, int64_t n_rows, int L) {
  int per_sm = (int)(kSmemPerSm / (smem + 1024));
  per_sm = per_sm < 1 ? 1 : (per_sm > max_per_sm ? max_per_sm : per_sm);
  const long long tiles = (n_rows + L - 1) / L;
  const long long grid = (long long)kNumSMs * per_sm;
  return (unsigned)(grid < tiles ? grid : tiles);
}

// x pass: the register form for rows of <= 16 or 32 segments of kColLen (832 samples), then the shared-memory sweep
// of 16 rows per tile while they fit kPipeSmemMax (879 samples), of 8 rows beyond
static int launch_rows_pipe(const float* in, int64_t in_pitch, double* out, int64_t out_pitch, int n, int nx,
                            int64_t n_rows, const Tap* tx, cudaStream_t st) {
  if (n <= 32 * kColLen) {
    const int segs = n <= 16 * kColLen ? 16 : 32;
    const size_t smem = rows_pipe_smem(n, 16);
    int len = (n + segs - 1) / segs;
    if (len % 2 == 0 && len < kColLen) ++len;      // odd segment length: the lanes of a row hit distinct banks
    return launch_pass(kPassX, segs == 16 ? MICA_RS_ROWS_REG16 : MICA_RS_ROWS_REG32, "rows_reg_interp_kernel",
                       segs == 16 ? rows_reg_interp_kernel<16> : rows_reg_interp_kernel<32>,
                       rows_grid(smem, 512 / (16 * segs), n_rows, 16), 16 * segs, smem, st, in, in_pitch, out,
                       out_pitch, n, nx, n_rows, tx, len);
  }
  const int L = rows_pipe_smem(n, 16) <= kPipeSmemMax ? 16 : 8;
  const size_t smem = rows_pipe_smem(n, L);
  return launch_pass(kPassX, L == 16 ? MICA_RS_ROWS_PIPE_16_512 : MICA_RS_ROWS_PIPE_8_512, "rows_pipe_interp_kernel",
                     L == 16 ? rows_pipe_interp_kernel<16, 512> : rows_pipe_interp_kernel<8, 512>,
                     rows_grid(smem, 2048 / 512, n_rows, L), 512, smem, st, in, in_pitch, out, out_pitch, n, nx,
                     n_rows, tx);
}

extern "C" size_t mica_resample_workspace_bytes(int src_nz_local, int sy, int sx, int nz, int ny, int nx, int order) {
  size_t taps = align_up((size_t)(nz + ny + nx) * sizeof(Tap), 256) + align_up((size_t)nz * sizeof(ZWin), 256);
  size_t coeff = 0;
  if (order == 3) {
    coeff = align_up((size_t)src_nz_local * sy * sx * sizeof(double), 256);                 // general path
    const size_t fast = align_up((size_t)2 * src_nz_local * sy * pitch_f32(sx) * sizeof(float), 256) +
                        align_up((size_t)src_nz_local * sy * pitch_f64(nx) * sizeof(double), 256);
    if (fast > coeff) coeff = fast;
  }
  return taps + coeff + 512;
}

// grid of a march: a CTA owns an [8 y x 64 x] output column and marches zchunk planes of it; the planes are cut into
// enough chunks of >= 16 for 8 CTAs per SM
static int march_grid(int ny, int nx, int nz_local, dim3* grid, int* zchunk) {
  const int xt = (nx + 63) / 64, yt = (ny + 7) / 8;
  int nzc = (8 * kNumSMs + xt * yt - 1) / (xt * yt);
  nzc = nzc < 1 ? 1 : nzc;
  if (nzc > (nz_local + 15) / 16) nzc = (nz_local + 15) / 16;
  *zchunk = (nz_local + nzc - 1) / nzc;
  *grid = dim3(xt, yt, (nz_local + *zchunk - 1) / *zchunk);
  MICA_REQUIRE(yt <= 65535 && grid->z <= 65535, "output too large for the launch grid");
  return MICA_OK;
}

// TMA descriptor of the float64 volume [nz][ny][pitch] at base, read in boxes of [box_y][box_x] of one plane
static CUresult encode_f64_3d(CUtensorMap* map, double* base, int64_t pitch, int ny, int nz, int box_x, int box_y) {
  const TensorMapEncodeFn enc = tensor_map_encode_fn();
  if (!enc) return CUDA_ERROR_NOT_SUPPORTED;
  const cuuint64_t gdim[3] = {(cuuint64_t)pitch, (cuuint64_t)ny, (cuuint64_t)nz};
  const cuuint64_t gstr[2] = {(cuuint64_t)pitch * 8, (cuuint64_t)ny * pitch * 8};
  const cuuint32_t box[3] = {(cuuint32_t)box_x, (cuuint32_t)box_y, 1}, estr[3] = {1, 1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

// the fast order-3 path, on a float32 map that fast_path_ok accepts
template <typename Taps>
static int resample_fast(const float* src, int sz, int sy, int sx, int src_z0, int src_nz_local, float* dst, int nz,
                         int ny, int nx, int dst_z0, int dst_nz_local, const Tap* tz, const Tap* ty, const Tap* tx,
                         ZWin* zw, double* coeff, cudaStream_t st, const Taps& taps) {
  const int64_t plane = (int64_t)sy * sx;
  MICA_REQUIRE(plane <= 0x7fffffffLL && src_nz_local <= 65535 && sy <= 65535, "source plane too large");
  const int64_t p32 = pitch_f32(sx), p64 = pitch_f64(nx);
  float* c32 = (float*)coeff;
  float* c32b = c32 + (size_t)src_nz_local * sy * p32;      // second float32 volume (the register pass is not in place)
  double* xr = (double*)((char*)coeff + align_up((size_t)2 * src_nz_local * sy * p32 * sizeof(float), 256));
  // source planes whose coefficients the z taps of this output slab can touch (global numbers, one plane of
  // margin): the whole line for a whole map; for a z-slab the planes beyond them are prefilter horizon only
  // and take no part in the y and x passes
  int c_lo, c_hi;
  needed_planes(sz, nz, dst_z0, dst_nz_local, src_z0, src_nz_local, &c_lo, &c_hi);
  const int l0 = c_lo - src_z0, cnt = c_hi - c_lo + 1;
  MICA_REQUIRE(sy <= 65535 && cnt <= 65535, "too many outer lines for the launch grid");   // grid z of cols_reg
  dim3 mgrid;
  int zchunk;
  if (int rc = march_grid(ny, nx, dst_nz_local, &mgrid, &zchunk)) return rc;
  const int rows = y_span(sy, ny) <= 12 ? 12 : 16;
  CUtensorMap tmap;
  const CUresult cr = encode_f64_3d(&tmap, xr, p64, sy, src_nz_local, 64, rows);
  if (cr != CUDA_SUCCESS) return set_error(MICA_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)cr);

  if (int rc = taps()) return rc;
  const ColStrides Sz{plane, sy * p32, sx, p32}, Sy{p32, p32, sy * p32, sy * p32};
  const size_t l0_f32 = (size_t)l0 * sy * p32;
  // axis 0 (z): float32 in (row pitch sx) -> c32b (row pitch p32); axis 1 (y): c32b -> c32
  if (int rc = launch_cols_reg(src, c32b, src_nz_local, sx, sy, Sz, st, kPassZ, src_z0, sz, c_lo, c_hi)) return rc;
  if (int rc = launch_cols_reg(c32b + l0_f32, c32 + l0_f32, sy, sx, cnt, Sy, st, kPassY, 0, sy, 0, sy - 1)) return rc;
  // axis 2 (x): prefilter + interpolate the rows -> x-resampled float64 volume
  if (int rc = launch_rows_pipe(c32 + l0_f32, p32, xr + (size_t)l0 * sy * p64, p64, sx, nx, (int64_t)cnt * sy, tx, st))
    return rc;
  zwin_kernel<<<(dst_nz_local + 127) / 128, 128, 0, st>>>(tz, zw, dst_nz_local, src_nz_local);
  MICA_LAUNCH_CHECK("zwin_kernel");
  return launch_pass(kPassInterp, rows == 12 ? MICA_RS_MARCH_YZ_TMA3 : MICA_RS_MARCH_YZ_TMA4, "march_yz_tma_kernel",
                     rows == 12 ? march_yz_tma_kernel<3> : march_yz_tma_kernel<4>, mgrid, 256,
                     (size_t)kYzStages * rows * 64 * 8 + 128, st, tmap, zw, ty, dst, ny, nx, dst_nz_local, zchunk);
}

// general order-3 path: float64 coefficients prefiltered in place along z, y and x; then the marching gather when the
// y span of an 8-row output tile fits the staged rows and every axis has a full 4-sample window, else one thread per
// output voxel.  The y and x passes run on the planes the z taps read (needed_planes) only.  An integer map given a
// block of a longer z line runs its z pass on the whole line's segment grid (seg16_plan): the block's planes come out
// with the whole map's bits.  A float32 block is prefiltered as a line of its own, as it always has been.
template <typename T, typename Taps>
static int resample_general(const T* src, int sz, int sy, int sx, int src_z0, int src_nz_local, T* dst, int nz, int ny,
                            int nx, int dst_z0, int dst_nz_local, const Tap* tz, const Tap* ty, const Tap* tx, ZWin* zw,
                            double* coeff, cudaStream_t st, const Taps& taps) {
  const int64_t plane = (int64_t)sy * sx;
  MICA_REQUIRE(plane <= 0x7fffffffLL && src_nz_local <= 65535, "source plane too large");
  int c_lo, c_hi;
  needed_planes(sz, nz, dst_z0, dst_nz_local, src_z0, src_nz_local, &c_lo, &c_hi);
  const int l0 = c_lo - src_z0, cnt = c_hi - c_lo + 1;
  const bool block = !std::is_same<T, float>::value && src_nz_local < sz;
  Seg16Plan zp{};
  if (block) {
    MICA_REQUIRE(sz >= kMinSegLine && sz <= kMaxSeg16Line,
                 "an integer map's z line of %d samples is prefiltered in one piece: a block of it cannot give the "
                 "whole map's bits (only lines of %d..%d samples can be cut)", sz, kMinSegLine, kMaxSeg16Line);
    zp = seg16_plan(sz, c_lo, c_hi);
    MICA_REQUIRE(src_z0 <= zp.raw_lo && src_z0 + src_nz_local >= zp.raw_hi,
                 "source planes [%d, %d) do not hold the prefilter windows [%d, %d) of output planes [%d, %d) "
                 "(mica_resample_slab_source_planes_general)", src_z0, src_z0 + src_nz_local, zp.raw_lo, zp.raw_hi,
                 dst_z0, dst_z0 + dst_nz_local);
  }
  const int span_y = y_span(sy, ny);
  const bool march = !g_force_generic && src_nz_local >= 4 && sy >= 4 && sx >= 4 && span_y <= 16;
  dim3 mgrid;
  int zchunk = 0;
  if (march) {
    if (int rc = march_grid(ny, nx, dst_nz_local, &mgrid, &zchunk)) return rc;
  }
  // TMA-fed ring when the coefficient rows are 16-byte multiples and the x span of a 64-wide output tile fits one
  // box; else the register-prefetch variant
  const double zoom_x = nx > 1 ? (double)(sx - 1) / (double)(nx - 1) : 1.0;
  const int xb = (((int)floor(63.0 * zoom_x) + 5) + 1 + 1) & ~1;   // span + 1 (even box start), even width
  const int rows = span_y <= 12 ? 12 : 16;
  CUtensorMap tmap;
  const bool tma = march && sx % 2 == 0 && xb <= 256 && !getenv("MICA_NO_TMA") &&
                   encode_f64_3d(&tmap, coeff, sx, sy, src_nz_local, xb, rows) == CUDA_SUCCESS;

  if (int rc = taps()) return rc;
  // axis 0 (z): lines of length src_nz_local, stride plane; reads the map's type, writes float64
  if (block) {
    if (int rc = launch_cols_seg_block<T>(src, coeff, src_nz_local, plane, src_z0, sz, zp, st)) return rc;
  } else if (int rc = launch_cols_f64<T>(src, coeff, src_nz_local, plane, (int)plane, 0, 1, st, kPassZ)) {
    return rc;
  }
  // axis 1 (y): per needed z plane, lines of length sy, stride sx
  double* c0 = coeff + (size_t)l0 * plane;
  if (int rc = launch_cols_f64<double>(c0, c0, sy, sx, sx, plane, cnt, st, kPassY)) return rc;
  // axis 2 (x): contiguous rows
  if (int rc = launch_rows(c0, sx, (int64_t)cnt * sy, st)) return rc;
  if (!march)
    return launch_pass(kPassInterp, MICA_RS_GATHER3, "gather3_kernel", gather3_kernel<T>,
                       dim3((nx + 127) / 128, ny, dst_nz_local), 128, 0, st, coeff, sy, sx, tz, ty, tx, dst, ny, nx);
  zwin_kernel<<<(dst_nz_local + 127) / 128, 128, 0, st>>>(tz, zw, dst_nz_local, src_nz_local);
  MICA_LAUNCH_CHECK("zwin_kernel");
  if (tma)
    return launch_pass(kPassInterp, rows == 12 ? MICA_RS_MARCH3_TMA3 : MICA_RS_MARCH3_TMA4, "march3_tma_kernel",
                       rows == 12 ? march3_tma_kernel<3, T> : march3_tma_kernel<4, T>, mgrid, 256,
                       (size_t)kMarchStages * (((size_t)rows * xb + 15) / 16 * 16) * 8 + 128, st, tmap, xb, zw, ty, tx,
                       dst, ny, nx, dst_nz_local, zchunk);
  return launch_pass(kPassInterp, rows == 12 ? MICA_RS_MARCH3_3 : MICA_RS_MARCH3_4, "march3_kernel",
                     rows == 12 ? march3_kernel<3, T> : march3_kernel<4, T>, mgrid, 256, 0, st, coeff, sy, sx, zw, ty,
                     tx, dst, ny, nx, dst_nz_local, zchunk);
}

// T = the map's sample type, in and out.  Integer maps never take the fast path (see the file header).
template <typename T>
static int resample_impl(const T* src, int sz, int sy, int sx, int src_z0, int src_nz_local, T* dst, int nz, int ny,
                         int nx, int dst_z0, int dst_nz_local, void* workspace, size_t workspace_bytes, int order,
                         mica_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  MICA_REQUIRE(src && dst && workspace, "null pointer");
  MICA_REQUIRE(order == 3 || order == 1, "order must be 3 or 1 (got %d)", order);
  MICA_REQUIRE(sz > 0 && sy > 0 && sx > 0 && nz > 0 && ny > 0 && nx > 0, "empty shape");
  MICA_REQUIRE(src_z0 >= 0 && src_nz_local > 0 && src_z0 + src_nz_local <= sz, "bad source slab");
  MICA_REQUIRE(dst_z0 >= 0 && dst_nz_local >= 0 && dst_z0 + dst_nz_local <= nz, "bad output slab");
  MICA_REQUIRE(ny <= 65535 && dst_nz_local <= 65535, "output too large for the launch grid");
  MICA_REQUIRE(order != 3 || row_fits_smem(sx) || (int64_t)src_nz_local * sy <= 65535,
               "rows of %d samples are prefiltered one per CTA: at most 65535 of them fit the launch grid (got %lld)",
               sx, (long long)src_nz_local * sy);
  if (workspace_bytes < mica_resample_workspace_bytes(src_nz_local, sy, sx, nz, ny, nx, order))
    return set_error(MICA_ERR_WORKSPACE, "resample workspace too small");
  if (dst_nz_local == 0) return MICA_OK;

  char* ws = (char*)(((uintptr_t)workspace + 255) / 256 * 256);
  Tap* tz = (Tap*)ws;
  Tap* ty = tz + nz;
  Tap* tx = ty + ny;
  ZWin* zw = (ZWin*)(ws + align_up((size_t)(nz + ny + nx) * sizeof(Tap), 256));
  double* coeff = (double*)((char*)zw + align_up((size_t)nz * sizeof(ZWin), 256));
  // each path calls taps() once its own checks have passed and its tensor map is encoded: a refused call launches
  // nothing
  auto taps = [&]() -> int {
    taps_kernel<<<(dst_nz_local + 127) / 128, 128, 0, st>>>(tz, dst_nz_local, dst_z0, sz, nz, order, src_z0,
                                                             src_nz_local);
    MICA_LAUNCH_CHECK("taps_kernel(z)");
    taps_kernel<<<(ny + 127) / 128, 128, 0, st>>>(ty, ny, 0, sy, ny, order, 0, sy);
    MICA_LAUNCH_CHECK("taps_kernel(y)");
    taps_kernel<<<(nx + 127) / 128, 128, 0, st>>>(tx, nx, 0, sx, nx, order, 0, sx);
    MICA_LAUNCH_CHECK("taps_kernel(x)");
    return MICA_OK;
  };

  if (order == 1) {
    if (int rc = taps()) return rc;
    return launch_pass(kPassInterp, MICA_RS_GATHER1, "gather1_kernel", gather1_kernel<T, T>,
                       dim3((nx + 127) / 128, ny, dst_nz_local), 128, 0, st, src, sy, sx, tz, ty, tx, dst, ny, nx);
  }
  if constexpr (std::is_same<T, float>::value) {
    if (fast_path_ok(sz, src_nz_local, sy, sx, ny))
      return resample_fast(src, sz, sy, sx, src_z0, src_nz_local, dst, nz, ny, nx, dst_z0, dst_nz_local, tz, ty, tx,
                           zw, coeff, st, taps);
  }
  return resample_general(src, sz, sy, sx, src_z0, src_nz_local, dst, nz, ny, nx, dst_z0, dst_nz_local, tz, ty, tx, zw,
                          coeff, st, taps);
}

extern "C" int mica_resample(const void* src, int src_dtype, int sz, int sy, int sx, int src_z0, int src_nz_local,
                             void* dst, int dst_dtype, int nz, int ny, int nx, int dst_z0, int dst_nz_local,
                             void* workspace, size_t workspace_bytes, int order, mica_stream_t stream) {
  for (int& k : g_resample_path) k = -1;
  MICA_REQUIRE(src_dtype == dst_dtype, "resample writes the source's own type (src dtype %d, dst dtype %d)", src_dtype,
               dst_dtype);
#define MICA_RESAMPLE_AS(T)                                                                                          \
  resample_impl<T>((const T*)src, sz, sy, sx, src_z0, src_nz_local, (T*)dst, nz, ny, nx, dst_z0, dst_nz_local,     \
                   workspace, workspace_bytes, order, stream)
  switch (src_dtype) {
    case MICA_DTYPE_F32: return MICA_RESAMPLE_AS(float);
    case MICA_DTYPE_I8: return MICA_RESAMPLE_AS(int8_t);
    case MICA_DTYPE_I16: return MICA_RESAMPLE_AS(int16_t);
    case MICA_DTYPE_U16: return MICA_RESAMPLE_AS(uint16_t);
    default: return set_error(MICA_ERR_INVALID, "unknown dtype code %d", src_dtype);
  }
#undef MICA_RESAMPLE_AS
}

extern "C" int mica_bspline_resample_f32(const float* src, int sz, int sy, int sx, int src_z0, int src_nz_local,
                                         float* dst, int nz, int ny, int nx, int dst_z0, int dst_nz_local,
                                         void* workspace, size_t workspace_bytes, int order, mica_stream_t stream) {
  return mica_resample(src, MICA_DTYPE_F32, sz, sy, sx, src_z0, src_nz_local, dst, MICA_DTYPE_F32, nz, ny, nx, dst_z0,
                       dst_nz_local, workspace, workspace_bytes, order, stream);
}

extern "C" int mica_last_resample_path(int pass) { return pass >= 0 && pass < 4 ? g_resample_path[pass] : -1; }
