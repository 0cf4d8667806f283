// R2/R3 for integer maps (DESIGN.md D12): exact median / 99.9-percentile and the float64 normalisation.
//
// The reference normalises the integer array scipy.ndimage.zoom returns for an int8 / int16 / uint16 map:
//   med = np.median(x)                      float64: the middle element or the mean of the two middle ones
//   m = (x > med) * (x - med)               float64, multiples of 0.5
//   p = np.percentile(m[m > 0], 99.9)       float64 interpolation, vi = (npos - 1) * (99.9 / 100)
//   y = ((m < p) * m + (m >= p) * p) / p    float64, cast to float32
// Values have at most 16 bits, so ONE exact histogram of 2^8 or 2^16 bins gives every order statistic; this is
// kept apart from the float32 radix select (select.cu), which is built around sampled 32-bit float keys.
//
// Kernels:
//   int_hist_kernel      one pass over the map.  A CTA privatises the whole key range in shared memory as 16-bit
//                        counters, two to a 32-bit word (2^16 bins = 128 KB), and histograms slices of at most
//                        kSlice < 2^16 voxels, so no counter can carry into its neighbour; after each slice the
//                        non-zero counters are added to the uint64 histogram in global memory.
//   int_pick_kernel      one CTA: prefix sums of the histogram, the four order statistics, the float64 median and
//                        percentile and the status word.
//   int_normalize_kernel the float64 expression per voxel, float32 out.
// Several GPUs (a z-slab partition) sum their histograms between hist and pick: over NCCL (mica_int_stats_hist_ptr)
// or over NVLink peer memory with int_peer_publish_kernel + int_peer_sum_kernel (below).
#include "common.cuh"

namespace mica {

constexpr int kIntMaxBins = 1 << 16;
constexpr int kSlice = 65520;          // voxels per flush: < 2^16, and 16-byte chunks of int8 and int16 alike
constexpr int kIntHistThreads = 1024;
constexpr int kIntPickThreads = 1024;

struct IntStatsState {
  unsigned long long hist[kIntMaxBins];
  long long n_total;
  long long n_le_med;
  // the result record (MICA_INT_STATS_RESULT_BYTES), copied out in one piece
  double median;
  double p;
  long long n_pos;
  int status;
  int zero;
};
static_assert(offsetof(IntStatsState, zero) + sizeof(int) - offsetof(IntStatsState, median) ==
                  MICA_INT_STATS_RESULT_BYTES, "result record size");

template <typename T>
struct IntKey;
template <>
struct IntKey<int8_t> {
  static constexpr int kBits = 8, kOffset = -128;
};
template <>
struct IntKey<int16_t> {
  static constexpr int kBits = 16, kOffset = -32768;
};
template <>
struct IntKey<uint16_t> {
  static constexpr int kBits = 16, kOffset = 0;
};
// key = value - smallest value of the type: order-preserving, 0 .. 2^bits - 1
template <typename T>
__device__ __forceinline__ unsigned int_key(T v) {
  return (unsigned)((int)v - IntKey<T>::kOffset);
}

__global__ void int_stats_init_kernel(IntStatsState* s, int bins, long long n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < bins) s->hist[i] = 0ull;
  if (i == 0) {
    s->n_total = n;
    s->n_le_med = 0;
    s->median = 0.0;
    s->p = 0.0;
    s->n_pos = 0;
    s->status = MICA_NORM_PENDING;
    s->zero = 0;
  }
}

// grid-stride over slices of kSlice voxels; dynamic smem = 2^bits * 2 bytes
template <typename T>
__global__ void __launch_bounds__(kIntHistThreads)
int_hist_kernel(const T* __restrict__ x, long long n, IntStatsState* __restrict__ s) {
  constexpr int kWords = (1 << IntKey<T>::kBits) / 2;
  constexpr int kPerChunk = 16 / (int)sizeof(T);
  extern __shared__ unsigned cnt[];   // bins 2w (low half) and 2w + 1 (high half)
  for (int w = threadIdx.x; w < kWords; w += blockDim.x) cnt[w] = 0u;
  __syncthreads();
  auto add = [&](T v) {
    const unsigned k = int_key(v);
    atomicAdd(&cnt[k >> 1], 1u << ((k & 1u) * 16u));
  };
  const bool vec = ((uintptr_t)x & 15) == 0;
  const long long n_slices = (n + kSlice - 1) / kSlice;
  for (long long sl = blockIdx.x; sl < n_slices; sl += gridDim.x) {
    const long long s0 = sl * kSlice, len = min((long long)kSlice, n - s0);
    const T* p = x + s0;
    long long done = 0;
    if (vec) {   // s0 * sizeof(T) is a multiple of 16: whole slices stay aligned
      const int chunks = (int)(len / kPerChunk);
      const uint4* p4 = reinterpret_cast<const uint4*>(p);
      for (int c = threadIdx.x; c < chunks; c += blockDim.x) {
        union {
          uint4 u;
          T v[kPerChunk];
        } b;
        b.u = __ldg(p4 + c);
#pragma unroll
        for (int e = 0; e < kPerChunk; ++e) add(b.v[e]);
      }
      done = (long long)chunks * kPerChunk;
    }
    for (long long i = done + threadIdx.x; i < len; i += blockDim.x) add(p[i]);
    __syncthreads();
    for (int w = threadIdx.x; w < kWords; w += blockDim.x) {
      const unsigned c = cnt[w];
      if (c) {
        if (c & 0xffffu) atomicAdd(&s->hist[2 * w], (unsigned long long)(c & 0xffffu));
        if (c >> 16) atomicAdd(&s->hist[2 * w + 1], (unsigned long long)(c >> 16));
        cnt[w] = 0u;
      }
    }
    __syncthreads();
  }
}

// The bins of order statistics r[0..nq) (0-based ranks) and count(key <= that bin).  All threads call it; `pre` holds
// the exclusive prefix of the per-thread bin sums, thread t owning bins [t * per, (t + 1) * per).
__device__ void int_pick_ranks(const unsigned long long* h, int bins, int per, const long long* pre,
                               const long long* r, int nq, int* key, long long* cum) {
  const int b0 = threadIdx.x * per, b1 = min(bins, b0 + per);
  for (int q = 0; q < nq; ++q) {
    long long c = pre[threadIdx.x];
    if (b0 < b1 && r[q] >= c && r[q] < pre[threadIdx.x + 1]) {
      for (int b = b0; b < b1; ++b) {
        c += (long long)h[b];
        if (c > r[q]) {
          key[q] = b;
          cum[q] = c;
          break;
        }
      }
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kIntPickThreads)
int_pick_kernel(IntStatsState* s, int bins, int offset) {
  __shared__ long long pre[kIntPickThreads + 1];
  __shared__ int key[2];
  __shared__ long long cum[2];
  if (s->status != MICA_NORM_PENDING) return;   // a peer sum that timed out left a partial histogram
  const long long n = s->n_total;
  if (n <= 0) {
    if (threadIdx.x == 0) s->status = MICA_NORM_NO_POSITIVE;
    return;
  }
  const int per = (bins + kIntPickThreads - 1) / kIntPickThreads;
  const int b0 = threadIdx.x * per, b1 = min(bins, b0 + per);
  long long mine = 0;
  for (int b = b0; b < b1; ++b) mine += (long long)s->hist[b];
  pre[threadIdx.x + 1] = mine;
  if (threadIdx.x == 0) pre[0] = 0;
  __syncthreads();
  for (int d = 1; d < kIntPickThreads; d <<= 1) {   // inclusive scan of pre[1..]
    const long long v = threadIdx.x >= d ? pre[threadIdx.x + 1 - d] : 0;
    __syncthreads();
    pre[threadIdx.x + 1] += v;
    __syncthreads();
  }
  // np.median: order statistics (n - 1) / 2 and n / 2, their float64 mean
  const long long rm[2] = {(n - 1) / 2, n / 2};
  int_pick_ranks(s->hist, bins, per, pre, rm, 2, key, cum);
  const double a = (double)(key[0] + offset), b = (double)(key[1] + offset);
  const double med = (n & 1) ? b : __ddiv_rn(__dadd_rn(a, b), 2.0);
  // count(x <= med): a and b are adjacent order statistics, a <= med <= b
  const long long n_le = (med >= b) ? cum[1] : cum[0];
  const long long npos = n - n_le;
  __syncthreads();
  if (npos <= 0) {
    if (threadIdx.x == 0) {
      s->median = med;
      s->n_le_med = n_le;
      s->n_pos = 0;
      s->status = MICA_NORM_NO_POSITIVE;
    }
    return;
  }
  // np.percentile(pos, 99.9) on float64: vi = (npos - 1) * q, g = vi - floor(vi), linear interpolation
  const double q = __ddiv_rn(99.9, 100.0);
  const double vi = __dmul_rn((double)(npos - 1), q);
  const double prev = floor(vi);
  long long lo, hi;
  if (vi >= (double)(npos - 1)) {
    lo = hi = npos - 1;
  } else {
    lo = (long long)prev;
    hi = lo + 1 < npos - 1 ? lo + 1 : npos - 1;
  }
  const double g = __dsub_rn(vi, prev);
  const long long rp[2] = {n_le + lo, n_le + hi};
  int_pick_ranks(s->hist, bins, per, pre, rp, 2, key, cum);
  if (threadIdx.x == 0) {
    const double pa = __dsub_rn((double)(key[0] + offset), med), pb = __dsub_rn((double)(key[1] + offset), med);
    const double d = __dsub_rn(pb, pa);
    const double r = (g >= 0.5) ? __dsub_rn(pb, __dmul_rn(d, __dsub_rn(1.0, g))) : __dadd_rn(pa, __dmul_rn(d, g));
    s->median = med;
    s->p = r;
    s->n_le_med = n_le;
    s->n_pos = npos;
    s->status = (r != 0.0) ? MICA_NORM_OK : MICA_NORM_ZERO_PCTL;
  }
}

// ((m < p) * m + (m >= p) * p) / p with m = (x > med) * (x - med), all float64 as NumPy evaluates it, then float32:
//   x <= med       m = +-0, the sum is +0 + 0 = +0: y = +0
//   x - med >= p   the sum is p: y = 1
//   otherwise      the sum is m: y = float32(m / p), the float64 quotient rounded once more
template <typename T>
__device__ __forceinline__ float int_normalize_one(T v, double med, double p) {
  const double x = (double)v;
  if (!(x > med)) return 0.0f;
  const double m = __dsub_rn(x, med);
  if (m >= p) return 1.0f;
  return __double2float_rn(__ddiv_rn(m, p));
}

template <typename T>
__global__ void __launch_bounds__(256)
int_normalize_kernel(const T* __restrict__ x, float* __restrict__ y, long long n, const IntStatsState* __restrict__ s) {
  if (s->status != MICA_NORM_OK) return;
  const double med = s->median, p = s->p;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  struct alignas(4 * sizeof(T)) T4 {
    T v[4];
  };
  const bool vec = ((((uintptr_t)x) & (4 * sizeof(T) - 1)) | (((uintptr_t)y) & 15)) == 0;
  const long long n4 = vec ? (n >> 2) : 0;
  const T4* x4 = reinterpret_cast<const T4*>(x);
  float4* y4 = reinterpret_cast<float4*>(y);
  for (long long i = tid; i < n4; i += stride) {
    const T4 v = x4[i];
    st_stream4(y4 + i, make_float4(int_normalize_one(v.v[0], med, p), int_normalize_one(v.v[1], med, p),
                                   int_normalize_one(v.v[2], med, p), int_normalize_one(v.v[3], med, p)));
  }
  for (long long i = n4 * 4 + tid; i < n; i += stride) y[i] = int_normalize_one(x[i], med, p);
}

static IntStatsState* int_state_of(const void* ws) { return (IntStatsState*)(((uintptr_t)ws + 255) / 256 * 256); }

static bool int_dtype_ok(int dtype) {
  return dtype == MICA_DTYPE_I8 || dtype == MICA_DTYPE_I16 || dtype == MICA_DTYPE_U16;
}

template <typename T>
static int int_hist_t(const T* x, int64_t n, IntStatsState* s, cudaStream_t st) {
  constexpr int bins = 1 << IntKey<T>::kBits;
  if (n <= 0) return MICA_OK;
  const size_t smem = (size_t)bins * sizeof(unsigned short);
  // per device/context attribute: set it on every call
  MICA_CUDA(cudaFuncSetAttribute(int_hist_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t slices = ceil_div64(n, kSlice);
  const int64_t cap = (int64_t)kNumSMs * (bins > 256 ? 1 : 2);   // 128 KB of counters: one CTA per SM
  int_hist_kernel<T><<<(unsigned)(slices < cap ? slices : cap), kIntHistThreads, smem, st>>>(x, (long long)n, s);
  MICA_LAUNCH_CHECK("int_hist_kernel");
  return MICA_OK;
}

// ---------------------------------------------------- histogram sum over peer memory
// A z-slab partition needs the SUM of every rank's histogram between hist and pick.  Every rank owns one exported
// buffer (mica_ipc_alloc of mica_int_peer_buffer_bytes) that all peers have mapped.  Two kernels, so that no kernel
// waits for a flag another CTA of its own grid raises:
//   int_peer_publish_kernel  copies the local histogram into this rank's slot `parity`; the last CTA to finish raises
//                            this rank's epoch flag in every peer's buffer (st.release.sys).  It never waits.
//   int_peer_sum_kernel      every CTA waits (ld.acquire.sys, bounded) for every peer's flag, then sums its slice of
//                            bins from every peer's slot into the local state.  A peer that never arrives sets the
//                            status to MICA_NORM_PEER_TIMEOUT, and int_pick_kernel leaves such a state alone.
// Only the live bins travel: 2^8 for int8, 2^16 for int16 / uint16.
// Slots alternate with the call epoch.  Rank r rewrites slot `parity` two calls later, in the publish of epoch e + 2.
// It gets there only after its sum of epoch e + 1, which waited for every peer's flag of e + 1; a peer raises that
// flag in its publish of e + 1, which its stream runs after its sum of epoch e has finished reading the slot.
// The two kernels have entry points of their own: ranks emulated on ONE GPU (tests) must enqueue every rank's
// publish before any rank's sum, or the spinning sum CTAs of one rank can hold the SMs (or a hardware queue) that
// another rank's histogram and publish are waiting for.
constexpr int kIntPeerMaxWorld = 64;
constexpr int kIntPeerBinsPerCta = 2048;   // 32 CTAs for 2^16 bins: few CTAs spin while the peers publish

struct IntPeerBuffer {
  unsigned long long slot[2][kIntMaxBins];
  int flag[kIntPeerMaxWorld];     // flag[p] = last epoch rank p has published
  unsigned done[2];               // publish bookkeeping: CTAs finished, per parity
  int pad[kIntPeerMaxWorld - 2];
};

__global__ void __launch_bounds__(256)
int_peer_publish_kernel(const IntStatsState* __restrict__ s, IntPeerBuffer* const* __restrict__ peers, int rank,
                        int world, int parity, int epoch, int bins) {
  IntPeerBuffer* mine = peers[rank];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < bins; i += gridDim.x * blockDim.x)
    mine->slot[parity][i] = s->hist[i];
  __threadfence();
  __syncthreads();
  __shared__ bool last;
  if (threadIdx.x == 0) last = (atomicAdd(&mine->done[parity], 1u) == gridDim.x - 1);
  __syncthreads();
  if (!last) return;
  if (threadIdx.x == 0) mine->done[parity] = 0;   // ready for this slot's next use (two calls later)
  __threadfence_system();                         // every CTA's bins (observed through the counter) before the flags
  __syncthreads();
  if (threadIdx.x < world) st_release_sys(&peers[threadIdx.x]->flag[rank], epoch);
}

// grid = ceil(bins / kIntPeerBinsPerCta), block = 256: eight bins per thread
__global__ void __launch_bounds__(256)
int_peer_sum_kernel(IntStatsState* __restrict__ s, IntPeerBuffer* const* __restrict__ peers, int rank, int world,
                    int parity, int epoch, int bins, long long timeout_cycles) {
  __shared__ int ok;
  __shared__ const unsigned long long* base[kIntPeerMaxWorld];
  if (threadIdx.x == 0) ok = 1;
  __syncthreads();
  if (threadIdx.x < world) {     // wait for peer threadIdx.x
    const int* f = &peers[rank]->flag[threadIdx.x];
    const long long t0 = clock64();
    while (ld_acquire_sys(f) - epoch < 0) {
      if (clock64() - t0 > timeout_cycles) {
        ok = 0;
        break;
      }
    }
    base[threadIdx.x] = peers[threadIdx.x]->slot[parity];
  }
  __threadfence_system();
  __syncthreads();
  if (!ok) {
    if (threadIdx.x == 0) s->status = MICA_NORM_PEER_TIMEOUT;
    return;
  }
  constexpr int kPer = kIntPeerBinsPerCta / 256;
  const int b0 = blockIdx.x * kIntPeerBinsPerCta + threadIdx.x;
  unsigned long long sum[kPer];
#pragma unroll
  for (int k = 0; k < kPer; ++k) sum[k] = 0ull;
  for (int p = 0; p < world; ++p) {   // the kPer loads of one peer are issued before they are consumed
    unsigned long long v[kPer];
#pragma unroll
    for (int k = 0; k < kPer; ++k) v[k] = b0 + k * 256 < bins ? __ldcv(base[p] + b0 + k * 256) : 0ull;
#pragma unroll
    for (int k = 0; k < kPer; ++k) sum[k] += v[k];
  }
#pragma unroll
  for (int k = 0; k < kPer; ++k)
    if (b0 + k * 256 < bins) s->hist[b0 + k * 256] = sum[k];
}

template <typename T>
static int int_normalize_t(const T* x, float* y, int64_t n, const IntStatsState* s, cudaStream_t st) {
  const int64_t want = ceil_div64(ceil_div64(n, 4), 256);
  const int grid = (int)(want < (int64_t)kNumSMs * 8 ? want : (int64_t)kNumSMs * 8);
  int_normalize_kernel<T><<<grid, 256, 0, st>>>(x, y, (long long)n, s);
  MICA_LAUNCH_CHECK("int_normalize_kernel");
  return MICA_OK;
}

}  // namespace mica

using namespace mica;

extern "C" size_t mica_int_stats_workspace_bytes(void) { return sizeof(IntStatsState) + 256; }

static int int_bins(int dtype) { return dtype == MICA_DTYPE_I8 ? 256 : kIntMaxBins; }

extern "C" int mica_int_stats_init(void* workspace, int dtype, int64_t n_total, mica_stream_t stream) {
  MICA_REQUIRE(workspace, "null pointer");
  MICA_REQUIRE(n_total >= 0, "negative n");
  MICA_REQUIRE(int_dtype_ok(dtype), "integer order statistics take MICA_DTYPE_I8 / I16 / U16 (got dtype %d)", dtype);
  const int bins = int_bins(dtype);
  int_stats_init_kernel<<<(bins + 255) / 256, 256, 0, (cudaStream_t)stream>>>(int_state_of(workspace), bins,
                                                                             (long long)n_total);
  MICA_LAUNCH_CHECK("int_stats_init_kernel");
  return MICA_OK;
}

extern "C" int mica_int_stats_hist(const void* x, int dtype, int64_t n_local, void* workspace, mica_stream_t stream) {
  MICA_REQUIRE(workspace && (x || n_local == 0), "null pointer");
  MICA_REQUIRE(n_local >= 0, "negative n");
  MICA_REQUIRE(int_dtype_ok(dtype), "integer order statistics take MICA_DTYPE_I8 / I16 / U16 (got dtype %d)", dtype);
  IntStatsState* s = int_state_of(workspace);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == MICA_DTYPE_I8) return int_hist_t((const int8_t*)x, n_local, s, st);
  if (dtype == MICA_DTYPE_I16) return int_hist_t((const int16_t*)x, n_local, s, st);
  return int_hist_t((const uint16_t*)x, n_local, s, st);
}

extern "C" int64_t* mica_int_stats_hist_ptr(void* workspace) {
  return workspace ? reinterpret_cast<int64_t*>(int_state_of(workspace)->hist) : nullptr;
}

extern "C" int mica_int_stats_pick(void* workspace, int dtype, mica_stream_t stream) {
  MICA_REQUIRE(workspace, "null pointer");
  MICA_REQUIRE(int_dtype_ok(dtype), "integer order statistics take MICA_DTYPE_I8 / I16 / U16 (got dtype %d)", dtype);
  const int offset = dtype == MICA_DTYPE_I8 ? IntKey<int8_t>::kOffset
                                            : (dtype == MICA_DTYPE_I16 ? IntKey<int16_t>::kOffset : IntKey<uint16_t>::kOffset);
  int_pick_kernel<<<1, kIntPickThreads, 0, (cudaStream_t)stream>>>(int_state_of(workspace), int_bins(dtype), offset);
  MICA_LAUNCH_CHECK("int_pick_kernel");
  return MICA_OK;
}

extern "C" int mica_int_order_stats(const void* x, int dtype, int64_t n, void* workspace, mica_stream_t stream) {
  MICA_REQUIRE(workspace && (x || n == 0), "null pointer");
  MICA_REQUIRE(n >= 0, "negative n");
  MICA_REQUIRE(int_dtype_ok(dtype), "integer order statistics take MICA_DTYPE_I8 / I16 / U16 (got dtype %d)", dtype);
  if (int rc = mica_int_stats_init(workspace, dtype, n, stream)) return rc;
  if (int rc = mica_int_stats_hist(x, dtype, n, workspace, stream)) return rc;
  return mica_int_stats_pick(workspace, dtype, stream);
}

extern "C" size_t mica_int_peer_buffer_bytes(void) { return sizeof(IntPeerBuffer); }

static int int_peer_args(void* workspace, int dtype, void* const* peer_bufs, int rank, int world, int parity) {
  MICA_REQUIRE(workspace && peer_bufs, "null pointer");
  MICA_REQUIRE(int_dtype_ok(dtype), "integer order statistics take MICA_DTYPE_I8 / I16 / U16 (got dtype %d)", dtype);
  MICA_REQUIRE(world >= 1 && world <= kIntPeerMaxWorld && rank >= 0 && rank < world, "bad rank/world");
  MICA_REQUIRE(parity == 0 || parity == 1, "parity must be 0 or 1");
  return MICA_OK;
}

static unsigned int_peer_grid(int dtype) {
  return (unsigned)((int_bins(dtype) + kIntPeerBinsPerCta - 1) / kIntPeerBinsPerCta);
}

extern "C" int mica_int_stats_peer_publish(const void* workspace, int dtype, void* const* peer_bufs, int rank,
                                           int world, int parity, int epoch, mica_stream_t stream) {
  if (int rc = int_peer_args((void*)workspace, dtype, peer_bufs, rank, world, parity)) return rc;
  if (world == 1) return MICA_OK;
  int_peer_publish_kernel<<<int_peer_grid(dtype), 256, 0, (cudaStream_t)stream>>>(
      int_state_of(workspace), reinterpret_cast<IntPeerBuffer* const*>(peer_bufs), rank, world, parity, epoch,
      int_bins(dtype));
  MICA_LAUNCH_CHECK("int_peer_publish_kernel");
  return MICA_OK;
}

extern "C" int mica_int_stats_peer_sum(void* workspace, int dtype, void* const* peer_bufs, int rank, int world,
                                       int parity, int epoch, mica_stream_t stream) {
  if (int rc = int_peer_args(workspace, dtype, peer_bufs, rank, world, parity)) return rc;
  if (world == 1) return MICA_OK;
  int_peer_sum_kernel<<<int_peer_grid(dtype), 256, 0, (cudaStream_t)stream>>>(
      int_state_of(workspace), reinterpret_cast<IntPeerBuffer* const*>(peer_bufs), rank, world, parity, epoch,
      int_bins(dtype), mica::peer_timeout_cycles());
  MICA_LAUNCH_CHECK("int_peer_sum_kernel");
  return MICA_OK;
}

extern "C" int mica_int_stats_result_async(const void* workspace, void* host_record, mica_stream_t stream) {
  MICA_REQUIRE(workspace && host_record, "null pointer");
  const IntStatsState* s = int_state_of(workspace);
  MICA_CUDA(cudaMemcpyAsync(host_record, &s->median, MICA_INT_STATS_RESULT_BYTES, cudaMemcpyDeviceToHost,
                            (cudaStream_t)stream));
  return MICA_OK;
}

extern "C" int mica_int_stats_result(const void* workspace, double* median, double* p999, int64_t* n_pos,
                                     int* norm_status, mica_stream_t stream) {
  struct {
    double median, p;
    long long n_pos;
    int status, zero;
  } r;
  static_assert(sizeof(r) == MICA_INT_STATS_RESULT_BYTES, "result record size");
  int rc = mica_int_stats_result_async(workspace, &r, stream);
  if (rc) return rc;
  MICA_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  if (median) *median = r.median;
  if (p999) *p999 = r.p;
  if (n_pos) *n_pos = r.n_pos;
  if (norm_status) *norm_status = r.status;
  return MICA_OK;
}

extern "C" int mica_normalize_apply_int(const void* x, int dtype, float* y, int64_t n, const void* workspace,
                                        mica_stream_t stream) {
  MICA_REQUIRE(x && y && workspace, "null pointer");
  MICA_REQUIRE(int_dtype_ok(dtype), "integer normalisation takes MICA_DTYPE_I8 / I16 / U16 (got dtype %d)", dtype);
  if (n <= 0) return MICA_OK;
  const IntStatsState* s = int_state_of(workspace);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == MICA_DTYPE_I8) return int_normalize_t((const int8_t*)x, y, n, s, st);
  if (dtype == MICA_DTYPE_I16) return int_normalize_t((const int16_t*)x, y, n, s, st);
  return int_normalize_t((const uint16_t*)x, y, n, s, st);
}
