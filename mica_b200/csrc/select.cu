// R2/R3: exact median / 99.9-percentile normalisation.
//
// Replaces utils/preprocessing.py:122-133 (reference root):
//   norm = nan_to_num(x); med = np.median(norm); m = (norm > med) * (norm - med)
//   p = np.percentile(m[m > 0], 99.9); m = min(m, p) / p
// np.median / np.percentile are exact order statistics; they are found here by a
// most-significant-digit radix select (11 + 11 + 10 bits) over order-preserving
// uint32 keys with warp-ballot (match_any) aggregated shared-memory histograms.
// The interpolation between the two bracketing order statistics follows the
// installed NumPy 2.x float32 arithmetic (SURVEY.md 8a R3).  Because float32
// subtraction is monotone, the percentile of the positives m is selected on x at
// rank count(x <= med) + lo and the median subtracted afterwards.
//
// All state lives in a device workspace; the host only sequences launches, so a
// multi-GPU run can all-reduce hist[] between `hist` and `pick` on the stream.
#include <string.h>

#include "common.cuh"

namespace mica {

constexpr int kBins = 2048;
constexpr int kDigitRounds = 5;   // digit passes: median 0,1,2 + percentile 1,2 (digit 0 of the percentile reuses hist0)

struct SelectState {
  // histograms first: this is the region the multi-GPU all-reduce covers
  long long hist[2][kBins];   // MICA_SELECT_HIST_WORDS int64
  long long hist0[kBins];     // saved digit-0 histogram of the whole array
  long long n_total;
  long long rank[2];          // remaining rank of each target inside its prefix bucket
  long long below[2];         // number of keys strictly below the prefix bucket
  long long count_eq[2];      // multiplicity of the selected key (after the last pass)
  unsigned prefix[2];         // key bits fixed so far (right-aligned)
  int round;                  // 0..4 = next hist/pick round; 5 = done
  int status;                 // MICA_NORM_*
  long long n_le_med;         // count(x <= median)
  long long n_pos;            // count(x > median)
  float median;
  float p;
  float g;                    // percentile interpolation weight
  int phase0;                 // digit 0: 0 = sample pending, 1 = guided pass pending, 2 = full pass pending, 3 = done
  int cand[3];                // candidate digit-0 bins from the sample: median in [cand0, cand1], percentile >= cand2
  int comp_ok;                // 1 = the compact buffer holds every voxel of the candidate bins (digits 1, 2 read it)
  // compact buffer (follows the state in the workspace): the voxels the guided pass found in the candidate
  // bins -- a few percent of the map -- so that the four later digit passes do not stream the map again
  long long comp_cap;         // capacity in floats; set once per workspace (mica_select_set_compact), survives init
  unsigned long long comp_count;   // floats appended by the guided pass (> comp_cap = overflow: not usable)
  // the candidate bins as float thresholds (smallest float of bin cand[0], of bin cand[1] + 1, of bin cand[2]):
  // the compacting guided pass classifies a voxel with three float compares instead of building its key
  float thr[3];
  int guided_compact;         // 1 = digit 0 came from the compacting guided pass (histogram built from the buffer)
};

constexpr int kCompStage = 160;   // per-warp staging slots of the guided pass (flushed when < 32 are free)

__host__ __device__ __forceinline__ float* comp_buffer(SelectState* s) {
  return reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(s + 1) + 255) / 256 * 256);
}

static_assert(sizeof(long long) * 2 * kBins == MICA_SELECT_HIST_WORDS * 8, "hist words");

__device__ __forceinline__ float nan_to_num_f32(float v) {
  // np.nan_to_num defaults: nan -> 0, +inf -> FLT_MAX, -inf -> -FLT_MAX
  if (v != v) return 0.0f;
  if (v == __int_as_float(0x7f800000)) return __int_as_float(0x7f7fffff);
  if (v == __int_as_float(0xff800000)) return __int_as_float(0xff7fffff);
  return v;
}

// order-preserving key; -0.0 and +0.0 share a key (they compare equal in NumPy's sort)
__device__ __forceinline__ unsigned f32_key(float v) {
  unsigned u = __float_as_uint(v);
  if (u == 0x80000000u) u = 0u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_f32(unsigned k) {
  unsigned u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(u);
}

// round r -> which digit: rounds 0,1,2 = median digits 0,1,2; rounds 3,4 = percentile digits 1,2
__device__ __forceinline__ int round_digit(int r) { return r < 3 ? r : r - 2; }

__device__ __forceinline__ void warp_hist_add(unsigned* h, unsigned bin, bool pred) {
  unsigned act = __ballot_sync(0xffffffffu, pred);
  if (act == 0u) return;
  if (__popc(act) <= 8) {          // a few candidates: plain shared atomics
    if (pred) atomicAdd(&h[bin], 1u);
  } else if (pred) {               // many (ties): one atomic per distinct bin
    unsigned peers = __match_any_sync(act, bin);
    if ((threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&h[bin], (unsigned)__popc(peers));
  }
}

__device__ __forceinline__ void hist_one(float v, int digit, unsigned p0, unsigned p1, bool same, unsigned* h) {
  unsigned k = f32_key(nan_to_num_f32(v));
  if (digit == 0) {
    warp_hist_add(h, k >> 21, true);
  } else if (digit == 1) {
    unsigned hi = k >> 21, bin = (k >> 10) & 0x7ffu;
    warp_hist_add(h, bin, hi == p0);
    if (!same) warp_hist_add(h + kBins, bin, hi == p1);
  } else {
    unsigned hi = k >> 10, bin = k & 0x3ffu;
    warp_hist_add(h, bin, hi == p0);
    if (!same) warp_hist_add(h + kBins, bin, hi == p1);
  }
}

// raw float bits whose order-preserving key has `hi` as its top bits (width = number of prefix bits)
__host__ __device__ __forceinline__ unsigned raw_prefix_of(unsigned hi, int width) {
  const unsigned top = 1u << (width - 1), mask = (top << 1) - 1u;
  return (hi & top) ? (hi & (top - 1u)) : (~hi & mask);   // positive floats: drop the set bit; negative: complement
}

// persistent grid-stride histogram pass for digits 1 and 2; float4 loads when aligned.
// These digits only count the elements inside the one or two prefix buckets found so far, so the
// common case is decided on the RAW bits
// (two shifts and compares per element); the key transform, nan_to_num and the ballot histogram
// run only for warps that hold a candidate or a special value (NaN, +-inf, +-0).
__global__ void __launch_bounds__(512)
select_hist_kernel(const float* __restrict__ x, long long n, SelectState* __restrict__ s) {
  __shared__ unsigned h[2 * kBins];
  const int round = s->round;
  if (round == 0 || round >= kDigitRounds || s->phase0 != 3 || s->status != MICA_NORM_PENDING) return;   // digit 0 has its own kernels
  if (s->comp_ok) {   // every voxel these digits can count was compacted by the guided pass
    x = comp_buffer(s);
    n = (long long)s->comp_count;
    if ((long long)blockIdx.x * blockDim.x * 4 >= n) return;   // the grid is sized for the whole map
  }
  for (int i = threadIdx.x; i < 2 * kBins; i += blockDim.x) h[i] = 0;
  __syncthreads();
  const int digit = round_digit(round);
  const unsigned p0 = s->prefix[0], p1 = s->prefix[1];
  const bool same = (p0 == p1);
  const int shift = digit == 1 ? 21 : 10, width = digit == 1 ? 11 : 22;
  const unsigned r0 = digit ? raw_prefix_of(p0, width) : 0u, r1 = digit ? raw_prefix_of(p1, width) : 0u;
  unsigned* h0 = h;

  const long long n4 = (((uintptr_t)x & 15) == 0) ? (n >> 2) : 0;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  const long long stride = (long long)gridDim.x * blockDim.x;
  // whole warps iterate together (match_any needs converged lanes): pad the loop to the warp
  const long long n4_pad = (n4 + 31) & ~31LL;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4_pad; i += stride) {
    bool ok = i < n4;
    float4 v = ok ? ld_stream4(x4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (__ballot_sync(0xffffffffu, ok) == 0xffffffffu) {
      if (digit != 0) {
        const unsigned u[4] = {__float_as_uint(v.x), __float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(v.w)};
        bool cand = false;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const unsigned r = u[c] >> shift, e = u[c] << 1;
          cand |= (r == r0) | (r == r1) | (e >= 0xff000000u) | (e == 0u);
        }
        if (!__any_sync(0xffffffffu, cand)) continue;
      }
      hist_one(v.x, digit, p0, p1, same, h0);
      hist_one(v.y, digit, p0, p1, same, h0);
      hist_one(v.z, digit, p0, p1, same, h0);
      hist_one(v.w, digit, p0, p1, same, h0);
    } else if (ok) {  // ragged last warp: plain atomics
      float vv[4] = {v.x, v.y, v.z, v.w};
      for (int c = 0; c < 4; ++c) {
        unsigned k = f32_key(nan_to_num_f32(vv[c]));
        if (digit == 0) {
          atomicAdd(&h[k >> 21], 1u);
        } else {
          unsigned hi = digit == 1 ? (k >> 21) : (k >> 10);
          unsigned bin = digit == 1 ? ((k >> 10) & 0x7ffu) : (k & 0x3ffu);
          if (hi == p0) atomicAdd(&h[bin], 1u);
          if (!same && hi == p1) atomicAdd(&h[kBins + bin], 1u);
        }
      }
    }
  }
  // scalar tail (and the whole array when it is not 16-byte aligned)
  for (long long i = n4 * 4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    unsigned k = f32_key(nan_to_num_f32(x[i]));
    if (digit == 0) {
      atomicAdd(&h[k >> 21], 1u);
    } else {
      unsigned hi = digit == 1 ? (k >> 21) : (k >> 10);
      unsigned bin = digit == 1 ? ((k >> 10) & 0x7ffu) : (k & 0x3ffu);
      if (hi == p0) atomicAdd(&h[bin], 1u);
      if (!same && hi == p1) atomicAdd(&h[kBins + bin], 1u);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * kBins; i += blockDim.x) {
    unsigned c = h[i];
    if (c) atomicAdd(reinterpret_cast<unsigned long long*>(&s->hist[0][0]) + i, (unsigned long long)c);
  }
}


// ---- digit 0 (every element counts): warp-private 16-bit histograms, no atomics in the loop.
// Every warp owns a [2048] uint16 histogram: after match_any the leader lanes hold DISTINCT bins, so
// a plain load-add-store per leader is race-free (no shared-memory atomics, no inter-warp contention
// on the few hot bins), and a warp never sees more than kHist0MaxPerWarp elements (the host sizes
// the grid), so 16 bits cannot overflow.  grid x 512 threads, 64 KB dynamic shared memory.
// Measured on B200: this pass stays ~3x slower than the others whatever does the aggregation
// (shared atomics, this scheme, 11 ballots instead of MATCH): ~50 warp-wide MIO operations per
// float4 bound it, not DRAM.  Next step (DESIGN.md): a sampled pivot so that ~99 % of the
// elements only bump a register counter.
constexpr int kHist0Warps = 16;
constexpr long long kHist0MaxPerWarp = 60000;

__global__ void __launch_bounds__(512)
select_hist0_kernel(const float* __restrict__ x, long long n, SelectState* __restrict__ s) {
  extern __shared__ unsigned short hw_all[];   // [kHist0Warps][kBins]
  if (s->phase0 != 2 || s->status != MICA_NORM_PENDING) return;   // the fallback of the guided pass
  for (int i = threadIdx.x; i < kHist0Warps * kBins / 2; i += blockDim.x) reinterpret_cast<unsigned*>(hw_all)[i] = 0u;
  __syncthreads();
  unsigned short* hw = hw_all + (threadIdx.x >> 5) * kBins;
  unsigned long long* gh = reinterpret_cast<unsigned long long*>(&s->hist[0][0]);

  // head: scalars up to the first 16-byte boundary; body: float4; tail: the rest
  long long head = (4 - (long long)(((uintptr_t)x >> 2) & 3)) & 3;
  if (head > n) head = n;
  const float4* x4 = reinterpret_cast<const float4*>(x + head);
  const long long n4 = (n - head) >> 2;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  if (tid < head) atomicAdd(gh + (f32_key(nan_to_num_f32(x[tid])) >> 21), 1ull);
  for (long long i = head + n4 * 4 + tid; i < n; i += stride) atomicAdd(gh + (f32_key(nan_to_num_f32(x[i])) >> 21), 1ull);

  const long long n4_pad = (n4 + 31) & ~31LL;
  for (long long i = tid; i < n4_pad; i += stride) {
    const bool ok = i < n4;
    const float4 v = ok ? ld_stream4(x4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    const unsigned act = __ballot_sync(0xffffffffu, ok);
    if (!ok) continue;
    const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const unsigned bin = f32_key(nan_to_num_f32(vv[c])) >> 21;
      const unsigned peers = __match_any_sync(act, bin);
      if ((threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) hw[bin] = (unsigned short)(hw[bin] + __popc(peers));
      __syncwarp(act);   // the next round's leaders may touch the bins written here
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kBins; i += blockDim.x) {
    unsigned c = 0;
#pragma unroll
    for (int w = 0; w < kHist0Warps; ++w) c += hw_all[w * kBins + i];
    if (c) atomicAdd(gh + i, (unsigned long long)c);
  }
}

// ---- digit 0 from a sampled pivot.  A 1/64 sample (select_sample_kernel, same histogram) tells where
// the median and the 99.9 % tail will fall: a few candidate bins [A_lo, A_hi] around the sample
// median and everything from P_lo (sample quantile 0.997) upwards.  The guided pass then histograms
// only the voxels inside the candidate bins exactly; every other voxel just bumps one of two
// register counters ("below A_lo", "between A_hi and P_lo"), whose totals are lumped into bins
// A_lo-1 and P_lo-1.  The pick verifies on these EXACT counts that both median ranks fall inside
// [A_lo, A_hi] and that the tail from P_lo holds more voxels than any percentile rank can skip;
// otherwise select_hist0_kernel (the full histogram) runs as the fallback round.  ~96 % of the
// voxels of a density map take the two-instruction path.
constexpr int kSampleStride = 64;   // float4 stride of the sample

__global__ void __launch_bounds__(512)
select_sample_kernel(const float* __restrict__ x, long long n, SelectState* __restrict__ s) {
  __shared__ unsigned h[kBins];
  if (s->phase0 != 0 || s->status != MICA_NORM_PENDING) return;
  for (int i = threadIdx.x; i < kBins; i += blockDim.x) h[i] = 0;
  __syncthreads();
  long long head = (4 - (long long)(((uintptr_t)x >> 2) & 3)) & 3;
  if (head > n) head = n;
  const float4* x4 = reinterpret_cast<const float4*>(x + head);
  const long long n4 = (n - head) >> 2, ns4 = (n4 + kSampleStride - 1) / kSampleStride;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < ns4; i += stride) {
    const float4 v = x4[i * kSampleStride];
    atomicAdd(&h[f32_key(nan_to_num_f32(v.x)) >> 21], 1u);
    atomicAdd(&h[f32_key(nan_to_num_f32(v.y)) >> 21], 1u);
    atomicAdd(&h[f32_key(nan_to_num_f32(v.z)) >> 21], 1u);
    atomicAdd(&h[f32_key(nan_to_num_f32(v.w)) >> 21], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kBins; i += blockDim.x) {
    unsigned c = h[i];
    if (c) atomicAdd(reinterpret_cast<unsigned long long*>(&s->hist[0][0]) + i, (unsigned long long)c);
  }
}

__global__ void __launch_bounds__(512)
select_hist0_guided_kernel(const float* __restrict__ x, long long n, SelectState* __restrict__ s, int allow_compacting) {
  __shared__ unsigned h[kBins];
  __shared__ unsigned long long lump[2];
  __shared__ float stage_all[16][kCompStage];
  if (s->phase0 != 1 || s->status != MICA_NORM_PENDING) return;
  if (allow_compacting && s->comp_cap > 0) return;   // select_guided_compact_kernel serves this workspace
  for (int i = threadIdx.x; i < kBins; i += blockDim.x) h[i] = 0;
  if (threadIdx.x < 2) lump[threadIdx.x] = 0ull;
  __syncthreads();
  // candidate voxels are appended to the compact buffer: staged per warp (ballot-ranked, no atomics), one
  // global atomic per ~130 candidates reserves the run, the warp writes it coalesced
  float* const comp = comp_buffer(s);
  const long long comp_cap = s->comp_cap;
  float* const stage = stage_all[threadIdx.x >> 5];
  const unsigned lane = threadIdx.x & 31, lt_mask = (1u << lane) - 1u;
  int staged = 0;   // warp-uniform
  auto flush = [&]() {
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(&s->comp_count, (unsigned long long)staged);
    base = __shfl_sync(0xffffffffu, base, 0);
    __syncwarp();
    if ((long long)(base + staged) <= comp_cap)
      for (int i = lane; i < staged; i += 32) comp[base + i] = stage[i];
    __syncwarp();
    staged = 0;
  };
  auto append = [&](unsigned m, bool mine, float v) {   // m = ballot of `mine` over the (converged) warp
    if (comp_cap == 0) return;
    if (mine) stage[staged + __popc(m & lt_mask)] = v;
    staged += __popc(m);
    if (staged > kCompStage - 32) flush();
  };
  const unsigned a_lo = (unsigned)s->cand[0], a_w = (unsigned)(s->cand[1] - s->cand[0]), p_lo = (unsigned)s->cand[2];
  unsigned c0 = 0, c1 = 0;   // voxels below A_lo / between A_hi and P_lo seen by this thread
  auto classify = [&](float v, unsigned& bin) -> bool {
    bin = f32_key(nan_to_num_f32(v)) >> 21;
    const bool below = bin < a_lo, exact = (bin - a_lo <= a_w) | (bin >= p_lo);
    c0 += below ? 1u : 0u;
    c1 += (below | exact) ? 0u : 1u;
    return exact;
  };
  long long head = (4 - (long long)(((uintptr_t)x >> 2) & 3)) & 3;
  if (head > n) head = n;
  const float4* x4 = reinterpret_cast<const float4*>(x + head);
  const long long n4 = (n - head) >> 2;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  unsigned bin;
  // head (< 4 scalars) and tail (< 4 scalars): only the first lanes of block 0's first warp see them; the
  // whole warp walks through the append so that the ballots stay converged
  {
    const long long n_edge = head + (n - head - n4 * 4);   // <= 6
    if (blockIdx.x == 0 && threadIdx.x < 32) {
      const long long e = threadIdx.x;
      const bool have = e < n_edge;
      const long long idx = e < head ? e : head + n4 * 4 + (e - head);
      const float v = have ? x[idx] : 0.f;
      const bool exact = have && classify(v, bin);
      if (exact) atomicAdd(&h[bin], 1u);
      append(__ballot_sync(0xffffffffu, exact), exact, v);
    }
  }
  const long long n4_pad = (n4 + 31) & ~31LL;
  for (long long i = tid; i < n4_pad; i += stride) {
    const bool ok = i < n4;
    const float4 v = ok ? ld_stream4(x4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const bool exact = ok && classify(vv[c], bin);
      const unsigned m = __ballot_sync(0xffffffffu, exact);
      if (m == 0u) continue;
      append(m, exact, vv[c]);
      if (__popc(m) <= 8) {            // a few candidates: plain shared atomics
        if (exact) atomicAdd(&h[bin], 1u);
      } else if (exact) {              // many (ties, masked maps): one atomic per distinct bin
        const unsigned peers = __match_any_sync(m, bin);
        if ((threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&h[bin], (unsigned)__popc(peers));
      }
    }
  }
  if (staged > 0) flush();
  // block totals of the two counters
  for (int o = 16; o > 0; o >>= 1) {
    c0 += __shfl_xor_sync(0xffffffffu, c0, o);
    c1 += __shfl_xor_sync(0xffffffffu, c1, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (c0) atomicAdd(&lump[0], (unsigned long long)c0);
    if (c1) atomicAdd(&lump[1], (unsigned long long)c1);
  }
  __syncthreads();
  unsigned long long* gh = reinterpret_cast<unsigned long long*>(&s->hist[0][0]);
  for (int i = threadIdx.x; i < kBins; i += blockDim.x) {
    unsigned c = h[i];
    if (c) atomicAdd(gh + i, (unsigned long long)c);
  }
  if (threadIdx.x == 0) {
    if (lump[0]) atomicAdd(gh + (a_lo > 0 ? a_lo - 1 : 0), lump[0]);
    if (lump[1]) atomicAdd(gh + (p_lo > 0 ? p_lo - 1 : 0), lump[1]);
  }
}

// ---- digit 0, compacting form (workspaces with a compact buffer).  ncu on the kernel above: 66 instructions
// per voxel, 72 % issue-bound -- every voxel pays for the key transform although ~95 % of them only bump a
// counter.  Here the candidate bins arrive as three float thresholds (pick step 0): a voxel is classified with
// three compares, the candidates are only APPENDED to the compact buffer (lane-private shared-memory queues,
// flushed warp-wide) and
// their digit-0 histogram is built afterwards from the buffer (select_hist0_compact_kernel: a few percent of
// the map).  NaN fails every compare and -0 compares equal to +0, so both take the candidate route, where the
// key is exact; bins outside the candidate ranges that receive such strays are at or below the lumped bins, so
// every cumulative count the pick uses stays exact.
constexpr int kLaneQueue = 8;     // candidate slots per lane between two warp-wide flushes

__global__ void __launch_bounds__(512)
select_guided_compact_kernel(const float* __restrict__ x, long long n, SelectState* __restrict__ s) {
  __shared__ unsigned long long lump[2];
  __shared__ float queue_all[512 * kLaneQueue];   // [slot][thread]: lane-private queues, conflict-free
  __shared__ float gather_all[16][32 * kLaneQueue];   // per warp: the queues packed for a coalesced flush
  if (s->phase0 != 1 || s->status != MICA_NORM_PENDING || s->comp_cap <= 0) return;
  if (threadIdx.x < 2) lump[threadIdx.x] = 0ull;
  __syncthreads();
  const float lo = s->thr[0], hi = s->thr[1], pt = s->thr[2];
  float* const comp = comp_buffer(s);
  const long long comp_cap = s->comp_cap;
  float* const queue = queue_all + threadIdx.x;    // slot q of this lane: queue[q * 512]
  const unsigned lane = threadIdx.x & 31;
  int queued = 0;                                  // this lane's candidates waiting for the next flush
  unsigned c0 = 0, c1 = 0;
  // A candidate costs its lane one predicated shared store and one add -- no ballot per value.  When some
  // lane's queue could overflow in the next iteration (>= kLaneQueue - 4 entries) the warp flushes: a shuffle
  // scan of the 32 counts, one global atomic for the warp, every lane copies its entries to its range.
  auto flush = [&]() {
    int incl = queued;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int up = __shfl_up_sync(0xffffffffu, incl, o);
      if ((int)lane >= o) incl += up;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(&s->comp_count, (unsigned long long)total);
    base = __shfl_sync(0xffffffffu, base, 0);
    float* const pack = gather_all[threadIdx.x >> 5];
    const int at = incl - queued;
    for (int q = 0; q < queued; ++q) pack[at + q] = queue[q * 512];
    __syncwarp();
    if ((long long)(base + total) <= comp_cap)
      for (int i = lane; i < total; i += 32) comp[base + i] = pack[i];
    __syncwarp();
    queued = 0;
  };
  auto take = [&](float v, bool ok) {
    const bool below = v < lo, between = (v >= hi) & (v < pt);
    c0 += (ok & below) ? 1u : 0u;
    c1 += (ok & between) ? 1u : 0u;
    // branch-free append: the value always lands in the lane's next free slot (the flush keeps at least
    // four free), the slot is only kept when the voxel is a candidate
    queue[queued * 512] = v;
    queued += (ok & !(below | between)) ? 1 : 0;
  };
  long long head = (4 - (long long)(((uintptr_t)x >> 2) & 3)) & 3;
  if (head > n) head = n;
  const float4* x4 = reinterpret_cast<const float4*>(x + head);
  const long long n4 = (n - head) >> 2;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  if (blockIdx.x == 0 && threadIdx.x < 32) {   // the < 4 scalars before and after the float4 body
    const long long n_edge = head + (n - head - n4 * 4);
    const long long e = threadIdx.x;
    const bool have = e < n_edge;
    const long long idx = e < head ? e : head + n4 * 4 + (e - head);
    take(have ? x[idx] : 0.f, have);
  }
  const long long n4_pad = (n4 + 31) & ~31LL;      // whole warps iterate together (the flush is warp-wide)
  // four independent 16-byte loads in flight per thread: with one, 32 warps/SM keep only ~16 KB per SM on the
  // way, half of what the HBM latency-bandwidth product asks for (ncu: 31 % of DRAM peak, long-scoreboard stalls)
  constexpr int kDepth = 4;
  for (long long i = tid; i < n4_pad; i += kDepth * stride) {
    float4 v[kDepth];
    bool ok[kDepth];
#pragma unroll
    for (int u = 0; u < kDepth; ++u) {
      const long long iu = i + u * stride;
      ok[u] = iu < n4;
      v[u] = ok[u] ? ld_stream4(x4 + iu) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < kDepth; ++u) {
      if (i + u * stride >= n4_pad) break;         // warp-uniform: i and stride are multiples of 32 apart per warp
      take(v[u].x, ok[u]);
      take(v[u].y, ok[u]);
      take(v[u].z, ok[u]);
      take(v[u].w, ok[u]);
      if (__any_sync(0xffffffffu, queued > kLaneQueue - 4)) flush();
    }
  }
  if (__any_sync(0xffffffffu, queued > 0)) flush();
  for (int o = 16; o > 0; o >>= 1) {
    c0 += __shfl_xor_sync(0xffffffffu, c0, o);
    c1 += __shfl_xor_sync(0xffffffffu, c1, o);
  }
  if (lane == 0) {
    if (c0) atomicAdd(&lump[0], (unsigned long long)c0);
    if (c1) atomicAdd(&lump[1], (unsigned long long)c1);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long* gh = reinterpret_cast<unsigned long long*>(&s->hist[0][0]);
    const int a_lo = s->cand[0], p_lo = s->cand[2];
    if (lump[0]) atomicAdd(gh + (a_lo > 0 ? a_lo - 1 : 0), lump[0]);
    if (lump[1]) atomicAdd(gh + (p_lo > 0 ? p_lo - 1 : 0), lump[1]);
    s->guided_compact = 1;
  }
}

// digit-0 histogram of the compacted candidates (exact keys), added to the lumped counts
__global__ void __launch_bounds__(512)
select_hist0_compact_kernel(SelectState* __restrict__ s) {
  __shared__ unsigned h[kBins];
  if (s->phase0 != 1 || s->status != MICA_NORM_PENDING || s->comp_cap <= 0) return;
  const long long n = (long long)s->comp_count;
  if (n > s->comp_cap) {
    // overflow: this rank's candidate histogram is incomplete.  Word hist[1][0] (unused while digit 0 is being
    // found) carries the fact through the multi-GPU histogram sum, so EVERY rank's pick asks for the full pass
    if (blockIdx.x == 0 && threadIdx.x == 0)
      atomicAdd(reinterpret_cast<unsigned long long*>(&s->hist[1][0]), 1ull);
    return;
  }
  if ((long long)blockIdx.x * blockDim.x >= n) return;
  for (int i = threadIdx.x; i < kBins; i += blockDim.x) h[i] = 0;
  __syncthreads();
  const float* c = comp_buffer(s);
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long n_pad = (n + 31) & ~31LL;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_pad; i += stride) {
    const bool ok = i < n;
    const unsigned bin = ok ? (f32_key(nan_to_num_f32(c[i])) >> 21) : 0u;
    warp_hist_add(h, bin, ok);
  }
  __syncthreads();
  unsigned long long* gh = reinterpret_cast<unsigned long long*>(&s->hist[0][0]);
  for (int i = threadIdx.x; i < kBins; i += blockDim.x) {
    const unsigned v = h[i];
    if (v) atomicAdd(gh + i, (unsigned long long)v);
  }
}

// 1 block x kPickThreads threads, two bins per thread.  Finds the bucket holding `rank`.
constexpr int kPickThreads = kBins / 2;

// Finds, for up to three ranks at once, the bin holding the rank (one scan of the 2048 bins:
// warp-shuffle scan of the per-thread pair sums + a scan of the 32 warp totals).
__device__ void pick_buckets(const long long* hist, const long long* ranks, int n_ranks, int* bucket, long long* below,
                             long long* count, long long* scratch /* [kPickThreads] shared */) {
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const long long v0 = hist[2 * t], v1 = hist[2 * t + 1];
  long long incl = v0 + v1;
  for (int off = 1; off < 32; off <<= 1) {
    const long long up = __shfl_up_sync(0xffffffffu, incl, off);
    if (lane >= off) incl += up;
  }
  if (lane == 31) scratch[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    long long w = scratch[lane];
    for (int off = 1; off < 32; off <<= 1) {
      const long long up = __shfl_up_sync(0xffffffffu, w, off);
      if (lane >= off) w += up;
    }
    scratch[32 + lane] = w;          // inclusive totals of the warps
  }
  __syncthreads();
  const long long excl0 = incl - v0 - v1 + (warp ? scratch[32 + warp - 1] : 0), excl1 = excl0 + v0;
  for (int q = 0; q < n_ranks; ++q) {
    const long long rank = ranks[q];
    if (v0 > 0 && rank >= excl0 && rank < excl0 + v0) {
      bucket[q] = 2 * t;
      below[q] = excl0;
      count[q] = v0;
    }
    if (v1 > 0 && rank >= excl1 && rank < excl1 + v1) {
      bucket[q] = 2 * t + 1;
      below[q] = excl1;
      count[q] = v1;
    }
  }
  __syncthreads();
}

__device__ void pick_bucket(const long long* hist, long long rank, int* bucket, long long* below,
                            long long* count, long long* scratch) {
  pick_buckets(hist, &rank, 1, bucket, below, count, scratch);
}

// Host step t (0 .. MICA_SELECT_PASSES-1) -> what the pick does, gated on the device-side state so that
// a step whose pass did not run (e.g. the fallback round after a successful guided pass) is a no-op:
//   t = 0  sample histogram     -> candidate bins (phase0 0 -> 1)
//   t = 1  guided digit-0 pass  -> verify; commit digit 0 (phase0 1 -> 3, round 0 -> 1) or ask for the fallback (1 -> 2)
//   t = 2  full digit-0 pass    -> commit digit 0 (phase0 2 -> 3); no-op unless phase0 == 2
//   t = 3..6                    -> digit rounds 1..4 (median digits 1, 2; percentile digits 1, 2)
__global__ void __launch_bounds__(kPickThreads)
select_pick_kernel(SelectState* s, int t) {
  __shared__ long long scratch[kPickThreads];
  __shared__ int bucket[3];
  __shared__ long long below[3], count[3];
  __shared__ long long tail_count;
  __shared__ int verdict;
  if (s->status != MICA_NORM_PENDING) return;
  const int phase0 = s->phase0;
  int round;   // digit round to commit, or -1
  if (t == 0) {
    if (phase0 != 0) return;
    round = -1;
  } else if (t == 1) {
    if (phase0 != 1) return;
    round = 0;
  } else if (t == 2) {
    if (phase0 != 2) return;
    round = 0;
  } else {
    round = t - 2;
    if (phase0 != 3 || s->round != round || round >= kDigitRounds) return;
  }
  if (threadIdx.x < 3) {
    bucket[threadIdx.x] = -1;
    below[threadIdx.x] = 0;
    count[threadIdx.x] = 0;
  }
  if (threadIdx.x == 0) {
    tail_count = 0;
    verdict = 1;
  }
  __syncthreads();

  if (t == 0) {
    // ---- candidate bins from the sample: sample quantiles 0.48 / 0.52 bracket the median, 0.997 the tail
    long long part = s->hist[0][2 * threadIdx.x] + s->hist[0][2 * threadIdx.x + 1];
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if ((threadIdx.x & 31) == 0 && part) atomicAdd(reinterpret_cast<unsigned long long*>(&tail_count), (unsigned long long)part);
    __syncthreads();
    const long long ns = tail_count;
    long long ranks[3] = {(long long)(0.48 * (double)ns), (long long)(0.52 * (double)ns), (long long)(0.997 * (double)ns)};
    for (int q = 0; q < 3; ++q) ranks[q] = ranks[q] < ns ? ranks[q] : ns - 1;
    if (ns >= 4096) pick_buckets(s->hist[0], ranks, 3, bucket, below, count, scratch);
    __syncthreads();
    if (threadIdx.x == 0) {
      int a_lo = 0, a_hi = kBins - 1, p_lo = 0;   // tiny inputs: everything is histogrammed exactly
      if (ns >= 4096 && bucket[0] >= 0 && bucket[1] >= bucket[0] && bucket[2] >= 0) {
        a_lo = bucket[0];
        a_hi = bucket[1];
        p_lo = bucket[2] > a_hi ? bucket[2] : a_hi + 1;
      }
      s->cand[0] = a_lo;
      s->cand[1] = a_hi;
      s->cand[2] = p_lo;
      // float form of the bin edges; an edge that is not an ordinary float (bin 0, NaN patterns) becomes an
      // infinity so that the compare it feeds is never true and the voxel takes the exact (key) route
      auto edge = [](int bin, float fallback) {
        if (bin <= 0 || bin >= kBins) return fallback;
        const float f = key_f32((unsigned)bin << 21);
        return (f == f) ? f : fallback;
      };
      s->thr[0] = edge(a_lo, -__int_as_float(0x7f800000));        // below  <=> v <  thr[0]
      s->thr[1] = edge(a_hi + 1, __int_as_float(0x7f800000));     // between <=> thr[1] <= v < thr[2]
      s->thr[2] = edge(p_lo, __int_as_float(0x7f800000));
      s->phase0 = 1;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kBins; i += kPickThreads) {
      s->hist[0][i] = 0;
      s->hist[1][i] = 0;
    }
    return;
  }

  const int digit = round_digit(round);
  const bool same = (s->prefix[0] == s->prefix[1]);
  if (digit == 0 || same) {
    const long long ranks2[2] = {s->rank[0], s->rank[1]};
    pick_buckets(s->hist[0], ranks2, 2, bucket, below, count, scratch);
  } else {
    for (int q = 0; q < 2; ++q) pick_bucket(s->hist[q], s->rank[q], &bucket[q], &below[q], &count[q], scratch);
  }
  __syncthreads();
  if (t == 1) {
    // ---- verify the guided pass on its exact counts
    const int a_lo = s->cand[0], a_hi = s->cand[1], p_lo = s->cand[2];
    long long part = 0;
    for (int i = threadIdx.x; i < kBins; i += kPickThreads)
      if (i >= p_lo) part += s->hist[0][i];
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if ((threadIdx.x & 31) == 0 && part) atomicAdd(reinterpret_cast<unsigned long long*>(&tail_count), (unsigned long long)part);
    __syncthreads();
    if (threadIdx.x == 0) {
      // every percentile rank is >= 0.9995 N - 1 (at least half of the voxels are <= the median);
      // the margin covers the float32 virtual index of NumPy 2
      const long long need = (long long)(0.00052 * (double)s->n_total) + 64;
      // the compacting guided pass builds its histogram from the buffer: an overflow on ANY rank (counted in
      // hist[1][0], summed with the histograms) leaves it incomplete
      const bool hist_ok = s->hist[1][0] == 0;
      const bool med_ok = hist_ok && bucket[0] >= a_lo && bucket[0] <= a_hi && bucket[1] >= a_lo && bucket[1] <= a_hi;
      const bool tail_ok = (p_lo == 0) || tail_count >= need;
      if (!(med_ok && tail_ok)) {
        verdict = 0;
        s->phase0 = 2;      // run the full histogram (host step 2)
      }
      // the compact buffer is usable when the guided pass was accepted and nothing overflowed; in a
      // multi-GPU run every rank decides for its own buffer (the reduced histograms do not depend on it)
      s->comp_ok = (med_ok && tail_ok && s->comp_cap > 0 && s->comp_count <= (unsigned long long)s->comp_cap) ? 1 : 0;
    }
    __syncthreads();
    if (!verdict) {
      for (int i = threadIdx.x; i < kBins; i += kPickThreads) {
        s->hist[0][i] = 0;
        s->hist[1][i] = 0;
      }
      return;
    }
  }
  if (round == 0) {  // keep the digit-0 histogram for the percentile phase
    s->hist0[threadIdx.x] = s->hist[0][threadIdx.x];
    s->hist0[threadIdx.x + kPickThreads] = s->hist[0][threadIdx.x + kPickThreads];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (round == 0) s->phase0 = 3;
    for (int q = 0; q < 2; ++q) {
      int b = bucket[q] < 0 ? 0 : bucket[q];  // unreachable for consistent counts
      s->prefix[q] = digit == 0 ? (unsigned)b : ((s->prefix[q] << (digit == 1 ? 11 : 10)) | (unsigned)b);
      s->rank[q] -= below[q];
      s->below[q] += below[q];
      s->count_eq[q] = count[q];
    }
    if (round == 2) {
      // ---- median (np.median on float32): N odd -> s[N/2]; N even -> f32((a + b) / 2)
      float a = key_f32(s->prefix[0]), b = key_f32(s->prefix[1]);
      float med = (s->n_total & 1) ? b : __fdiv_rn(__fadd_rn(a, b), 2.0f);
      s->median = med;
      // count(x <= med): a and b are adjacent order statistics, a <= med <= b
      long long n_le = (med >= b) ? s->below[1] + s->count_eq[1] : s->below[0] + s->count_eq[0];
      s->n_le_med = n_le;
      long long npos = s->n_total - n_le;
      s->n_pos = npos;
      if (npos <= 0) {
        s->status = MICA_NORM_NO_POSITIVE;
        s->round = kDigitRounds;
      } else {
        // ---- np.percentile(pos, 99.9), float32 virtual index (NumPy >= 2)
        float q = __fdiv_rn(99.9f, 100.0f);
        float vi = __fmul_rn((float)(npos - 1), q);
        float prev = floorf(vi);
        float next = __fadd_rn(prev, 1.0f);
        long long lo, hi;
        if (vi >= (float)(npos - 1)) {
          lo = hi = npos - 1;
        } else {
          lo = (long long)prev;
          hi = (long long)next;
        }
        if (hi > npos - 1) hi = npos - 1;
        s->g = __fsub_rn(vi, prev);
        s->rank[0] = n_le + lo;
        s->rank[1] = n_le + hi;
        s->below[0] = s->below[1] = 0;
        s->prefix[0] = s->prefix[1] = 0;
      }
    } else if (round == 4) {
      float med = s->median;
      float a = __fsub_rn(key_f32(s->prefix[0]), med);
      float b = __fsub_rn(key_f32(s->prefix[1]), med);
      float g = s->g;
      float d = __fsub_rn(b, a);
      float r = __fadd_rn(a, __fmul_rn(d, g));
      if (g >= 0.5f) r = __fsub_rn(b, __fmul_rn(d, __fsub_rn(1.0f, g)));
      s->p = r;
      s->status = (r != 0.0f) ? MICA_NORM_OK : MICA_NORM_ZERO_PCTL;
    }
    if (s->round < kDigitRounds) s->round = round + 1;
  }
  __syncthreads();
  // clear the exchange histograms for the next round
  for (int i = threadIdx.x; i < kBins; i += kPickThreads) {
    s->hist[0][i] = 0;
    s->hist[1][i] = 0;
  }
  __syncthreads();
  if (round == 2 && s->status == MICA_NORM_PENDING) {
    // percentile digit 0 comes from the saved whole-array histogram (no extra data pass); after a
    // guided pass its bins below cand[2] are lumped, and the verification guarantees the ranks lie above
    __shared__ int b2[2];
    __shared__ long long bl2[2], c2[2];
    const long long ranks2[2] = {s->rank[0], s->rank[1]};
    pick_buckets(s->hist0, ranks2, 2, b2, bl2, c2, scratch);
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int q = 0; q < 2; ++q) {
        s->prefix[q] = (unsigned)b2[q];
        s->rank[q] -= bl2[q];
        s->below[q] = bl2[q];
        s->count_eq[q] = c2[q];
      }
    }
  }
}

// ---------------------------------------------------- histogram all-reduce over peer memory
// Multi-GPU order statistics need the SUM of every rank's histogram between `hist` and `pick`
// (5 times per map).  Through NCCL that is 5 small collectives with a stream hand-over each
// (measured: +1.7 ms per step on 8 GPUs).  Here the exchange is one single-CTA kernel over
// NVLink peer memory: every rank owns a small buffer that all peers have mapped (CUDA IPC);
// the kernel publishes the local histogram in the round's slot, raises a flag in every peer's
// buffer, waits for the peers' flags and sums their slots (P2P loads) into the local state.
// Slots alternate with the call epoch: a slot is rewritten two calls later, and a rank can only
// get there after every peer has signalled the call in between, i.e. finished reading.
constexpr int kPeerSlotWords = MICA_SELECT_HIST_WORDS;          // int64 words per slot
constexpr int kPeerMaxWorld = 64;
constexpr size_t kPeerBufferBytes = 2 * kPeerSlotWords * sizeof(long long) + kPeerMaxWorld * sizeof(int) * 2;

struct PeerBuffer {
  long long slot[2][kPeerSlotWords];
  int flag[kPeerMaxWorld];     // flag[p] = last epoch rank p has published
  int pad[kPeerMaxWorld];
};

__global__ void __launch_bounds__(1024)
select_peer_reduce_kernel(SelectState* __restrict__ s, PeerBuffer* const* __restrict__ peers, int rank, int world,
                          int parity, int epoch, int step, long long timeout_cycles) {
  __shared__ int ok;
  // a host step whose data pass did not run has nothing to exchange: the full-histogram fallback (step 2)
  // after an accepted guided pass, or anything once the status is final.  The state that decides this is
  // derived from the reduced histograms, so it is the same on every rank and all ranks skip together.
  if (s->status != MICA_NORM_PENDING || (step == 2 && s->phase0 != 2)) return;
  PeerBuffer* mine = peers[rank];
  long long* local = &s->hist[0][0];
  for (int i = threadIdx.x; i < kPeerSlotWords; i += blockDim.x) mine->slot[parity][i] = local[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x < world)     // raise my flag in every peer's buffer (and my own)
    st_release_sys(&peers[threadIdx.x]->flag[rank], epoch);
  if (threadIdx.x == 0) ok = 1;
  __syncthreads();
  if (threadIdx.x < world) {   // wait for peer threadIdx.x
    const int* f = &mine->flag[threadIdx.x];
    const long long t0 = clock64();
    while (ld_acquire_sys(f) - epoch < 0) {
      if (clock64() - t0 > timeout_cycles) {
        ok = 0;
        break;
      }
    }
  }
  __threadfence_system();
  __syncthreads();
  if (!ok) {                   // a peer never arrived: fail the normalisation instead of hanging the GPU
    if (threadIdx.x == 0) {
      s->status = MICA_NORM_PEER_TIMEOUT;
      s->round = kDigitRounds;
    }
    return;
  }
  // sum the peers' slots: all loads of a thread (4 words x up to 4 peers) are issued before the first
  // is consumed -- one NVLink round trip per group of 4 peers instead of one per load
  __shared__ const long long* base[kPeerMaxWorld];
  if (threadIdx.x < world) base[threadIdx.x] = peers[threadIdx.x]->slot[parity];
  __syncthreads();
  constexpr int kPer = kPeerSlotWords / 1024;
  long long sum[kPer];
#pragma unroll
  for (int k = 0; k < kPer; ++k) sum[k] = 0;
  for (int p0 = 0; p0 < world; p0 += 4) {
    long long v[kPer][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const long long* b = base[p0 + j < world ? p0 + j : rank];
#pragma unroll
      for (int k = 0; k < kPer; ++k)
        asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v[k][j]) : "l"(b + threadIdx.x + k * 1024));
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (p0 + j < world) {
#pragma unroll
        for (int k = 0; k < kPer; ++k) sum[k] += v[k][j];
      }
  }
#pragma unroll
  for (int k = 0; k < kPer; ++k) local[threadIdx.x + k * 1024] = sum[k];
}

__global__ void select_init_kernel(SelectState* s, long long n_total) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < kBins) {
    s->hist[0][t] = 0;
    s->hist[1][t] = 0;
    s->hist0[t] = 0;
  }
  if (t == 0) {
    s->n_total = n_total;
    // np.median: order statistics (N-1)/2 and N/2 (equal when N is odd)
    s->rank[0] = (n_total - 1) / 2;
    s->rank[1] = n_total / 2;
    s->below[0] = s->below[1] = 0;
    s->count_eq[0] = s->count_eq[1] = 0;
    s->prefix[0] = s->prefix[1] = 0;
    s->round = 0;
    s->phase0 = 0;
    s->cand[0] = 0;
    s->cand[1] = kBins - 1;
    s->cand[2] = 0;
    s->comp_ok = 0;
    s->comp_count = 0ull;
    s->guided_compact = 0;
    s->thr[0] = s->thr[1] = s->thr[2] = 0.f;
    s->status = n_total > 0 ? MICA_NORM_PENDING : MICA_NORM_NO_POSITIVE;
    s->n_le_med = 0;
    s->n_pos = 0;
    s->median = 0.f;
    s->p = 0.f;
    s->g = 0.f;
  }
}

// y = ((m < p) * m + (m >= p) * p) / p,  m = (v > med) * (v - med): every product and
// sum is a separate IEEE float32 operation, exactly as NumPy evaluates the expression
__device__ __forceinline__ float normalize_one(float x, float med, float p) {
  float v = nan_to_num_f32(x);
  float m = __fmul_rn((v > med) ? 1.0f : 0.0f, __fsub_rn(v, med));
  float r = __fadd_rn(__fmul_rn((m < p) ? 1.0f : 0.0f, m), __fmul_rn((m >= p) ? 1.0f : 0.0f, p));
  return __fdiv_rn(r, p);
}

// The same value with a handful of instructions for ordinary inputs.  Walking the NumPy expression:
//   v <= med            -> m = 0 * (v - med) = +-0, r = +-0 + 0 = +0, y = +0
//   v - med >= p        -> r = 0 * m + p = p, y = p / p = 1
//   0 < v - med < p     -> r = m, y = RN(m / p): q0 = RN(m * RN(1/p)), rem = m - q0 * p (exact in an
//                          fma), y = RN(q0 + rem * RN(1/p)) is the correctly rounded quotient
//                          (Markstein's division-by-reciprocal step) as long as nothing underflows.
// Huge / non-finite inputs (v - med could overflow, nan_to_num applies), quotients near the
// denormal range and a divisor whose significand is all ones take normalize_one().
__device__ __forceinline__ float normalize_fast(float x, float med, float p, float rcp, bool rcp_ok) {
  const unsigned a = __float_as_uint(x) & 0x7fffffffu;
  if (a >= 0x7e000000u || !rcp_ok) return normalize_one(x, med, p);
  if (!(x > med)) return 0.0f;
  const float d = __fsub_rn(x, med);
  if (d >= p) return 1.0f;
  const float q0 = __fmul_rn(d, rcp);
  if (q0 < 1e-30f) return __fdiv_rn(d, p);
  const float rem = __fmaf_rn(-q0, p, d);
  return __fmaf_rn(rem, rcp, q0);
}

template <bool FAST>
__global__ void __launch_bounds__(256)
normalize_apply_kernel(const float* __restrict__ x, float* __restrict__ y, long long n,
                       const SelectState* __restrict__ s) {
  if (s->status != MICA_NORM_OK) return;
  const float med = s->median, p = s->p;
  const float rcp = __fdiv_rn(1.0f, p);
  // the reciprocal step needs finite, normal operands and a divisor that is not 2 - ulp
  const unsigned pu = __float_as_uint(p), ru = __float_as_uint(rcp);
  const bool rcp_ok = FAST && p > 1e-30f && p < 1e30f && (pu & 0x7fffffu) != 0x7fffffu && (ru & 0x7f800000u) != 0u &&
                      fabsf(med) < 1e30f;
  const bool vec = ((((uintptr_t)x) | ((uintptr_t)y)) & 15) == 0;
  const long long n4 = vec ? (n >> 2) : 0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  float4* y4 = reinterpret_cast<float4*>(y);
  for (long long i = tid; i < n4; i += stride) {
    float4 v = x4[i];
    v.x = normalize_fast(v.x, med, p, rcp, rcp_ok);
    v.y = normalize_fast(v.y, med, p, rcp, rcp_ok);
    v.z = normalize_fast(v.z, med, p, rcp, rcp_ok);
    v.w = normalize_fast(v.w, med, p, rcp, rcp_ok);
    y4[i] = v;
  }
  for (long long i = n4 * 4 + tid; i < n; i += stride) y[i] = normalize_fast(x[i], med, p, rcp, rcp_ok);
}

}  // namespace mica

using namespace mica;

extern "C" size_t mica_select_workspace_bytes(void) { return sizeof(SelectState) + 256; }

// capacity of the compact buffer for n_local voxels per rank: the candidate bins hold ~4 % of a density map
// (sample quantiles 0.48-0.52 and the top 0.3 %) plus whatever shares their digit-0 bins; 1/8 of the map
// leaves room for coarse bins, and an overflow only means the digit passes stream the map as before
static long long compact_capacity(int64_t n_local) {
  if (n_local < (1 << 22)) return 0;              // small inputs: the full passes cost microseconds
  return (long long)(n_local / 8 + 4095) / 4096 * 4096;
}

extern "C" size_t mica_select_workspace_bytes_for(int64_t n_local) {
  return mica_select_workspace_bytes() + 256 + (size_t)compact_capacity(n_local) * sizeof(float);
}

__global__ void select_set_compact_kernel(SelectState* s, long long cap) { s->comp_cap = cap; }

// Tell a (zero-initialised) workspace how large it is: everything beyond the state becomes the compact
// buffer.  Once per allocation; mica_select_init keeps the setting.
extern "C" int mica_select_set_compact(void* workspace, size_t workspace_bytes, mica_stream_t stream) {
  MICA_REQUIRE(workspace, "null workspace");
  MICA_REQUIRE(workspace_bytes >= mica_select_workspace_bytes(), "workspace smaller than the select state");
  SelectState* s = (SelectState*)(((uintptr_t)workspace + 255) / 256 * 256);
  const uintptr_t end = (uintptr_t)workspace + workspace_bytes;
  const uintptr_t buf = (uintptr_t)comp_buffer(s);
  const long long cap = end > buf ? (long long)((end - buf) / sizeof(float)) : 0;
  select_set_compact_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(s, cap);
  MICA_LAUNCH_CHECK("select_set_compact_kernel");
  return MICA_OK;
}

static SelectState* state_of(const void* ws) { return (SelectState*)(((uintptr_t)ws + 255) / 256 * 256); }

extern "C" int64_t* mica_select_hist_ptr(void* workspace) {
  return workspace ? (int64_t*)&state_of(workspace)->hist[0][0] : nullptr;
}

extern "C" int mica_select_init(void* workspace, int64_t n_total, mica_stream_t stream) {
  MICA_REQUIRE(workspace, "null workspace");
  MICA_REQUIRE(n_total >= 0, "negative n");
  select_init_kernel<<<kBins / 256, 256, 0, (cudaStream_t)stream>>>(state_of(workspace), n_total);
  MICA_LAUNCH_CHECK("select_init_kernel");
  return MICA_OK;
}

// One data pass of host step t (see select_pick_kernel).  Every kernel re-checks the device-side state and
// returns at once when the step is not due (the fallback step 2 after a successful guided pass), so
// the host never reads the state back between steps.
extern "C" int mica_select_hist(const float* x, int64_t n_local, void* workspace, int step, mica_stream_t stream) {
  MICA_REQUIRE(workspace && (x || n_local == 0), "null pointer");
  MICA_REQUIRE(n_local >= 0, "negative n");
  MICA_REQUIRE(step >= 0 && step < MICA_SELECT_PASSES, "select step %d out of range", step);
  if (n_local == 0) return MICA_OK;
  cudaStream_t st = (cudaStream_t)stream;
  SelectState* s = state_of(workspace);
  const int64_t want = ceil_div64(ceil_div64(n_local, 4), 512);
  const int grid = (int)(want < (int64_t)kNumSMs * 4 ? want : (int64_t)kNumSMs * 4);
  if (step == 0) {
    const int64_t ws = ceil_div64(ceil_div64(n_local, 4 * kSampleStride), 512);
    select_sample_kernel<<<(unsigned)(ws < kNumSMs ? (ws > 0 ? ws : 1) : kNumSMs), 512, 0, st>>>(x, n_local, s);
    MICA_LAUNCH_CHECK("select_sample_kernel");
  } else if (step == 1) {
    // which form runs is decided on the device (whether the workspace has a compact buffer): the other
    // kernels return at once.  Small inputs never have one, so they only get the histogramming form.
    const int compacting = !getenv("MICA_SELECT_OLD_GUIDED");
    if (compacting && n_local >= (1 << 22)) {
      select_guided_compact_kernel<<<grid, 512, 0, st>>>(x, n_local, s);
      MICA_LAUNCH_CHECK("select_guided_compact_kernel");
      select_hist0_compact_kernel<<<kNumSMs * 2, 512, 0, st>>>(s);
      MICA_LAUNCH_CHECK("select_hist0_compact_kernel");
    }
    select_hist0_guided_kernel<<<grid, 512, 0, st>>>(x, n_local, s, compacting);
    MICA_LAUNCH_CHECK("select_hist0_guided_kernel");
  } else if (step == 2) {
    // full digit-0 histogram: at most kHist0MaxPerWarp elements per warp (16-bit counters), >= two CTAs per SM
    int64_t grid0 = ceil_div64(n_local, kHist0Warps * kHist0MaxPerWarp);
    if (grid0 < 2 * kNumSMs) grid0 = want < 2 * kNumSMs ? want : 2 * kNumSMs;
    const size_t smem0 = (size_t)kHist0Warps * kBins * sizeof(unsigned short);
    // per device/context attribute: set it on every call (a process-wide flag would leave the other GPUs unset)
    MICA_CUDA(cudaFuncSetAttribute(select_hist0_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem0));
    select_hist0_kernel<<<(unsigned)grid0, 512, smem0, st>>>(x, n_local, s);
    MICA_LAUNCH_CHECK("select_hist0_kernel");
  } else {
    select_hist_kernel<<<grid, 512, 0, st>>>(x, n_local, s);
    MICA_LAUNCH_CHECK("select_hist_kernel");
  }
  return MICA_OK;
}

static int g_select_force_fallback;
__global__ void select_spoil_candidates_kernel(SelectState* s);

extern "C" int mica_select_pick(void* workspace, int step, mica_stream_t stream) {
  MICA_REQUIRE(workspace, "null workspace");
  MICA_REQUIRE(step >= 0 && step < MICA_SELECT_PASSES, "select step %d out of range", step);
  select_pick_kernel<<<1, kPickThreads, 0, (cudaStream_t)stream>>>(state_of(workspace), step);
  MICA_LAUNCH_CHECK("select_pick_kernel");
  if (step == 0 && g_select_force_fallback) {
    select_spoil_candidates_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(state_of(workspace));
    MICA_LAUNCH_CHECK("select_spoil_candidates_kernel");
  }
  return MICA_OK;
}

// test hook: 1 forces the guided pass to be rejected (exercises the full-histogram fallback)
__global__ void select_spoil_candidates_kernel(SelectState* s) {
  if (s->phase0 == 1) {   // candidates that cannot contain the median
    s->cand[0] = kBins - 1;
    s->cand[1] = kBins - 1;
    s->cand[2] = kBins - 1;
  }
}
extern "C" int mica_select_force_fallback(int on) {
  const int was = g_select_force_fallback;
  g_select_force_fallback = on ? 1 : 0;
  return was;
}

// ---- peer buffers (CUDA IPC) and the fused exchange
extern "C" size_t mica_peer_buffer_bytes(void) { return kPeerBufferBytes; }

extern "C" int mica_peer_alloc(void** dev_ptr, void* ipc_handle_out) {
  MICA_REQUIRE(dev_ptr, "null pointer");
  void* p = nullptr;
  MICA_CUDA(cudaMalloc(&p, kPeerBufferBytes));
  MICA_CUDA(cudaMemset(p, 0, kPeerBufferBytes));
  if (ipc_handle_out) {
    cudaIpcMemHandle_t h;
    MICA_CUDA(cudaIpcGetMemHandle(&h, p));
    memcpy(ipc_handle_out, &h, sizeof(h));
  }
  *dev_ptr = p;
  return MICA_OK;
}

extern "C" int mica_peer_open(const void* ipc_handle, void** dev_ptr) {
  MICA_REQUIRE(ipc_handle && dev_ptr, "null pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, ipc_handle, sizeof(h));
  MICA_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return MICA_OK;
}

extern "C" int mica_peer_enable(int device, int peer_device) {
  MICA_REQUIRE(device >= 0 && peer_device >= 0, "bad device pair (%d, %d)", device, peer_device);
  if (device == peer_device) return MICA_OK;
  int can = 0;
  MICA_CUDA(cudaDeviceCanAccessPeer(&can, device, peer_device));
  MICA_REQUIRE(can, "device %d cannot access the memory of device %d (no peer path between them)", device,
               peer_device);
  int prev = 0;
  MICA_CUDA(cudaGetDevice(&prev));
  MICA_CUDA(cudaSetDevice(device));
  cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) {   // e.g. enabled by PyTorch for a copy: not an error, and
    cudaGetLastError();                           // must not be reported by a later launch check
    e = cudaSuccess;
  }
  const cudaError_t restore = cudaSetDevice(prev);
  MICA_CUDA(e);
  MICA_CUDA(restore);
  return MICA_OK;
}

extern "C" int mica_peer_close(void* dev_ptr) {
  if (dev_ptr) MICA_CUDA(cudaIpcCloseMemHandle(dev_ptr));
  return MICA_OK;
}

extern "C" int mica_peer_free(void* dev_ptr) {
  if (dev_ptr) MICA_CUDA(cudaFree(dev_ptr));
  return MICA_OK;
}

extern "C" int mica_select_peer_reduce(void* workspace, void* const* peer_bufs, int rank, int world, int parity,
                                       int epoch, int step, mica_stream_t stream) {
  MICA_REQUIRE(workspace && peer_bufs, "null pointer");
  MICA_REQUIRE(world >= 1 && world <= kPeerMaxWorld && rank >= 0 && rank < world, "bad rank/world");
  MICA_REQUIRE(parity == 0 || parity == 1, "parity must be 0 or 1");
  const long long timeout_cycles = mica::peer_timeout_cycles();
  select_peer_reduce_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(
      state_of(workspace), reinterpret_cast<PeerBuffer* const*>(peer_bufs), rank, world, parity, epoch, step,
      timeout_cycles);
  MICA_LAUNCH_CHECK("select_peer_reduce_kernel");
  return MICA_OK;
}

extern "C" int mica_order_stats_f32(const float* x, int64_t n, void* workspace, mica_stream_t stream) {
  int rc = mica_select_init(workspace, n, stream);
  for (int t = 0; t < MICA_SELECT_PASSES && rc == MICA_OK; ++t) {
    rc = mica_select_hist(x, n, workspace, t, stream);
    if (rc == MICA_OK) rc = mica_select_pick(workspace, t, stream);
  }
  return rc;
}

// [n_le_med i64][n_pos i64][median f32][p f32][g f32][status i32]
struct SelectResultRecord {
  long long n_le_med, n_pos;
  float median, p, g;
  int status;
};
static_assert(sizeof(SelectResultRecord) == MICA_SELECT_RESULT_BYTES, "result record size");

extern "C" int mica_select_result_async(const void* workspace, void* host_record, mica_stream_t stream) {
  MICA_REQUIRE(workspace && host_record, "null pointer");
  const SelectState* s = state_of(workspace);
  cudaStream_t st = (cudaStream_t)stream;
  SelectResultRecord* r = (SelectResultRecord*)host_record;
  MICA_CUDA(cudaMemcpyAsync(r, &s->n_le_med, 28, cudaMemcpyDeviceToHost, st));
  MICA_CUDA(cudaMemcpyAsync(&r->status, &s->status, sizeof(int), cudaMemcpyDeviceToHost, st));
  return MICA_OK;
}

extern "C" int mica_select_result(const void* workspace, float* median, float* p999, int64_t* n_pos, int* norm_status,
                                  mica_stream_t stream) {
  SelectResultRecord r;
  int rc = mica_select_result_async(workspace, &r, stream);
  if (rc) return rc;
  MICA_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  if (median) *median = r.median;
  if (p999) *p999 = r.p;
  if (n_pos) *n_pos = r.n_pos;
  if (norm_status) *norm_status = r.status;
  return MICA_OK;
}

// test / diagnostics hook: {comp_ok, comp_count, comp_cap} of a workspace (synchronises the stream)
extern "C" int mica_select_compact_info(const void* workspace, int64_t out[3], mica_stream_t stream) {
  MICA_REQUIRE(workspace && out, "null pointer");
  const SelectState* s = state_of(workspace);
  int ok = 0;
  long long cap = 0;
  unsigned long long cnt = 0;
  cudaStream_t st = (cudaStream_t)stream;
  MICA_CUDA(cudaMemcpyAsync(&ok, &s->comp_ok, sizeof(int), cudaMemcpyDeviceToHost, st));
  MICA_CUDA(cudaMemcpyAsync(&cap, &s->comp_cap, sizeof(cap), cudaMemcpyDeviceToHost, st));
  MICA_CUDA(cudaMemcpyAsync(&cnt, &s->comp_count, sizeof(cnt), cudaMemcpyDeviceToHost, st));
  MICA_CUDA(cudaStreamSynchronize(st));
  out[0] = ok;
  out[1] = (int64_t)cnt;
  out[2] = cap;
  return MICA_OK;
}

static int g_normalize_reference_arith = 0;

// test hook: on != 0 evaluates the NumPy expression operation by operation for every voxel
// (normalize_one) instead of the short equivalent path; returns the previous setting
extern "C" int mica_normalize_force_reference_arith(int on) {
  const int was = g_normalize_reference_arith;
  g_normalize_reference_arith = on ? 1 : 0;
  return was;
}

// test hook: stores median / percentile into a select workspace as if mica_order_stats_f32 had found them
__global__ void select_set_thresholds_kernel(SelectState* s, float median, float p) {
  s->median = median;
  s->p = p;
  s->status = MICA_NORM_OK;
  s->round = kDigitRounds;
  s->phase0 = 3;
}
extern "C" int mica_select_set_thresholds(void* workspace, float median, float p, mica_stream_t stream) {
  MICA_REQUIRE(workspace, "null workspace");
  select_set_thresholds_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(state_of(workspace), median, p);
  MICA_LAUNCH_CHECK("select_set_thresholds_kernel");
  return MICA_OK;
}

extern "C" int mica_normalize_apply_f32(const float* x, float* y, int64_t n, const void* workspace, mica_stream_t stream) {
  MICA_REQUIRE(x && y && workspace, "null pointer");
  if (n <= 0) return MICA_OK;
  int64_t want = ceil_div64(ceil_div64(n, 4), 256);
  int grid = (int)(want < (int64_t)kNumSMs * 8 ? want : (int64_t)kNumSMs * 8);
  if (g_normalize_reference_arith)
    normalize_apply_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, n, state_of(workspace));
  else
    normalize_apply_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, n, state_of(workspace));
  MICA_LAUNCH_CHECK("normalize_apply_kernel");
  return MICA_OK;
}
