// R7/R8: fused softmax / argmax post-processing and volume stitching.
//
// Replaces, in one pass over the model's logits, the block at utils/predict.py:342-349
// (reference root)
//     bb = softmax(cat(bb[:, :1], bb[:, 2:]))[:, 2]        (3-way, class 1 dropped)
//     ca = softmax(cat(ca[:, :1], ca[:, 2:]))[:, 2]
//     aa_scores = softmax(aa[:, 1:]); aa_pred = argmax(aa_scores)
// the per-cube .cpu().numpy() + np.savez round trip (:353-369) and reconstruct_volume
// (:439-512): vol[i:i+di, j:j+dj, k:k+dk] = cube[pad:pad+di, pad:pad+dj, pad:pad+dk].
// Only the disjoint cores are read (the halo predictions are discarded by the
// reference too), so each output voxel is written exactly once: no atomics, no weights.
// One thread per core voxel, the cube's fastest axis across the warp: 26 coalesced
// channel reads (stride W^3) and 23 coalesced writes per voxel.
#include "common.cuh"

namespace mica {

constexpr int kStitchMaxWorld = 64;

// multi-GPU ownership of the output along cube axis 0 (x): rank r owns planes [bounds[r], bounds[r+1]) and
// holds them as 23 channels of [bounds[r+1]-bounds[r], Y, Z] floats at base[r] (peer memory, mapped here):
// [backbone | carbon_alpha | amino_acid_prediction | amino_acid_probability x 20]
struct StitchOwners {
  float* const* base;
  int world;
  int bounds[kStitchMaxWorld + 1];
};

struct StitchParams {
  const void* bb;  // logits of the kernels' element type T (float or __nv_bfloat16)
  const void* ca;
  const void* aa;
  const int32_t* ijk;
  int X, Y, Z;
  int org[3], ext[3];
  int S, pad, W;
  float* bb_vol;
  float* ca_vol;
  float* aa_prob_vol;
  float* aa_pred_vol;
};

// exp(x) for x <= 0 on the SFU: ex2.approx is good to ~2 ulp, far inside the 1e-5 bar on
// probabilities; the kernel is issue-limited otherwise (libm expf + IEEE division cost ~20
// instructions per channel, 29 channels per voxel)
__device__ __forceinline__ float exp_neg(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
  return y;
}

__device__ __forceinline__ float softmax3_last(float l0, float l1, float l2) {
  float m = fmaxf(l0, fmaxf(l1, l2));
  float e0 = exp_neg(l0 - m), e1 = exp_neg(l1 - m), e2 = exp_neg(l2 - m);
  return e2 * __frcp_rn((e0 + e1) + e2);
}

// grid = (B, S [core plane a] * ceil(S*S / 256)), block = 256: one core voxel per thread, so a batch
// is thousands of small CTAs and the last wave over the 148 SMs is short.  The cube is the FASTEST
// grid index: cubes that follow each other in the batch are neighbours along the volume's fastest
// axis (k), so CTAs resident together write adjacent 128-byte runs of the same output rows
// PEER: the destination of a core plane is the volume block of the rank that owns its x plane -- the
// local one or a peer's, written over NVLink (coalesced 128-byte runs, fire and forget).  The owner is
// uniform per CTA (a CTA handles one core plane), so the lookup costs nothing per voxel.
// T: the logits' element type, float or __nv_bfloat16 -- bf16 is widened exactly on load, the rest is the same
template <bool PEER, typename T>
__global__ void __launch_bounds__(256)
postproc_stitch_kernel(StitchParams P, StitchOwners O) {
  const int S = P.S, W = P.W;
  const int chunks = (S * S + 255) >> 8;
  const int a = blockIdx.y / chunks, b = blockIdx.x;
  const int i = P.ijk[3 * b + 0], j = P.ijk[3 * b + 1], k = P.ijk[3 * b + 2];
  const int gx = i + a;
  if (gx >= P.X || gx < P.org[0] || gx >= P.org[0] + P.ext[0]) return;
  const int64_t W3 = (int64_t)W * W * W;
  const T* bb = static_cast<const T*>(P.bb) + (int64_t)b * 4 * W3;
  const T* ca = static_cast<const T*>(P.ca) + (int64_t)b * 4 * W3;
  const T* aa = static_cast<const T*>(P.aa) + (int64_t)b * 21 * W3;
  int64_t vol_n = (int64_t)P.ext[0] * P.ext[1] * P.ext[2];
  int x_org = P.org[0];
  if (PEER) {
    int r = 0;
    while (r + 1 < O.world && gx >= O.bounds[r + 1]) ++r;
    x_org = O.bounds[r];
    vol_n = (int64_t)(O.bounds[r + 1] - O.bounds[r]) * P.ext[1] * P.ext[2];
    float* base = O.base[r];
    P.bb_vol = base;
    P.ca_vol = base + vol_n;
    P.aa_pred_vol = base + 2 * vol_n;
    P.aa_prob_vol = base + 3 * vol_n;
  }
  {
    const int e = (blockIdx.y - a * chunks) * 256 + threadIdx.x;
    if (e >= S * S) return;
    const int bj = e / S, c = e - bj * S;
    const int gy = j + bj, gz = k + c;
    if (gy >= P.Y || gz >= P.Z) return;
    const int ly = gy - P.org[1], lz = gz - P.org[2];
    if ((unsigned)ly >= (unsigned)P.ext[1] || (unsigned)lz >= (unsigned)P.ext[2]) return;
    const int64_t src = ((int64_t)(a + P.pad) * W + (bj + P.pad)) * W + (c + P.pad);
    const int64_t dst = ((int64_t)(gx - x_org) * P.ext[1] + ly) * P.ext[2] + lz;
    // issue every load before the math: 26 independent requests in flight per thread
    const float b0 = ld_stream_core_el(bb + src), b2 = ld_stream_core_el(bb + 2 * W3 + src), b3 = ld_stream_core_el(bb + 3 * W3 + src);
    const float c0 = ld_stream_core_el(ca + src), c2 = ld_stream_core_el(ca + 2 * W3 + src), c3 = ld_stream_core_el(ca + 3 * W3 + src);
    float l[20];
#pragma unroll
    for (int t = 0; t < 20; ++t) l[t] = ld_stream_core_el(aa + (int64_t)(t + 1) * W3 + src);
    st_stream(P.bb_vol + dst, softmax3_last(b0, b2, b3));
    st_stream(P.ca_vol + dst, softmax3_last(c0, c2, c3));
    // argmax on the logits (softmax is monotone); first maximum wins, as torch.max
    float m = l[0];
    int arg = 0;
#pragma unroll
    for (int t = 1; t < 20; ++t) {
      if (l[t] > m) {
        m = l[t];
        arg = t;
      }
    }
    float s = 0.f;
#pragma unroll
    for (int t = 0; t < 20; ++t) {
      l[t] = exp_neg(l[t] - m);
      s += l[t];
    }
    const float r = __frcp_rn(s);
#pragma unroll
    for (int t = 0; t < 20; ++t) st_stream(P.aa_prob_vol + (int64_t)t * vol_n + dst, l[t] * r);
    st_stream(P.aa_pred_vol + dst, (float)arg);
  }
}

// ---------------------------------------------------------------- overlap-weighted stitching (north_star variant)
// NOT the reference's arithmetic: the reference pastes disjoint cores (utils/predict.py:494-501, DESIGN.md D2).
// BASELINE.json's north_star words the stage as "overlap-averaged stitching ... accumulate prediction plus
// weight volumes in one pass"; this is that mode, offered next to the reference one.
//
// The result does not depend on the order of the contributions (batch size, launch, GPU, partition):
//  - the normaliser comes from the cube lattice, not from an accumulated weight volume.  The weight sum at a voxel
//    is separable, Wx[x] Wy[y] Wz[z]; the host computes the three 1-D tables in float64 from the FULL lattice and
//    passes their reciprocals N (0 where the sum is 0);
//  - every window voxel adds q = rint(p * (((w1[a] w1[b]) w1[c]) ((Nx Ny) Nz) 2^31)) to a uint32 sum
//    (red.global.add.u32), p the probability the paste would store.  Integer addition is associative, so the sums
//    are the same bits whatever the order.  A voxel's sum is at most 2^31 + n_cover / 2 (no overflow); its error
//    against the exact weighted mean is at most n_cover 2^-32;
//  - overlap_finalize_kernel turns each sum s into float(s) 2^-31 in place and takes the arg-max of the 20 integer
//    amino-acid sums (first maximum wins).
// The accumulator is the 23-channel block of StitchedVolumes.from_block, read as uint32:
// [backbone | carbon_alpha | amino_acid_prediction (unused until finalize) | amino_acid_probability x 20].
// The 1-on-the-core window is not run here: the fixed-point grid would round every probability below 2^-8, so
// callers route it to the reference paste (postproc_stitch), which it equals by definition.
constexpr int kOverlapMaxW = 128;
struct OverlapWindow {
  float w1[kOverlapMaxW];
};

struct OverlapParams {
  const void* bb;  // logits of the kernels' element type T (float or __nv_bfloat16)
  const void* ca;
  const void* aa;
  const int32_t* ijk;
  int X, Y, Z, pad, W;
  const double* norm;  // [X | Y | Z] reciprocals of the lattice weight sums
  uint32_t* block;     // local destination: 23 channels of [X, Y, Z]
  int obase, os[3];    // logits of window voxel v at obase + v . os (Orientation; W^2, W, 1 for orientation 0)
};

// owners of the output along one cube axis (0 = x, 2 = k): rank r holds planes [bounds[r], bounds[r+1]) of that
// axis as the 23-channel block at base[r] (local or peer memory), the other two axes whole
struct OverlapOwners {
  uint32_t* const* base;
  int axis;
  int world;
  int bounds[kStitchMaxWorld + 1];
};

// The one rounding recipe of a contribution: every product correctly rounded in float64, in this order, so that
// every instantiation (local, peer) and every partition produces the same bits whatever contraction the compiler
// would otherwise choose.  The scale by 2^31 is exact.
__device__ __forceinline__ double overlap_scale(float wa, float wb, float wc, double nx, double ny, double nz) {
  const double w = __dmul_rn(__dmul_rn((double)wa, (double)wb), (double)wc);
  const double n = __dmul_rn(__dmul_rn(nx, ny), nz);
  return __dmul_rn(__dmul_rn(w, n), 2147483648.0);
}
__device__ __forceinline__ uint32_t overlap_fixed(float p, double scale) {
  return __double2uint_rn(__dmul_rn((double)p, scale));
}
__device__ __forceinline__ void red_add_u32(uint32_t* p, uint32_t v) {
  if (v) asm volatile("red.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// where the contributions of window voxel (gx, gy, gz) go: the local block, or (PEER) the block of the rank that
// owns its plane along O.axis.  Returns the channel-0 address; channels are vol_n apart.
template <bool PEER>
__device__ __forceinline__ uint32_t* overlap_dest(const OverlapParams& P, const OverlapOwners& O, int gx, int gy,
                                                  int gz, int64_t* vol_n) {
  if (!PEER) {
    *vol_n = (int64_t)P.X * P.Y * P.Z;
    return P.block + ((int64_t)gx * P.Y + gy) * P.Z + gz;
  }
  const int g = O.axis == 0 ? gx : gz;
  int r = 0;
  while (r + 1 < O.world && g >= O.bounds[r + 1]) ++r;
  const int lo = O.bounds[r], n = O.bounds[r + 1] - lo;
  if (O.axis == 0) {
    *vol_n = (int64_t)n * P.Y * P.Z;
    return O.base[r] + ((int64_t)(gx - lo) * P.Y + gy) * P.Z + gz;
  }
  *vol_n = (int64_t)P.X * P.Y * n;
  return O.base[r] + ((int64_t)gx * P.Y + gy) * n + (gz - lo);
}

// the 22 contributions (backbone, carbon_alpha, amino_acid_probability x 20) of the logits at offset src of cube
// b's [4 | 4 | 21] x W^3 channels: the softmax of the paste (postproc_stitch_kernel), maximum taken the same way.
// T: the logits' element type (bf16 widened exactly on load)
constexpr int kOverlapQ = 22;
template <typename T>
__device__ __forceinline__ void overlap_contrib(const OverlapParams& P, int b, int64_t src, double scale,
                                                uint32_t q[kOverlapQ]) {
  const int64_t W3 = (int64_t)P.W * P.W * P.W;
  const T* bb = static_cast<const T*>(P.bb) + (int64_t)b * 4 * W3;
  const T* ca = static_cast<const T*>(P.ca) + (int64_t)b * 4 * W3;
  const T* aa = static_cast<const T*>(P.aa) + (int64_t)b * 21 * W3;
  const float b0 = ld_stream_el(bb + src), b2 = ld_stream_el(bb + 2 * W3 + src), b3 = ld_stream_el(bb + 3 * W3 + src);
  const float c0 = ld_stream_el(ca + src), c2 = ld_stream_el(ca + 2 * W3 + src), c3 = ld_stream_el(ca + 3 * W3 + src);
  float l[20];
#pragma unroll
  for (int t = 0; t < 20; ++t) l[t] = ld_stream_el(aa + (int64_t)(t + 1) * W3 + src);
  q[0] = overlap_fixed(softmax3_last(b0, b2, b3), scale);
  q[1] = overlap_fixed(softmax3_last(c0, c2, c3), scale);
  float m = l[0];
#pragma unroll
  for (int t = 1; t < 20; ++t) {
    if (l[t] > m) m = l[t];
  }
  float s = 0.f;
#pragma unroll
  for (int t = 0; t < 20; ++t) {
    l[t] = exp_neg(l[t] - m);
    s += l[t];
  }
  const float rs = __frcp_rn(s);
#pragma unroll
  for (int t = 0; t < 20; ++t) q[2 + t] = overlap_fixed(l[t] * rs, scale);
}

// block channel of contribution ch: [backbone | carbon_alpha | (prediction) | probability x 20]
__device__ __forceinline__ int64_t overlap_channel(int ch, int64_t vol_n) { return (ch < 2 ? ch : ch + 1) * vol_n; }

// grid = (B, W [window plane a] * ceil(W*W / 256)), block = 256: one window voxel per thread, lanes along window
// axis 2.  The logits are those of the window in orientation P.orient (test-time augmentation; orientation 0 = the
// window itself): window voxel v reads them at the oriented offset obase + v . os, which for the orientations
// run here (|os[2]| == 1: the fastest axis stays, possibly reversed) keeps the reads coalesced.
// PEER: each contribution goes to the block of the rank that owns its plane along O.axis, locally or over NVLink
template <bool PEER, typename T>
__global__ void __launch_bounds__(256)
overlap_accumulate_kernel(OverlapParams P, OverlapWindow Wn, OverlapOwners O) {
  const int W = P.W;
  const int chunks = (W * W + 255) >> 8;
  const int a = blockIdx.y / chunks, b = blockIdx.x;
  const float wa = Wn.w1[a];
  if (wa == 0.f) return;
  const int i = P.ijk[3 * b + 0], j = P.ijk[3 * b + 1], k = P.ijk[3 * b + 2];
  const int gx = i - P.pad + a;
  if ((unsigned)gx >= (unsigned)P.X) return;
  const int e = (blockIdx.y - a * chunks) * 256 + threadIdx.x;
  if (e >= W * W) return;
  const int bj = e / W, c = e - bj * W;
  const int gy = j - P.pad + bj, gz = k - P.pad + c;
  if ((unsigned)gy >= (unsigned)P.Y || (unsigned)gz >= (unsigned)P.Z) return;
  const float wb = Wn.w1[bj], wc = Wn.w1[c];
  if (wb == 0.f || wc == 0.f) return;
  const double scale = overlap_scale(wa, wb, wc, P.norm[gx], P.norm[P.X + gy], P.norm[P.X + P.Y + gz]);
  int64_t vol_n;
  uint32_t* dst = overlap_dest<PEER>(P, O, gx, gy, gz, &vol_n);
  const int64_t src = P.obase + (int64_t)a * P.os[0] + (int64_t)bj * P.os[1] + (int64_t)c * P.os[2];
  uint32_t q[kOverlapQ];
  overlap_contrib<T>(P, b, src, scale, q);
#pragma unroll
  for (int t = 0; t < kOverlapQ; ++t) red_add_u32(dst + overlap_channel(t, vol_n), q[t]);
}

// The orientations that move the fastest axis (|os[2]| != 1): the logits are contiguous along window axis K (0 or 1),
// the block along window axis 2.  One CTA = a 32 (axis K) x 32 (axis 2) tile of one plane of the remaining window
// axis L: the 22 contributions are computed with lanes along K (coalesced logit reads), parked in shared memory
// ([22][32][33] uint32, conflict-free both ways) and added with lanes along axis 2 (coalesced red.global.add).
// grid = (B, W [plane of L] * ceil(W/32)^2), block = 256
constexpr int kOverlapTileSmem = kOverlapQ * 32 * 33 * 4;
template <bool PEER, typename T>
__global__ void __launch_bounds__(256)
overlap_accumulate_tiled_kernel(OverlapParams P, OverlapWindow Wn, OverlapOwners O, int K) {
  extern __shared__ uint32_t tq[];
  const int W = P.W, nt = (W + 31) >> 5;
  const int b = blockIdx.x, l = blockIdx.y / (nt * nt), t = blockIdx.y - l * nt * nt;
  if (Wn.w1[l] == 0.f) return;  // uniform over the CTA
  const int tk = (t / nt) << 5, t2 = (t % nt) << 5;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int i0 = P.ijk[3 * b + 0] - P.pad, j0 = P.ijk[3 * b + 1] - P.pad, k0 = P.ijk[3 * b + 2] - P.pad;
#pragma unroll 1
  for (int r = 0; r < 4; ++r) {
    const int vk = tk + tx, v2 = t2 + ty + 8 * r;
    uint32_t q[kOverlapQ];
#pragma unroll
    for (int c = 0; c < kOverlapQ; ++c) q[c] = 0u;
    if (vk < W && v2 < W) {
      const int v0 = K == 0 ? vk : l, v1 = K == 0 ? l : vk;
      const int gx = i0 + v0, gy = j0 + v1, gz = k0 + v2;
      const float w0 = Wn.w1[v0], w1 = Wn.w1[v1], w2 = Wn.w1[v2];
      if ((unsigned)gx < (unsigned)P.X && (unsigned)gy < (unsigned)P.Y && (unsigned)gz < (unsigned)P.Z &&
          w0 != 0.f && w1 != 0.f && w2 != 0.f) {
        const double scale = overlap_scale(w0, w1, w2, P.norm[gx], P.norm[P.X + gy], P.norm[P.X + P.Y + gz]);
        const int64_t src = P.obase + (int64_t)v0 * P.os[0] + (int64_t)v1 * P.os[1] + (int64_t)v2 * P.os[2];
        overlap_contrib<T>(P, b, src, scale, q);
      }
    }
#pragma unroll
    for (int c = 0; c < kOverlapQ; ++c) tq[(c * 32 + ty + 8 * r) * 33 + tx] = q[c];
  }
  __syncthreads();
#pragma unroll 1
  for (int r = 0; r < 4; ++r) {
    const int v2 = t2 + tx, vk = tk + ty + 8 * r;
    if (vk >= W || v2 >= W) continue;
    const int v0 = K == 0 ? vk : l, v1 = K == 0 ? l : vk;
    const int gx = i0 + v0, gy = j0 + v1, gz = k0 + v2;
    if ((unsigned)gx >= (unsigned)P.X || (unsigned)gy >= (unsigned)P.Y || (unsigned)gz >= (unsigned)P.Z) continue;
    int64_t vol_n;
    uint32_t* dst = overlap_dest<PEER>(P, O, gx, gy, gz, &vol_n);
#pragma unroll
    for (int c = 0; c < kOverlapQ; ++c) red_add_u32(dst + overlap_channel(c, vol_n), tq[(c * 32 + tx) * 33 + ty + 8 * r]);
  }
}

// in place over one 23-channel block of n voxels: sums -> float(s) 2^-31, arg-max of the 20 amino-acid sums
// (first maximum wins) into channel 2.  A voxel no weighted window reached has all sums 0 and stays 0.
__global__ void __launch_bounds__(256)
overlap_finalize_kernel(uint32_t* __restrict__ block, int64_t n) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  float* out = reinterpret_cast<float*>(block);
  const float kScale = 4.656612873077392578125e-10f;  // 2^-31
  out[v] = __fmul_rn(__uint2float_rn(block[v]), kScale);
  out[n + v] = __fmul_rn(__uint2float_rn(block[n + v]), kScale);
  uint32_t best = 0;
  int arg = 0;
#pragma unroll
  for (int t = 0; t < 20; ++t) {
    const uint32_t s = block[(3 + t) * n + v];
    if (s > best) {
      best = s;
      arg = t;
    }
    out[(3 + t) * n + v] = __fmul_rn(__uint2float_rn(s), kScale);
  }
  out[2 * n + v] = (float)arg;
}

// grid = (S, n_ch, B), block = 256: vol[ch, core] = cubes[b, ch, core]
__global__ void __launch_bounds__(256)
stitch_cubes_kernel(const float* __restrict__ cubes, int n_ch, const int32_t* __restrict__ ijk, int X, int Y,
                    int Z, int o0, int o1, int o2, int e0, int e1, int e2, int S, int pad, int W,
                    float* __restrict__ vol) {
  const int a = blockIdx.x, ch = blockIdx.y, b = blockIdx.z;
  const int i = ijk[3 * b + 0], j = ijk[3 * b + 1], k = ijk[3 * b + 2];
  const int gx = i + a;
  if (gx >= X || gx < o0 || gx >= o0 + e0) return;
  const int64_t W3 = (int64_t)W * W * W;
  const float* cube = cubes + ((int64_t)b * n_ch + ch) * W3;
  float* v = vol + (int64_t)ch * e0 * e1 * e2;
  for (int e = threadIdx.x; e < S * S; e += blockDim.x) {
    const int bj = e / S, c = e - bj * S;
    const int gy = j + bj, gz = k + c;
    if (gy >= Y || gz >= Z) continue;
    const int ly = gy - o1, lz = gz - o2;
    if ((unsigned)ly >= (unsigned)e1 || (unsigned)lz >= (unsigned)e2) continue;
    const int64_t src = ((int64_t)(a + pad) * W + (bj + pad)) * W + (c + pad);
    v[((int64_t)(gx - o0) * e1 + ly) * e2 + lz] = ld_stream_half_line(cube + src);
  }
}

}  // namespace mica

using namespace mica;

static int check_box(int X, int Y, int Z, const int org[3], const int ext[3]) {
  MICA_REQUIRE(org && ext, "null box");
  MICA_REQUIRE(X > 0 && Y > 0 && Z > 0, "empty volume");
  const int G[3] = {X, Y, Z};
  for (int m = 0; m < 3; ++m)
    MICA_REQUIRE(org[m] >= 0 && ext[m] > 0 && org[m] + ext[m] <= G[m], "box outside the volume on axis %d", m);
  return MICA_OK;
}

// byte offset of cube b0's logits in a [B, n_ch, W^3] batch of `esize`-byte elements
static inline const void* cube_offset(const void* p, int64_t b0, int n_ch, int64_t W3, int esize) {
  return static_cast<const char*>(p) + b0 * n_ch * W3 * esize;
}

extern "C" int mica_postproc_stitch_as(const void* bb, const void* ca, const void* aa, int logit_dtype,
                                       const int32_t* ijk, int n_cubes, int X, int Y, int Z, const int org[3],
                                       const int ext[3], int grid_size, int padding, float* bb_vol, float* ca_vol,
                                       float* aa_prob_vol, float* aa_pred_vol, mica_stream_t stream) {
  const int esize = model_dtype_bytes(logit_dtype);
  MICA_REQUIRE(esize, "logit dtype %d: must be MICA_DTYPE_F32 or MICA_DTYPE_BF16", logit_dtype);
  MICA_REQUIRE(bb_vol && ca_vol && aa_prob_vol && aa_pred_vol, "null output volume");
  MICA_REQUIRE(n_cubes == 0 || (bb && ca && aa && ijk), "null input");
  MICA_REQUIRE(grid_size > 0 && padding >= 0, "bad grid_size/padding");
  int rc = check_box(X, Y, Z, org, ext);
  if (rc) return rc;
  if (n_cubes <= 0) return MICA_OK;
  StitchParams P;
  P.bb = bb;
  P.ca = ca;
  P.aa = aa;
  P.X = X;
  P.Y = Y;
  P.Z = Z;
  for (int m = 0; m < 3; ++m) {
    P.org[m] = org[m];
    P.ext[m] = ext[m];
  }
  P.S = grid_size;
  P.pad = padding;
  P.W = grid_size + 2 * padding;
  P.bb_vol = bb_vol;
  P.ca_vol = ca_vol;
  P.aa_prob_vol = aa_prob_vol;
  P.aa_pred_vol = aa_pred_vol;
  const int64_t W3 = (int64_t)P.W * P.W * P.W;
  const int kMaxY = 32768;
  for (int b0 = 0; b0 < n_cubes; b0 += kMaxY) {
    const int nb = (n_cubes - b0 < kMaxY) ? n_cubes - b0 : kMaxY;
    P.bb = cube_offset(bb, b0, 4, W3, esize);
    P.ca = cube_offset(ca, b0, 4, W3, esize);
    P.aa = cube_offset(aa, b0, 21, W3, esize);
    P.ijk = ijk + 3 * (int64_t)b0;
    const int chunks = (grid_size * grid_size + 255) / 256;
    const dim3 grid(nb, grid_size * chunks);
    if (logit_dtype == MICA_DTYPE_BF16)
      postproc_stitch_kernel<false, __nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(P, StitchOwners());
    else
      postproc_stitch_kernel<false, float><<<grid, 256, 0, (cudaStream_t)stream>>>(P, StitchOwners());
    MICA_LAUNCH_CHECK("postproc_stitch_kernel");
  }
  return MICA_OK;
}

extern "C" int mica_postproc_stitch(const float* bb, const float* ca, const float* aa,
                                    const int32_t* ijk, int n_cubes, int X, int Y, int Z,
                                    const int org[3], const int ext[3], int grid_size, int padding,
                                    float* bb_vol, float* ca_vol, float* aa_prob_vol, float* aa_pred_vol,
                                    mica_stream_t stream) {
  return mica_postproc_stitch_as(bb, ca, aa, MICA_DTYPE_F32, ijk, n_cubes, X, Y, Z, org, ext, grid_size, padding,
                                 bb_vol, ca_vol, aa_prob_vol, aa_pred_vol, stream);
}

// the paste of cubes the model did not run on (the keep rule of ops.select_cubes): their cores, clipped to the box,
// become 0 in all 23 channels -- what the reference's stitcher leaves where a cube has no grid file.
// grid = (n_cubes, grid_size [core plane a]), block = 256 over the (b, c) plane of the core.
__global__ void __launch_bounds__(256)
zero_cores_kernel(StitchParams P) {
  const int S = P.S, b = blockIdx.x, a = blockIdx.y;
  const int gx = P.ijk[3 * b + 0] + a, j = P.ijk[3 * b + 1], k = P.ijk[3 * b + 2];
  if (gx >= P.X || gx < P.org[0] || gx >= P.org[0] + P.ext[0]) return;
  const int64_t vol_n = (int64_t)P.ext[0] * P.ext[1] * P.ext[2];
  for (int e = threadIdx.x; e < S * S; e += blockDim.x) {
    const int gy = j + e / S, gz = k + e % S;
    if (gy >= P.Y || gz >= P.Z) continue;
    const int ly = gy - P.org[1], lz = gz - P.org[2];
    if (ly < 0 || ly >= P.ext[1] || lz < 0 || lz >= P.ext[2]) continue;
    const int64_t o = ((int64_t)(gx - P.org[0]) * P.ext[1] + ly) * P.ext[2] + lz;
    P.bb_vol[o] = 0.f;
    P.ca_vol[o] = 0.f;
    P.aa_pred_vol[o] = 0.f;
#pragma unroll 4
    for (int t = 0; t < 20; ++t) P.aa_prob_vol[t * vol_n + o] = 0.f;
  }
}

extern "C" int mica_zero_cores(const int32_t* ijk, int n_cubes, int X, int Y, int Z, const int org[3],
                               const int ext[3], int grid_size, float* bb_vol, float* ca_vol, float* aa_prob_vol,
                               float* aa_pred_vol, mica_stream_t stream) {
  MICA_REQUIRE(bb_vol && ca_vol && aa_prob_vol && aa_pred_vol, "null output volume");
  MICA_REQUIRE(n_cubes == 0 || ijk, "null input");
  MICA_REQUIRE(grid_size > 0 && grid_size <= 65535, "bad grid_size");
  MICA_REQUIRE(n_cubes >= 0, "bad cube count %d", n_cubes);
  int rc = check_box(X, Y, Z, org, ext);
  if (rc) return rc;
  if (n_cubes == 0) return MICA_OK;
  StitchParams P = {};
  P.ijk = ijk;
  P.X = X;
  P.Y = Y;
  P.Z = Z;
  for (int m = 0; m < 3; ++m) {
    P.org[m] = org[m];
    P.ext[m] = ext[m];
  }
  P.S = grid_size;
  P.bb_vol = bb_vol;
  P.ca_vol = ca_vol;
  P.aa_prob_vol = aa_prob_vol;
  P.aa_pred_vol = aa_pred_vol;
  zero_cores_kernel<<<dim3(n_cubes, grid_size), 256, 0, (cudaStream_t)stream>>>(P);
  MICA_LAUNCH_CHECK("zero_cores_kernel");
  return MICA_OK;
}

extern "C" int mica_postproc_stitch_peer_as(const void* bb, const void* ca, const void* aa, int logit_dtype,
                                            const int32_t* ijk, int n_cubes, int X, int Y, int Z, int grid_size,
                                            int padding, void* const* owner_base, const int* x_bounds, int world,
                                            mica_stream_t stream) {
  const int esize = model_dtype_bytes(logit_dtype);
  MICA_REQUIRE(esize, "logit dtype %d: must be MICA_DTYPE_F32 or MICA_DTYPE_BF16", logit_dtype);
  MICA_REQUIRE(owner_base && x_bounds, "null owner table");
  MICA_REQUIRE(world >= 1 && world <= kStitchMaxWorld, "bad world size %d", world);
  MICA_REQUIRE(n_cubes == 0 || (bb && ca && aa && ijk), "null input");
  MICA_REQUIRE(grid_size > 0 && padding >= 0 && X > 0 && Y > 0 && Z > 0, "bad geometry");
  MICA_REQUIRE(x_bounds[0] == 0 && x_bounds[world] == X, "x_bounds must run from 0 to X");
  for (int r = 0; r < world; ++r) MICA_REQUIRE(x_bounds[r] <= x_bounds[r + 1], "x_bounds must not decrease");
  if (n_cubes <= 0) return MICA_OK;
  StitchParams P;
  P.X = X;
  P.Y = Y;
  P.Z = Z;
  P.org[0] = P.org[1] = P.org[2] = 0;
  P.ext[0] = X;
  P.ext[1] = Y;
  P.ext[2] = Z;
  P.S = grid_size;
  P.pad = padding;
  P.W = grid_size + 2 * padding;
  P.bb_vol = P.ca_vol = P.aa_prob_vol = P.aa_pred_vol = nullptr;
  StitchOwners O;
  O.base = reinterpret_cast<float* const*>(owner_base);
  O.world = world;
  for (int r = 0; r <= world; ++r) O.bounds[r] = x_bounds[r];
  for (int r = world + 1; r <= kStitchMaxWorld; ++r) O.bounds[r] = X;
  const int64_t W3 = (int64_t)P.W * P.W * P.W;
  const int kMaxY = 32768;
  for (int b0 = 0; b0 < n_cubes; b0 += kMaxY) {
    const int nb = (n_cubes - b0 < kMaxY) ? n_cubes - b0 : kMaxY;
    P.bb = cube_offset(bb, b0, 4, W3, esize);
    P.ca = cube_offset(ca, b0, 4, W3, esize);
    P.aa = cube_offset(aa, b0, 21, W3, esize);
    P.ijk = ijk + 3 * (int64_t)b0;
    const int chunks = (grid_size * grid_size + 255) / 256;
    const dim3 grid(nb, grid_size * chunks);
    if (logit_dtype == MICA_DTYPE_BF16)
      postproc_stitch_kernel<true, __nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(P, O);
    else
      postproc_stitch_kernel<true, float><<<grid, 256, 0, (cudaStream_t)stream>>>(P, O);
    MICA_LAUNCH_CHECK("postproc_stitch_kernel<peer>");
  }
  return MICA_OK;
}

extern "C" int mica_postproc_stitch_peer(const float* bb, const float* ca, const float* aa, const int32_t* ijk,
                                         int n_cubes, int X, int Y, int Z, int grid_size, int padding,
                                         void* const* owner_base, const int* x_bounds, int world,
                                         mica_stream_t stream) {
  return mica_postproc_stitch_peer_as(bb, ca, aa, MICA_DTYPE_F32, ijk, n_cubes, X, Y, Z, grid_size, padding,
                                      owner_base, x_bounds, world, stream);
}

extern "C" int mica_stitch_cubes(const float* cubes, int n_ch, const int32_t* ijk, int n_cubes,
                                 int X, int Y, int Z, const int org[3], const int ext[3],
                                 int grid_size, int padding, float* vol, mica_stream_t stream) {
  MICA_REQUIRE(vol, "null output volume");
  MICA_REQUIRE(n_cubes == 0 || (cubes && ijk), "null input");
  MICA_REQUIRE(n_ch > 0 && n_ch <= 65535, "bad channel count");
  MICA_REQUIRE(grid_size > 0 && padding >= 0, "bad grid_size/padding");
  int rc = check_box(X, Y, Z, org, ext);
  if (rc) return rc;
  if (n_cubes <= 0) return MICA_OK;
  const int W = grid_size + 2 * padding;
  const int64_t W3 = (int64_t)W * W * W;
  const int kMaxZ = 32768;
  for (int b0 = 0; b0 < n_cubes; b0 += kMaxZ) {
    const int nb = (n_cubes - b0 < kMaxZ) ? n_cubes - b0 : kMaxZ;
    stitch_cubes_kernel<<<dim3(grid_size, n_ch, nb), 256, 0, (cudaStream_t)stream>>>(
        cubes + (int64_t)b0 * n_ch * W3, n_ch, ijk + 3 * (int64_t)b0, X, Y, Z, org[0], org[1], org[2], ext[0],
        ext[1], ext[2], grid_size, padding, W, vol);
    MICA_LAUNCH_CHECK("stitch_cubes_kernel");
  }
  return MICA_OK;
}

static int overlap_setup(const void* bb, const void* ca, const void* aa, const int32_t* ijk, int n_cubes, int X,
                         int Y, int Z, int grid_size, int padding, const float* window_w1, const double* norm,
                         int orientation, OverlapParams* P, OverlapWindow* Wn) {
  MICA_REQUIRE(window_w1 && norm, "null pointer");
  Orientation ori;
  MICA_REQUIRE(orientation_decode(orientation, grid_size + 2 * padding, &ori), "orientation %d is not in 0..47",
               orientation);
  P->obase = ori.base;
  for (int m = 0; m < 3; ++m) P->os[m] = ori.s[m];
  MICA_REQUIRE(n_cubes == 0 || (bb && ca && aa && ijk), "null input");
  MICA_REQUIRE(grid_size > 0 && padding >= 0 && X > 0 && Y > 0 && Z > 0, "bad geometry");
  const int W = grid_size + 2 * padding;
  MICA_REQUIRE(W <= kOverlapMaxW, "window of %d voxels exceeds the %d the weight table holds", W, kOverlapMaxW);
  bool any = false;
  for (int u = 0; u < W; ++u) {
    const float w = window_w1[u];
    MICA_REQUIRE(w >= 0.f && w <= 3.4028234663852886e38f, "window weight %d is %g: weights must be finite and >= 0",
                 u, (double)w);
    any = any || w > 0.f;
  }
  MICA_REQUIRE(any, "window weights are all 0");
  P->bb = bb;
  P->ca = ca;
  P->aa = aa;
  P->ijk = ijk;
  P->X = X;
  P->Y = Y;
  P->Z = Z;
  P->pad = padding;
  P->W = W;
  P->norm = norm;
  P->block = nullptr;
  for (int u = 0; u < kOverlapMaxW; ++u) Wn->w1[u] = u < W ? window_w1[u] : 0.f;
  return MICA_OK;
}

template <bool PEER, typename T>
static int overlap_launch(OverlapParams P, const OverlapWindow& Wn, const OverlapOwners& O, int n_cubes,
                          cudaStream_t stream) {
  const int64_t W3 = (int64_t)P.W * P.W * P.W;
  const void *bb = P.bb, *ca = P.ca, *aa = P.aa;
  const int32_t* ijk = P.ijk;
  const int kMaxX = 32768;
  for (int b0 = 0; b0 < n_cubes; b0 += kMaxX) {
    const int nb = (n_cubes - b0 < kMaxX) ? n_cubes - b0 : kMaxX;
    P.bb = cube_offset(bb, b0, 4, W3, sizeof(T));
    P.ca = cube_offset(ca, b0, 4, W3, sizeof(T));
    P.aa = cube_offset(aa, b0, 21, W3, sizeof(T));
    P.ijk = ijk + 3 * (int64_t)b0;
    if (P.os[2] == 1 || P.os[2] == -1) {
      const int chunks = (P.W * P.W + 255) / 256;
      overlap_accumulate_kernel<PEER, T><<<dim3(nb, P.W * chunks), 256, 0, stream>>>(P, Wn, O);
      MICA_LAUNCH_CHECK(PEER ? "overlap_accumulate_kernel<peer>" : "overlap_accumulate_kernel");
    } else {
      const int nt = (P.W + 31) / 32, K = (P.os[0] == 1 || P.os[0] == -1) ? 0 : 1;
      MICA_CUDA(cudaFuncSetAttribute(overlap_accumulate_tiled_kernel<PEER, T>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, kOverlapTileSmem));
      overlap_accumulate_tiled_kernel<PEER, T><<<dim3(nb, P.W * nt * nt), 256, kOverlapTileSmem, stream>>>(P, Wn, O, K);
      MICA_LAUNCH_CHECK(PEER ? "overlap_accumulate_tiled_kernel<peer>" : "overlap_accumulate_tiled_kernel");
    }
  }
  return MICA_OK;
}

extern "C" int mica_overlap_accumulate_fixed_as(const void* bb, const void* ca, const void* aa, int logit_dtype,
                                                const int32_t* ijk, int n_cubes, int X, int Y, int Z, int grid_size,
                                                int padding, const float* window_w1, const double* norm,
                                                int orientation, void* block, mica_stream_t stream) {
  MICA_REQUIRE(model_dtype_bytes(logit_dtype), "logit dtype %d: must be MICA_DTYPE_F32 or MICA_DTYPE_BF16",
               logit_dtype);
  MICA_REQUIRE(block, "null block");
  OverlapParams P;
  OverlapWindow Wn;
  int rc = overlap_setup(bb, ca, aa, ijk, n_cubes, X, Y, Z, grid_size, padding, window_w1, norm, orientation, &P,
                         &Wn);
  if (rc) return rc;
  if (n_cubes <= 0) return MICA_OK;
  P.block = static_cast<uint32_t*>(block);
  OverlapOwners O;
  O.base = nullptr;
  O.axis = 0;
  O.world = 1;
  if (logit_dtype == MICA_DTYPE_BF16)
    return overlap_launch<false, __nv_bfloat16>(P, Wn, O, n_cubes, (cudaStream_t)stream);
  return overlap_launch<false, float>(P, Wn, O, n_cubes, (cudaStream_t)stream);
}

extern "C" int mica_overlap_accumulate_fixed_peer_as(const void* bb, const void* ca, const void* aa, int logit_dtype,
                                                     const int32_t* ijk, int n_cubes, int X, int Y, int Z,
                                                     int grid_size, int padding, const float* window_w1,
                                                     const double* norm, int orientation, void* const* owner_base,
                                                     int axis, const int* bounds, int world, mica_stream_t stream) {
  MICA_REQUIRE(model_dtype_bytes(logit_dtype), "logit dtype %d: must be MICA_DTYPE_F32 or MICA_DTYPE_BF16",
               logit_dtype);
  MICA_REQUIRE(owner_base && bounds, "null owner table");
  MICA_REQUIRE(world >= 1 && world <= kStitchMaxWorld, "bad world size %d", world);
  MICA_REQUIRE(axis == 0 || axis == 2, "owner axis must be 0 (x) or 2 (k), got %d", axis);
  OverlapParams P;
  OverlapWindow Wn;
  int rc = overlap_setup(bb, ca, aa, ijk, n_cubes, X, Y, Z, grid_size, padding, window_w1, norm, orientation, &P,
                         &Wn);
  if (rc) return rc;
  const int G = axis == 0 ? X : Z;
  MICA_REQUIRE(bounds[0] == 0 && bounds[world] == G, "bounds must run from 0 to %d", G);
  for (int r = 0; r < world; ++r) MICA_REQUIRE(bounds[r] <= bounds[r + 1], "bounds must not decrease");
  if (n_cubes <= 0) return MICA_OK;
  OverlapOwners O;
  O.base = reinterpret_cast<uint32_t* const*>(owner_base);
  O.axis = axis;
  O.world = world;
  for (int r = 0; r <= world; ++r) O.bounds[r] = bounds[r];
  for (int r = world + 1; r <= kStitchMaxWorld; ++r) O.bounds[r] = G;
  if (logit_dtype == MICA_DTYPE_BF16)
    return overlap_launch<true, __nv_bfloat16>(P, Wn, O, n_cubes, (cudaStream_t)stream);
  return overlap_launch<true, float>(P, Wn, O, n_cubes, (cudaStream_t)stream);
}

extern "C" int mica_overlap_accumulate_fixed_oriented(const float* bb, const float* ca, const float* aa,
                                                      const int32_t* ijk, int n_cubes, int X, int Y, int Z,
                                                      int grid_size, int padding, const float* window_w1,
                                                      const double* norm, int orientation, void* block,
                                                      mica_stream_t stream) {
  return mica_overlap_accumulate_fixed_as(bb, ca, aa, MICA_DTYPE_F32, ijk, n_cubes, X, Y, Z, grid_size, padding,
                                          window_w1, norm, orientation, block, stream);
}

extern "C" int mica_overlap_accumulate_fixed_peer_oriented(const float* bb, const float* ca, const float* aa,
                                                           const int32_t* ijk, int n_cubes, int X, int Y, int Z,
                                                           int grid_size, int padding, const float* window_w1,
                                                           const double* norm, int orientation,
                                                           void* const* owner_base, int axis, const int* bounds,
                                                           int world, mica_stream_t stream) {
  return mica_overlap_accumulate_fixed_peer_as(bb, ca, aa, MICA_DTYPE_F32, ijk, n_cubes, X, Y, Z, grid_size, padding,
                                               window_w1, norm, orientation, owner_base, axis, bounds, world, stream);
}

extern "C" int mica_overlap_accumulate_fixed(const float* bb, const float* ca, const float* aa, const int32_t* ijk,
                                             int n_cubes, int X, int Y, int Z, int grid_size, int padding,
                                             const float* window_w1, const double* norm, void* block,
                                             mica_stream_t stream) {
  return mica_overlap_accumulate_fixed_oriented(bb, ca, aa, ijk, n_cubes, X, Y, Z, grid_size, padding, window_w1, norm,
                                                0, block, stream);
}

extern "C" int mica_overlap_accumulate_fixed_peer(const float* bb, const float* ca, const float* aa,
                                                  const int32_t* ijk, int n_cubes, int X, int Y, int Z,
                                                  int grid_size, int padding, const float* window_w1,
                                                  const double* norm, void* const* owner_base, int axis,
                                                  const int* bounds, int world, mica_stream_t stream) {
  return mica_overlap_accumulate_fixed_peer_oriented(bb, ca, aa, ijk, n_cubes, X, Y, Z, grid_size, padding, window_w1,
                                                     norm, 0, owner_base, axis, bounds, world, stream);
}

extern "C" int mica_overlap_finalize_fixed(void* block, int64_t n_voxels, mica_stream_t stream) {
  MICA_REQUIRE(block && n_voxels >= 0, "bad arguments");
  if (n_voxels == 0) return MICA_OK;
  overlap_finalize_kernel<<<(unsigned)ceil_div64(n_voxels, 256), 256, 0, (cudaStream_t)stream>>>(
      static_cast<uint32_t*>(block), n_voxels);
  MICA_LAUNCH_CHECK("overlap_finalize_kernel");
  return MICA_OK;
}

extern "C" int mica_peer_atomics_supported(int device, int peer_device) {
  MICA_REQUIRE(device >= 0 && peer_device >= 0, "bad device pair (%d, %d)", device, peer_device);
  if (device == peer_device) return 1;
  int can = 0;
  MICA_CUDA(cudaDeviceGetP2PAttribute(&can, cudaDevP2PAttrNativeAtomicSupported, device, peer_device));
  return can ? 1 : 0;
}
