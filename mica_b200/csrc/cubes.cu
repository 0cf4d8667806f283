// R5/R6: fused cube extraction into the model's input batch.
//
// Replaces GridCreator.transpose + create_grids_from_mrc (utils/create_grids.py:67-176,
// reference root), the five training twins (scripts_for_training_data/create_grids_for_*.py)
// and CryoEMTestDataset.__getitem__ (dataset/dataset.py:194-224): instead of np.pad +
// one .npz per cube per channel + 25 np.load per cube, every W^3 window (W = grid_size +
// 2*padding) is cut straight from the resident (nz,ny,nx) volumes into the
// [B, C, W, W, W] tensor the model consumes, zero-filled outside the map.
//
// The reference cuts cubes from an axis-permuted view (D6): cube axis m walks memory
// axis perm[m].  For the standard MRC axis order perm = (2,1,0), i.e. the cube's slowest
// axis is the memory-contiguous one, so the copy is a tiled transpose through shared
// memory (32x33 tiles: coalesced 128-byte reads along x, coalesced 128-byte writes
// along the cube's fastest axis).  Pure index work: bit-exact.
#include <cuda.h>
#include <math_constants.h>

#include <stdlib.h>

#include "common.cuh"

namespace mica {

struct ExtractParams {
  const float* vol;
  int64_t chan_stride;
  int T[3];            // cube-space global dims: T[m] = memdims[perm[m]]
  int64_t sstride[3];  // memory stride walked by cube axis m
  int slab_axis;       // cube axis that walks memory axis 0 (the slab axis)
  int z0, nzl;         // slab: memory planes [z0, z0 + nzl)
  int W, pad;
  const int32_t* ijk;
  void* out;               // float or __nv_bfloat16 (the kernels' T), out_cube_stride in elements
  int64_t out_cube_stride;
  int32_t* nonzero;
  float* cube_max;
};

__device__ __forceinline__ void atomic_max_f32(float* addr, float v) {
  if (v >= 0.f)
    atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else
    atomicMin(reinterpret_cast<unsigned*>(addr), __float_as_uint(v));
}

__device__ __forceinline__ void block_flags(const ExtractParams& P, int cube, bool any_nz, float vmax) {
  if (P.nonzero) {
    if (__syncthreads_or(any_nz) && threadIdx.x == 0 && threadIdx.y == 0) atomicOr(&P.nonzero[cube], 1);
  }
  if (P.cube_max && blockIdx.z == 0) {
    for (int o = 16; o > 0; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    if (threadIdx.x == 0) atomic_max_f32(&P.cube_max[cube], vmax);
  }
}

// memory offset of cube-space position p (relative to the local slab), or -1 outside the map
__device__ __forceinline__ bool in_map(const ExtractParams& P, int p0, int p1, int p2) {
  return (unsigned)p0 < (unsigned)P.T[0] && (unsigned)p1 < (unsigned)P.T[1] && (unsigned)p2 < (unsigned)P.T[2];
}

// ---- cube's fastest axis (2) is the memory-contiguous one: row copy.
// grid = (W [u0], B, C), block = (32, 8)
// T (here and in the other extract kernels): the element type of the output, float or __nv_bfloat16; the flags are
// taken on the float32 values before st_stream_el rounds them
template <typename T>
__global__ void __launch_bounds__(256)
extract_rows_kernel(ExtractParams P) {
  const int u0 = blockIdx.x, c = blockIdx.z, b = blockIdx.y;
  const int W = P.W;
  const int i0 = P.ijk[3 * b + 0] - P.pad, j0 = P.ijk[3 * b + 1] - P.pad, k0 = P.ijk[3 * b + 2] - P.pad;
  const float* src = P.vol + (int64_t)c * P.chan_stride;
  T* dst = static_cast<T*>(P.out) + (int64_t)b * P.out_cube_stride + (int64_t)c * W * W * W + (int64_t)u0 * W * W;
  const int p0 = i0 + u0;
  const int zsub[3] = {P.slab_axis == 0 ? P.z0 : 0, P.slab_axis == 1 ? P.z0 : 0, P.slab_axis == 2 ? P.z0 : 0};
  bool any_nz = false;
  float vmax = -CUDART_INF_F;
  for (int u1 = threadIdx.y; u1 < W; u1 += blockDim.y) {
    const int p1 = j0 + u1;
    for (int u2 = threadIdx.x; u2 < W; u2 += 32) {
      const int p2 = k0 + u2;
      float v = 0.f;
      if (in_map(P, p0, p1, p2)) {
        int q0 = p0 - zsub[0], q1 = p1 - zsub[1], q2 = p2 - zsub[2];
        int qs = P.slab_axis == 0 ? q0 : (P.slab_axis == 1 ? q1 : q2);
        if ((unsigned)qs < (unsigned)P.nzl) v = src[q0 * P.sstride[0] + q1 * P.sstride[1] + q2 * P.sstride[2]];
      }
      any_nz |= (v != 0.f);
      vmax = fmaxf(vmax, v);
      st_stream_el(dst + (int64_t)u1 * W + u2, v);
    }
  }
  block_flags(P, b, any_nz, vmax);
}

// ---- cube axis MC (0 or 1) is memory-contiguous: tiled transpose MC <-> 2.
// grid = (W [u_o, the other slow axis], B, C), block = (32, 8)
template <int MC, typename T>
__global__ void __launch_bounds__(256)
extract_transpose_kernel(ExtractParams P) {
  __shared__ float tile[32][33];
  constexpr int OA = 1 - MC;
  const int uo = blockIdx.x, c = blockIdx.z, b = blockIdx.y;
  const int W = P.W;
  int org[3] = {P.ijk[3 * b + 0] - P.pad, P.ijk[3 * b + 1] - P.pad, P.ijk[3 * b + 2] - P.pad};
  const float* src = P.vol + (int64_t)c * P.chan_stride;
  T* dst = static_cast<T*>(P.out) + (int64_t)b * P.out_cube_stride + (int64_t)c * W * W * W;
  const int64_t out_mc = (MC == 0) ? (int64_t)W * W : W;   // output stride of cube axis MC
  const int64_t out_oa = (MC == 0) ? W : (int64_t)W * W;   // output stride of the other slow axis
  const int po = org[OA] + uo;
  const bool ok_o = (unsigned)po < (unsigned)P.T[OA];
  const int zs_o = (P.slab_axis == OA) ? P.z0 : 0, zs_c = (P.slab_axis == MC) ? P.z0 : 0,
            zs_2 = (P.slab_axis == 2) ? P.z0 : 0;
  const bool slab_o = (P.slab_axis != OA) || ((unsigned)(po - P.z0) < (unsigned)P.nzl);
  const int64_t base_o = (int64_t)(po - zs_o) * P.sstride[OA];
  const int tx = threadIdx.x, ty = threadIdx.y;
  bool any_nz = false;
  float vmax = -CUDART_INF_F;
  for (int t2 = 0; t2 < W; t2 += 32) {
    for (int tc = 0; tc < W; tc += 32) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int u2 = t2 + ty + 8 * r, uc = tc + tx;
        const int p2 = org[2] + u2, pc = org[MC] + uc;
        float v = 0.f;
        if (ok_o && slab_o && u2 < W && uc < W && (unsigned)p2 < (unsigned)P.T[2] && (unsigned)pc < (unsigned)P.T[MC]) {
          const int q2 = p2 - zs_2, qc = pc - zs_c;
          const bool slab_ok = (P.slab_axis == 2) ? ((unsigned)q2 < (unsigned)P.nzl)
                                                  : (P.slab_axis == MC ? ((unsigned)qc < (unsigned)P.nzl) : true);
          if (slab_ok) v = __ldg(src + base_o + (int64_t)q2 * P.sstride[2] + (int64_t)qc * P.sstride[MC]);
        }
        any_nz |= (v != 0.f);
        vmax = fmaxf(vmax, v);
        tile[ty + 8 * r][tx] = v;
      }
      __syncthreads();
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int uc = tc + ty + 8 * r, u2 = t2 + tx;
        if (uc < W && u2 < W) st_stream_el(dst + uc * out_mc + uo * out_oa + u2, tile[tx][ty + 8 * r]);
      }
      __syncthreads();
    }
  }
  block_flags(P, b, any_nz, vmax);
}


// ---- oriented windows (test-time augmentation, orientation code != 0, ops.orientation): P is expressed in OUTPUT
// axes -- T, sstride and slab_axis of output axis a are those of window axis pi[a] -- and output axis a starts at
// cube coordinate ijk[cax[a]] - pad, walked forwards (dir +1) or, flipped, backwards from the far end of the window.
// MC = the output axis that walks memory x: 2 -> row copy (a flipped row only reverses the lanes: still one
// 128-byte line per warp); 0 / 1 -> tiled transpose MC <-> 2 through shared memory as extract_transpose_kernel, so
// loads along x and streaming stores along the output's fastest axis both stay 128-byte coalesced.
struct OrientAxes {
  int cax[3];
  int dir[3];
};

__device__ __forceinline__ float load_oriented(const ExtractParams& P, const float* src, int p0, int p1, int p2) {
  if (!in_map(P, p0, p1, p2)) return 0.f;
  const int q0 = p0 - (P.slab_axis == 0 ? P.z0 : 0), q1 = p1 - (P.slab_axis == 1 ? P.z0 : 0),
            q2 = p2 - (P.slab_axis == 2 ? P.z0 : 0);
  const int qs = P.slab_axis == 0 ? q0 : (P.slab_axis == 1 ? q1 : q2);
  if ((unsigned)qs >= (unsigned)P.nzl) return 0.f;
  return __ldg(src + q0 * P.sstride[0] + q1 * P.sstride[1] + q2 * P.sstride[2]);
}

// grid = (W [output axis 0 for MC == 2, else the slow output axis that is not MC], B, C), block = (32, 8)
template <int MC, typename T>
__global__ void __launch_bounds__(256)
extract_oriented_kernel(ExtractParams P, OrientAxes A) {
  __shared__ float tile[32][33];
  const int uo = blockIdx.x, c = blockIdx.z, b = blockIdx.y;
  const int W = P.W;
  int org[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) org[a] = P.ijk[3 * b + A.cax[a]] - P.pad + (A.dir[a] < 0 ? W - 1 : 0);
  const float* src = P.vol + (int64_t)c * P.chan_stride;
  T* dst = static_cast<T*>(P.out) + (int64_t)b * P.out_cube_stride + (int64_t)c * W * W * W;
  const int tx = threadIdx.x, ty = threadIdx.y;
  bool any_nz = false;
  float vmax = -CUDART_INF_F;
  if (MC == 2) {
    const int p0 = org[0] + A.dir[0] * uo;
    for (int u1 = ty; u1 < W; u1 += 8) {
      const int p1 = org[1] + A.dir[1] * u1;
      for (int u2 = tx; u2 < W; u2 += 32) {
        const float v = load_oriented(P, src, p0, p1, org[2] + A.dir[2] * u2);
        any_nz |= (v != 0.f);
        vmax = fmaxf(vmax, v);
        st_stream_el(dst + ((int64_t)uo * W + u1) * W + u2, v);
      }
    }
  } else {
    constexpr int OA = 1 - (MC & 1);
    const int64_t out_mc = (MC == 0) ? (int64_t)W * W : W;
    const int64_t out_oa = (MC == 0) ? W : (int64_t)W * W;
    const int po = org[OA] + A.dir[OA] * uo;
    for (int t2 = 0; t2 < W; t2 += 32) {
      for (int tc = 0; tc < W; tc += 32) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int u2 = t2 + ty + 8 * r, uc = tc + tx;
          float v = 0.f;
          if (u2 < W && uc < W) {
            const int p2 = org[2] + A.dir[2] * u2, pc = org[MC] + A.dir[MC] * uc;
            v = MC == 0 ? load_oriented(P, src, pc, po, p2) : load_oriented(P, src, po, pc, p2);
          }
          any_nz |= (v != 0.f);
          vmax = fmaxf(vmax, v);
          tile[ty + 8 * r][tx] = v;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int uc = tc + ty + 8 * r, u2 = t2 + tx;
          if (uc < W && u2 < W) st_stream_el(dst + uc * out_mc + uo * out_oa + u2, tile[tx][ty + 8 * r]);
        }
        __syncthreads();
      }
    }
  }
  block_flags(P, b, any_nz, vmax);
}

// ---- TMA path for the standard layout (cube axis 0 is memory-contiguous, W % 32 == 0,
// 16-byte aligned rows): one CTA = one [32 a] x [BT b] x [W c] tile of one (cube, channel).
// A single elected thread issues ONE cp.async.bulk.tensor box load of a rank-4 tensor map
// whose dims are ordered (x, c-axis, b-axis, channel), so the box lands in shared memory as
// [b][c][32 x] rows of exactly 128 bytes with the 128-byte hardware swizzle; negative or
// too-large coordinates are zero-filled by the TMA unit, which IS the reference's np.pad.
// Consumers read float4 (4 consecutive a) along lanes = c -- conflict-free thanks to the
// swizzle -- and issue four fully coalesced 128-byte streaming stores per warp.
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

struct TmaExtractParams {
  const int32_t* ijk;
  void* out;
  int64_t out_cube_stride;
  int32_t* nonzero;
  float* cube_max;
  int W, pad;
  int off_c, off_b;  // slab offsets subtracted from the tensor-map coordinates of dims 1 and 2
};

template <int BT, typename T>
__global__ void __launch_bounds__(256)
extract_tma_kernel(const __grid_constant__ CUtensorMap tmap, TmaExtractParams P) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  uint8_t* tile = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int W = P.W;
  const int a_tiles = W >> 5;
  const int a0 = (blockIdx.x % a_tiles) << 5, b0 = (blockIdx.x / a_tiles) * BT;
  // channel is the slowest grid index: CTAs resident at the same time cut overlapping windows of ONE
  // channel, so the 8x window overlap is served by L2 instead of DRAM
  const int ch = blockIdx.z, cube = blockIdx.y;
  const int i0 = P.ijk[3 * cube + 0] - P.pad, j0 = P.ijk[3 * cube + 1] - P.pad, k0 = P.ijk[3 * cube + 2] - P.pad;
  const uint32_t bar_a = smem_u32(&bar), tile_a = smem_u32(tile);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t bytes = (uint32_t)BT * W * 128u;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(bytes) : "memory");
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
        ::"r"(tile_a), "l"(&tmap), "r"(i0 + a0), "r"(k0 - P.off_c), "r"(j0 + b0 - P.off_b), "r"(ch), "r"(bar_a)
        : "memory");
  }
  {  // wait for the box (phase 0)
    uint32_t done = 0;
    while (!done) {
      asm volatile(
          "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(done) : "r"(bar_a) : "memory");
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c_groups = W >> 5;
  const int64_t W2 = (int64_t)W * W;
  T* dst = static_cast<T*>(P.out) + (int64_t)cube * P.out_cube_stride + (int64_t)ch * W2 * W + (int64_t)a0 * W2 +
           (int64_t)b0 * W;
  bool any_nz = false;
  float vmax = -CUDART_INF_F;
  const int items = BT * c_groups * 8;
#pragma unroll 4
  for (int it = warp; it < items; it += 8) {
    const int j = it & 7, cg = (it >> 3) % c_groups, y = (it >> 3) / c_groups;
    const int z = (cg << 5) + lane;
    const int R = y * W + z;
    const float4 v = *reinterpret_cast<const float4*>(tile + (size_t)R * 128 + (((j ^ (R & 7))) << 4));
    T* o = dst + (int64_t)(4 * j) * W2 + (int64_t)y * W + z;
    st_stream_el(o, v.x);
    st_stream_el(o + W2, v.y);
    st_stream_el(o + 2 * W2, v.z);
    st_stream_el(o + 3 * W2, v.w);
    any_nz |= (v.x != 0.f) | (v.y != 0.f) | (v.z != 0.f) | (v.w != 0.f);
    vmax = fmaxf(fmaxf(vmax, fmaxf(v.x, v.y)), fmaxf(v.z, v.w));
  }
  if (P.nonzero) {
    if (__syncthreads_or(any_nz) && threadIdx.x == 0) atomicOr(&P.nonzero[cube], 1);
  }
  if (P.cube_max && ch == 0) {
    for (int o = 16; o > 0; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    if (lane == 0) atomic_max_f32(&P.cube_max[cube], vmax);
  }
}

constexpr int kTmaBT = 4;  // b-rows per tile: 4 * 64 * 128 B = 32 KB of shared memory per CTA

// ---- window maximum (inference keep rule, ops.select_cubes): out[b] = max of cube b's W^3 window, zeros standing
// for the parts outside the map (np.pad), NaN if the window holds one (np.max).  The maximum does not depend on the
// element order, so the window is walked as the axis-aligned box it covers in MEMORY order, whatever the perm: rows
// along x stay coalesced, and nothing is written per voxel.  One CTA per cube; warps take (z, y, 32-wide x chunk)
// items, four independent loads in flight per thread.
struct WindowMaxParams {
  const float* vol;     // [nz_local, ny, nx]
  int ny, nx;
  int lo_z, hi_z;       // the planes the block holds, global: [z0, z0 + nz_local)
  int z0;
  int inv[3];           // inv[a] = cube axis that walks memory axis a (0 = z, 1 = y, 2 = x)
  int W, pad;
  const int32_t* ijk;
  float* out;
};

__global__ void __launch_bounds__(256)
cube_window_max_kernel(WindowMaxParams P) {
  const int b = blockIdx.x;
  int lo[3], n[3];
  bool clipped = false;
  const int dim_lo[3] = {P.lo_z, 0, 0}, dim_hi[3] = {P.hi_z, P.ny, P.nx};
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const int w0 = P.ijk[3 * b + P.inv[a]] - P.pad;
    const int a0 = max(w0, dim_lo[a]), a1 = min(w0 + P.W, dim_hi[a]);
    lo[a] = a0;
    n[a] = max(0, a1 - a0);
    clipped |= n[a] < P.W;
  }
  float vmax = clipped ? 0.f : -CUDART_INF_F;
  bool nan = false;
  const int chunks = (n[2] + 31) >> 5;
  const int items = n[0] * n[1] * chunks;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float* base = P.vol + ((int64_t)(lo[0] - P.z0) * P.ny + lo[1]) * P.nx + lo[2];
#pragma unroll 4
  for (int it = warp; it < items; it += 8) {
    const int c = it % chunks, row = it / chunks;
    const int x = (c << 5) + lane;
    if (x < n[2]) {
      const int y = row % n[1], z = row / n[1];
      const float v = __ldg(base + ((int64_t)z * P.ny + y) * P.nx + x);
      nan |= v != v;
      vmax = fmaxf(vmax, v);
    }
  }
  __shared__ float red[8];
  __shared__ int any_nan;
  if (threadIdx.x == 0) any_nan = 0;
  for (int o = 16; o > 0; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
  if (lane == 0) red[warp] = vmax;
  __syncthreads();
  if (nan) any_nan = 1;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = red[0];
    for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
    P.out[b] = any_nan ? CUDART_NAN_F : m;
  }
}

__global__ void init_flags_kernel(int32_t* nonzero, float* cube_max, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (nonzero) nonzero[i] = 0;
  if (cube_max) cube_max[i] = -CUDART_INF_F;
}

}  // namespace mica

using namespace mica;

static thread_local int g_last_extract_path = -1;
extern "C" int mica_last_extract_path(void) { return g_last_extract_path; }

template <typename T>
static int extract_cubes_impl(const float* vol, int64_t chan_stride, int n_channels, int nz, int ny, int nx, int z0,
                              int nz_local, const int perm[3], int grid_size, int padding, const int32_t* ijk,
                              int n_cubes, T* out, int64_t out_cube_stride, int32_t* nonzero, float* cube_max,
                              int orientation, cudaStream_t st) {
  Orientation ori;
  MICA_REQUIRE(orientation_decode(orientation, 1, &ori), "orientation %d is not in 0..47", orientation);
  MICA_REQUIRE(vol && perm && out && (ijk || n_cubes == 0), "null pointer");
  MICA_REQUIRE(n_channels > 0 && n_channels <= 65535, "bad channel count %d", n_channels);
  MICA_REQUIRE(nz > 0 && ny > 0 && nx > 0, "empty volume");
  MICA_REQUIRE(z0 >= 0 && nz_local > 0 && z0 + nz_local <= nz, "bad slab");
  MICA_REQUIRE(grid_size > 0 && padding >= 0, "bad grid_size/padding");
  int seen = 0;
  for (int m = 0; m < 3; ++m) {
    MICA_REQUIRE(perm[m] >= 0 && perm[m] < 3, "perm must be a permutation of 0,1,2");
    seen |= 1 << perm[m];
  }
  MICA_REQUIRE(seen == 7, "perm must be a permutation of 0,1,2");
  const int W = grid_size + 2 * padding;
  MICA_REQUIRE(W <= 65535, "window too large");
  if (n_cubes <= 0) return MICA_OK;

  ExtractParams P;
  const int memdims[3] = {nz, ny, nx};
  const int64_t memstride[3] = {(int64_t)ny * nx, nx, 1};
  P.vol = vol;
  P.chan_stride = chan_stride;
  P.slab_axis = 0;
  for (int m = 0; m < 3; ++m) {
    P.T[m] = memdims[perm[m]];
    P.sstride[m] = memstride[perm[m]];
    if (perm[m] == 0) P.slab_axis = m;
  }
  P.z0 = z0;
  P.nzl = nz_local;
  P.W = W;
  P.pad = padding;
  P.out = out;
  P.out_cube_stride = out_cube_stride;
  P.nonzero = nonzero;
  P.cube_max = cube_max;

  const int contiguous_axis = perm[0] == 2 ? 0 : (perm[1] == 2 ? 1 : 2);
  if (orientation != 0) {
    ExtractParams Q = P;  // in output axes: output axis a walks window axis ori.perm[a]
    OrientAxes A;
    for (int a = 0; a < 3; ++a) {
      Q.T[a] = P.T[ori.perm[a]];
      Q.sstride[a] = P.sstride[ori.perm[a]];
      A.cax[a] = ori.perm[a];
      A.dir[a] = ori.flip[a] ? -1 : 1;
    }
    Q.slab_axis = ori.inv[P.slab_axis];
    const int mc = ori.inv[contiguous_axis];
    const int kMaxZ = 32768;
    for (int b0 = 0; b0 < n_cubes; b0 += kMaxZ) {
      const int nb = (n_cubes - b0 < kMaxZ) ? n_cubes - b0 : kMaxZ;
      Q.ijk = ijk + 3 * (int64_t)b0;
      Q.out = out + (int64_t)b0 * out_cube_stride;
      Q.nonzero = nonzero ? nonzero + b0 : nullptr;
      Q.cube_max = cube_max ? cube_max + b0 : nullptr;
      if (nonzero || cube_max) {
        init_flags_kernel<<<(nb + 255) / 256, 256, 0, st>>>(Q.nonzero, Q.cube_max, nb);
        MICA_LAUNCH_CHECK("init_flags_kernel");
      }
      dim3 grid(W, nb, n_channels), block(32, 8);
      if (mc == 2)
        extract_oriented_kernel<2, T><<<grid, block, 0, st>>>(Q, A);
      else if (mc == 0)
        extract_oriented_kernel<0, T><<<grid, block, 0, st>>>(Q, A);
      else
        extract_oriented_kernel<1, T><<<grid, block, 0, st>>>(Q, A);
      g_last_extract_path = 3;
      MICA_LAUNCH_CHECK("extract_oriented_kernel");
    }
    return MICA_OK;
  }

  // TMA path: standard layout, window a multiple of 32, 16-byte aligned base / rows / channels
  CUtensorMap tmap;
  bool use_tma = false;
  const size_t tma_smem = (size_t)kTmaBT * W * 128 + 1024;
  if (contiguous_axis == 0 && W % 32 == 0 && W <= 256 && nx % 4 == 0 && chan_stride % 4 == 0 &&
      ((uintptr_t)vol & 15) == 0 && !getenv("MICA_NO_TMA")) {
    TensorMapEncodeFn enc = tensor_map_encode_fn();
    if (enc) {
      const int local[3] = {nz_local, ny, nx};
      // dims: (x, axis walked by c, axis walked by b, channel)
      cuuint64_t gdim[4] = {(cuuint64_t)nx, (cuuint64_t)local[perm[2]], (cuuint64_t)local[perm[1]],
                            (cuuint64_t)n_channels};
      cuuint64_t gstr[3] = {(cuuint64_t)memstride[perm[2]] * 4, (cuuint64_t)memstride[perm[1]] * 4,
                            (cuuint64_t)(n_channels > 1 ? chan_stride : (int64_t)nz_local * ny * nx) * 4};
      cuuint32_t box[4] = {32, (cuuint32_t)W, (cuuint32_t)kTmaBT, 1};
      cuuint32_t estr[4] = {1, 1, 1, 1};
      // L2 promotion: 64B measured best of none / 64B / 128B / 256B on B200
      CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)vol, gdim, gstr, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_64B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r == CUDA_SUCCESS) {
        use_tma = true;
        MICA_CUDA(cudaFuncSetAttribute(extract_tma_kernel<kTmaBT, T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)tma_smem));
      }
    }
  }
  const int kMaxZ = 32768;
  for (int b0 = 0; b0 < n_cubes; b0 += kMaxZ) {
    const int nb = (n_cubes - b0 < kMaxZ) ? n_cubes - b0 : kMaxZ;
    P.ijk = ijk + 3 * (int64_t)b0;
    P.out = out + (int64_t)b0 * out_cube_stride;
    P.nonzero = nonzero ? nonzero + b0 : nullptr;
    P.cube_max = cube_max ? cube_max + b0 : nullptr;
    if (nonzero || cube_max) {
      init_flags_kernel<<<(nb + 255) / 256, 256, 0, st>>>(P.nonzero, P.cube_max, nb);
      MICA_LAUNCH_CHECK("init_flags_kernel");
    }
    dim3 grid(W, nb, n_channels), block(32, 8);
    if (use_tma) {
      TmaExtractParams TP;
      TP.ijk = P.ijk;
      TP.out = P.out;
      TP.out_cube_stride = out_cube_stride;
      TP.nonzero = P.nonzero;
      TP.cube_max = P.cube_max;
      TP.W = W;
      TP.pad = padding;
      TP.off_c = perm[2] == 0 ? z0 : 0;
      TP.off_b = perm[1] == 0 ? z0 : 0;
      dim3 tgrid((W / 32) * (W / kTmaBT), nb, n_channels);
      extract_tma_kernel<kTmaBT, T><<<tgrid, 256, tma_smem, st>>>(tmap, TP);
    } else if (contiguous_axis == 2)
      extract_rows_kernel<T><<<grid, block, 0, st>>>(P);
    else if (contiguous_axis == 0)
      extract_transpose_kernel<0, T><<<grid, block, 0, st>>>(P);
    else
      extract_transpose_kernel<1, T><<<grid, block, 0, st>>>(P);
    g_last_extract_path = use_tma ? 2 : (contiguous_axis == 2 ? 0 : 1);
    MICA_LAUNCH_CHECK("extract_cubes kernel");
  }
  return MICA_OK;
}

extern "C" int mica_extract_cubes_as(const float* vol, int64_t chan_stride, int n_channels, int nz, int ny, int nx,
                                     int z0, int nz_local, const int perm[3], int grid_size, int padding,
                                     const int32_t* ijk, int n_cubes, void* out, int out_dtype,
                                     int64_t out_cube_stride, int32_t* nonzero, float* cube_max, int orientation,
                                     mica_stream_t stream) {
  MICA_REQUIRE(model_dtype_bytes(out_dtype), "cube output dtype %d: must be MICA_DTYPE_F32 or MICA_DTYPE_BF16",
               out_dtype);
  if (out_dtype == MICA_DTYPE_BF16)
    return extract_cubes_impl(vol, chan_stride, n_channels, nz, ny, nx, z0, nz_local, perm, grid_size, padding, ijk,
                              n_cubes, static_cast<__nv_bfloat16*>(out), out_cube_stride, nonzero, cube_max,
                              orientation, (cudaStream_t)stream);
  return extract_cubes_impl(vol, chan_stride, n_channels, nz, ny, nx, z0, nz_local, perm, grid_size, padding, ijk,
                            n_cubes, static_cast<float*>(out), out_cube_stride, nonzero, cube_max, orientation,
                            (cudaStream_t)stream);
}

extern "C" int mica_extract_cubes_oriented(const float* vol, int64_t chan_stride, int n_channels,
                                           int nz, int ny, int nx, int z0, int nz_local, const int perm[3],
                                           int grid_size, int padding, const int32_t* ijk, int n_cubes,
                                           float* out, int64_t out_cube_stride, int32_t* nonzero, float* cube_max,
                                           int orientation, mica_stream_t stream) {
  return mica_extract_cubes_as(vol, chan_stride, n_channels, nz, ny, nx, z0, nz_local, perm, grid_size, padding, ijk,
                               n_cubes, out, MICA_DTYPE_F32, out_cube_stride, nonzero, cube_max, orientation, stream);
}

extern "C" int mica_cube_window_max(const float* vol, int nz, int ny, int nx, int z0, int nz_local,
                                    const int perm[3], int grid_size, int padding, const int32_t* ijk, int n_cubes,
                                    float* out, mica_stream_t stream) {
  MICA_REQUIRE(vol && perm && (out || n_cubes == 0) && (ijk || n_cubes == 0), "null pointer");
  MICA_REQUIRE(nz > 0 && ny > 0 && nx > 0, "empty volume");
  MICA_REQUIRE(z0 >= 0 && nz_local > 0 && z0 + nz_local <= nz, "bad slab");
  MICA_REQUIRE(grid_size > 0 && padding >= 0, "bad grid_size/padding");
  MICA_REQUIRE(n_cubes >= 0, "bad cube count %d", n_cubes);
  WindowMaxParams P;
  int seen = 0;
  for (int m = 0; m < 3; ++m) {
    MICA_REQUIRE(perm[m] >= 0 && perm[m] < 3, "perm must be a permutation of 0,1,2");
    seen |= 1 << perm[m];
    P.inv[perm[m]] = m;
  }
  MICA_REQUIRE(seen == 7, "perm must be a permutation of 0,1,2");
  const int64_t W = (int64_t)grid_size + 2 * (int64_t)padding;
  MICA_REQUIRE(W <= 65535, "window too large");
  if (n_cubes == 0) return MICA_OK;
  P.vol = vol;
  P.ny = ny;
  P.nx = nx;
  P.lo_z = z0;
  P.hi_z = z0 + nz_local;
  P.z0 = z0;
  P.W = (int)W;
  P.pad = padding;
  P.ijk = ijk;
  P.out = out;
  cube_window_max_kernel<<<n_cubes, 256, 0, (cudaStream_t)stream>>>(P);
  MICA_LAUNCH_CHECK("cube_window_max_kernel");
  return MICA_OK;
}

extern "C" int mica_extract_cubes(const float* vol, int64_t chan_stride, int n_channels,
                                  int nz, int ny, int nx, int z0, int nz_local, const int perm[3],
                                  int grid_size, int padding, const int32_t* ijk, int n_cubes,
                                  float* out, int64_t out_cube_stride, int32_t* nonzero, float* cube_max,
                                  mica_stream_t stream) {
  return mica_extract_cubes_oriented(vol, chan_stride, n_channels, nz, ny, nx, z0, nz_local, perm, grid_size,
                                     padding, ijk, n_cubes, out, out_cube_stride, nonzero, cube_max, 0, stream);
}
