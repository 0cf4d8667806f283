// R4: 24-channel AF3 rasteriser.
//
// Replaces transform_coordinates + the per-atom Python loop at
// utils/preprocessing.py:172-178,275-298 (reference root).  Each atom marks one
// voxel in its backbone channel (CA,N,C,O) and one in its residue-type channel.
// Stores of 1.0f are idempotent, so the scatter needs no atomics and is
// order-independent (bit-exact).  Traffic is the zero fill (96 B/voxel); the
// scatter itself touches < 2 sectors per atom.
#include "common.cuh"

namespace mica {

__global__ void __launch_bounds__(256)
fill_zero_kernel(float4* __restrict__ p4, long long n4, float* __restrict__ tail, int ntail) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) p4[i] = z;
  if (blockIdx.x == 0 && threadIdx.x < ntail) tail[threadIdx.x] = 0.f;
}

int fill_zero(float* p, long long n, cudaStream_t st) {
  if (n <= 0) return MICA_OK;
  // align the head to 16 bytes with the scalar tail path (cudaMalloc'd buffers already are)
  long long head = (((uintptr_t)p & 15) == 0) ? 0 : ((16 - ((uintptr_t)p & 15)) / 4);
  if (head > n) head = n;
  if (head) {
    fill_zero_kernel<<<1, 32, 0, st>>>(nullptr, 0, p, (int)head);
    MICA_LAUNCH_CHECK("fill_zero_kernel(head)");
  }
  float* q = p + head;
  long long m = n - head, n4 = m >> 2;
  int64_t want = ceil_div64(n4 > 0 ? n4 : 1, 256 * 4);
  int grid = (int)(want < (int64_t)kNumSMs * 8 ? want : (int64_t)kNumSMs * 8);
  fill_zero_kernel<<<grid, 256, 0, st>>>((float4*)q, n4, q + n4 * 4, (int)(m & 3));
  MICA_LAUNCH_CHECK("fill_zero_kernel");
  return MICA_OK;
}

__global__ void __launch_bounds__(256)
af3_scatter_kernel(const float* __restrict__ xyz, const int8_t* __restrict__ bb_ch,
                   const int8_t* __restrict__ aa_ch, long long n_atoms, float ox, float oy, float oz,
                   int clip_x, int clip_y, int clip_z, int nz, int ny, int nx, int z0, int nz_local,
                   float* __restrict__ vol, int* __restrict__ status_oob) {
  long long a = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n_atoms) return;
  // np.round(coord - origin) in float32, round-half-even; then clip(., 0, shape - 1)
  float fx = rintf(__fsub_rn(xyz[3 * a + 0], ox));
  float fy = rintf(__fsub_rn(xyz[3 * a + 1], oy));
  float fz = rintf(__fsub_rn(xyz[3 * a + 2], oz));
  // float -> int64 as numpy astype(int); clamp in float first so the cast cannot overflow
  long long ix = (long long)fminf(fmaxf(fx, -4.0e18f), 4.0e18f);
  long long iy = (long long)fminf(fmaxf(fy, -4.0e18f), 4.0e18f);
  long long iz = (long long)fminf(fmaxf(fz, -4.0e18f), 4.0e18f);
  ix = ix < 0 ? 0 : (ix > clip_x ? clip_x : ix);
  iy = iy < 0 ? 0 : (iy > clip_y ? clip_y : iy);
  iz = iz < 0 ? 0 : (iz > clip_z ? clip_z : iz);
  const int b = bb_ch[a], r = aa_ch[a];
  if (b < 0 && r < 0) return;                 // the reference indexes the volume only when it writes
  if (ix >= nx || iy >= ny || iz >= nz) {     // numpy would raise IndexError (D7) -> encoding fails
    atomicExch(status_oob, 1);
    return;
  }
  const long long zl = iz - z0;
  if (zl < 0 || zl >= nz_local) return;       // another rank's slab
  const long long chan = (long long)nz_local * ny * nx;
  const long long off = (zl * ny + iy) * nx + ix;
  if (b >= 0) vol[b * chan + off] = 1.0f;
  if (r >= 0) vol[r * chan + off] = 1.0f;
}

}  // namespace mica

using namespace mica;

extern "C" int mica_af3_encode(const float* xyz, const int8_t* bb_ch, const int8_t* aa_ch, int64_t n_atoms,
                               float ox, float oy, float oz, int clip_x, int clip_y, int clip_z,
                               int nz, int ny, int nx, int z0, int nz_local,
                               float* vol24, int* status_oob, mica_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  MICA_REQUIRE(vol24 && status_oob, "null pointer");
  MICA_REQUIRE(n_atoms == 0 || (xyz && bb_ch && aa_ch), "null atom arrays");
  MICA_REQUIRE(nz > 0 && ny > 0 && nx > 0, "empty grid");
  MICA_REQUIRE(z0 >= 0 && nz_local >= 0 && z0 + nz_local <= nz, "bad slab");
  MICA_REQUIRE(clip_x >= 0 && clip_y >= 0 && clip_z >= 0, "negative clip bound");
  MICA_CUDA(cudaMemsetAsync(status_oob, 0, sizeof(int), st));
  int rc = fill_zero(vol24, 24LL * nz_local * ny * nx, st);
  if (rc) return rc;
  if (n_atoms > 0 && nz_local > 0) {
    af3_scatter_kernel<<<(unsigned)ceil_div64(n_atoms, 256), 256, 0, st>>>(
        xyz, bb_ch, aa_ch, n_atoms, ox, oy, oz, clip_x, clip_y, clip_z, nz, ny, nx, z0, nz_local, vol24,
        status_oob);
    MICA_LAUNCH_CHECK("af3_scatter_kernel");
  }
  return MICA_OK;
}

// ===========================================================================
// R4 + R5 fused: AF3 channels of the cube batch straight from the atoms.
//
// The 24-channel volume is ~1e-4 dense (one voxel per atom per channel), yet the reference
// materialises it densely (utils/preprocessing.py:268), writes 24 MRC files, re-reads them,
// pads them and cuts 24 x n_cubes windows out of them (utils/create_grids.py:269-352).
// Here the atoms are binned per cube once per map (count -> scan -> fill), and each batch's
// [B,24,W,W,W] model input is kept as "all zeros except this batch's atom voxels": a slot's
// previous cube is un-scattered (0.0f at its listed voxels) and the new cube scattered
// (1.0f).  The tensor handed to the model is bit-identical to extract(encode(atoms)).
namespace mica {

struct BinParams {
  int T[3];        // cube-space dims
  int ncube[3];    // cubes per axis
  int S, pad, W;
  int perm[3];     // cube axis m walks memory axis perm[m]; memory index = (z, y, x)
};

struct BinWorkspace {
  int* counts;          // [n_cubes + 1]
  int* offsets;         // [n_cubes + 1]
  int* cursor;          // [n_cubes]
  unsigned* entries;    // [capacity]
  long long capacity;
};

__device__ __forceinline__ bool atom_voxel(const float* __restrict__ xyz, long long a, float ox, float oy, float oz,
                                           int clip_x, int clip_y, int clip_z, int nz, int ny, int nx, int mem[3]) {
  float fx = rintf(__fsub_rn(xyz[3 * a + 0], ox));
  float fy = rintf(__fsub_rn(xyz[3 * a + 1], oy));
  float fz = rintf(__fsub_rn(xyz[3 * a + 2], oz));
  long long ix = (long long)fminf(fmaxf(fx, -4.0e18f), 4.0e18f);
  long long iy = (long long)fminf(fmaxf(fy, -4.0e18f), 4.0e18f);
  long long iz = (long long)fminf(fmaxf(fz, -4.0e18f), 4.0e18f);
  ix = ix < 0 ? 0 : (ix > clip_x ? clip_x : ix);
  iy = iy < 0 ? 0 : (iy > clip_y ? clip_y : iy);
  iz = iz < 0 ? 0 : (iz > clip_z ? clip_z : iz);
  mem[0] = (int)iz;
  mem[1] = (int)iy;
  mem[2] = (int)ix;
  return !(ix >= nx || iy >= ny || iz >= nz);
}

// FILL == false: count entries per cube; FILL == true: write the packed entries
template <bool FILL>
__global__ void __launch_bounds__(256)
af3_bin_kernel(const float* __restrict__ xyz, const int8_t* __restrict__ bb_ch, const int8_t* __restrict__ aa_ch,
               long long n_atoms, float ox, float oy, float oz, int clip_x, int clip_y, int clip_z, int nz, int ny,
               int nx, BinParams P, BinWorkspace ws, int* __restrict__ status_oob) {
  long long a = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n_atoms) return;
  const int b = bb_ch[a], r = aa_ch[a];
  if (b < 0 && r < 0) return;
  int mem[3];
  if (!atom_voxel(xyz, a, ox, oy, oz, clip_x, clip_y, clip_z, nz, ny, nx, mem)) {
    if (!FILL) atomicExch(status_oob, 1);
    return;
  }
  const int p[3] = {mem[P.perm[0]], mem[P.perm[1]], mem[P.perm[2]]};
  // cubes whose window [o - pad, o - pad + W) contains p, o a multiple of S inside the volume
  int lo[3], hi[3];
  for (int m = 0; m < 3; ++m) {
    int first = p[m] + P.pad - P.W + 1;                    // smallest admissible origin
    lo[m] = first <= 0 ? 0 : (first + P.S - 1) / P.S;      // as a cube index
    hi[m] = min((p[m] + P.pad) / P.S, P.ncube[m] - 1);
  }
  const unsigned chan = (unsigned)(b + 1) | ((unsigned)(r < 0 ? 0 : r - 3) << 3);   // 3 + 5 bits
  for (int c0 = lo[0]; c0 <= hi[0]; ++c0)
    for (int c1 = lo[1]; c1 <= hi[1]; ++c1)
      for (int c2 = lo[2]; c2 <= hi[2]; ++c2) {
        const int id = (c0 * P.ncube[1] + c1) * P.ncube[2] + c2;
        // the atoms of a residue are neighbours in the array and in space: lanes that hit the same
        // cube elect one leader for a single atomic (consecutive atoms would otherwise serialise)
        const unsigned peers = __match_any_sync(__activemask(), id);
        const int leader = __ffs(peers) - 1, lane = threadIdx.x & 31;
        const int rank = __popc(peers & ((1u << lane) - 1u));
        if (!FILL) {
          if (lane == leader) atomicAdd(&ws.counts[id], __popc(peers));
        } else {
          const int u0 = p[0] - (c0 * P.S - P.pad), u1 = p[1] - (c1 * P.S - P.pad), u2 = p[2] - (c2 * P.S - P.pad);
          const unsigned off = (unsigned)((u0 * P.W + u1) * P.W + u2);
          int base = 0;
          if (lane == leader) base = atomicAdd(&ws.cursor[id], __popc(peers));
          base = __shfl_sync(peers, base, leader);
          const long long pos = (long long)ws.offsets[id] + base + rank;
          if (pos < ws.capacity) ws.entries[pos] = (off << 8) | chan;
        }
      }
}

// single block: offsets = exclusive scan of counts; counts[n] / offsets[n] = total
__global__ void __launch_bounds__(1024)
af3_scan_kernel(BinWorkspace ws, int n) {
  __shared__ int warp_sums[32];
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < n; base += 1024) {
    const int i = base + threadIdx.x;
    const int v = i < n ? ws.counts[i] : 0;
    int incl = v;
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, incl, o);
      if ((threadIdx.x & 31) >= o) incl += t;
    }
    if ((threadIdx.x & 31) == 31) warp_sums[threadIdx.x >> 5] = incl;
    __syncthreads();
    if (threadIdx.x < 32) {
      int w = warp_sums[threadIdx.x];
      for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, w, o);
        if (threadIdx.x >= o) w += t;
      }
      warp_sums[threadIdx.x] = w;
    }
    __syncthreads();
    const int warp_off = (threadIdx.x >> 5) ? warp_sums[(threadIdx.x >> 5) - 1] : 0;
    if (i < n) {
      ws.offsets[i] = carry + warp_off + incl - v;
      ws.cursor[i] = 0;
    }
    __syncthreads();
    if (threadIdx.x == 1023) carry += warp_off + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) ws.offsets[n] = carry;
}

constexpr int kFillBlocks = 16;

__device__ __forceinline__ int cube_id_of(const BinParams& P, const int32_t* __restrict__ ijk, int slot) {
  return ((ijk[3 * slot] / P.S) * P.ncube[1] + ijk[3 * slot + 1] / P.S) * P.ncube[2] + ijk[3 * slot + 2] / P.S;
}

// grid = (kFillBlocks, slots), launched twice on the stream: SET == false clears the voxels of the cube
// slot b currently shows (ijk_prev[b], b < n_prev; clean otherwise), SET == true then sets those of
// ijk_next[b] (b < n_next; left clean otherwise).  A voxel can be in both lists, so "clear, then set"
// must stay ordered -- the kernel boundary does that, and inside a launch every entry is independent:
// the entries of a slot spread over kFillBlocks CTAs, which keeps densely populated cubes cheap.
// Stateless: the caller says what the slots hold, and in which orientation (test-time augmentation: the slots
// show every cube of the batch in one orientation, ops.orientation): an entry's window offset v is moved to the
// oriented offset base + v0 s[0] + v1 s[1] + v2 s[2] (Orientation), the identity for orientation 0.  A slot that
// keeps its cube but changes orientation is cleared and set again.
struct FillOrient {
  int oriented;  // 0: orientation 0, offsets used as binned
  int base, s[3];
};

// T: the buffer's element type, float or __nv_bfloat16 (1.0 and 0.0 are exact in both)
template <bool SET, typename T>
__global__ void __launch_bounds__(256)
af3_fill_cubes_kernel(BinWorkspace ws, BinParams P, const int32_t* __restrict__ ijk_prev, int n_prev,
                      const int32_t* __restrict__ ijk_next, int n_next, T* __restrict__ out,
                      int64_t out_cube_stride, int32_t* __restrict__ nonzero, FillOrient o, bool same_orientation) {
  const int slot = blockIdx.y;
  const int prev = slot < n_prev ? cube_id_of(P, ijk_prev, slot) : -1;
  const int next = slot < n_next ? cube_id_of(P, ijk_next, slot) : -1;
  if (SET && blockIdx.x == 0 && threadIdx.x == 0 && nonzero && next >= 0)
    nonzero[slot] = (ws.offsets[next + 1] > ws.offsets[next]) ? 1 : 0;
  const int id = SET ? next : prev;
  if (id < 0 || (prev == next && same_orientation)) return;
  T* cube = out + (int64_t)slot * out_cube_stride;
  const int64_t W3 = (int64_t)P.W * P.W * P.W;
  const float val = SET ? 1.0f : 0.0f;
  const int e0 = ws.offsets[id], e1 = ws.offsets[id + 1];
  for (int e = e0 + blockIdx.x * 256 + threadIdx.x; e < e1; e += kFillBlocks * 256) {
    const unsigned v = ws.entries[e];
    const unsigned b = v & 7u, r = (v >> 3) & 31u;
    unsigned off = v >> 8;
    if (o.oriented) {
      const int W = P.W, v0 = (int)off / (W * W), v1 = ((int)off / W) % W, v2 = (int)off % W;
      off = (unsigned)(o.base + v0 * o.s[0] + v1 * o.s[1] + v2 * o.s[2]);
    }
    if (b) st_plain_el(cube + (int64_t)(b - 1) * W3 + off, val);
    if (r) st_plain_el(cube + (int64_t)(r + 3) * W3 + off, val);
  }
}

static size_t a256(size_t v) { return (v + 255) / 256 * 256; }

static BinWorkspace carve(void* workspace, int n_cubes, long long capacity) {
  char* p = (char*)(((uintptr_t)workspace + 255) / 256 * 256);
  BinWorkspace ws;
  ws.counts = (int*)p;
  p += a256(sizeof(int) * (n_cubes + 1));
  ws.offsets = (int*)p;
  p += a256(sizeof(int) * (n_cubes + 1));
  ws.cursor = (int*)p;
  p += a256(sizeof(int) * (n_cubes + 1));
  ws.entries = (unsigned*)p;
  ws.capacity = capacity;
  return ws;
}

static int make_bin_params(BinParams& P, int nz, int ny, int nx, const int perm[3], int grid_size, int padding) {
  MICA_REQUIRE(perm, "null perm");
  int seen = 0;
  const int memdims[3] = {nz, ny, nx};
  for (int m = 0; m < 3; ++m) {
    MICA_REQUIRE(perm[m] >= 0 && perm[m] < 3, "perm must be a permutation of 0,1,2");
    seen |= 1 << perm[m];
    P.perm[m] = perm[m];
    P.T[m] = memdims[perm[m]];
    P.ncube[m] = (P.T[m] + grid_size - 1) / grid_size;
  }
  MICA_REQUIRE(seen == 7, "perm must be a permutation of 0,1,2");
  MICA_REQUIRE(grid_size > 0 && padding >= 0, "bad grid_size/padding");
  P.S = grid_size;
  P.pad = padding;
  P.W = grid_size + 2 * padding;
  MICA_REQUIRE(P.W <= 256, "window larger than 256 is not supported by the packed atom entries");
  MICA_REQUIRE((long long)P.ncube[0] * P.ncube[1] * P.ncube[2] < (1LL << 30), "too many cubes");
  return MICA_OK;
}

static long long bin_capacity(long long n_atoms, int grid_size, int padding) {
  const int W = grid_size + 2 * padding;
  const long long per_axis = (W + grid_size - 1) / grid_size;
  return n_atoms * per_axis * per_axis * per_axis;
}

}  // namespace mica

extern "C" size_t mica_af3_bins_workspace_bytes(int64_t n_atoms, int nz, int ny, int nx, const int perm[3],
                                                int grid_size, int padding) {
  BinParams P;
  if (make_bin_params(P, nz, ny, nx, perm, grid_size, padding) != MICA_OK) return 0;
  const long long n_cubes = (long long)P.ncube[0] * P.ncube[1] * P.ncube[2];
  return 3 * a256(sizeof(int) * (n_cubes + 1)) + a256(sizeof(unsigned) * (size_t)bin_capacity(n_atoms, grid_size, padding)) + 512;
}

extern "C" int mica_af3_bin_atoms(const float* xyz, const int8_t* bb_ch, const int8_t* aa_ch, int64_t n_atoms,
                                  float ox, float oy, float oz, int clip_x, int clip_y, int clip_z,
                                  int nz, int ny, int nx, const int perm[3], int grid_size, int padding,
                                  void* workspace, size_t workspace_bytes, int* status_oob, mica_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  MICA_REQUIRE(workspace && status_oob, "null pointer");
  MICA_REQUIRE(n_atoms == 0 || (xyz && bb_ch && aa_ch), "null atom arrays");
  MICA_REQUIRE(nz > 0 && ny > 0 && nx > 0, "empty grid");
  BinParams P;
  int rc = make_bin_params(P, nz, ny, nx, perm, grid_size, padding);
  if (rc) return rc;
  if (workspace_bytes < mica_af3_bins_workspace_bytes(n_atoms, nz, ny, nx, perm, grid_size, padding))
    return set_error(MICA_ERR_WORKSPACE, "af3 bins workspace too small");
  const int n_cubes = P.ncube[0] * P.ncube[1] * P.ncube[2];
  BinWorkspace ws = carve(workspace, n_cubes, bin_capacity(n_atoms, grid_size, padding));
  MICA_CUDA(cudaMemsetAsync(status_oob, 0, sizeof(int), st));
  MICA_CUDA(cudaMemsetAsync(ws.counts, 0, sizeof(int) * (n_cubes + 1), st));
  const unsigned blocks = (unsigned)ceil_div64(n_atoms > 0 ? n_atoms : 1, 256);
  if (n_atoms > 0) {
    af3_bin_kernel<false><<<blocks, 256, 0, st>>>(xyz, bb_ch, aa_ch, n_atoms, ox, oy, oz, clip_x, clip_y, clip_z, nz,
                                                  ny, nx, P, ws, status_oob);
    MICA_LAUNCH_CHECK("af3_bin_kernel<count>");
  }
  af3_scan_kernel<<<1, 1024, 0, st>>>(ws, n_cubes);
  MICA_LAUNCH_CHECK("af3_scan_kernel");
  if (n_atoms > 0) {
    af3_bin_kernel<true><<<blocks, 256, 0, st>>>(xyz, bb_ch, aa_ch, n_atoms, ox, oy, oz, clip_x, clip_y, clip_z, nz,
                                                 ny, nx, P, ws, status_oob);
    MICA_LAUNCH_CHECK("af3_bin_kernel<fill>");
  }
  return MICA_OK;
}

static FillOrient fill_orient(int code, int W) {
  Orientation ori;
  orientation_decode(code, W, &ori);
  FillOrient o;
  o.oriented = code != 0;
  o.base = ori.base;
  for (int m = 0; m < 3; ++m) o.s[m] = ori.s[m];
  return o;
}

template <typename T>
static int af3_fill_cubes_impl(const void* workspace, int64_t n_atoms, int nz, int ny, int nx, const int perm[3],
                               int grid_size, int padding, const int32_t* ijk_prev, int n_prev,
                               const int32_t* ijk_next, int n_next, T* out, int64_t out_cube_stride,
                               int32_t* nonzero, int orientation_prev, int orientation_next, cudaStream_t stream) {
  MICA_REQUIRE(workspace && out, "null pointer");
  Orientation ori;
  MICA_REQUIRE(orientation_decode(orientation_prev, 1, &ori) && orientation_decode(orientation_next, 1, &ori),
               "orientations %d, %d: each must be in 0..47", orientation_prev, orientation_next);
  MICA_REQUIRE(n_prev >= 0 && n_next >= 0 && (ijk_prev || n_prev == 0) && (ijk_next || n_next == 0), "bad slot lists");
  BinParams P;
  int rc = make_bin_params(P, nz, ny, nx, perm, grid_size, padding);
  if (rc) return rc;
  const int n_slots = n_prev > n_next ? n_prev : n_next;
  if (n_slots <= 0) return MICA_OK;
  MICA_REQUIRE(n_slots <= 65535, "too many slots");
  const int n_cubes = P.ncube[0] * P.ncube[1] * P.ncube[2];
  BinWorkspace ws = carve(const_cast<void*>(workspace), n_cubes, bin_capacity(n_atoms, grid_size, padding));
  if (n_prev > 0) {
    af3_fill_cubes_kernel<false, T><<<dim3(kFillBlocks, n_prev), 256, 0, stream>>>(
        ws, P, ijk_prev, n_prev, ijk_next, n_next, out, out_cube_stride, nonzero, fill_orient(orientation_prev, P.W),
        orientation_prev == orientation_next);
    MICA_LAUNCH_CHECK("af3_fill_cubes_kernel<clear>");
  }
  if (n_next > 0) {
    af3_fill_cubes_kernel<true, T><<<dim3(kFillBlocks, n_next), 256, 0, stream>>>(
        ws, P, ijk_prev, n_prev, ijk_next, n_next, out, out_cube_stride, nonzero, fill_orient(orientation_next, P.W),
        orientation_prev == orientation_next);
    MICA_LAUNCH_CHECK("af3_fill_cubes_kernel<set>");
  }
  return MICA_OK;
}

extern "C" int mica_af3_fill_cubes_as(const void* workspace, int64_t n_atoms, int nz, int ny, int nx,
                                      const int perm[3], int grid_size, int padding, const int32_t* ijk_prev,
                                      int n_prev, const int32_t* ijk_next, int n_next, void* out, int out_dtype,
                                      int64_t out_cube_stride, int32_t* nonzero, int orientation_prev,
                                      int orientation_next, mica_stream_t stream) {
  MICA_REQUIRE(model_dtype_bytes(out_dtype), "AF3 cube dtype %d: must be MICA_DTYPE_F32 or MICA_DTYPE_BF16",
               out_dtype);
  if (out_dtype == MICA_DTYPE_BF16)
    return af3_fill_cubes_impl(workspace, n_atoms, nz, ny, nx, perm, grid_size, padding, ijk_prev, n_prev, ijk_next,
                               n_next, static_cast<__nv_bfloat16*>(out), out_cube_stride, nonzero, orientation_prev,
                               orientation_next, (cudaStream_t)stream);
  return af3_fill_cubes_impl(workspace, n_atoms, nz, ny, nx, perm, grid_size, padding, ijk_prev, n_prev, ijk_next,
                             n_next, static_cast<float*>(out), out_cube_stride, nonzero, orientation_prev,
                             orientation_next, (cudaStream_t)stream);
}

extern "C" int mica_af3_fill_cubes_oriented(const void* workspace, int64_t n_atoms, int nz, int ny, int nx,
                                            const int perm[3], int grid_size, int padding, const int32_t* ijk_prev,
                                            int n_prev, const int32_t* ijk_next, int n_next, float* out,
                                            int64_t out_cube_stride, int32_t* nonzero, int orientation_prev,
                                            int orientation_next, mica_stream_t stream) {
  return mica_af3_fill_cubes_as(workspace, n_atoms, nz, ny, nx, perm, grid_size, padding, ijk_prev, n_prev, ijk_next,
                                n_next, out, MICA_DTYPE_F32, out_cube_stride, nonzero, orientation_prev,
                                orientation_next, stream);
}

extern "C" int mica_af3_fill_cubes(const void* workspace, int64_t n_atoms, int nz, int ny, int nx, const int perm[3],
                                   int grid_size, int padding, const int32_t* ijk_prev, int n_prev,
                                   const int32_t* ijk_next, int n_next, float* out, int64_t out_cube_stride,
                                   int32_t* nonzero, mica_stream_t stream) {
  return mica_af3_fill_cubes_oriented(workspace, n_atoms, nz, ny, nx, perm, grid_size, padding, ijk_prev, n_prev,
                                      ijk_next, n_next, out, out_cube_stride, nonzero, 0, 0, stream);
}
