// Prediction maps: the four stitched volumes (cube space [X,Y,Z], the working map's memory axes permuted by perm)
// resampled trilinearly onto a target grid in the target's memory order [c][nz][ny][nx] -- the input map's grid or the
// working grid -- with the amino-acid label taken as the arg-max of the 20 resampled probabilities.
// Definition: oracle/prediction_maps_oracle.py (float64 weights, products and sums rounded in the oracle's order).
//
// One CTA per target tile.  Target x is the tile's fastest axis (coalesced stores); the memory axis that is the cube
// volumes' fastest axis gets a long edge too, so the support box each channel needs is loaded along rows of the
// volume.  Per channel the box goes to shared memory once and every target voxel of the tile reads its 8 corners
// there: a working voxel comes from DRAM about once per channel whatever the perm.
#include "common.cuh"

namespace mica {
namespace {

constexpr int kMapsThreads = 256;
constexpr int kMapsTileX = 32;          // target x per tile: one warp stores 32 consecutive floats
constexpr int kMapsOutPerThread = 4;    // a tile holds at most 32 * 32 targets
constexpr int kMapsChannels = 22;       // backbone, C-alpha, 20 amino-acid probabilities (the stitched label unread)
constexpr int kMapsTableBytes = 3 * kMapsTileX * (2 * 8 + 2 * 4);
constexpr size_t kMapsSmemDefault = 48 * 1024;
constexpr size_t kMapsSmemMax = 200 * 1024;

struct MapsParams {
  const float *bb, *ca, *prob;      // cube space [X,Y,Z]; prob [20][X,Y,Z]
  float *out_bb, *out_ca, *out_pred, *out_prob;  // target memory order [nz,ny,nx]; out_prob [20][nz,ny,nx]
  int64_t n_w, n_s;                 // voxels of one working / target channel
  int cdim[3];                      // X, Y, Z
  int perm[3];                      // cube axis a walks memory axis perm[a]
  int nw[3], ns[3];                 // working / target shape, memory axes (z, y, x)
  int tile[3], ntile[3];            // targets per tile and tiles, memory axes
  int sstride[3];                   // shared-memory stride of memory axis m in the box
  int pad[2];                       // padded box extents of cube axes 1 and 2
};

// oracle/prediction_maps_oracle.py::axis_coords: the integer product, one float64 division, no other rounding
__host__ __device__ __forceinline__ void maps_axis_coord(int s, int n_s, int n_w, int* i0, int* i1, double* t) {
  double c = 0.0;
#ifdef __CUDA_ARCH__
  if (n_s > 1) c = __ddiv_rn((double)((long long)s * (n_w - 1)), (double)(n_s - 1));
#else
  if (n_s > 1) c = (double)((long long)s * (n_w - 1)) / (double)(n_s - 1);
#endif
  const int f = (int)floor(c);
  const int top = n_w - 2 > 0 ? n_w - 2 : 0;
  *i0 = f < top ? f : top;
  *i1 = *i0 + 1 < n_w - 1 ? *i0 + 1 : n_w - 1;
#ifdef __CUDA_ARCH__
  *t = __dsub_rn(c, (double)*i0);
#else
  *t = c - (double)*i0;
#endif
}

__global__ void __launch_bounds__(kMapsThreads, 3)
volumes_to_grid_kernel(MapsParams P) {
  extern __shared__ __align__(16) unsigned char maps_smem[];
  double* tw = reinterpret_cast<double*>(maps_smem);       // [3][32] t
  double* tw1 = tw + 3 * kMapsTileX;                       // [3][32] 1 - t
  int* toff = reinterpret_cast<int*>(tw1 + 3 * kMapsTileX);  // [3][32] (i0 - box origin) * shared stride
  int* tdel = toff + 3 * kMapsTileX;                       // [3][32] (i1 - i0) * shared stride
  float* buf = reinterpret_cast<float*>(maps_smem + kMapsTableBytes);

  int64_t b = blockIdx.x;
  int tc[3];
  tc[2] = (int)(b % P.ntile[2]);
  b /= P.ntile[2];
  tc[1] = (int)(b % P.ntile[1]);
  tc[0] = (int)(b / P.ntile[1]);
  int s0[3], cnt[3], lo[3], span[3];
#pragma unroll
  for (int m = 0; m < 3; ++m) {
    s0[m] = tc[m] * P.tile[m];
    cnt[m] = min(P.tile[m], P.ns[m] - s0[m]);
    int a0, a1, b0, b1;
    double t;
    maps_axis_coord(s0[m], P.ns[m], P.nw[m], &a0, &a1, &t);
    maps_axis_coord(s0[m] + cnt[m] - 1, P.ns[m], P.nw[m], &b0, &b1, &t);
    lo[m] = a0;
    span[m] = b1 - a0 + 1;
  }
  if (threadIdx.x < 3 * kMapsTileX) {
    const int m = threadIdx.x / kMapsTileX, j = threadIdx.x % kMapsTileX;
    if (j < cnt[m]) {
      int i0, i1;
      double t;
      maps_axis_coord(s0[m] + j, P.ns[m], P.nw[m], &i0, &i1, &t);
      tw[threadIdx.x] = t;
      tw1[threadIdx.x] = __dsub_rn(1.0, t);
      toff[threadIdx.x] = (i0 - lo[m]) * P.sstride[m];
      tdel[threadIdx.x] = (i1 - i0) * P.sstride[m];
    }
  }
  // the box in cube order: extents B, origin L (cube coordinates), padded extents for cube axes 1 and 2
  const int B0 = span[P.perm[0]], B1 = span[P.perm[1]], B2 = span[P.perm[2]];
  const int L0 = lo[P.perm[0]], L1 = lo[P.perm[1]], L2 = lo[P.perm[2]];
  const int nbox = B0 * B1 * B2;
  __syncthreads();

  // the targets of this thread: o = threadIdx.x + 256 k, target x fastest in the tile, so a warp stores 32 consecutive
  // x and a thread's x (its lane) is the same for every k: the x weights live in registers, the y and z ones are the
  // same across the warp and come from the shared tables as broadcasts
  const int jx = threadIdx.x % kMapsTileX;
  const double wx = tw[2 * kMapsTileX + jx], ux = tw1[2 * kMapsTileX + jx];
  const int dx = tdel[2 * kMapsTileX + jx];
  int jyz[kMapsOutPerThread];         // y | z << 8 tile indices, -1 outside the target grid
  int base[kMapsOutPerThread];
#pragma unroll
  for (int k = 0; k < kMapsOutPerThread; ++k) {
    const int r = threadIdx.x / kMapsTileX + k * (kMapsThreads / kMapsTileX);
    const int jy = r % P.tile[1], jz = r / P.tile[1];
    const bool ok = jz < cnt[0] && jy < cnt[1] && jx < cnt[2];
    jyz[k] = ok ? (jy | jz << 8) : -1;
    base[k] = ok ? toff[jz] + toff[kMapsTileX + jy] + toff[2 * kMapsTileX + jx] : 0;
  }
  float best[kMapsOutPerThread];
  int arg[kMapsOutPerThread];

  for (int ch = 0; ch < kMapsChannels; ++ch) {
    const float* src = ch == 0 ? P.bb : (ch == 1 ? P.ca : P.prob + (int64_t)(ch - 2) * P.n_w);
    if (ch) __syncthreads();            // every thread is done with the previous channel's box
    for (int e = threadIdx.x; e < nbox; e += kMapsThreads) {
      const int i2 = e % B2, r = e / B2, i1 = r % B1, i0 = r / B1;
      const int64_t g = ((int64_t)(L0 + i0) * P.cdim[1] + (L1 + i1)) * P.cdim[2] + (L2 + i2);
      buf[(i0 * P.pad[0] + i1) * P.pad[1] + i2] = __ldg(src + g);
    }
    __syncthreads();
    float* dst = ch == 0 ? P.out_bb : (ch == 1 ? P.out_ca : P.out_prob + (int64_t)(ch - 2) * P.n_s);
#pragma unroll
    for (int k = 0; k < kMapsOutPerThread; ++k) {
      if (jyz[k] < 0) continue;
      const int jy = jyz[k] & 255, jz = jyz[k] >> 8;
      const double wy = tw[kMapsTileX + jy], uy = tw1[kMapsTileX + jy], wz = tw[jz], uz = tw1[jz];
      const int dy = tdel[kMapsTileX + jy], dz = tdel[jz];
      const float* p = buf + base[k];
      const double v000 = p[0], v001 = p[dx], v010 = p[dy], v011 = p[dy + dx];
      const double v100 = p[dz], v101 = p[dz + dx], v110 = p[dz + dy], v111 = p[dz + dy + dx];
      const double f00 = __dadd_rn(__dmul_rn(v000, ux), __dmul_rn(v001, wx));
      const double f01 = __dadd_rn(__dmul_rn(v010, ux), __dmul_rn(v011, wx));
      const double f10 = __dadd_rn(__dmul_rn(v100, ux), __dmul_rn(v101, wx));
      const double f11 = __dadd_rn(__dmul_rn(v110, ux), __dmul_rn(v111, wx));
      const double g0 = __dadd_rn(__dmul_rn(f00, uy), __dmul_rn(f01, wy));
      const double g1 = __dadd_rn(__dmul_rn(f10, uy), __dmul_rn(f11, wy));
      const float f = __double2float_rn(__dadd_rn(__dmul_rn(g0, uz), __dmul_rn(g1, wz)));
      st_stream(dst + (((int64_t)(s0[0] + jz) * P.ns[1] + (s0[1] + jy)) * P.ns[2] + (s0[2] + jx)), f);
      if (ch == 2) {
        best[k] = f;
        arg[k] = 0;
      } else if (ch > 2 && !isnan(best[k]) && (f > best[k] || isnan(f))) {   // np.argmax: first max, NaN largest
        best[k] = f;
        arg[k] = ch - 2;
      }
    }
  }
#pragma unroll
  for (int k = 0; k < kMapsOutPerThread; ++k)
    if (jyz[k] >= 0) {
      const int jy = jyz[k] & 255, jz = jyz[k] >> 8;
      st_stream(P.out_pred + (((int64_t)(s0[0] + jz) * P.ns[1] + (s0[1] + jy)) * P.ns[2] + (s0[2] + jx)),
                (float)arg[k]);
    }
}

// the largest box extent along one memory axis over its tiles of `tile` targets
int max_span(int n_s, int n_w, int tile) {
  int best = 0;
  for (int s0 = 0; s0 < n_s; s0 += tile) {
    const int s1 = (s0 + tile < n_s ? s0 + tile : n_s) - 1;
    int a0, a1, b0, b1;
    double t;
    maps_axis_coord(s0, n_s, n_w, &a0, &a1, &t);
    maps_axis_coord(s1, n_s, n_w, &b0, &b1, &t);
    if (b1 - a0 + 1 > best) best = b1 - a0 + 1;
  }
  return best;
}

inline int odd_up(int v) { return v | 1; }

}  // namespace
}  // namespace mica

using namespace mica;

extern "C" int mica_volumes_to_grid(const float* bb, const float* ca, const float* aa_pred, const float* aa_prob,
                                    int X, int Y, int Z, const int org[3], const int ext[3], const int perm[3],
                                    const int working_zyx[3], const int target_zyx[3], float* out_bb, float* out_ca,
                                    float* out_pred, float* out_prob, mica_stream_t stream) {
  MICA_REQUIRE(bb && ca && aa_pred && aa_prob, "null input volume");
  MICA_REQUIRE(out_bb && out_ca && out_pred && out_prob, "null output volume");
  MICA_REQUIRE(org && ext && perm && working_zyx && target_zyx, "null shape argument");
  MICA_REQUIRE(X >= 1 && Y >= 1 && Z >= 1, "bad cube shape (%d, %d, %d)", X, Y, Z);
  for (int m = 0; m < 3; ++m) {
    MICA_REQUIRE(working_zyx[m] >= 1 && target_zyx[m] >= 1, "bad shape: working (%d, %d, %d), target (%d, %d, %d)",
                 working_zyx[0], working_zyx[1], working_zyx[2], target_zyx[0], target_zyx[1], target_zyx[2]);
  }
  MICA_REQUIRE(perm[0] >= 0 && perm[0] < 3 && perm[1] >= 0 && perm[1] < 3 && perm[2] >= 0 && perm[2] < 3 &&
                   perm[0] != perm[1] && perm[0] != perm[2] && perm[1] != perm[2],
               "perm (%d, %d, %d) is not a permutation of (0, 1, 2)", perm[0], perm[1], perm[2]);
  const int cdim[3] = {X, Y, Z};
  for (int a = 0; a < 3; ++a) {
    MICA_REQUIRE(org[a] == 0 && ext[a] == cdim[a],
                 "the box org (%d, %d, %d) ext (%d, %d, %d) is not the whole cube space (%d, %d, %d)", org[0], org[1],
                 org[2], ext[0], ext[1], ext[2], X, Y, Z);
    MICA_REQUIRE(cdim[a] == working_zyx[perm[a]],
                 "cube shape (%d, %d, %d) is not the working shape (%d, %d, %d) permuted by (%d, %d, %d)", X, Y, Z,
                 working_zyx[0], working_zyx[1], working_zyx[2], perm[0], perm[1], perm[2]);
  }

  MapsParams P = {};
  P.bb = bb;
  P.ca = ca;
  P.prob = aa_prob;
  P.out_bb = out_bb;
  P.out_ca = out_ca;
  P.out_pred = out_pred;
  P.out_prob = out_prob;
  P.n_w = (int64_t)X * Y * Z;
  P.n_s = (int64_t)target_zyx[0] * target_zyx[1] * target_zyx[2];
  for (int m = 0; m < 3; ++m) {
    P.cdim[m] = cdim[m];
    P.perm[m] = perm[m];
    P.nw[m] = working_zyx[m];
    P.ns[m] = target_zyx[m];
  }
  // target x (memory axis 2) always 32 wide; the memory axis the volumes store fastest (perm[2]) gets the other long
  // edge when it is not x, else the tile grows 8 x 4 in y, z.  Edges other than x halve while the box is too large
  // (downsampling by a large ratio).
  P.tile[2] = kMapsTileX;
  if (perm[2] != 2) {
    P.tile[perm[2]] = kMapsTileX;
    P.tile[3 - perm[2] - 2] = 1;
  } else {
    P.tile[1] = 8;
    P.tile[0] = 4;
  }
  int span[3], pad[2];
  size_t bytes = 0;
  for (;;) {
    for (int m = 0; m < 3; ++m) span[m] = max_span(P.ns[m], P.nw[m], P.tile[m]);
    pad[0] = odd_up(span[perm[1]]);
    pad[1] = odd_up(span[perm[2]]);
    bytes = kMapsTableBytes + (size_t)span[perm[0]] * pad[0] * pad[1] * sizeof(float);
    if (bytes <= kMapsSmemDefault) break;
    const int m = P.tile[0] >= P.tile[1] ? 0 : 1;
    if (P.tile[m] == 1) break;
    P.tile[m] /= 2;
  }
  MICA_REQUIRE(bytes <= kMapsSmemMax, "a target tile needs %zu bytes of shared memory (working (%d, %d, %d) -> target "
               "(%d, %d, %d)): the ratio is too large", bytes, working_zyx[0], working_zyx[1], working_zyx[2],
               target_zyx[0], target_zyx[1], target_zyx[2]);
  P.pad[0] = pad[0];
  P.pad[1] = pad[1];
  const int cstride[3] = {pad[0] * pad[1], pad[1], 1};
  for (int a = 0; a < 3; ++a) P.sstride[perm[a]] = cstride[a];
  int64_t blocks = 1;
  for (int m = 0; m < 3; ++m) {
    P.ntile[m] = (P.ns[m] + P.tile[m] - 1) / P.tile[m];
    blocks *= P.ntile[m];
  }
  MICA_REQUIRE(blocks <= 0x7fffffff, "target grid too large");
  if (bytes > kMapsSmemDefault)
    MICA_CUDA(cudaFuncSetAttribute(volumes_to_grid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  volumes_to_grid_kernel<<<(unsigned)blocks, kMapsThreads, bytes, (cudaStream_t)stream>>>(P);
  MICA_LAUNCH_CHECK("volumes_to_grid_kernel");
  return MICA_OK;
}
