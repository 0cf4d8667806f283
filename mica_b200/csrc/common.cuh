// Shared helpers for the mica_b200 kernels (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/mica_b200.h"

namespace mica {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

extern thread_local char g_last_error[512];
extern std::atomic<int64_t> g_launches;

int set_error(int code, const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);

// How long a kernel waits for a flag another rank raises over NVLink before it gives up with a status word
// (clock64 ticks).  Ranks of one job can be SECONDS apart -- one still allocating 10 GB of pinned host memory,
// another draining its volumes over a shared PCIe switch -- so the bound only has to beat "forever":
// MICA_PEER_TIMEOUT_MS, default 60 s.
long long peer_timeout_cycles();

inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

#define MICA_CUDA(call)                                      \
  do {                                                       \
    int _rc = ::mica::check_cuda((call), #call);             \
    if (_rc != MICA_OK) return _rc;                          \
  } while (0)

#define MICA_LAUNCH_CHECK(name)                              \
  do {                                                       \
    ::mica::count_launch();                                  \
    int _rc = ::mica::check_cuda(cudaGetLastError(), name);  \
    if (_rc != MICA_OK) return _rc;                          \
  } while (0)

#define MICA_REQUIRE(cond, ...)                                            \
  do {                                                                     \
    if (!(cond)) return ::mica::set_error(MICA_ERR_INVALID, __VA_ARGS__);  \
  } while (0)

// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda at link time)
typedef CUresult (*TensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                      const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
TensorMapEncodeFn tensor_map_encode_fn();

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// streaming (read-once / write-once) accesses: keep L1 for the data with reuse
__device__ __forceinline__ float ld_stream(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
// same, for 128-byte runs that start in the middle of a 128-byte line (cube cores at stride 32):
// by default a miss makes L2 fetch the whole 128-byte line from DRAM (measured on B200: 2.0x the
// requested bytes, tools/micro/overfetch.cu); .L2::64B caps the fill at the 64-byte half that is used
__device__ __forceinline__ float ld_stream_half_line(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::64B.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float4 ld_stream4(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ void st_stream(float* p, float v) {
  asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ void st_stream4(float4* p, float4 v) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

// Model-facing buffers (cube batches, logits) are float32 or bfloat16 (MICA_DTYPE_F32 / MICA_DTYPE_BF16); source
// maps and output volumes are always float32.  A bf16 store rounds the float32 value once, to nearest even; a bf16
// load widens exactly (the 16 bits become the high half of the float32).
__device__ __forceinline__ void st_stream_el(float* p, float v) { st_stream(p, v); }
__device__ __forceinline__ void st_stream_el(__nv_bfloat16* p, float v) {
  const unsigned short h = __bfloat16_as_ushort(__float2bfloat16_rn(v));
  asm volatile("st.global.cs.b16 [%0], %1;" ::"l"(p), "h"(h) : "memory");
}
__device__ __forceinline__ void st_plain_el(float* p, float v) { *p = v; }
__device__ __forceinline__ void st_plain_el(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ float bf16_bits_to_float(unsigned short h) { return __uint_as_float((unsigned)h << 16); }
__device__ __forceinline__ float ld_stream_el(const float* p) { return ld_stream(p); }
__device__ __forceinline__ float ld_stream_el(const __nv_bfloat16* p) {
  unsigned short h;
  asm volatile("ld.global.nc.L1::no_allocate.b16 %0, [%1];" : "=h"(h) : "l"(p));
  return bf16_bits_to_float(h);
}
// ld_stream_half_line for bf16 logits: at stride 32 a bf16 core row is the 64 bytes [32, 96) of a 128-byte line,
// which straddles both 64-byte halves, so the float32 helper's .L2::64B cap does not apply.  No L2 prefetch-size
// qualifier: on B200 none / 64B / 128B / 256B read these cores within 0.4 % of each other, none marginally fastest
// (tools/micro/bf16_core_read.cu, profiles/bf16_core_read_microbench.txt).
__device__ __forceinline__ float ld_stream_core_el(const float* p) { return ld_stream_half_line(p); }
__device__ __forceinline__ float ld_stream_core_el(const __nv_bfloat16* p) { return ld_stream_el(p); }

// host side: the element size of a model-facing dtype code, 0 if the code is not one of them
static inline int model_dtype_bytes(int dtype) {
  return dtype == MICA_DTYPE_F32 ? 4 : (dtype == MICA_DTYPE_BF16 ? 2 : 0);
}

// Test-time-augmentation orientation of a W^3 window (code 0..47, ops.orientation): code = 8 p + f, p the index
// of the axis permutation pi in lexicographic order, bit a of f flips output axis a.  The oriented window is
// O[u0,u1,u2] = C[v] with v[pi[a]] = (f_a ? W-1-u_a : u_a).
constexpr int kNumOrientations = 48;
struct Orientation {
  int perm[3];  // pi: output axis a reads window axis perm[a]
  int flip[3];  // 1 where output axis a is reversed
  int inv[3];   // pi^-1: window axis m is output axis inv[m]
  // flat offset of the ORIENTED position of window position v: base + v0 s[0] + v1 s[1] + v2 s[2]
  int base, s[3];
};
static inline bool orientation_decode(int code, int W, Orientation* o) {
  static const int kPerms[6][3] = {{0, 1, 2}, {0, 2, 1}, {1, 0, 2}, {1, 2, 0}, {2, 0, 1}, {2, 1, 0}};
  if (code < 0 || code >= kNumOrientations) return false;
  const int p = code >> 3, f = code & 7;
  const int pw[3] = {W * W, W, 1};
  o->base = 0;
  for (int a = 0; a < 3; ++a) {
    o->perm[a] = kPerms[p][a];
    o->flip[a] = (f >> a) & 1;
    o->inv[kPerms[p][a]] = a;
  }
  for (int a = 0; a < 3; ++a) {
    o->s[o->perm[a]] = o->flip[a] ? -pw[a] : pw[a];
    if (o->flip[a]) o->base += (W - 1) * pw[a];
  }
  return true;
}

// system-scope release / acquire on a flag word in (possibly peer) global memory: the PTX-model form of
// "data, fence, flag" between GPUs
__device__ __forceinline__ void st_release_sys(int* p, int v) {
  asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_sys(const int* p) {
  int v;
  asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

}  // namespace mica
