// Multi-GPU (SURVEY.md 8e): the z-halo exchange of the source map over NVLink peer memory.
//
// A rank resamples its output slab from its own block of source planes plus a few planes of each
// neighbour's block (interpolation taps + prefilter horizon, mica_b200/slab.py::SlabPlan).  There is
// no reference counterpart (the reference is single-process).  Through NCCL the exchange is a
// batch_isend_irecv whose cost is the rendezvous, not the 37 MB (measured round 1: 1.2 ms waited for
// a 0.18 ms transfer).  Here it is two kernels on the caller's stream and no host involvement:
//
//   publish   copy the boundary planes the neighbours need into this rank's EXPORTED buffer
//             (cudaMalloc + CUDA IPC, mapped by both neighbours); the last CTA to finish makes the
//             data visible system-wide and raises a flag IN THE NEIGHBOUR's buffer (st.release.sys),
//             so the neighbour polls local memory;
//   pull      wait (ld.acquire.sys, bounded) for the neighbour's flag, then copy its published
//             planes over NVLink straight into this rank's assembled source buffer.
//
// publish never waits, so ranks cannot deadlock; a neighbour that never arrives turns into a status
// word, not a hang.  Slots alternate with the call epoch: a slot is rewritten two exchanges later,
// and between two exchanges every rank takes part in the order-statistics histogram exchange of the
// map in between (a barrier in effect), so the neighbour has finished reading by then.
#include <string.h>

#include "common.cuh"

namespace mica {

constexpr int kHaloFlagWords = 64;

struct HaloHeader {
  int ready_from_lo;   // last epoch published by the LOWER neighbour (rank - 1), written by it
  int ready_from_hi;   // same for the UPPER neighbour (rank + 1)
  unsigned done[2];    // publish bookkeeping: CTAs finished, per parity
  int pad[kHaloFlagWords - 4];
};
static_assert(sizeof(HaloHeader) == kHaloFlagWords * sizeof(int), "header size");

// buffer layout: HaloHeader | slot[parity 0..1][side 0..1][slot_bytes] ; side 0 = planes for the lower neighbour
// (the low end of my block), side 1 = planes for the upper neighbour.  Slots are counted in bytes, so that planes of
// any sample type (float32, int16, int8) fit; slot_bytes is a multiple of 16 here.
__host__ __device__ __forceinline__ char* halo_slot(void* buf, int parity, int side, int64_t slot_bytes) {
  return reinterpret_cast<char*>(buf) + sizeof(HaloHeader) + (int64_t)(parity * 2 + side) * slot_bytes;
}

// n bytes in words of W, then the tail bytes
template <typename W>
__device__ __forceinline__ void copy_words(char* __restrict__ dst, const char* __restrict__ src, int64_t n,
                                           int64_t tid, int64_t stride, bool remote) {
  const int64_t nw = n / (int64_t)sizeof(W);
  const W* s = reinterpret_cast<const W*>(src);
  W* d = reinterpret_cast<W*>(dst);
  for (int64_t i = tid; i < nw; i += stride) d[i] = remote ? __ldcv(s + i) : s[i];
  for (int64_t i = nw * (int64_t)sizeof(W) + tid; i < n; i += stride)
    dst[i] = remote ? (char)__ldcv(reinterpret_cast<const unsigned char*>(src) + i) : src[i];
}

// 16-byte vectors when both ends are 16-byte aligned (float32 planes always are: the assembled buffers and the slots
// are), 4-byte words when they are 4-byte aligned, bytes otherwise
__device__ __forceinline__ void copy_bytes(char* __restrict__ dst, const char* __restrict__ src, int64_t n,
                                           int64_t tid, int64_t stride, bool remote) {
  const uintptr_t a = ((uintptr_t)dst) | ((uintptr_t)src);
  if ((a & 15) == 0)
    copy_words<uint4>(dst, src, n, tid, stride, remote);
  else if ((a & 3) == 0)
    copy_words<unsigned>(dst, src, n, tid, stride, remote);
  else
    copy_words<unsigned char>(dst, src, n, tid, stride, remote);
}

// own: this rank's block of source planes.  n_lo / n_hi bytes go to the lower / upper neighbour from byte offsets
// off_lo / off_hi of the block.
__global__ void __launch_bounds__(256)
halo_publish_kernel(const char* __restrict__ own, int64_t off_lo, int64_t n_lo, int64_t off_hi, int64_t n_hi,
                    void* const* __restrict__ peers, int rank, int world, int parity, int epoch, int64_t slot_bytes) {
  void* mine = peers[rank];
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  if (rank > 0 && n_lo > 0) copy_bytes(halo_slot(mine, parity, 0, slot_bytes), own + off_lo, n_lo, tid, stride, false);
  if (rank + 1 < world && n_hi > 0)
    copy_bytes(halo_slot(mine, parity, 1, slot_bytes), own + off_hi, n_hi, tid, stride, false);
  __threadfence();
  __syncthreads();
  __shared__ bool last;
  HaloHeader* h = reinterpret_cast<HaloHeader*>(mine);
  if (threadIdx.x == 0) last = (atomicAdd(&h->done[parity], 1u) == gridDim.x - 1);
  __syncthreads();
  if (!last) return;
  if (threadIdx.x == 0) {
    h->done[parity] = 0;                 // ready for this slot's next use (two exchanges later)
    __threadfence_system();              // every CTA's planes (observed through the counter) before the flags
    if (rank > 0) st_release_sys(&reinterpret_cast<HaloHeader*>(peers[rank - 1])->ready_from_hi, epoch);
    if (rank + 1 < world) st_release_sys(&reinterpret_cast<HaloHeader*>(peers[rank + 1])->ready_from_lo, epoch);
  }
}

// dst_lo receives n_lo bytes published by the lower neighbour (its side 1), dst_hi n_hi bytes published by the upper
// neighbour (its side 0).  status: set to 1 when a neighbour timed out.
__global__ void __launch_bounds__(256)
halo_pull_kernel(char* __restrict__ dst_lo, int64_t n_lo, char* __restrict__ dst_hi, int64_t n_hi,
                 void* const* __restrict__ peers, int rank, int world, int parity, int epoch, int64_t slot_bytes,
                 long long timeout_cycles, int* __restrict__ status) {
  __shared__ int ok;
  const HaloHeader* h = reinterpret_cast<const HaloHeader*>(peers[rank]);
  const bool want_lo = rank > 0 && n_lo > 0, want_hi = rank + 1 < world && n_hi > 0;
  if (threadIdx.x == 0) {
    int good = 1;
    const long long t0 = clock64();
    if (want_lo)
      while (ld_acquire_sys(&h->ready_from_lo) - epoch < 0)
        if (clock64() - t0 > timeout_cycles) { good = 0; break; }
    if (want_hi && good)
      while (ld_acquire_sys(&h->ready_from_hi) - epoch < 0)
        if (clock64() - t0 > timeout_cycles) { good = 0; break; }
    ok = good;
  }
  __syncthreads();
  if (!ok) {
    if (threadIdx.x == 0) atomicExch(status, 1);
    return;
  }
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  if (want_lo) copy_bytes(dst_lo, halo_slot(peers[rank - 1], parity, 1, slot_bytes), n_lo, tid, stride, true);
  if (want_hi) copy_bytes(dst_hi, halo_slot(peers[rank + 1], parity, 0, slot_bytes), n_hi, tid, stride, true);
}

}  // namespace mica

using namespace mica;

extern "C" size_t mica_halo_buffer_bytes(int64_t slot_elems) {
  if (slot_elems < 0) return 0;
  const int64_t padded = (slot_elems + 3) / 4 * 4;
  return sizeof(HaloHeader) + (size_t)4 * padded * sizeof(float);
}

// cudaMalloc'd, zeroed, IPC-exportable buffer of any size (the histogram exchange has its own fixed-size
// mica_peer_alloc); open / close / free with mica_peer_open / mica_peer_close / mica_peer_free
extern "C" int mica_ipc_alloc(size_t bytes, void** dev_ptr, void* ipc_handle_out) {
  MICA_REQUIRE(dev_ptr && bytes > 0, "bad arguments");
  void* p = nullptr;
  MICA_CUDA(cudaMalloc(&p, bytes));
  MICA_CUDA(cudaMemset(p, 0, bytes));
  if (ipc_handle_out) {
    cudaIpcMemHandle_t h;
    MICA_CUDA(cudaIpcGetMemHandle(&h, p));
    memcpy(ipc_handle_out, &h, sizeof(h));
  }
  *dev_ptr = p;
  return MICA_OK;
}

// one 16-byte vector per thread and pass, at most two CTAs per SM
static int halo_grid(int64_t bytes) {
  int64_t want = ceil_div64(ceil_div64(bytes, 16), 256 * 4);
  if (want < 1) want = 1;
  return (int)(want < 2 * kNumSMs ? want : 2 * kNumSMs);
}

static int64_t slot_stride(int64_t slot_bytes) { return (slot_bytes + 15) / 16 * 16; }

extern "C" int mica_halo_publish_bytes(const void* own, int64_t off_lo, int64_t n_lo, int64_t off_hi, int64_t n_hi,
                                       void* const* peer_bufs, int rank, int world, int parity, int epoch,
                                       int64_t slot_bytes, mica_stream_t stream) {
  MICA_REQUIRE(peer_bufs && (own || (n_lo == 0 && n_hi == 0)), "null pointer");
  MICA_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bad rank/world");
  MICA_REQUIRE(parity == 0 || parity == 1, "parity must be 0 or 1");
  MICA_REQUIRE(n_lo >= 0 && n_hi >= 0 && n_lo <= slot_bytes && n_hi <= slot_bytes, "halo larger than the slot");
  if (world == 1) return MICA_OK;
  halo_publish_kernel<<<halo_grid(n_lo + n_hi), 256, 0, (cudaStream_t)stream>>>(
      (const char*)own, off_lo, n_lo, off_hi, n_hi, peer_bufs, rank, world, parity, epoch, slot_stride(slot_bytes));
  MICA_LAUNCH_CHECK("halo_publish_kernel");
  return MICA_OK;
}

extern "C" int mica_halo_pull_bytes(void* dst_lo, int64_t n_lo, void* dst_hi, int64_t n_hi, void* const* peer_bufs,
                                    int rank, int world, int parity, int epoch, int64_t slot_bytes, int* status,
                                    mica_stream_t stream) {
  MICA_REQUIRE(peer_bufs && status, "null pointer");
  MICA_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bad rank/world");
  MICA_REQUIRE(parity == 0 || parity == 1, "parity must be 0 or 1");
  MICA_REQUIRE(n_lo >= 0 && n_hi >= 0 && n_lo <= slot_bytes && n_hi <= slot_bytes, "halo larger than the slot");
  MICA_REQUIRE((n_lo == 0 || dst_lo) && (n_hi == 0 || dst_hi), "null destination");
  if (world == 1) return MICA_OK;
  const long long timeout_cycles = mica::peer_timeout_cycles();
  halo_pull_kernel<<<halo_grid(n_lo + n_hi), 256, 0, (cudaStream_t)stream>>>(
      (char*)dst_lo, n_lo, (char*)dst_hi, n_hi, peer_bufs, rank, world, parity, epoch, slot_stride(slot_bytes),
      timeout_cycles, status);
  MICA_LAUNCH_CHECK("halo_pull_kernel");
  return MICA_OK;
}

extern "C" int mica_halo_publish(const float* own, int64_t off_lo, int64_t n_lo, int64_t off_hi, int64_t n_hi,
                                 void* const* peer_bufs, int rank, int world, int parity, int epoch,
                                 int64_t slot_elems, mica_stream_t stream) {
  return mica_halo_publish_bytes(own, off_lo * 4, n_lo * 4, off_hi * 4, n_hi * 4, peer_bufs, rank, world, parity,
                                 epoch, slot_elems * 4, stream);
}

extern "C" int mica_halo_pull(float* dst_lo, int64_t n_lo, float* dst_hi, int64_t n_hi, void* const* peer_bufs,
                              int rank, int world, int parity, int epoch, int64_t slot_elems, int* status,
                              mica_stream_t stream) {
  return mica_halo_pull_bytes(dst_lo, n_lo * 4, dst_hi, n_hi * 4, peer_bufs, rank, world, parity, epoch,
                              slot_elems * 4, status, stream);
}
