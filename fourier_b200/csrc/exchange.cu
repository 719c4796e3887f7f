// exchange.cu -- the exchange step of the distributed six-step transform (BASELINE configs[4]) as ONE kernel
// over NVLink peer memory, plus the CUDA-IPC plumbing that gives every rank (one process per GPU) the
// addresses of its peers' buffers.
//
// An exchange transposes a matrix whose rows are block-distributed over the P ranks: rank `me` holds
// rows_loc rows of `ld` = P*cb columns and must deliver columns [q*cb, (q+1)*cb) to rank q, where they
// become rows of length P*rows_loc.  The NCCL formulation (fourier_b200/distributed.py, exchange="nccl")
// needs three sweeps over the data per rank: pack (local transpose), all_to_all, unpack (axis swap).
// Here the transposing kernel stores its tiles straight into the destination rank's buffer, already in
// the final layout
//     dst_q[(c * P + me) * rows_loc + r] = src[r][q*cb + c] * w_N^{(row0 + r) * (q*cb + c)}
// so the data is read once from local HBM and written once over NVLink (1/P of it stays local); the
// inter-step twiddle of the six-step algorithm rides along.  Blocks rotate over the destinations
// (q = me+1, me+2, ... per consecutive block) so that every rank feeds all its peers at the same rate and no
// receiver's ingress is oversubscribed.  Ordering between ranks (all tiles have landed / the source may be
// overwritten) is a stream-ordered barrier issued by the caller after the kernel.
#include <cstdlib>
#include <cstring>

#include "plan.h"

namespace fb200 {
namespace {

struct PeerPtrs { void* p[kMaxPeers]; };

// PERSIST: a fixed number of blocks walks over the tiles (grid-stride), so that the kernel occupies only part of
// the GPU and kernels on other streams (the row FFTs of the next block of rows) run beside it; enough blocks must
// stay in flight to cover the NVLink latency (~2 MB of tiles).  Experiment knob, see launch_exchange.
template <typename T, int TW, bool PERSIST>
__global__ void __launch_bounds__(256)
exchange_kernel(const cpx<T>* __restrict__ in, PeerPtrs outs, int nranks, int me, size_t rows, size_t cb, size_t ld,
                size_t out_ld, size_t out_off, unsigned tiles_c, unsigned long long row0, unsigned long long n_total,
                unsigned total_tiles) {
  using V = cpx<T>;
  __shared__ V tile[32][33];
  for (unsigned id = blockIdx.x; PERSIST ? id < total_tiles : id == blockIdx.x; id += gridDim.x) {
  if (PERSIST && id != blockIdx.x) __syncthreads();   // the previous tile has left shared memory
  const int q = (me + 1 + (int)(id % (unsigned)nranks)) % nranks;
  const unsigned t = id / (unsigned)nranks;
  const size_t c0 = (size_t)(t % tiles_c) * 32, r0 = (size_t)(t / tiles_c) * 32;
  const V* src = in + (size_t)q * cb;
  V* dst = reinterpret_cast<V*>(outs.p[q]) + out_off;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  double wr = 1.0, wi = 0.0, sr = 1.0, si = 0.0;
  if constexpr (TW != 0) {
    // row and column indices are < 2^32 (checked by the launcher): the products fit 64 bits
    const unsigned long long cg = ((unsigned long long)q * cb + c0 + tx) % n_total;
    const unsigned long long m0 = ((row0 + r0 + ty) % n_total) * cg % n_total, ms = 8ull * cg % n_total;
    sincospi(2.0 * (double)m0 / (double)n_total, &wi, &wr);
    sincospi(2.0 * (double)ms / (double)n_total, &si, &sr);
    if (TW == 1) { wi = -wi; si = -si; }
  }
  for (int i = ty; i < 32; i += 8) {
    if (r0 + i < rows && c0 + tx < cb) {
      V v = src[(r0 + i) * ld + c0 + tx];
      if constexpr (TW != 0) {
        const double xr = (double)v.x, xi = (double)v.y;
        v = mk<T>((T)(xr * wr - xi * wi), (T)(xr * wi + xi * wr));
      }
      tile[i][tx] = v;
    }
    if constexpr (TW != 0) {
      const double nr = wr * sr - wi * si;
      wi = wr * si + wi * sr;
      wr = nr;
    }
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8)
    if (c0 + i < cb && r0 + tx < rows) dst[(c0 + i) * out_ld + r0 + tx] = tile[tx][i];
  }
}

}  // namespace

template <typename T>
cudaError_t launch_exchange(const cpx<T>* in, void* const* outs, int nranks, int me, size_t rows, size_t cb, size_t ld,
                            size_t out_ld, size_t out_off, int twiddle, unsigned long long row0,
                            unsigned long long n_total, cudaStream_t s) {
  if (nranks < 1 || nranks > kMaxPeers || me < 0 || me >= nranks || !in || !outs || twiddle < 0 || twiddle > 2) {
    set_last_error("exchange: bad arguments");
    return cudaErrorInvalidValue;
  }
  if (rows == 0 || cb == 0) return cudaSuccess;
  const size_t tiles_c = (cb + 31) / 32, tiles_r = (rows + 31) / 32;
  if (tiles_c * tiles_r * (size_t)nranks >= (1ull << 31) || tiles_c >= (1ull << 32) ||
      (twiddle != 0 && (n_total == 0 || row0 + rows > (1ull << 32) || (size_t)nranks * cb > (1ull << 32)))) {
    set_last_error("exchange: matrix too large");
    return cudaErrorInvalidValue;
  }
  PeerPtrs p;
  for (int i = 0; i < kMaxPeers; ++i) p.p[i] = i < nranks ? outs[i] : nullptr;
  const unsigned total = (unsigned)(tiles_c * tiles_r * (size_t)nranks);
  // FOURIER_B200_EXCHANGE_BLOCKS=n (experiment, not yet measured): n persistent blocks instead of one block per tile.
  // Unlike the plans' knobs (Tuning) this one is read on every call: the exchange has no plan to hold it, and callers
  // switch it between calls.
  const char* blocks = env_value("FOURIER_B200_EXCHANGE_BLOCKS");
  const int limit = blocks ? atoi(blocks) : 0;
#define FB_EXCHANGE_LAUNCH(TW)                                                                                      \
  do {                                                                                                               \
    if (limit > 0 && (unsigned)limit < total)                                                                        \
      exchange_kernel<T, TW, true><<<(unsigned)limit, 256, 0, s>>>(in, p, nranks, me, rows, cb, ld, out_ld, out_off, \
                                                                   (unsigned)tiles_c, row0, n_total, total);         \
    else                                                                                                             \
      exchange_kernel<T, TW, false><<<total, 256, 0, s>>>(in, p, nranks, me, rows, cb, ld, out_ld, out_off,          \
                                                          (unsigned)tiles_c, row0, n_total, total);                  \
  } while (0)
  if (twiddle == 0) FB_EXCHANGE_LAUNCH(0);
  else if (twiddle == 1) FB_EXCHANGE_LAUNCH(1);
  else FB_EXCHANGE_LAUNCH(2);
#undef FB_EXCHANGE_LAUNCH
  return cudaGetLastError();
}
template cudaError_t launch_exchange<float>(const cpx<float>*, void* const*, int, int, size_t, size_t, size_t, size_t,
                                            size_t, int, unsigned long long, unsigned long long, cudaStream_t);
template cudaError_t launch_exchange<double>(const cpx<double>*, void* const*, int, int, size_t, size_t, size_t, size_t,
                                             size_t, int, unsigned long long, unsigned long long, cudaStream_t);

// ---- peer memory: cudaMalloc'ed buffers shared between the ranks of one box through CUDA IPC -----------------
static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the C ABI passes IPC handles as 64 opaque bytes");

cudaError_t peer_alloc(size_t bytes, void** ptr, void* handle64) {
  if (!ptr || !handle64 || bytes == 0) return cudaErrorInvalidValue;
  cudaError_t e = cudaMalloc(ptr, bytes);
  if (e != cudaSuccess) { set_last_error(std::string("peer_alloc: cudaMalloc: ") + cudaGetErrorString(e)); return e; }
  cudaIpcMemHandle_t h;
  e = cudaIpcGetMemHandle(&h, *ptr);
  if (e != cudaSuccess) {
    set_last_error(std::string("peer_alloc: cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
    cudaFree(*ptr);
    *ptr = nullptr;
    return e;
  }
  std::memcpy(handle64, &h, sizeof h);
  return cudaSuccess;
}

cudaError_t peer_open(const void* handle64, void** ptr) {
  if (!ptr || !handle64) return cudaErrorInvalidValue;
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle64, sizeof h);
  const cudaError_t e = cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) set_last_error(std::string("peer_open: cudaIpcOpenMemHandle: ") + cudaGetErrorString(e));
  return e;
}

cudaError_t peer_close(void* ptr) { return ptr ? cudaIpcCloseMemHandle(ptr) : cudaSuccess; }
cudaError_t peer_free(void* ptr) { return ptr ? cudaFree(ptr) : cudaSuccess; }

}  // namespace fb200
