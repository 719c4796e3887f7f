// dist_fft.cu -- row FFTs of the distributed six-step transform with the exchange folded into the store of their
// last register stage (dist_kernels.cuh): pass 1 of the two-pass tile kernels as it is, pass 2 on tiles of C
// adjacent transforms that store over NVLink peer memory.  Chunks rotate over the caller's stream and
// plan-owned ones (lanes), each with its own intermediate, so that pass 1 of one chunk (HBM reads, no NVLink
// traffic) runs beside pass 2 of another (NVLink stores).
#include <algorithm>
#include <type_traits>

#include "dist_kernels.cuh"
#include "plan.h"
#include "twopass_kernels.cuh"

namespace fb200 {

namespace {

template <typename T> struct RowsExchangeCall {
  const cpx<T>* scratch; const void* twa; void* const* outs; int nranks; size_t groups, out_ld, out_off;
  int twiddle, cb_shift; unsigned long long row0, n_total; bool fwd; cudaStream_t s;
  size_t r0, out_bs; int rb_shift; size_t rpb, rows_valid;
};

// Tiles of twice as many transforms where the configuration's pass-2 tile has 16 (f32) / 8 (f64): a warp's store is then
// one 256-byte run instead of two 128-byte pieces.  Measured (profiles/r02_rows_exchange_knobs.txt, r02_c5_modes_8gpu.json):
// N = 2^30 on 2 GPUs 12.64 -> 12.27 ms, on 8 GPUs 5.13 -> 5.15 ms (no change), one GPU (three-pass path) no change.
// Paddings are the bank-conflict-free ones (tools/emulate.cu).  The narrow tiles remain for row counts that are not a
// multiple of the wide tile.
template <class S, typename T> struct WideShape { using type = S; };
template <> struct WideShape<twopass::Shape<8, 16, 16, 16, 2>, float> { using type = twopass::Shape<8, 16, 16, 32, 2>; };
template <> struct WideShape<twopass::Shape<16, 16, 16, 16, 1>, float> { using type = twopass::Shape<16, 16, 16, 32, 1>; };
template <> struct WideShape<twopass::Shape<8, 16, 16, 8, 1>, double> { using type = twopass::Shape<8, 16, 16, 16, 1>; };
template <> struct WideShape<twopass::Shape<16, 16, 16, 8, 1>, double> { using type = twopass::Shape<16, 16, 16, 16, 1>; };

template <class G, bool WIDE, typename T> struct ExchangeTile {
  using S = typename std::conditional<WIDE, typename WideShape<typename G::Shape2, T>::type, typename G::Shape2>::type;
  template <bool FWD> using Tile = TileFFT<T, S::RA, S::RB, S::E, S::C, FWD>;
  using Lay = ExLayout<S::RA * S::C + S::PAD, S::C, 1>;
  static constexpr int C = S::C;
  static constexpr size_t smem = sizeof(cpx<T>) * Tile<true>::template smem_elems<Lay>();
  // resident CTAs per SM: the configuration's pass-2 setting scaled to the tile's threads
  static constexpr int kMinBlocks = (G::kMinBlocks2 * G::C2 + C - 1) / C;
};

// MORE: resident CTAs per SM beyond the configuration's pass-2 setting (the kernel waits on L2 / NVLink, not on
// registers: ptxas fits 80 instead of 112 registers per thread without spilling)
template <class G, bool FWD, int TW, int MORE, bool WIDE, typename T>
cudaError_t launch_rows_exchange(const RowsExchangeCall<T>& c) {
  using X = ExchangeTile<G, WIDE, T>;
  using Tile = typename X::template Tile<FWD>;
  using Body = dist::RowsExchangeBody<Tile, typename X::Lay, G::N1, G::N2, TW>;
  auto kernel = &dist::rows_exchange_kernel<Body, Tile, X::kMinBlocks + (WIDE ? MORE / 2 : MORE)>;
  static std::atomic<unsigned long long> prepared{0};
  if (cudaError_t e = ensure_dynamic_smem(kernel, X::smem, prepared)) return e;
  typename Body::Args a;
  a.scratch = c.scratch;
  a.twa = (const TwPair<T>*)c.twa;
  for (int i = 0; i < kMaxPeers; ++i) a.outs.p[i] = i < c.nranks ? c.outs[i] : nullptr;
  a.out_ld = c.out_ld; a.out_off = c.out_off; a.row0 = c.row0; a.n_total = c.n_total;
  a.groups = (unsigned)c.groups; a.cb_shift = c.cb_shift;
  a.r0 = c.r0; a.out_bs = c.out_bs; a.rb_shift = c.rb_shift; a.rpb = c.rpb; a.rows_valid = c.rows_valid;
  kernel<<<(unsigned)(c.groups * (size_t)G::N1), Tile::THREADS, X::smem, c.s>>>(a);
  return cudaGetLastError();
}

template <class G, bool WIDE, typename T> cudaError_t dispatch_rows_exchange(const RowsExchangeCall<T>& c) {
  constexpr int MORE = 2;   // +1 .. 6 % on the three-pass path, neutral on the distributed one (profiles/r02_rows_exchange_knobs.txt)
  if (c.fwd) return c.twiddle ? launch_rows_exchange<G, true, 1, MORE, WIDE>(c) : launch_rows_exchange<G, true, 0, MORE, WIDE>(c);
  return c.twiddle ? launch_rows_exchange<G, false, 2, MORE, WIDE>(c) : launch_rows_exchange<G, false, 0, MORE, WIDE>(c);
}

}  // namespace

template <typename T>
cudaError_t Plan<T>::exec_rows_exchange(const C* in, size_t rows, bool forward, void* const* outs, int nranks,
                                        size_t out_ld, size_t out_off, int twiddle, unsigned long long row0,
                                        unsigned long long n_total, cudaStream_t s, size_t rows_per_batch,
                                        size_t out_batch_stride, size_t rows_valid) {
  if (path_ != Path::kTwoPass || !fast_ops_) {
    set_last_error("rows_exchange: the plan is not a two-pass plan (power-of-two sizes 2^11 .. 2^20 (f32), 2^9 .. 2^16 (f64))");
    return cudaErrorNotSupported;
  }
  if (!in || !outs || nranks < 1 || nranks > kMaxPeers || (nranks & (nranks - 1)) || n_ % (size_t)nranks ||
      twiddle < 0 || twiddle > 2 || (twiddle == 1 && !forward) || (twiddle == 2 && forward)) {
    set_last_error("rows_exchange: bad arguments (ranks must be a power of two dividing the size; twiddle 1 goes with "
                   "the forward, 2 with the inverse direction)");
    return cudaErrorInvalidValue;
  }
  if (twiddle != 0 && (n_total == 0 || n_total > (1ull << 32) || row0 + rows > (1ull << 32))) {
    set_last_error("rows_exchange: twiddle index out of range");
    return cudaErrorInvalidValue;
  }
  int rb_shift = 63;
  size_t rpb = 0;                                   // rows per batch when that is not a power of two
  if (rows_per_batch) {
    if (rows_per_batch & (rows_per_batch - 1)) rpb = rows_per_batch;
    else for (rb_shift = 0; ((size_t)1 << rb_shift) < rows_per_batch; ++rb_shift) {}
  }
  if (rows_valid == 0 || rows_valid > rows) rows_valid = rows;
  if (rows == 0) return cudaSuccess;
  const auto* ops = static_cast<const twopass::TwoPassOps<T>*>(fast_ops_);
  int c2 = 0, c2w = 0;
  twopass::visit_config<T>(n_, [&](auto g) {
    c2 = decltype(g)::C2;
    c2w = ExchangeTile<decltype(g), true, T>::C;
  });
  const bool wide = c2w != c2 && rows % (size_t)c2w == 0;
  if (wide) c2 = c2w;
  if (c2 == 0 || rows % (size_t)c2) {
    set_last_error("rows_exchange: the number of rows must be a multiple of " + std::to_string(c2));
    return cudaErrorInvalidValue;
  }
  DeviceGuard guard(device_);
  int cb_shift = 0;
  while (((size_t)1 << cb_shift) < n_ / (size_t)nranks) ++cb_shift;
  // chunks of whole tiles, two of them in flight.  Measured on 2 B200s (N = 2^28, profiles/r02_c5_fused_ab_2gpu.txt):
  // 16 MB chunks 3.60 ms per transform, 32 MB 3.23, 64 MB 3.07 -- NVLink, not the L2 residency of the intermediate,
  // bounds this path, and longer kernels overlap better across the two streams (tuning_.dist_chunk_mb, 64 by default).
  const size_t want = std::max<size_t>(1, (tuning_.dist_chunk_mb << 20) / (n_ * sizeof(C)));
  size_t chunk = std::max<size_t>((size_t)c2, std::min(want, rows) / (size_t)c2 * (size_t)c2);
  // lanes: chunks rotate over the caller's stream and up to three plan-owned ones, each with its own intermediate
  const int nlanes = (int)std::min<size_t>((size_t)tuning_.dist_lanes, (rows + chunk - 1) / chunk);
  FB_CHECK(work_.reserve((size_t)nlanes * chunk * n_ * sizeof(C)));
  cudaStream_t lanes[4] = {s, s, s, s};
  if (nlanes > 1) {
    FB_CHECK(host_resources());
    FB_CHECK(cudaEventRecord(events_[0], s));
    for (int l = 1; l < nlanes; ++l) {
      lanes[l] = streams_[l - 1];
      FB_CHECK(cudaStreamWaitEvent(lanes[l], events_[0], 0));
    }
  }
  launches_ = 0;
  size_t i = 0;
  for (size_t b0 = 0; b0 < rows; b0 += chunk, ++i) {
    const size_t nb = std::min(chunk, rows - b0);
    const int lane = (int)(i % (size_t)nlanes);
    C* scratch = (C*)work_.data() + (size_t)lane * chunk * n_;
    cudaStream_t st = lanes[lane];
    FB_CHECK(ops->pass1(in + b0 * n_, scratch, tw_a_.data(), (const C*)tw2_.data(), nb, forward, st));
    RowsExchangeCall<T> c{scratch, tw_b_.data(), outs, nranks, nb / (size_t)c2, out_ld, out_off, twiddle, cb_shift,
                          row0, n_total, forward, st, b0, out_batch_stride, rb_shift, rpb, rows_valid};
    cudaError_t e = cudaErrorNotSupported;
    twopass::visit_config<T>(n_, [&](auto g) {
      e = wide ? dispatch_rows_exchange<decltype(g), true>(c) : dispatch_rows_exchange<decltype(g), false>(c);
    });
    FB_CHECK(e);
    launches_ += 2;
  }
  for (int l = 1; l < nlanes; ++l) {
    FB_CHECK(cudaEventRecord(events_[l], lanes[l]));
    FB_CHECK(cudaStreamWaitEvent(s, events_[l], 0));
  }
  return cudaSuccess;
}

template cudaError_t Plan<float>::exec_rows_exchange(const C*, size_t, bool, void* const*, int, size_t, size_t, int,
                                                     unsigned long long, unsigned long long, cudaStream_t, size_t, size_t,
                                                     size_t);
template cudaError_t Plan<double>::exec_rows_exchange(const C*, size_t, bool, void* const*, int, size_t, size_t, int,
                                                      unsigned long long, unsigned long long, cudaStream_t, size_t, size_t,
                                                      size_t);

}  // namespace fb200
