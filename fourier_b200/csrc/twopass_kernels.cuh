// twopass_kernels.cuh -- kernels, per-size configurations and table builders of the two-pass (four-step)
// path.  Shared by twopass.cu (the product) and tools/emulate.cu (CPU emulation of the same code).
#pragma once

#include <vector>

#include "plan.h"
#include "tables.cuh"
#include "tilefft.cuh"

namespace fb200 {
namespace twopass {

// ---- kernels ------------------------------------------------------------------------------------------
// One CTA = one tile of Tile::C FFTs of one transform of the chunk.
// The body of one tile, split at the CTA barrier so that tools/emulate.cu can run the identical code on
// the CPU: phase1 for every thread, then phase2 for every thread.
template <class Tile, class LAY, long NS, long CS, bool LOAD_UF, long KS, long OCS, bool TW2>
struct TileBody {
  using V = typename Tile::V;
  using T = decltype(V::x);
  struct Args {
    const V* in; V* out; const TwPair<T>* twa; const V* tw2;
    long tile_stride_in, tile_stride_out, batch_stride; int tiles_per_fft; T scale; int do_scale;
  };
  static FB_HD void phase1(Tile& f, const Args& a, long block, int t, V* smem) {
    const int tile = (int)(block % a.tiles_per_fft);
    const long b = block / a.tiles_per_fft;
    const V* src = a.in + b * a.batch_stride + (long)tile * a.tile_stride_in;
    f.template load<LOAD_UF, NS, CS>(t, src);
    f.template stage_a<LOAD_UF>(t, a.twa);
    f.template scatter<LOAD_UF, LAY>(t, smem);
  }
  static FB_HD void phase2(Tile& f, const Args& a, long block, int t, const V* smem) {
    const int tile = (int)(block % a.tiles_per_fft);
    const long b = block / a.tiles_per_fft;
    V* dst = a.out + b * a.batch_stride + (long)tile * a.tile_stride_out;
    const V* t2 = TW2 ? a.tw2 + (long)tile * a.tile_stride_out : nullptr;
    f.template gather<false, LAY>(t, smem);
    f.stage_b();
    if (a.do_scale) f.template store<false, KS, OCS, TW2, true>(t, dst, t2, a.scale);
    else f.template store<false, KS, OCS, TW2, false>(t, dst, t2, a.scale);
  }
};

// One CTA = one tile of Tile::C FFTs of one transform of the chunk.
template <class Tile, class LAY, long NS, long CS, bool LOAD_UF, long KS, long OCS, bool TW2, int MINB>
__global__ void __launch_bounds__(Tile::THREADS, MINB)
tile_kernel(const typename TileBody<Tile, LAY, NS, CS, LOAD_UF, KS, OCS, TW2>::Args a) {
  using Body = TileBody<Tile, LAY, NS, CS, LOAD_UF, KS, OCS, TW2>;
  using V = typename Tile::V;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  V* smem = reinterpret_cast<V*>(smem_raw);
  Tile f;
  Body::phase1(f, a, blockIdx.x, threadIdx.x, smem);
  __syncthreads();
  Body::phase2(f, a, blockIdx.x, threadIdx.x, smem);
}

template <typename T> struct TwoPassOps {
  size_t n1, n2;
  int ra1, rb1, ra2, rb2;
  cudaError_t (*pass1)(const cpx<T>*, cpx<T>*, const void*, const cpx<T>*, size_t, bool, cudaStream_t);
  cudaError_t (*pass2)(const cpx<T>*, cpx<T>*, const void*, size_t, bool, T, bool, cudaStream_t);
  cudaError_t (*prepare)();
};

// Shape of one pass: length L = RA*RB, E samples per thread, C FFTs per tile, PAD = padding of the
// exchange row (chosen so that the scatter is bank-conflict free; checked by tools/emulate.cu).
template <int RA_, int RB_, int E_, int C_, int PAD_> struct Shape {
  static constexpr int RA = RA_, RB = RB_, E = E_, C = C_, PAD = PAD_;
  static constexpr long L = (long)RA * RB;
};

// Configuration of one supported size N = N1*N2: pass 1 = column tiles of shape S1, pass 2 = row tiles S2.
template <typename T, class S1, class S2, int MINB1, int MINB2>
struct TwoPassG {
  static constexpr long N1 = S1::L, N2 = S2::L, N = N1 * N2;
  static constexpr int C1 = S1::C, C2 = S2::C;
  static constexpr int kMinBlocks1 = MINB1, kMinBlocks2 = MINB2;
  using Shape1 = S1;
  using Shape2 = S2;
  // pass 1: FFT length N1 over n1 (stride N2), C1 adjacent columns; both stages "col fast"
  template <bool FWD> using Tile1 = TileFFT<T, S1::RA, S1::RB, S1::E, C1, FWD>;
  using Lay1 = ExLayout<S1::RA * C1 + S1::PAD, C1, 1>;
  // pass 2: FFT length N2 over contiguous rows, C2 adjacent rows; stage A "u fast", stage B "col fast"
  template <bool FWD> using Tile2 = TileFFT<T, S2::RA, S2::RB, S2::E, C2, FWD>;
  using Lay2 = ExLayout<S2::RA * C2 + S2::PAD, C2, 1>;
  template <bool FWD> using Body1 = TileBody<Tile1<FWD>, Lay1, N2, 1, false, N2, 1, true>;
  template <bool FWD> using Body2 = TileBody<Tile2<FWD>, Lay2, 1, N2, true, N1, 1, false>;
  template <bool FWD> static constexpr auto k1() {
    return &tile_kernel<Tile1<FWD>, Lay1, N2, 1, false, N2, 1, true, MINB1>;
  }
  template <bool FWD> static constexpr auto k2() {
    return &tile_kernel<Tile2<FWD>, Lay2, 1, N2, true, N1, 1, false, MINB2>;
  }
  template <bool FWD>
  static typename Body1<FWD>::Args args1(const cpx<T>* in, cpx<T>* scratch, const void* twa, const cpx<T>* tw2) {
    return {in, scratch, (const TwPair<T>*)twa, tw2, C1, C1, N, (int)(N2 / C1), (T)1, 0};
  }
  template <bool FWD>
  static typename Body2<FWD>::Args args2(const cpx<T>* scratch, cpx<T>* out, const void* twa, T scale,
                                         bool do_scale) {
    return {scratch, out, (const TwPair<T>*)twa, nullptr, (long)C2 * N2, C2, N, (int)(N1 / C2), scale,
            do_scale ? 1 : 0};
  }
  static constexpr size_t smem1 = sizeof(cpx<T>) * Tile1<true>::template smem_elems<Lay1>();
  static constexpr size_t smem2 = sizeof(cpx<T>) * Tile2<true>::template smem_elems<Lay2>();

  static cudaError_t prepare() {
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(k1<true>(), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1))) return e;
    if ((e = cudaFuncSetAttribute(k1<false>(), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1))) return e;
    if ((e = cudaFuncSetAttribute(k2<true>(), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2))) return e;
    if ((e = cudaFuncSetAttribute(k2<false>(), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2))) return e;
    return cudaSuccess;
  }
  static cudaError_t pass1(const cpx<T>* in, cpx<T>* scratch, const void* twa, const cpx<T>* tw2, size_t nb,
                           bool fwd, cudaStream_t s) {
    const unsigned grid = (unsigned)(nb * (N2 / C1));
    if (fwd) k1<true>()<<<grid, Tile1<true>::THREADS, smem1, s>>>(args1<true>(in, scratch, twa, tw2));
    else k1<false>()<<<grid, Tile1<true>::THREADS, smem1, s>>>(args1<false>(in, scratch, twa, tw2));
    return cudaGetLastError();
  }
  static cudaError_t pass2(const cpx<T>* scratch, cpx<T>* out, const void* twa, size_t nb, bool fwd, T scale,
                           bool do_scale, cudaStream_t s) {
    const unsigned grid = (unsigned)(nb * (N1 / C2));
    if (fwd) k2<true>()<<<grid, Tile2<true>::THREADS, smem2, s>>>(args2<true>(scratch, out, twa, scale, do_scale));
    else k2<false>()<<<grid, Tile2<true>::THREADS, smem2, s>>>(args2<false>(scratch, out, twa, scale, do_scale));
    return cudaGetLastError();
  }
  static const TwoPassOps<T>* ops() {
    static const TwoPassOps<T> o = {(size_t)N1, (size_t)N2, S1::RA, S1::RB, S2::RA, S2::RB, &pass1, &pass2, &prepare};
    return &o;
  }
};

// square shorthand used by the original configurations: both passes R x R register stages
template <typename T, int R1, int R2, int C1, int C2, int PAD1, int MINB1, int MINB2>
using TwoPass = TwoPassG<T, Shape<R1, R1, R1, C1, PAD1>, Shape<R2, R2, R2, C2, 1>, MINB1, MINB2>;

// Supported sizes.  f32: 32x32 register stages (1024-point tiles); f64: 16x16 (256-point tiles).
// visit_config<T>(n, f) calls f with a value of the configuration type of size n (false when there is none): the one
// list of sizes behind lookup() here and behind the distributed variant of pass 2 (dist_fft.cu).
template <class F> bool visit_config_f32(size_t n, F&& f) {
  switch (n) {
    case (size_t)1 << 20: f(TwoPass<float, 32, 32, 8, 8, 8, 2, 2>{}); return true;
    case (size_t)1 << 11: f(TwoPassG<float, Shape<4, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>{}); return true;
    case (size_t)1 << 12: f(TwoPassG<float, Shape<8, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>{}); return true;
    case (size_t)1 << 13: f(TwoPassG<float, Shape<8, 8, 8, 32, 0>, Shape<8, 16, 16, 16, 2>, 4, 4>{}); return true;
    case (size_t)1 << 14: f(TwoPassG<float, Shape<8, 16, 16, 16, 0>, Shape<8, 16, 16, 16, 2>, 4, 4>{}); return true;
    case (size_t)1 << 15: f(TwoPassG<float, Shape<8, 16, 16, 16, 0>, Shape<16, 16, 16, 16, 1>, 4, 2>{}); return true;
    case (size_t)1 << 16: f(TwoPass<float, 16, 16, 16, 16, 0, 2, 2>{}); return true;
    case (size_t)1 << 17: f(TwoPassG<float, Shape<16, 16, 16, 16, 0>, Shape<16, 32, 32, 8, 1>, 2, 2>{}); return true;
    case (size_t)1 << 19: f(TwoPassG<float, Shape<16, 32, 32, 8, 8>, Shape<32, 32, 32, 8, 1>, 2, 2>{}); return true;
    case (size_t)1 << 18: f(TwoPass<float, 16, 32, 16, 8, 0, 2, 2>{}); return true;
    default: return false;
  }
}
template <class F> bool visit_config_f64(size_t n, F&& f) {
  switch (n) {
    case (size_t)1 << 16: f(TwoPass<double, 16, 16, 8, 8, 4, 2, 2>{}); return true;
    case (size_t)1 << 9: f(TwoPassG<double, Shape<4, 4, 4, 16, 0>, Shape<4, 8, 8, 16, 2>, 4, 4>{}); return true;
    case (size_t)1 << 10: f(TwoPassG<double, Shape<4, 8, 8, 16, 0>, Shape<4, 8, 8, 16, 2>, 4, 4>{}); return true;
    case (size_t)1 << 11: f(TwoPassG<double, Shape<4, 8, 8, 16, 0>, Shape<8, 8, 8, 16, 1>, 4, 4>{}); return true;
    case (size_t)1 << 12: f(TwoPass<double, 8, 8, 16, 16, 0, 4, 4>{}); return true;
    case (size_t)1 << 13: f(TwoPassG<double, Shape<8, 8, 8, 16, 0>, Shape<8, 16, 16, 8, 1>, 4, 2>{}); return true;
    case (size_t)1 << 15: f(TwoPassG<double, Shape<8, 16, 16, 8, 4>, Shape<16, 16, 16, 8, 1>, 2, 2>{}); return true;
    case (size_t)1 << 14: f(TwoPass<double, 8, 16, 16, 8, 0, 4, 2>{}); return true;
    default: return false;
  }
}
template <typename T, class F> bool visit_config(size_t n, F&& f) {
  if constexpr (sizeof(T) == 4) return visit_config_f32(n, f);
  else return visit_config_f64(n, f);
}
template <typename T> const TwoPassOps<T>* lookup(size_t n) {
  const TwoPassOps<T>* o = nullptr;
  visit_config<T>(n, [&](auto g) { o = decltype(g)::ops(); });
  return o;
}

}  // namespace twopass
}  // namespace fb200
