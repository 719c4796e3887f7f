// onchip.cu -- plans and launchers for the transforms that fit on chip (onchip_kernels.cuh):
// batched power-of-two FFTs up to 1024 points and the fused Bluestein kernel for N <= 1024.
// Reference counterparts: Autosort for small sizes (autosort/mod.rs:141-166) and
// Bluesteins::transform_in_place / apply (bluesteins.rs:193-259).
#include <algorithm>

#include "onchip_kernels.cuh"
#include "plan.h"
#include "tables.cuh"  // make_twa

namespace fb200 {

namespace {

using onchip::OnChipCfg;

template <typename T> struct OnChipOps {
  int ra, rb;
  cudaError_t (*prepare)();
  cudaError_t (*fft)(const cpx<T>*, cpx<T>*, const void* twa, size_t batch, bool fwd, T scale, bool do_scale,
                     int sms, cudaStream_t);
  // Bluestein: nullptr when the size class has no fused kernel
  cudaError_t (*bluestein)(const cpx<T>*, cpx<T>*, const void* twa, const cpx<T>* chirp, const cpx<T>* wm,
                           const cpx<T>* wce, const cpx<T>* wco, size_t n, size_t batch, T scale, int sms,
                           cudaStream_t);
};

template <typename T, int RA, int RB, int E, int WARPS, int MINB, int BWARPS, bool LOCAL_STASH = false>
struct OnChipImpl {
  template <bool FWD> using Cfg = OnChipCfg<T, RA, RB, E, WARPS, FWD>;
  using BCfg = OnChipCfg<T, RA, RB, E, BWARPS, true>;
  static constexpr size_t smem_fft = Cfg<true>::EX_BYTES + Cfg<true>::TWA_BYTES;
  static constexpr size_t smem_blue =
      BCfg::EX_BYTES + BCfg::TWA_BYTES + sizeof(cpx<T>) * (4 * (size_t)BCfg::L + (LOCAL_STASH ? 0 : (size_t)E * BCfg::THREADS));
  static constexpr bool kHasBluestein = (RA == RB) && (E == RA);

  static cudaError_t prepare() {
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(onchip::onchip_fft_kernel<Cfg<true>, MINB>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_fft))) return e;
    if ((e = cudaFuncSetAttribute(onchip::onchip_fft_kernel<Cfg<false>, MINB>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_fft))) return e;
    if constexpr (kHasBluestein) {
      if ((e = cudaFuncSetAttribute(onchip::bluestein_fused_kernel<BCfg, 1, LOCAL_STASH>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_blue))) return e;
    }
    return cudaSuccess;
  }
  static cudaError_t fft(const cpx<T>* in, cpx<T>* out, const void* twa, size_t batch, bool fwd, T scale,
                         bool do_scale, int sms, cudaStream_t s) {
    const size_t groups = (batch + Cfg<true>::C - 1) / Cfg<true>::C;
    const unsigned grid = (unsigned)std::min<size_t>(groups, (size_t)sms * MINB * 4);
    if (fwd) {
      typename onchip::FftBody<Cfg<true>>::Args a = {in, out, (const TwPair<T>*)twa, (long)batch, scale, do_scale};
      onchip::onchip_fft_kernel<Cfg<true>, MINB><<<grid, Cfg<true>::THREADS, smem_fft, s>>>(a);
    } else {
      typename onchip::FftBody<Cfg<false>>::Args a = {in, out, (const TwPair<T>*)twa, (long)batch, scale, do_scale};
      onchip::onchip_fft_kernel<Cfg<false>, MINB><<<grid, Cfg<false>::THREADS, smem_fft, s>>>(a);
    }
    return cudaGetLastError();
  }
  static cudaError_t bluestein(const cpx<T>* in, cpx<T>* out, const void* twa, const cpx<T>* chirp,
                               const cpx<T>* wm, const cpx<T>* wce, const cpx<T>* wco, size_t n, size_t batch,
                               T scale, int sms, cudaStream_t s) {
    if constexpr (kHasBluestein) {
      const size_t groups = (batch + BCfg::C - 1) / BCfg::C;
      const unsigned grid = (unsigned)std::min<size_t>(groups, (size_t)sms * 2);
      typename onchip::BluesteinBody<BCfg>::Args a = {in, out, (const TwPair<T>*)twa, chirp, wm, wce, wco,
                                                      (long)n, (long)batch, scale};
      onchip::bluestein_fused_kernel<BCfg, 1, LOCAL_STASH><<<grid, BCfg::THREADS, smem_blue, s>>>(a);
      return cudaGetLastError();
    } else {
      return cudaErrorNotSupported;
    }
  }
  static const OnChipOps<T>* ops() {
    static const OnChipOps<T> o = {RA, RB, &prepare, &fft, kHasBluestein ? &bluestein : nullptr};
    return &o;
  }
};

// size classes: L -> (RA, RB, E, warps per CTA, CTAs per SM, warps per CTA of the Bluestein kernel)
template <typename T> const OnChipOps<T>* onchip_lookup(size_t l);
template <> const OnChipOps<float>* onchip_lookup<float>(size_t l) {
  switch (l) {
    case 64: return OnChipImpl<float, 8, 8, 8, 8, 4, 8>::ops();
    case 128: return OnChipImpl<float, 8, 16, 16, 8, 4, 8>::ops();
    case 256: return OnChipImpl<float, 16, 16, 16, 8, 3, 8>::ops();
    case 512: return OnChipImpl<float, 16, 32, 32, 8, 2, 8>::ops();
    case 1024:
      // The fused Bluestein kernel parks the even half in thread-local memory (16 warps per SM, measured
      // 1.16e11 samples/s at N=1009); the shared-memory stash (11 warps per SM) measured 1.01e11.
      return OnChipImpl<float, 32, 32, 32, 8, 2, 16, true>::ops();
    default: return nullptr;
  }
}
template <> const OnChipOps<double>* onchip_lookup<double>(size_t l) {
  switch (l) {
    case 64: return OnChipImpl<double, 8, 8, 8, 8, 3, 8>::ops();
    case 128: return OnChipImpl<double, 8, 16, 16, 8, 2, 8>::ops();
    case 256: return OnChipImpl<double, 16, 16, 16, 8, 1, 8>::ops();
    default: return nullptr;
  }
}

}  // namespace

template <typename T>
cudaError_t Plan<T>::init_onchip() {
  const OnChipOps<T>* ops = onchip_lookup<T>(n_);
  if (!ops) return cudaErrorNotSupported;
  FB_CHECK(ops->prepare());
  FB_CHECK(upload(tw_a_, twopass::make_twa<T>(ops->ra, ops->rb)));
  fast_ops_ = ops;
  return cudaSuccess;
}

template <typename T>
cudaError_t Plan<T>::exec_onchip(const C* in, C* out, size_t batch, int code, cudaStream_t s) {
  const auto* ops = static_cast<const OnChipOps<T>*>(fast_ops_);
  const bool fwd = transform_is_forward(code);
  const bool do_scale = !(code == kFft || code == kUnscaledIfft);
  const T scale = scale_for<T>(code, n_);
  FB_CHECK(ops->fft(in, out, tw_a_.data(), batch, fwd, scale, do_scale, sm_count_, s));
  launches_ += 1;
  return cudaSuccess;
}

// Tables of the fused Bluestein kernel (one set per direction), built from the same chirp and W that
// init_bluestein() computes in double precision.
template <typename T>
cudaError_t Plan<T>::init_bluestein_fused(const std::vector<double>& chirp_re, const std::vector<double>& chirp_im,
                                          const std::vector<double>& w_re, const std::vector<double>& w_im) {
  const size_t l = m_ / 2;
  const OnChipOps<T>* ops = onchip_lookup<T>(l);
  if (!ops || !ops->bluestein) return cudaErrorNotSupported;
  FB_CHECK(ops->prepare());
  FB_CHECK(upload(tw_a_, twopass::make_twa<T>(ops->ra, ops->rb)));
  // layout per direction d (0 forward, 1 inverse): [chirp | wm | wce | wco], L entries each
  std::vector<cpx<T>> tab(2 * 4 * l, mk<T>((T)0, (T)0));
  for (int d = 0; d < 2; ++d) {
    const double sgn = d == 0 ? 1.0 : -1.0;   // the inverse direction conjugates chirp and W
    cpx<T>* t = tab.data() + (size_t)d * 4 * l;
    for (size_t i = 0; i < l; ++i) {
      if (i < n_) t[i] = mk<T>((T)chirp_re[i], (T)(sgn * chirp_im[i]));
      double re, im;
      host_twiddle(i, m_, &re, &im);
      t[l + i] = mk<T>((T)re, (T)im);                                    // w_M^i (same for both directions)
      t[2 * l + i] = mk<T>((T)w_re[2 * i], (T)(-sgn * w_im[2 * i]));          // conj(W_dir[2k])
      t[3 * l + i] = mk<T>((T)w_re[2 * i + 1], (T)(-sgn * w_im[2 * i + 1]));  // conj(W_dir[2k+1])
    }
  }
  FB_CHECK(upload(tbase_, tab));
  fast_ops_ = ops;
  return cudaSuccess;
}

template <typename T>
cudaError_t Plan<T>::exec_bluestein_fused(const C* in, C* out, size_t batch, int code, cudaStream_t s) {
  const auto* ops = static_cast<const OnChipOps<T>*>(fast_ops_);
  const bool fwd = transform_is_forward(code);
  const T scale = scale_for<T>(code, n_) / (T)m_;
  const size_t l = m_ / 2;
  const C* t = (const C*)tbase_.data() + (fwd ? 0 : 4 * l);
  FB_CHECK(ops->bluestein(in, out, tw_a_.data(), t, t + l, t + 2 * l, t + 3 * l, n_, batch, scale, sm_count_, s));
  launches_ += 1;
  return cudaSuccess;
}

template cudaError_t Plan<float>::init_onchip();
template cudaError_t Plan<double>::init_onchip();
template cudaError_t Plan<float>::exec_onchip(const C*, C*, size_t, int, cudaStream_t);
template cudaError_t Plan<double>::exec_onchip(const C*, C*, size_t, int, cudaStream_t);
template cudaError_t Plan<float>::init_bluestein_fused(const std::vector<double>&, const std::vector<double>&,
                                                       const std::vector<double>&, const std::vector<double>&);
template cudaError_t Plan<double>::init_bluestein_fused(const std::vector<double>&, const std::vector<double>&,
                                                        const std::vector<double>&, const std::vector<double>&);
template cudaError_t Plan<float>::exec_bluestein_fused(const C*, C*, size_t, int, cudaStream_t);
template cudaError_t Plan<double>::exec_bluestein_fused(const C*, C*, size_t, int, cudaStream_t);

}  // namespace fb200
