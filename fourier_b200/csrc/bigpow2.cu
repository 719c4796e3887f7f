// bigpow2.cu -- three passes: power-of-two N beyond the two-pass kernels (f32 2^21 .. 2^30, f64 2^17 .. 2^24), and
// N = 3^b * 2^k (b <= 3) beyond the CTA kernel's shared memory.
//
//   N = Na * Nb:  an outer column pass of length Na over HBM (outer_kernels.cuh), then the Na rows of length Nb on the
//   two-pass tile kernels of an inner plan whose last register stage stores TRANSPOSED (dist_kernels.cuh with a single
//   destination: X[ka + Na * kb] leaves the row kernel at out[kb * Na + ka]) -- the autosort of the reference
//   (autosort/mod.rs:313-404) realised as two sweeps over HBM instead of one per radix-4/8 stage (11 sweeps at 2^24),
//   and without any table of N entries (the reference's twiddle table, autosort/mod.rs:24-46, would be 128 MB per
//   direction at N = 2^24; the general per-stage path of this library needs one too).
#include <algorithm>

#include "outer_kernels.cuh"
#include "plan.h"
#include "twopass_kernels.cuh"

namespace fb200 {

namespace {

template <typename T> struct ColumnOps {
  int ra, rb, c;
  cudaError_t (*launch)(const cpx<T>* in, cpx<T>* out, const void* twa, size_t nb, size_t batch, T scale, bool fwd,
                        cudaStream_t s);
};

// register tile Shape (twopass_kernels.cuh) of the outer pass, C columns per CTA
template <typename T, class S, int MINB> struct ColumnImpl {
  template <bool FWD> using Tile = TileFFT<T, S::RA, S::RB, S::E, S::C, FWD>;
  using Lay = ExLayout<S::RA * S::C + S::PAD, S::C, 1>;
  static constexpr size_t smem = sizeof(cpx<T>) * Tile<true>::template smem_elems<Lay>();
  template <bool FWD>
  static cudaError_t run(const cpx<T>* in, cpx<T>* out, const void* twa, size_t nb, size_t batch, T scale, cudaStream_t s) {
    using Body = outer::ColumnBody<Tile<FWD>, Lay>;
    auto kernel = &outer::column_kernel<Body, Tile<FWD>, MINB>;
    static std::atomic<unsigned long long> prepared{0};
    if (cudaError_t e = ensure_dynamic_smem(kernel, smem, prepared)) return e;
    typename Body::Args a;
    a.in = in; a.out = out; a.twa = (const TwPair<T>*)twa;
    a.nb = nb; a.n_total = (unsigned long long)S::L * nb; a.tiles = (unsigned)(nb / S::C); a.scale = scale;
    kernel<<<(unsigned)(batch * (nb / S::C)), Tile<FWD>::THREADS, smem, s>>>(a);
    return cudaGetLastError();
  }
  static cudaError_t launch(const cpx<T>* in, cpx<T>* out, const void* twa, size_t nb, size_t batch, T scale, bool fwd,
                            cudaStream_t s) {
    return fwd ? run<true>(in, out, twa, nb, batch, scale, s) : run<false>(in, out, twa, nb, batch, scale, s);
  }
  static const ColumnOps<T>* ops() {
    static const ColumnOps<T> o = {S::RA, S::RB, S::C, &launch};
    return &o;
  }
};

using twopass::Shape;
template <typename T> const ColumnOps<T>* column_lookup(int log2_na);
template <> const ColumnOps<float>* column_lookup<float>(int a) {
  switch (a) {   // the pass-1 shapes of the two-pass configurations (bank-conflict-free paddings checked by the emulator)
    case 5: return ColumnImpl<float, Shape<4, 8, 8, 32, 0>, 4>::ops();
    case 6: return ColumnImpl<float, Shape<8, 8, 8, 32, 0>, 4>::ops();
    case 7: return ColumnImpl<float, Shape<8, 16, 16, 16, 0>, 4>::ops();
    case 8: return ColumnImpl<float, Shape<16, 16, 16, 16, 0>, 2>::ops();
    case 9: return ColumnImpl<float, Shape<16, 32, 32, 8, 8>, 2>::ops();
    case 10: return ColumnImpl<float, Shape<32, 32, 32, 8, 8>, 2>::ops();
    default: return nullptr;
  }
}
template <> const ColumnOps<double>* column_lookup<double>(int a) {
  switch (a) {
    case 4: return ColumnImpl<double, Shape<4, 4, 4, 16, 0>, 4>::ops();
    case 5: return ColumnImpl<double, Shape<4, 8, 8, 16, 0>, 4>::ops();
    case 6: return ColumnImpl<double, Shape<8, 8, 8, 16, 0>, 4>::ops();
    case 7: return ColumnImpl<double, Shape<8, 16, 16, 8, 4>, 2>::ops();
    case 8: return ColumnImpl<double, Shape<16, 16, 16, 8, 4>, 2>::ops();
    default: return nullptr;
  }
}

// outer radix-3 / 9 / 27 pass: one thread per column
template <typename T, int B, bool FWD>
cudaError_t run_radix3(const cpx<T>* in, cpx<T>* out, size_t nb, size_t batch, T scale, cudaStream_t s) {
  using Body = outer::Radix3ColumnBody<T, B, FWD>;
  typename Body::Args a;
  a.in = in; a.out = out; a.nb = nb; a.n_total = (unsigned long long)B * nb; a.count = (unsigned long long)batch * nb;
  a.scale = scale;
  outer::radix3_column_kernel<Body><<<(unsigned)((a.count + 255) / 256), 256, 0, s>>>(a);
  return cudaGetLastError();
}
template <typename T>
cudaError_t launch_radix3(int b, const cpx<T>* in, cpx<T>* out, size_t nb, size_t batch, T scale, bool fwd, cudaStream_t s) {
  switch (b) {
    case 3: return fwd ? run_radix3<T, 3, true>(in, out, nb, batch, scale, s) : run_radix3<T, 3, false>(in, out, nb, batch, scale, s);
    case 9: return fwd ? run_radix3<T, 9, true>(in, out, nb, batch, scale, s) : run_radix3<T, 9, false>(in, out, nb, batch, scale, s);
    case 27: return fwd ? run_radix3<T, 27, true>(in, out, nb, batch, scale, s) : run_radix3<T, 27, false>(in, out, nb, batch, scale, s);
    default: return cudaErrorNotSupported;
  }
}

}  // namespace

// N = 3^b * 2^k, b = 1 .. 3, with 2^k a two-pass size: outer radix-3^b pass + two-pass rows (the reference's radix-3
// stages, autosort/mod.rs:20-21, taken first).  Covers the {2,3}-smooth sizes with a large power-of-two factor that do
// not fit the CTA kernel's shared memory (3 * 2^13 ... 27 * 2^20 f32); the rest stays on the per-stage path.
template <typename T>
cudaError_t Plan<T>::init_threepass_radix3() {
  size_t r = n_;
  int b = 1;
  while (r % 3 == 0 && b < 27) { r /= 3; b *= 3; }
  if (b == 1 || (r & (r - 1)) || r % 3 == 0) return cudaErrorNotSupported;
  inner_.reset(Plan<T>::create(r, device_, true, tuning_));
  if (!inner_ || inner_->path() != Path::kTwoPass) { inner_.reset(); return cudaErrorNotSupported; }
  n1_ = (size_t)b;
  n2_ = r;
  outer_radix3_ = b;
  return cudaSuccess;
}

template <typename T>
cudaError_t Plan<T>::init_bigpow2() {
  int k = 0;
  while (((size_t)1 << k) < n_) ++k;
  constexpr int a_min = sizeof(T) == 4 ? 5 : 4, a_max = sizeof(T) == 4 ? 10 : 8;
  constexpr int k_min = sizeof(T) == 4 ? 21 : 17, k_max = sizeof(T) == 4 ? 30 : 24;
  if (((size_t)1 << k) != n_ || k < k_min || k > k_max) return cudaErrorNotSupported;
  // rows of 2^14 where possible (the best tile-kernel size with 16-row tiles), the outer pass takes the rest
  int a = std::min(a_max, std::max(a_min, k - 14));
  if (tuning_.big_na) a = std::min(a_max, std::max(a_min, *tuning_.big_na));
  const ColumnOps<T>* col = column_lookup<T>(a);
  if (!col) return cudaErrorNotSupported;
  inner_.reset(Plan<T>::create((size_t)1 << (k - a), device_, true, tuning_));
  if (!inner_ || inner_->path() != Path::kTwoPass) { inner_.reset(); return cudaErrorNotSupported; }
  n1_ = (size_t)1 << a;
  n2_ = (size_t)1 << (k - a);
  FB_CHECK(upload(tw_a_, twopass::make_twa<T>(col->ra, col->rb)));
  fast_ops_ = col;
  return cudaSuccess;
}

template <typename T>
cudaError_t Plan<T>::exec_bigpow2(const C* in, C* out, size_t batch, int code, cudaStream_t s) {
  const auto* col = static_cast<const ColumnOps<T>*>(fast_ops_);   // nullptr with an outer radix-3 pass
  const bool fwd = transform_is_forward(code);
  const T scale = scale_for<T>(code, n_);
  // the intermediate A[ka][nb] of a few transforms at a time (at most 2 GB of scratch, at least one transform)
  const size_t chunk = std::min(batch, std::max<size_t>(1, ((size_t)2 << 30) / (n_ * sizeof(C))));
  // the row kernel works on whole tiles of up to 32 rows: 3 / 9 / 27 rows per transform are padded up (the padding rows
  // are transformed and dropped)
  const size_t rows_max = (chunk * n1_ + 31) / 32 * 32;
  FB_CHECK(work_.reserve(rows_max * n2_ * sizeof(C)));
  C* work = (C*)work_.data();
  for (size_t b0 = 0; b0 < batch; b0 += chunk) {
    const size_t nb = std::min(chunk, batch - b0);
    if (outer_radix3_) FB_CHECK(launch_radix3<T>(outer_radix3_, in + b0 * n_, work, n2_, nb, scale, fwd, s));
    else FB_CHECK(col->launch(in + b0 * n_, work, tw_a_.data(), n2_, nb, scale, fwd, s));
    ++launches_;
    void* dst = out + b0 * n_;   // the rows of all nb transforms in one call: batch b is stored n_ elements further on
    const size_t rows = nb * n1_, rows_pad = outer_radix3_ ? (rows + 31) / 32 * 32 : rows;
    FB_CHECK(inner_->exec_rows_exchange(work, rows_pad, fwd, &dst, 1, n1_, 0, 0, 0, 0, s, n1_, n_, rows));
    launches_ += inner_->launches();
  }
  return cudaSuccess;
}

template cudaError_t Plan<float>::init_threepass_radix3();
template cudaError_t Plan<double>::init_threepass_radix3();
template cudaError_t Plan<float>::init_bigpow2();
template cudaError_t Plan<double>::init_bigpow2();
template cudaError_t Plan<float>::exec_bigpow2(const C*, C*, size_t, int, cudaStream_t);
template cudaError_t Plan<double>::exec_bigpow2(const C*, C*, size_t, int, cudaStream_t);

}  // namespace fb200
