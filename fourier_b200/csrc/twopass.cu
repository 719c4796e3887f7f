// twopass.cu -- large power-of-two N: the four-step FFT as TWO fused kernels with the intermediate
// kept in L2.
//
//   N = N1*N2, input index n = n1*N2 + n2, output index k = k1 + N1*k2
//   pass 1 (column tiles): for every n2:  A[k1][n2] = w_N^{n2*k1} * sum_{n1} x[n1*N2+n2] w_N1^{n1*k1}
//   pass 2 (row tiles):    for every k1:  X[k1 + N1*k2] = sum_{n2} A[k1][n2] w_N2^{n2*k2}
//
// Each pass is one TileFFT (tilefft.cuh): every sample is read once from global memory into
// registers, transformed by two register radix-R stages with one shared-memory exchange, and written
// once.  The reference streams the whole array once per radix-4/8 stage -- seven sweeps at N = 2^20
// (autosort/mod.rs:338-379, SURVEY.md 3.2); here HBM sees one read and one write per sample as long
// as the intermediate A of a few transforms stays resident in the 126 MB L2, which is what the
// chunking in exec_twopass() arranges.  All global accesses are >= 128-byte contiguous pieces:
//   pass 1 reads  x  as C consecutive columns (C*8 B per row),  writes A[k1][n2] the same way;
//   pass 2 reads  A  as whole contiguous rows,                  writes X as C consecutive k1.
#include <cstdio>

#include "plan.h"
#include "fused_kernels.cuh"
#include "twopass_kernels.cuh"

namespace fb200 {

using namespace twopass;

namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}

template <typename T> struct FusedOps {
  size_t n1, n2;
  int ra, rb, ra2, rb2, tile_c;   // register tiles of pass 1 (ra x rb) and pass 2 (ra2 x rb2); columns per pass-1 tile
  size_t smem_bytes;
  int default_ring, default_lag;
  bool base_pcol;   // layout of the factored base table this configuration reads (tables.cuh)
  cudaError_t (*prepare)();
  cudaError_t (*launch)(const fused::FusedArgs<T>&, bool fwd, int grid, cudaStream_t);
};

template <class Cfg> struct FusedImpl {
  using T = typename Cfg::T;
  static cudaError_t prepare() {
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(fused::fused_twopass_kernel<Cfg, true>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM_BYTES)))
      return e;
    return cudaFuncSetAttribute(fused::fused_twopass_kernel<Cfg, false>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM_BYTES);
  }
  static cudaError_t launch(const fused::FusedArgs<T>& a, bool fwd, int grid, cudaStream_t s) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return cudaErrorNotSupported;
    CUtensorMap map;
    const cuuint64_t gdim[2] = {(cuuint64_t)(2 * Cfg::N2), (cuuint64_t)a.batch * (cuuint64_t)Cfg::N1};
    const cuuint64_t gstride[1] = {(cuuint64_t)(Cfg::N2 * sizeof(cpx<T>))};
    const cuuint32_t box[2] = {(cuuint32_t)(2 * Cfg::C1), (cuuint32_t)Cfg::BOX_ROWS};
    const cuuint32_t estr[2] = {1, 1};
    const CUtensorMapDataType dt = sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64;
    if (enc(&map, dt, 2, (void*)a.in, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
      set_last_error("cuTensorMapEncodeTiled failed");
      return cudaErrorInvalidValue;
    }
    if (fwd) fused::fused_twopass_kernel<Cfg, true><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, s>>>(map, a);
    else fused::fused_twopass_kernel<Cfg, false><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, s>>>(map, a);
    return cudaGetLastError();
  }
  static const FusedOps<T>* ops(int ring, int lag) {
    static const FusedOps<T> o = {(size_t)Cfg::N1, (size_t)Cfg::N2, Cfg::RA, Cfg::RB, Cfg::RA2, Cfg::RB2, Cfg::C1, Cfg::SMEM_BYTES, ring, lag,
                                  true, &prepare, &launch};
    return &o;
  }
};

template <typename T> const FusedOps<T>* fused_lookup(size_t n);
template <> const FusedOps<float>* fused_lookup<float>(size_t n) {
  if (n == ((size_t)1 << 20)) {
    // default: two 256-thread groups, TMA staging, one shared exchange buffer taken under a lock
    return FusedImpl<fused::FusedCfg<float, 32, 8, 2, 8, 1>>::ops(8, 4);
  }
  if (n == ((size_t)1 << 16)) {
    // 256 x 256 with 16 x 16 register tiles, four 128-thread groups, 64-byte tile rows as at 2^20.  Measured on B200
    // (profiles/r02_sizes_cta_and_2pow16.txt): TMA staging 56.5 %, direct loads 51.7 % (ring 128; 47 % at ring 64),
    // two launches per chunk 33.9 % of the measured HBM peak.
    return FusedImpl<fused::FusedCfg<float, 16, 8, 4, 8, 4>>::ops(128, 64);
  }
  if (n == ((size_t)1 << 18)) {
    // 512 x 512 with 32 x 16 register tiles: three 128-thread groups with TMA staging, or four with direct loads
    return FusedImpl<fused::FusedCfg<float, 32, 8, 3, 8, 3, false, 16>>::ops(32, 16);
  }
  if (n == ((size_t)1 << 14)) {
    // 128 x 128 with 16 x 8 register tiles: eight 64-thread groups
    return FusedImpl<fused::FusedCfg<float, 16, 8, 8, 8, 8, false, 8>>::ops(512, 256);
  }
  // Odd powers of two: N1 x 2 N1 with a different register tile per pass, same threads per FFT in both
  // (template arguments: <T, RA, C, G, PAD1, EXB, DIRECT, RB, RA2, RB2, E1, E2>).  Ring = 64 MB / transform size.
  if (n == ((size_t)1 << 19)) {   // 512 (32 x 16) x 1024 (32 x 32), 16-column pass-1 tiles: two 256-thread groups
    return FusedImpl<fused::FusedCfg<float, 32, 8, 2, 0, 1, false, 16, 32, 32, 32, 32, 16, true>>::ops(32, 16);   // 39 % (ring 16: 35 %, tile kernels 29 %)
  }
  if (n == ((size_t)1 << 17)) {   // 256 (16 x 16, 16 per thread) x 512 (32 x 16, 32 per thread): three 128-thread groups
    return FusedImpl<fused::FusedCfg<float, 16, 8, 3, 8, 3, false, 16, 32, 16, 16, 32>>::ops(64, 32);
  }
  if (n == ((size_t)1 << 15)) {   // 128 (16 x 8, 16 per thread) x 256 (16 x 16, 32 per thread): six 64-thread groups
    return FusedImpl<fused::FusedCfg<float, 16, 8, 6, 8, 6, false, 8, 16, 16, 16, 32>>::ops(256, 128);
  }
  // (f32 2^12 = 64 x 64 was tried on the persistent kernel: 39.0 % against 41.7 % for the two-launch tile kernels)
  if (n == ((size_t)1 << 13)) {   // 64 (8 x 8, 8 per thread) x 128 (16 x 8, 16 per thread): eight 64-thread groups
    return FusedImpl<fused::FusedCfg<float, 8, 8, 8, 8, 8, false, 8, 16, 8, 8, 16>>::ops(512, 256);
  }
  return nullptr;
}
template <> const FusedOps<double>* fused_lookup<double>(size_t n) {
  if (n == ((size_t)1 << 16)) {
    // Three 128-thread groups with TMA staging, or four loading directly from global memory.  Short runs are a tie
    // (62.5 % / 59.9 % at batch 2048, 57.9 % / 58.8 % at 16384); at the BASELINE batch of 65536, where the run is
    // power-capped at ~1760 MHz, staging wins twice out of two A/B pairs: 56.5 / 57.4 % against 54.3 / 54.4 %
    // (profiles/r02_c3_staged_vs_direct.txt).
    return FusedImpl<fused::FusedCfg<double, 16, 8, 3, 4, 3>>::ops(64, 32);
  }
  if (n == ((size_t)1 << 14)) {
    // 128 x 128 with 16 x 8 register tiles: four 64-thread groups with TMA staging, or eight loading directly
    // measured: four groups with TMA staging 62.0 %, eight groups loading directly 53.7 %, tile kernels 37.7 %
    return FusedImpl<fused::FusedCfg<double, 16, 8, 4, 4, 4, false, 8>>::ops(256, 128);
  }
  if (n == ((size_t)1 << 12)) {   // 64 x 64 with 8 x 8 register tiles
    return FusedImpl<fused::FusedCfg<double, 8, 8, 8, 4, 8, true>>::ops(1024, 512);
  }
  if (n == ((size_t)1 << 13)) {   // 64 (8 x 8) x 128 (16 x 8): eight 64-thread groups loading directly
    return FusedImpl<fused::FusedCfg<double, 8, 8, 8, 4, 8, true, 8, 16, 8, 8, 16>>::ops(512, 256);
  }
  return nullptr;
}

}  // namespace

template <typename T>
cudaError_t Plan<T>::init_twopass() {
  const TwoPassOps<T>* ops = lookup<T>(n_);
  if (!ops) return cudaErrorNotSupported;
  FB_CHECK(ops->prepare());
  n1_ = ops->n1;
  n2_ = ops->n2;
  FB_CHECK(upload(tw_a_, make_twa<T>(ops->ra1, ops->rb1)));
  FB_CHECK(upload(tw_b_, make_twa<T>(ops->ra2, ops->rb2)));
  // inter-pass twiddles in the layout of the intermediate: T[k1*N2 + n2] = w_N^{n2*k1}
  std::vector<cpx<T>> tw2(n_);
  for (size_t k1 = 0; k1 < n1_; ++k1)
    for (size_t c = 0; c < n2_; ++c) {
      double re, im;
      host_twiddle(k1 * c, n_, &re, &im);
      tw2[k1 * n2_ + c] = mk<T>((T)re, (T)im);
    }
  FB_CHECK(upload(tw2_, tw2));
  // transforms per chunk: the intermediate of one chunk should sit comfortably inside the L2
  chunk_ = std::max<size_t>(1, (tuning_.chunk_mb << 20) / (n_ * sizeof(C)));
  fast_ops_ = ops;
  // the persistent fused kernel (one launch for the whole batch) where a configuration exists
  fused_ops_ = nullptr;
  if (tuning_.fused) {
    const FusedOps<T>* f = fused_lookup<T>(n_);
    if (f && f->prepare() == cudaSuccess) {
      // the persistent kernel has its own split and register tile (the tile kernels above stay as its fallback)
      FB_CHECK(upload(tw_f_, make_twa<T>(f->ra, f->rb)));
      FB_CHECK(upload(tw_f2_, make_twa<T>(f->ra2, f->rb2)));
      // factored inter-pass twiddles, contiguous per pass-1 tile of `tile_c` columns:
      //   tbase[tile][col][p] = w_N^{n2*p},  tstep[tile][r][col] = w_N^{R*n2*r},  n2 = tile*tile_c + col
      std::vector<cpx<T>> tb, ts;
      make_factored_twiddles<T>(n_, f->n2, f->ra, f->rb, f->tile_c, tb, ts, f->base_pcol);
      FB_CHECK(upload(tbase_, tb));
      FB_CHECK(upload(tstep_, ts));
      fused_ops_ = f;
      ring_ = std::max(2, tuning_.ring.value_or(f->default_ring));
      while (ring_ & (ring_ - 1)) ++ring_;   // the kernel wants a power of two
      lag_ = std::min(ring_ - 1, std::max(1, tuning_.lag.value_or(f->default_lag)));
    }
  }
  return cudaSuccess;
}

template <typename T>
cudaError_t Plan<T>::exec_twopass(const C* in, C* out, size_t batch, int code, cudaStream_t s) {
  const auto* ops = static_cast<const TwoPassOps<T>*>(fast_ops_);
  const bool fwd = transform_is_forward(code);
  const bool do_scale = !(code == kFft || code == kUnscaledIfft);
  const T scale = scale_for<T>(code, n_);
  if (fused_ops_ && batch <= (size_t)1 << 24) {
    const auto* f = static_cast<const FusedOps<T>*>(fused_ops_);
    int ring = ring_;
    while (ring > 2 && (size_t)ring / 2 >= batch) ring /= 2;
    const int lag = std::min(lag_, ring - 1);
    FB_CHECK(work_.reserve((size_t)ring * n_ * sizeof(C)));
    const size_t cbytes = (1 + 2 * batch) * sizeof(unsigned);
    FB_CHECK(counters_.reserve(cbytes));
    FB_CHECK(cudaMemsetAsync(counters_.data(), 0, cbytes, s));
    fused::FusedArgs<T> a;
    a.in = in; a.out = out; a.scratch = (C*)work_.data();
    a.twa = (const TwPair<T>*)tw_f_.data();
    a.twa2 = (const TwPair<T>*)tw_f2_.data();
    a.tbase = (const C*)tbase_.data(); a.tstep = (const C*)tstep_.data();
    a.counters = (unsigned*)counters_.data();
    a.trace = nullptr;
    if (!tuning_.trace.empty()) {
      const size_t tbytes = sizeof(long long) * 64 * fused::kTraceTiles * fused::kTracePhases;
      FB_CHECK(trace_.reserve(tbytes));
      FB_CHECK(cudaMemsetAsync(trace_.data(), 0, tbytes, s));
      a.trace = (long long*)trace_.data();
    }
    a.batch = (int)batch; a.ring = ring; a.lag = lag; a.scale = scale; a.do_scale = do_scale ? 1 : 0;
    const size_t tiles = batch * (f->n2 / (size_t)f->tile_c + f->n1 / 8);
    const int grid = (int)std::min<size_t>((size_t)sm_count_, std::max<size_t>(1, tiles / 2));
    FB_CHECK(f->launch(a, fwd, grid, s));
    launches_ += 1;
    if (a.trace) {  // dump the timeline of CTA 0 (debug aid; synchronises)
      std::vector<long long> h(64 * fused::kTraceTiles * fused::kTracePhases);
      FB_CHECK(cudaStreamSynchronize(s));
      FB_CHECK(cudaMemcpy(h.data(), trace_.data(), h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
      if (FILE* fp = fopen(tuning_.trace.c_str(), "w")) {
        for (int w = 0; w < 40; ++w)
          for (int k = 0; k < fused::kTraceTiles; ++k) {
            const long long* r = &h[((size_t)w * fused::kTraceTiles + k) * fused::kTracePhases];
            fprintf(fp, "%d %d %lld %lld %lld %lld %lld %lld %lld %lld\n", w, k, r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7]);
          }
        fclose(fp);
      }
    }
    return cudaSuccess;
  }
  const size_t chunk = std::min(chunk_, batch);
  FB_CHECK(work_.reserve(chunk * n_ * sizeof(C)));
  C* scratch = (C*)work_.data();
  for (size_t b0 = 0; b0 < batch; b0 += chunk) {
    const size_t nb = std::min(chunk, batch - b0);
    FB_CHECK(ops->pass1(in + b0 * n_, scratch, tw_a_.data(), (const C*)tw2_.data(), nb, fwd, s));
    FB_CHECK(ops->pass2(scratch, out + b0 * n_, tw_b_.data(), nb, fwd, scale, do_scale, s));
    launches_ += 2;
  }
  return cudaSuccess;
}

template cudaError_t Plan<float>::init_twopass();
template cudaError_t Plan<double>::init_twopass();
template cudaError_t Plan<float>::exec_twopass(const C*, C*, size_t, int, cudaStream_t);
template cudaError_t Plan<double>::exec_twopass(const C*, C*, size_t, int, cudaStream_t);

}  // namespace fb200
