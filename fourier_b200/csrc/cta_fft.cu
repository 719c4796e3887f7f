// cta_fft.cu -- plans and launcher of the CTA-level shared-memory transforms (cta_kernels.cuh): any {2,3}-smooth N
// that fits two shared-memory buffers, and the fused Bluestein chirp-z for inner sizes above the warp-level kernel.
// Reference counterparts: Autosort::new's factorisation (autosort/mod.rs:104-117 -- here 16/8/4/2 and 9/3 instead of
// 4/8/4/3/2: wider butterflies mean fewer shared-memory sweeps) and Bluesteins::apply (bluesteins.rs:218-259).
#include <algorithm>
#include <cmath>

#include "cta_kernels.cuh"
#include "plan.h"

namespace fb200 {

namespace {

constexpr size_t kSmemLimit = 227 * 1024;

template <typename T> size_t smem_bytes(int group, int len) {
  return 2 * (size_t)cta::buffer_elems(group, len) * sizeof(cpx<T>);
}

// Transforms per CTA iteration: at most about 32 KB per buffer (three CTAs share an SM), and among the candidates
// the one whose stages leave the fewest of the 256 threads idle in their last round of butterflies.
template <typename T> int group_for(int len) {
  const int target = (int)(32768 / sizeof(cpx<T>));
  const int gmax = std::max(1, target / len);
  cta::Stages st;
  if (!cta::factorize((size_t)len, st)) return gmax;
  int best = gmax;
  double best_eff = 0;
  for (int g = gmax; g >= std::max(1, gmax / 2); --g) {
    double work = 0, slots = 0;
    for (int s = 0; s < st.count; ++s) {
      const double n = (double)g * (len / st.radix[s]);
      work += n * st.radix[s];
      slots += std::ceil(n / cta::kThreads) * cta::kThreads * st.radix[s];
    }
    const double eff = work / slots;
    if (eff > best_eff + 1e-9) { best_eff = eff; best = g; }
  }
  return best;
}

template <typename T, bool DIR, bool CHIRP>
cudaError_t launch(const cta::Args<T>& a, int sms, cudaStream_t s) {
  const size_t bytes = smem_bytes<T>(a.group, a.len);
  // several CTAs per SM need the full shared-memory carve-out (the default heuristic left room for two of three)
  static std::atomic<unsigned long long> prepared{0};
  if (cudaError_t e = ensure_dynamic_smem(cta::cta_fft_kernel<T, DIR, CHIRP>, kSmemLimit, prepared,
                                          (int)cudaSharedmemCarveoutMaxShared))
    return e;
  const size_t groups = ((size_t)a.batch + a.group - 1) / a.group;
  const size_t per_sm = std::max<size_t>(1, std::min<size_t>(8, kSmemLimit / (bytes + 1024)));
  const unsigned grid = (unsigned)std::min<size_t>(groups, (size_t)sms * per_sm);
  cta::cta_fft_kernel<T, DIR, CHIRP><<<grid, cta::kThreads, bytes, s>>>(a);
  return cudaGetLastError();
}

}  // namespace

// Largest on-chip transform length of the CTA kernel for precision T.
template <typename T> size_t cta_max_len() {
  size_t len = 1;
  while (smem_bytes<T>(1, (int)(len * 2)) <= kSmemLimit) len *= 2;
  // not only powers of two: the true bound is the byte count; this is the largest power of two that fits
  return len;
}

template <typename T>
bool cta_fits(size_t len) { return len >= 2 && len < ((size_t)1 << 20) && smem_bytes<T>(1, (int)len) <= kSmemLimit; }

template <typename T>
cudaError_t Plan<T>::init_cta(size_t len) {
  if (!is_23_smooth(len) || !cta_fits<T>(len)) return cudaErrorNotSupported;
  cta_len_ = len;
  cta::Stages st;
  if (!cta::factorize(len, st)) return cudaErrorNotSupported;
  radices_.assign(st.radix, st.radix + st.count);
  FB_CHECK(upload(wtab_, cta::make_stage_twiddles<T>(len, st, host_twiddle)));
  return cudaSuccess;
}

template <typename T>
cudaError_t Plan<T>::exec_cta(const C* in, C* out, size_t batch, int code, cudaStream_t s, bool chirp) {
  const bool fwd = transform_is_forward(code);
  cta::Args<T> a;
  a.in = in; a.out = out;
  a.wtab = (const C*)wtab_.data();
  a.chirp = (const C*)chirp_.data();
  a.wf = (const C*)wf_.data();
  a.batch = (long)batch;
  a.n = (int)n_;
  a.len = (int)cta_len_;
  a.group = group_for<T>(a.len);
  T scale = scale_for<T>(code, n_);
  if (chirp) scale /= (T)cta_len_;      // the unscaled inner inverse transform
  a.scale = scale;
  cta::factorize(cta_len_, a.st);
  a.pad = a.st.radix[0] % 2 == 0 ? 1 : 0;
  cudaError_t e;
  if (chirp) e = fwd ? launch<T, true, true>(a, sm_count_, s) : launch<T, false, true>(a, sm_count_, s);
  else e = fwd ? launch<T, true, false>(a, sm_count_, s) : launch<T, false, false>(a, sm_count_, s);
  FB_CHECK(e);
  launches_ += 1;
  return cudaSuccess;
}

template cudaError_t Plan<float>::init_cta(size_t);
template cudaError_t Plan<double>::init_cta(size_t);
template cudaError_t Plan<float>::exec_cta(const C*, C*, size_t, int, cudaStream_t, bool);
template cudaError_t Plan<double>::exec_cta(const C*, C*, size_t, int, cudaStream_t, bool);

}  // namespace fb200
