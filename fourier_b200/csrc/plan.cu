// plan.cu -- host side of the engine: plan construction (path selection, factorisation, twiddle and
// chirp tables), batched execution on device pointers, and the pipelined host-pointer path.
//
// Reference counterparts: create_fft_f32/f64 (fourier/src/lib.rs:31-60), Autosort::new +
// initialize_twiddles (fourier-algorithms/src/autosort/mod.rs:24-46,104-134), the stage driver
// apply_stages_* (mod.rs:313-404), Bluesteins::new_with_fft + initialize_{w,x}_twiddles
// (bluesteins.rs:18-61,109-130) and bluesteins::apply (bluesteins.rs:218-259).
#include "plan.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>

namespace fb200 {

// ---------------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
void set_last_error(const std::string& s) { g_last_error = s; }
const char* last_error() { return g_last_error.c_str(); }

const char* path_name(Path p) {
  switch (p) {
    case Path::kTrivial: return "trivial";
    case Path::kOnChip: return "onchip";
    case Path::kTwoPass: return "twopass";
    case Path::kGlobalStages: return "global_stages";
    case Path::kBluestein: return "bluestein";
    case Path::kBluesteinFused: return "bluestein_fused";
    case Path::kCta: return "onchip_cta";
    case Path::kThreePass: return "threepass";
  }
  return "?";
}

// ---------------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------------
bool is_23_smooth(size_t n) {
  if (n == 0) return false;
  while (n % 2 == 0) n /= 2;
  while (n % 3 == 0) n /= 3;
  return n == 1;
}

size_t bluestein_inner_size(size_t n) {
  size_t want = 2 * n - 1, m = 1;
  while (m < want) m <<= 1;
  return m;
}

const char* env_value(const char* name) { return std::getenv(name); }

Tuning Tuning::from_env() {
  auto env_int = [](const char* name) -> std::optional<int> {
    const char* e = env_value(name);
    if (!e) return std::nullopt;
    return atoi(e);
  };
  Tuning t;
  if (auto v = env_int("FOURIER_B200_TWOPASS"); v && *v == 0) t.twopass = false;
  if (auto v = env_int("FOURIER_B200_FUSED"); v && *v == 0) t.fused = false;
  t.ring = env_int("FOURIER_B200_RING");
  t.lag = env_int("FOURIER_B200_LAG");
  const auto chunk_mb = env_int("FOURIER_B200_CHUNK_MB");
  if (chunk_mb) t.chunk_mb = (size_t)std::max(1, *chunk_mb);
  if (auto v = env_int("FOURIER_B200_DIST_CHUNK_MB")) t.dist_chunk_mb = (size_t)std::max(1, *v);
  else if (chunk_mb) t.dist_chunk_mb = t.chunk_mb;
  if (auto v = env_int("FOURIER_B200_DIST_LANES")) t.dist_lanes = std::min(4, std::max(1, *v));
  if (auto v = env_int("FOURIER_B200_DIST_OVERLAP"); v && *v == 0) t.dist_lanes = 1;
  t.big_na = env_int("FOURIER_B200_BIG_NA");
  t.zero_copy = env_value("FOURIER_B200_NO_ZEROCOPY") == nullptr;
  if (const char* e = env_value("FOURIER_B200_TRACE")) t.trace = e;
  return t;
}

DeviceBuffer::~DeviceBuffer() { release(); }
void DeviceBuffer::release() {
  if (ptr_) cudaFree(ptr_);
  ptr_ = nullptr;
  bytes_ = 0;
}
cudaError_t DeviceBuffer::reserve(size_t bytes) {
  if (bytes <= bytes_) return cudaSuccess;
  release();
  cudaError_t e = cudaMalloc(&ptr_, bytes);
  if (e != cudaSuccess) { ptr_ = nullptr; return e; }
  bytes_ = bytes;
  return cudaSuccess;
}

namespace {

constexpr size_t kScratchTargetBytes = (size_t)512 << 20;  // per scratch buffer on the general path
constexpr size_t kHostChunkBytes = (size_t)64 << 20;       // host-pointer pipeline granule
constexpr size_t kHostSmallBytes = (size_t)1 << 20;        // below this a host call takes the single-stream latency path
constexpr size_t kHostZeroCopyBytes = (size_t)64 << 10;    // below this the kernel reads / writes mapped host memory itself

}  // namespace

// ---------------------------------------------------------------------------------------------------
// construction
// ---------------------------------------------------------------------------------------------------
template <typename T>
Plan<T>* Plan<T>::create(size_t n, int device, bool allow_fast_paths) {
  return create(n, device, allow_fast_paths, Tuning::from_env());
}

template <typename T>
Plan<T>* Plan<T>::create(size_t n, int device, bool allow_fast_paths, const Tuning& tuning) {
  if (n == 0) {
    set_last_error("size 0 is not a valid transform length");
    return nullptr;
  }
  Plan<T>* p = new (std::nothrow) Plan<T>();
  if (!p) return nullptr;
  p->tuning_ = tuning;
  cudaError_t e = cudaErrorUnknown;
  try {
    e = p->init(n, device, allow_fast_paths);
  } catch (const std::exception& ex) {   // e.g. bad_alloc while building an N-entry host table
    set_last_error(std::string("plan construction threw: ") + ex.what());
  }
  if (e != cudaSuccess) {
    delete p;
    return nullptr;
  }
  return p;
}

template <typename T>
const char* Plan<T>::kernel_name() const {
  switch (path_) {
    case Path::kTrivial: return "scale_copy_kernel";
    case Path::kOnChip: return "onchip::onchip_fft_kernel";
    case Path::kTwoPass: return fused_ops_ ? "fused::fused_twopass_kernel" : "twopass::tile_kernel (pass 1 + pass 2)";
    case Path::kGlobalStages: return "stockham_stage_kernel (one launch per radix stage)";
    case Path::kBluestein: return "chirp / pointwise kernels around the inner plan's kernels";
    case Path::kBluesteinFused: return cta_chirp_ ? "cta::cta_fft_kernel (chirp mode)" : "onchip::bluestein_fused_kernel";
    case Path::kCta: return "cta::cta_fft_kernel";
    case Path::kThreePass:
      return outer_radix3_ ? "outer::radix3_column_kernel + twopass::tile_kernel (pass 1) + dist::rows_exchange_kernel (transposed store)"
                           : "outer::column_kernel + twopass::tile_kernel (pass 1) + dist::rows_exchange_kernel (transposed store)";
  }
  return "?";
}

template <typename T>
Plan<T>::~Plan() {
  DeviceGuard g(device_);
  for (auto& s : streams_)
    if (s) cudaStreamDestroy(s);
  for (auto& e : events_)
    if (e) cudaEventDestroy(e);
  if (zc_in_) cudaFreeHost(zc_in_);
  if (zc_out_) cudaFreeHost(zc_out_);
}

template <typename T>
cudaError_t Plan<T>::init(size_t n, int device, bool allow_fast_paths) {
  n_ = n;
  device_ = device;
  DeviceGuard g(device_);
  if (!g.ok) { set_last_error("cudaSetDevice failed"); return cudaErrorInvalidDevice; }
  if (cudaDeviceGetAttribute(&sm_count_, cudaDevAttrMultiProcessorCount, device_) != cudaSuccess) sm_count_ = 148;
  if (n == 1) { path_ = Path::kTrivial; return cudaSuccess; }
  if (is_23_smooth(n)) {
    const bool pow2 = (n & (n - 1)) == 0;
    if (allow_fast_paths && pow2) {
      if (init_onchip() == cudaSuccess) { path_ = Path::kOnChip; return cudaSuccess; }
      // tuning_.twopass = false (experiment knob): skip the two-pass kernels, so that sizes the CTA kernel also
      // covers can be measured on it
      if (tuning_.twopass && init_twopass() == cudaSuccess) { path_ = Path::kTwoPass; return cudaSuccess; }
      // beyond the two-pass sizes: an outer column pass around two-pass rows (bigpow2.cu)
      if (tuning_.twopass && init_bigpow2() == cudaSuccess) { path_ = Path::kThreePass; return cudaSuccess; }
    }
    // everything else that fits two shared-memory buffers: one kernel, one HBM round trip
    if (allow_fast_paths && init_cta(n) == cudaSuccess) { path_ = Path::kCta; return cudaSuccess; }
    // 3^b * 2^k (b <= 3) with a two-pass power of two: outer radix-3^b pass + two-pass rows (bigpow2.cu); without
    // tuning_.twopass the per-stage path is measured instead
    if (allow_fast_paths && !pow2 && tuning_.twopass && init_threepass_radix3() == cudaSuccess) {
      path_ = Path::kThreePass;
      return cudaSuccess;
    }
    path_ = Path::kGlobalStages;
    return init_global_stages();
  }
  return init_bluestein(allow_fast_paths);
}

// Factorisation for the general path.  The reference uses [4, 8.., 4.., 3.., 2..]
// (autosort/mod.rs:104-117); any ordering of the same prime content is a valid Stockham plan, and
// on the GPU the widest register butterflies first minimises passes over HBM.
template <typename T>
cudaError_t Plan<T>::init_global_stages() {
  size_t r = n_;
  int twos = 0, threes = 0;
  while (r % 2 == 0) { r /= 2; ++twos; }
  while (r % 3 == 0) { r /= 3; ++threes; }
  radices_.clear();
  while (twos >= 5 || twos == 3) { radices_.push_back(8); twos -= 3; }
  while (twos >= 2) { radices_.push_back(4); twos -= 2; }
  if (twos == 1) radices_.push_back(2);
  for (int i = 0; i < threes; ++i) radices_.push_back(3);

  std::vector<cpx<T>> w(n_);
  for (size_t k = 0; k < n_; ++k) {
    double re, im;
    host_twiddle(k, n_, &re, &im);
    w[k] = mk<T>((T)re, (T)im);
  }
  FB_CHECK(upload(wtab_, w));
  return cudaSuccess;
}

template <typename T>
cudaError_t Plan<T>::init_bluestein(bool allow_fast_paths) {
  m_ = bluestein_inner_size(n_);

  // chirp[i] = exp(-i*pi*i^2/N) = w_{2N}^{i^2 mod 2N}.  The reference forms i^2 in f64 without the
  // reduction (bluesteins.rs:31,33,57), which costs accuracy for large N; reducing first is exact.
  std::vector<cpx<T>> chirp(n_);
  std::vector<double> wr(m_, 0.0), wi(m_, 0.0), cr(n_), ci(n_);
  for (size_t i = 0; i < n_; ++i) {
    const size_t idx = (size_t)(((unsigned __int128)i * i) % (2 * (unsigned __int128)n_));
    double re, im;
    host_twiddle(idx, 2 * n_, &re, &im);
    chirp[i] = mk<T>((T)re, (T)im);
    cr[i] = re; ci[i] = im;
    // wrapped conjugate chirp (bluesteins.rs:18-45): w[i] = w[M-i] = exp(+i*pi*i^2/N)
    wr[i] = re; wi[i] = -im;
    if (i != 0) { wr[m_ - i] = re; wi[m_ - i] = -im; }
  }
  // W = FFT_M(w).  The reference computes this with the inner plan in precision T
  // (bluesteins.rs:46-47); computing it in f64 and rounding once is at least as accurate.
  host_fft_pow2(wr, wi, false);
  std::vector<cpx<T>> wf(m_);
  for (size_t i = 0; i < m_; ++i) wf[i] = mk<T>((T)wr[i], (T)wi[i]);
  if (allow_fast_paths && init_bluestein_fused(cr, ci, wr, wi) == cudaSuccess) {
    inner_.reset();   // the fused kernel carries its own on-chip inner FFTs
    path_ = Path::kBluesteinFused;
    return cudaSuccess;
  }
  if (allow_fast_paths && init_cta(m_) == cudaSuccess) {
    // inner size above the warp-level kernel: the CTA-level kernel in chirp mode, still one launch
    FB_CHECK(upload(chirp_, chirp));
    FB_CHECK(upload(wf_, wf));
    cta_chirp_ = true;
    path_ = Path::kBluesteinFused;
    return cudaSuccess;
  }
  inner_.reset(Plan<T>::create(m_, device_, allow_fast_paths, tuning_));
  if (!inner_) return cudaErrorUnknown;
  FB_CHECK(upload(chirp_, chirp));
  FB_CHECK(upload(wf_, wf));
  path_ = Path::kBluestein;
  return cudaSuccess;
}

template <typename T>
PlanInfo Plan<T>::info() const {
  PlanInfo i;
  i.size = n_;
  i.path = (int)path_;
  i.inner_size = m_;
  i.inner_path = inner_ ? (int)inner_->path() : 0;
  i.n1 = n1_;
  i.n2 = n2_;
  i.precision_bytes = (int)sizeof(T);
  i.device = device_;
  i.table_bytes = wtab_.bytes() + tw_a_.bytes() + tw_b_.bytes() + chirp_.bytes() + wf_.bytes() +
                  (inner_ ? inner_->info().table_bytes : 0);
  return i;
}

// ---------------------------------------------------------------------------------------------------
// execution on device pointers
// ---------------------------------------------------------------------------------------------------
template <typename T>
cudaError_t Plan<T>::exec_device(const C* in, C* out, size_t batch, int code, cudaStream_t stream) {
  launches_ = 0;
  if (code < 0 || code > 4) { set_last_error("unknown transform code"); return cudaErrorInvalidValue; }
  if (batch == 0) return cudaSuccess;
  DeviceGuard g(device_);
  switch (path_) {
    case Path::kTrivial: {
      const T s = scale_for<T>(code, 1);
      if (in == out && s == (T)1) return cudaSuccess;
      ++launches_;
      return launch_scale_copy<T>(in, out, batch, s, stream);
    }
    case Path::kOnChip: return exec_onchip(in, out, batch, code, stream);
    case Path::kTwoPass: return exec_twopass(in, out, batch, code, stream);
    case Path::kGlobalStages: return exec_global_stages(in, out, batch, code, stream);
    case Path::kBluestein: return exec_bluestein(in, out, batch, code, stream);
    case Path::kBluesteinFused:
      return cta_chirp_ ? exec_cta(in, out, batch, code, stream, true) : exec_bluestein_fused(in, out, batch, code, stream);
    case Path::kCta: return exec_cta(in, out, batch, code, stream, false);
    case Path::kThreePass: return exec_bigpow2(in, out, batch, code, stream);
  }
  return cudaErrorUnknown;
}

// Stage driver of the general path (reference: apply_stages_*, autosort/mod.rs:318-400): ping-pong
// between scratch buffers, the last stage lands in `out` with the scale folded in.
template <typename T>
cudaError_t Plan<T>::exec_global_stages(const C* in, C* out, size_t batch, int code, cudaStream_t s) {
  const bool fwd = transform_is_forward(code);
  const T scale = scale_for<T>(code, n_);
  const size_t stages = radices_.size();
  const size_t bytes_per = n_ * sizeof(C);
  size_t chunk = std::max<size_t>(1, kScratchTargetBytes / bytes_per);
  chunk = std::min(chunk, batch);
  if (stages >= 2) FB_CHECK(work_.reserve(chunk * bytes_per));
  if (stages >= 3) FB_CHECK(work2_.reserve(chunk * bytes_per));
  for (size_t b0 = 0; b0 < batch; b0 += chunk) {
    const size_t nb = std::min(chunk, batch - b0);
    const C* src = in + b0 * n_;
    C* final_dst = out + b0 * n_;
    size_t sub = n_, stride = 1;
    for (size_t k = 0; k < stages; ++k) {
      const bool last = k + 1 == stages;
      C* dst = last ? final_dst : ((k % 2 == 0) ? (C*)work_.data() : (C*)work2_.data());
      FB_CHECK(launch_stockham_stage<T>(radices_[k], src, dst, (const C*)wtab_.data(), n_, sub, stride, nb,
                                        fwd, last, scale, s));
      ++launches_;
      sub /= radices_[k];
      stride *= radices_[k];
      src = dst;
    }
  }
  return cudaSuccess;
}

// bluesteins::apply (bluesteins.rs:218-259) with the 1/M of the inner IFFT folded into the last step.
template <typename T>
cudaError_t Plan<T>::exec_bluestein(const C* in, C* out, size_t batch, int code, cudaStream_t s) {
  const bool fwd = transform_is_forward(code);
  const T scale = scale_for<T>(code, n_) / (T)m_;
  const size_t bytes_per = m_ * sizeof(C);
  size_t chunk = std::max<size_t>(1, kScratchTargetBytes / bytes_per);
  chunk = std::min(chunk, batch);
  FB_CHECK(work_.reserve(chunk * bytes_per));
  C* work = (C*)work_.data();
  for (size_t b0 = 0; b0 < batch; b0 += chunk) {
    const size_t nb = std::min(chunk, batch - b0);
    FB_CHECK(launch_chirp_in<T>(in + b0 * n_, work, (const C*)chirp_.data(), n_, m_, nb, fwd, s));
    FB_CHECK(inner_->exec_device(work, work, nb, kFft, s));
    launches_ += inner_->launches();
    FB_CHECK(launch_pointwise<T>(work, (const C*)wf_.data(), m_, nb, fwd, s));
    FB_CHECK(inner_->exec_device(work, work, nb, kUnscaledIfft, s));
    launches_ += inner_->launches();
    FB_CHECK(launch_chirp_out<T>(work, out + b0 * n_, (const C*)chirp_.data(), n_, m_, nb, fwd, scale, s));
    launches_ += 3;
  }
  return cudaSuccess;
}

// ---------------------------------------------------------------------------------------------------
// execution on host pointers: H2D -> transform in place -> D2H, three slots in flight
// ---------------------------------------------------------------------------------------------------
template <typename T>
cudaError_t Plan<T>::host_resources() {
  for (int i = 0; i < 3; ++i)
    if (!streams_[i]) FB_CHECK(cudaStreamCreateWithFlags(&streams_[i], cudaStreamNonBlocking));
  for (int i = 0; i < 9; ++i)
    if (!events_[i]) FB_CHECK(cudaEventCreateWithFlags(&events_[i], cudaEventDisableTiming));
  return cudaSuccess;
}

template <typename T>
cudaError_t Plan<T>::exec_host(const C* in, C* out, size_t batch, int code) {
  if (code < 0 || code > 4) { set_last_error("unknown transform code"); return cudaErrorInvalidValue; }
  if (batch == 0) return cudaSuccess;
  DeviceGuard g(device_);
  constexpr int kSlots = 3;
  FB_CHECK(host_resources());
  const size_t bytes_per = n_ * sizeof(C);
  if (batch * bytes_per <= kHostSmallBytes) {
    // Latency path (the reference ABI's single small transform, fourier-ffi/src/lib.rs:46-59): nothing to
    // pipeline, so one stream, no events, one synchronisation: H2D, kernel(s), D2H back to back.
    cudaStream_t s = streams_[1];
    if (batch * bytes_per <= kHostZeroCopyBytes && tuning_.zero_copy) {
      // Smallest calls: the two DMA copies cost more than the transform.  The kernels read the input from and write
      // the result to a pinned, device-mapped bounce buffer over PCIe themselves (one launch, one synchronisation;
      // the CPU copies 2 x <= 64 KB).  Measured: 24 -> ~12 us per 1024-point call (profiles/r02_latency.txt).
      if (!zc_in_) {
        FB_CHECK(cudaHostAlloc(&zc_in_, kHostZeroCopyBytes, cudaHostAllocMapped));
        FB_CHECK(cudaHostAlloc(&zc_out_, kHostZeroCopyBytes, cudaHostAllocMapped));
      }
      std::memcpy(zc_in_, in, batch * bytes_per);
      void *din = nullptr, *dout = nullptr;
      FB_CHECK(cudaHostGetDevicePointer(&din, zc_in_, 0));
      FB_CHECK(cudaHostGetDevicePointer(&dout, zc_out_, 0));
      FB_CHECK(exec_device((const C*)din, (C*)dout, batch, code, s));
      FB_CHECK(cudaStreamSynchronize(s));
      std::memcpy(out, zc_out_, batch * bytes_per);
      return cudaSuccess;
    }
    FB_CHECK(stage_[0].reserve(std::max(batch * bytes_per, kHostSmallBytes)));
    C* dev = (C*)stage_[0].data();
    FB_CHECK(cudaMemcpyAsync(dev, in, batch * bytes_per, cudaMemcpyHostToDevice, s));
    FB_CHECK(exec_device(dev, dev, batch, code, s));
    FB_CHECK(cudaMemcpyAsync(out, dev, batch * bytes_per, cudaMemcpyDeviceToHost, s));
    FB_CHECK(cudaStreamSynchronize(s));
    return cudaSuccess;
  }
  cudaStream_t s_in = streams_[0], s_ex = streams_[1], s_out = streams_[2];
  cudaEvent_t* ev_in = &events_[0];    // [slot] H2D finished
  cudaEvent_t* ev_ex = &events_[3];    // [slot] transform finished
  cudaEvent_t* ev_free = &events_[6];  // [slot] D2H finished, slot reusable

  size_t chunk = std::max<size_t>(1, kHostChunkBytes / bytes_per);
  chunk = std::min(chunk, batch);
  const size_t nchunks = (batch + chunk - 1) / chunk;
  const int used = (int)std::min<size_t>(kSlots, nchunks);
  for (int i = 0; i < used; ++i) FB_CHECK(stage_[i].reserve(chunk * bytes_per));

  unsigned long long total_launches = 0;
  for (size_t c = 0; c < nchunks; ++c) {
    const int slot = (int)(c % kSlots);
    const size_t b0 = c * chunk, nb = std::min(chunk, batch - b0);
    C* dev = (C*)stage_[slot].data();
    // the slot's previous D2H must be done before it is overwritten
    if (c >= (size_t)kSlots) FB_CHECK(cudaStreamWaitEvent(s_in, ev_free[slot], 0));
    FB_CHECK(cudaMemcpyAsync(dev, in + b0 * n_, nb * bytes_per, cudaMemcpyHostToDevice, s_in));
    FB_CHECK(cudaEventRecord(ev_in[slot], s_in));
    FB_CHECK(cudaStreamWaitEvent(s_ex, ev_in[slot], 0));
    FB_CHECK(exec_device(dev, dev, nb, code, s_ex));
    total_launches += launches_;
    FB_CHECK(cudaEventRecord(ev_ex[slot], s_ex));
    FB_CHECK(cudaStreamWaitEvent(s_out, ev_ex[slot], 0));
    FB_CHECK(cudaMemcpyAsync(out + b0 * n_, dev, nb * bytes_per, cudaMemcpyDeviceToHost, s_out));
    FB_CHECK(cudaEventRecord(ev_free[slot], s_out));
  }
  FB_CHECK(cudaStreamSynchronize(s_out));
  FB_CHECK(cudaStreamSynchronize(s_ex));
  FB_CHECK(cudaStreamSynchronize(s_in));
  launches_ = total_launches;
  return cudaSuccess;
}

template class Plan<float>;
template class Plan<double>;

}  // namespace fb200
