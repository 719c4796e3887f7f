// plan.h -- host-side plan objects behind the C ABI (include/fourier.h, include/fourier_b200.h).
//
// A Plan<T> is what the reference boxes up as `Box<dyn Fft<Real = T> + Send>`
// (fourier/src/lib.rs:31-60): it owns the twiddle tables and scratch for one transform size and
// exposes the single required operation, transform_in_place / transform with a Transform code
// (fourier-algorithms/src/fft.rs:40-82).  Here the tables and scratch live in HBM, the operation
// is batched, and it is enqueued on a CUDA stream.
#pragma once

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstddef>
#include <memory>
#include <optional>
#include <string>
#include <vector>

#include "cplx.cuh"

namespace fb200 {

// thread-local error text for the C ABI
void set_last_error(const std::string& s);
const char* last_error();

#define FB_CHECK(expr)                                                                       \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      set_last_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                    \
      return _e;                                                                             \
    }                                                                                        \
  } while (0)

// Execution strategy chosen at plan time.
enum class Path : int {
  kTrivial = 0,         // N == 1
  kOnChip = 1,          // one shared-memory Stockham FFT per CTA-slice (pow2 N <= on-chip limit)
  kTwoPass = 2,         // four-step, two fused kernels, L2-resident intermediate (large pow2 N)
  kGlobalStages = 3,    // one kernel per Stockham stage over HBM ({2,3}-smooth N, any size)
  kBluestein = 4,       // chirp-z around a pow2 inner plan, separate kernels
  kBluesteinFused = 5,  // chirp-z with the inner FFTs on chip, one kernel
  kCta = 6,             // whole transforms in shared memory, one CTA per group of transforms, all Stockham stages
                        // in one kernel ({2,3}-smooth N, pow2 N between the on-chip and two-pass kernels)
  kThreePass = 7,       // pow2 N above the two-pass kernels: outer column pass + two-pass rows storing transposed
};

const char* path_name(Path p);

constexpr int kMaxPeers = 16;   // ranks of one box (peer-memory exchange, exchange.cu / dist_fft.cu)

// Selection rule of create_fft_f32/f64 (fourier/src/lib.rs:38-42 with autosort/mod.rs:104-117):
// Autosort iff N = 2^a * 3^b (N >= 1), else Bluestein with inner size next_pow2(2N-1).
bool is_23_smooth(size_t n);
size_t bluestein_inner_size(size_t n);  // bluesteins.rs:110

// Makes `dev` the current device for the lifetime of the guard.
struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a per-device setting: done once per kernel AND device (a process
// may hold plans on several GPUs).  `done` is the kernel's own bit mask of prepared devices.  carveout >= 0 also sets
// the preferred shared-memory carve-out (a cudaSharedmemCarveout value or a percentage).
template <class Kernel>
inline cudaError_t ensure_dynamic_smem(Kernel kernel, size_t bytes, std::atomic<unsigned long long>& done,
                                       int carveout = -1) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const unsigned long long bit = 1ull << (dev & 63);
  if (done.load(std::memory_order_acquire) & bit) return cudaSuccess;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess && carveout >= 0)
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carveout);
  if (e == cudaSuccess) done.fetch_or(bit, std::memory_order_release);
  return e;
}

// Scale factor of a Transform code for length n (autosort/mod.rs:381-385, bluesteins.rs:240-258).
template <typename T> T scale_for(int code, size_t n) {
  switch (code) {
    case kIfft: return (T)1 / (T)n;
    case kSqrtScaledFft:
    case kSqrtScaledIfft: return (T)1 / std::sqrt((T)n);
    default: return (T)1;
  }
}

// The library's one environment lookup: the value of variable `name`, nullptr when it is unset.
const char* env_value(const char* name);

// Experiment knobs (FOURIER_B200_* environment variables).  A plan reads them once, when it is created, and hands the
// same values to its inner plans, so that a plan and its exec calls never see two configurations.
struct Tuning {
  bool twopass = true;          // TWOPASS=0: skip the two-pass, three-pass and radix-3 three-pass paths
  bool fused = true;            // FUSED=0: the two tile kernels instead of the persistent kernel
  std::optional<int> ring, lag; // RING, LAG: staging ring of the persistent kernel; unset = the configuration's own
  size_t chunk_mb = 32;         // CHUNK_MB: L2-resident chunk of the two-pass tile kernels
  size_t dist_chunk_mb = 64;    // DIST_CHUNK_MB, else CHUNK_MB: chunk of the fused row FFT + exchange
  int dist_lanes = 2;           // DIST_LANES (1 .. 4), DIST_OVERLAP=0 forces 1: streams the chunks rotate over
  std::optional<int> big_na;    // BIG_NA: log2 of the outer pass length of the three-pass path
  bool zero_copy = true;        // NO_ZEROCOPY (set): the smallest host calls take the copy path
  std::string trace;            // TRACE=<file>: phase timeline of the persistent kernel, written after every call

  static Tuning from_env();
};

// Grow-only device allocation.
class DeviceBuffer {
 public:
  DeviceBuffer() = default;
  ~DeviceBuffer();
  DeviceBuffer(const DeviceBuffer&) = delete;
  DeviceBuffer& operator=(const DeviceBuffer&) = delete;
  cudaError_t reserve(size_t bytes);
  void* data() const { return ptr_; }
  size_t bytes() const { return bytes_; }
  void release();

 private:
  void* ptr_ = nullptr;
  size_t bytes_ = 0;
};

// Copies a host table into `buf`, grown as needed (an empty table still reserves one element).
template <typename U>
cudaError_t upload(DeviceBuffer& buf, const std::vector<U>& host) {
  cudaError_t e = buf.reserve(std::max<size_t>(host.size(), 1) * sizeof(U));
  if (e != cudaSuccess) return e;
  if (host.empty()) return cudaSuccess;
  return cudaMemcpy(buf.data(), host.data(), host.size() * sizeof(U), cudaMemcpyHostToDevice);
}

struct PlanInfo {
  size_t size = 0;
  int path = 0;
  size_t inner_size = 0;     // Bluestein inner FFT length, else 0
  int inner_path = 0;
  size_t n1 = 0, n2 = 0;     // two-pass split
  int precision_bytes = 0;   // 4 or 8
  int device = 0;
  size_t table_bytes = 0;    // twiddle / chirp tables resident in HBM
};

template <typename T>
class Plan {
 public:
  using C = cpx<T>;

  // Returns nullptr (and sets last_error) when the plan cannot be built; size 0 is refused
  // (the reference never returns for 0: autosort/mod.rs:112).  The Tuning knobs are read from the environment here.
  static Plan* create(size_t n, int device, bool allow_fast_paths = true);
  ~Plan();

  size_t size() const { return n_; }
  int device() const { return device_; }
  Path path() const { return path_; }
  PlanInfo info() const;

  // Batched transform on device-resident data: `batch` contiguous transforms of size() samples,
  // in == out allowed (in place).  Enqueued on `stream`; not synchronised.
  cudaError_t exec_device(const C* in, C* out, size_t batch, int code, cudaStream_t stream);

  // Same on host memory (the reference ABI's case): staged H2D -> transform -> D2H through the
  // plan's own streams, chunked and pipelined; returns after the result is in `out`.
  cudaError_t exec_host(const C* in, C* out, size_t batch, int code);

  // Distributed six-step transform (dist_fft.cu): batched FFT of `rows` contiguous rows of size() samples whose last
  // register stage stores the result transposed, and optionally twiddled, straight into the destination ranks'
  // buffers: outs[q][c * out_ld + out_off + r] = X_r[q * cb + c] * w_Ntot^{(row0 + r) * (q * cb + c)}, cb = size() / nranks
  // (what launch_exchange() delivers after exec_device() on the same rows).  Two-pass sizes only; `in` is left intact.
  // rows_per_batch != 0 (three-pass path): the rows come in batches of that many, batch b goes out_batch_stride
  // elements further on: outs[q][b * out_batch_stride + c * out_ld + out_off + r % rows_per_batch]; rows_valid != 0:
  // only the first rows_valid rows exist, the rest pads the last tile (read, transformed, not stored).
  cudaError_t exec_rows_exchange(const C* in, size_t rows, bool forward, void* const* outs, int nranks, size_t out_ld,
                                 size_t out_off, int twiddle, unsigned long long row0, unsigned long long n_total,
                                 cudaStream_t stream, size_t rows_per_batch = 0, size_t out_batch_stride = 0,
                                 size_t rows_valid = 0);

  // Number of kernel launches the last exec_* call issued (bench.py reports it).
  unsigned long long launches() const { return launches_; }

  // Name of the kernel that moves (nearly) all of this plan's bytes -- what a profiler will list first.
  const char* kernel_name() const;

 private:
  Plan() = default;
  // inner plans (three-pass rows, Bluestein inner transform) take their parent's knobs
  static Plan* create(size_t n, int device, bool allow_fast_paths, const Tuning& tuning);
  cudaError_t init(size_t n, int device, bool allow_fast_paths);

  cudaError_t exec_global_stages(const C* in, C* out, size_t batch, int code, cudaStream_t s);
  cudaError_t exec_onchip(const C* in, C* out, size_t batch, int code, cudaStream_t s);
  cudaError_t exec_twopass(const C* in, C* out, size_t batch, int code, cudaStream_t s);
  cudaError_t exec_bluestein(const C* in, C* out, size_t batch, int code, cudaStream_t s);
  cudaError_t exec_bluestein_fused(const C* in, C* out, size_t batch, int code, cudaStream_t s);
  cudaError_t exec_cta(const C* in, C* out, size_t batch, int code, cudaStream_t s, bool chirp);
  cudaError_t exec_bigpow2(const C* in, C* out, size_t batch, int code, cudaStream_t s);

  cudaError_t init_global_stages();
  cudaError_t init_onchip();
  cudaError_t init_twopass();
  cudaError_t init_bigpow2();
  cudaError_t init_threepass_radix3();
  cudaError_t init_cta(size_t len);   // len = n_, or the Bluestein inner size
  cudaError_t init_bluestein(bool allow_fast_paths);
  cudaError_t init_bluestein_fused(const std::vector<double>& chirp_re, const std::vector<double>& chirp_im,
                                   const std::vector<double>& w_re, const std::vector<double>& w_im);

  size_t n_ = 0;
  int device_ = 0;
  Path path_ = Path::kTrivial;
  unsigned long long launches_ = 0;
  Tuning tuning_;

  // kGlobalStages: radices of the Stockham stages and the full forward table w_N^k, k < N
  std::vector<int> radices_;
  DeviceBuffer wtab_;

  // kOnChip / kTwoPass: see onchip.cu / twopass.cu
  size_t n1_ = 0, n2_ = 0;
  DeviceBuffer tw_a_, tw_b_, tw2_, tw_f_, tw_f2_;   // tw_f_, tw_f2_: stage twiddles of the persistent kernel's two register tiles
  const void* fast_ops_ = nullptr;   // TwoPassOps<T> / OnChipOps<T> of the selected kernel family
  size_t chunk_ = 0;                 // transforms per L2-resident chunk (two-pass)
  const void* fused_ops_ = nullptr;  // FusedOps<T>: persistent single-launch variant
  int ring_ = 0, lag_ = 0, sm_count_ = 148;
  int outer_radix3_ = 0;             // kThreePass: 3 / 9 / 27 = the outer pass is a radix-3 DFT (N = 3^b * 2^k), 0 = power of two
  DeviceBuffer counters_, tbase_, tstep_, trace_;

  // kCta (and kBluesteinFused through the CTA kernel): on-chip transform length, radices_ and wtab_ as above
  size_t cta_len_ = 0;
  bool cta_chirp_ = false;

  // kBluestein*: chirp x[i] (N entries), W = FFT_M(wrapped chirp) (M entries), both forward;
  // the inverse direction uses their conjugate-symmetric counterparts computed at plan time.
  size_t m_ = 0;
  std::unique_ptr<Plan<T>> inner_;
  DeviceBuffer chirp_, wf_, wi_;

  // scratch (grow-only) and host staging
  DeviceBuffer work_, work2_;
  DeviceBuffer stage_[3];
  cudaStream_t streams_[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t events_[9] = {};
  cudaError_t host_resources();   // streams and events of the host-pointer path, created once
  void* zc_in_ = nullptr;         // pinned, device-mapped bounce buffers of the smallest host calls (64 KB each)
  void* zc_out_ = nullptr;
};

// ---- kernel launchers implemented in the .cu files ------------------------------------------------

// stockham_generic.cu
template <typename T>
cudaError_t launch_stockham_stage(int radix, const cpx<T>* in, cpx<T>* out, const cpx<T>* wtab, size_t n,
                                  size_t sub_size, size_t stride, size_t batch, bool forward, bool last,
                                  T scale, cudaStream_t s);
template <typename T>
cudaError_t launch_scale_copy(const cpx<T>* in, cpx<T>* out, size_t count, T scale, cudaStream_t s);
template <typename T>
cudaError_t launch_chirp_in(const cpx<T>* in, cpx<T>* work, const cpx<T>* chirp, size_t n, size_t m,
                            size_t batch, bool forward, cudaStream_t s);
template <typename T>
cudaError_t launch_pointwise(cpx<T>* work, const cpx<T>* w, size_t m, size_t batch, bool forward,
                             cudaStream_t s);
template <typename T>
cudaError_t launch_chirp_out(const cpx<T>* work, cpx<T>* out, const cpx<T>* chirp, size_t n, size_t m,
                             size_t batch, bool forward, T scale, cudaStream_t s);

// synth.cu: counter-hash synthetic input (same generator as oracle/fourier_oracle.c fo_fill_input_*)
template <typename T>
cudaError_t launch_fill_input(T* out, unsigned long long first_scalar, size_t count,
                              unsigned long long seed, cudaStream_t s);

// synth.cu: helpers of the distributed six-step transform
template <typename T>
cudaError_t launch_transpose(const cpx<T>* in, cpx<T>* out, size_t batch, size_t rows, size_t cols, cudaStream_t s);
template <typename T>
cudaError_t launch_pack(const cpx<T>* in, cpx<T>* out, size_t batch, size_t rows, size_t cols, size_t ld, size_t ibs,
                        size_t obs, int twiddle, unsigned long long row0, unsigned long long col0,
                        unsigned long long n_total, cudaStream_t s);
template <typename T>
cudaError_t launch_swap_leading(const cpx<T>* in, cpx<T>* out, size_t a, size_t b, size_t inner, cudaStream_t s);
template <typename T>
cudaError_t launch_twiddle_rows(cpx<T>* data, size_t rows, size_t cols, unsigned long long row0,
                                unsigned long long n_total, bool forward, cudaStream_t s);

// exchange.cu: exchange step of the distributed transform over NVLink peer memory + CUDA-IPC plumbing
template <typename T>
cudaError_t launch_exchange(const cpx<T>* in, void* const* outs, int nranks, int me, size_t rows, size_t cb, size_t ld,
                            size_t out_ld, size_t out_off, int twiddle, unsigned long long row0,
                            unsigned long long n_total, cudaStream_t s);
cudaError_t peer_alloc(size_t bytes, void** ptr, void* handle64);
cudaError_t peer_open(const void* handle64, void** ptr);
cudaError_t peer_close(void* ptr);
cudaError_t peer_free(void* ptr);

// host math helpers (plan_math.cpp part of plan.cu)
void host_twiddle(size_t k, size_t n, double* re, double* im);            // exp(-2*pi*i*k/n), long-double accurate
void host_fft_pow2(std::vector<double>& re, std::vector<double>& im, bool inverse);  // unscaled, in place

}  // namespace fb200
