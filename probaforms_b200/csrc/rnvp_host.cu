// Host side of ingestion / egress (no device code in this file): what the reference does with
// torch.tensor(X, dtype=torch.float32) (realnvp.py:226-228) and .cpu().detach().numpy() (realnvp.py:281) once the
// kernels are fast enough for those copies to be the wall-clock bound (SURVEY 8f-2).
//
// rnvp_host_gather_xc: dst_x[r][:] = (float) src_x[idx ? idx[r] : row0 + r][:], and the same rows of src_c into dst_c
// unless src_c is NULL -- the rows of one optimisation step (a slice of the epoch permutation) or of one upload chunk,
// converted from the caller's float64 / float32 numpy arrays straight into pinned staging buffers, split over a few
// host threads.  RealNVP.fit streams these buffers to the GPU one step ahead of the kernels, so every rank uploads
// only the rows of its own shard.
// rnvp_host_copy: multi-threaded memcpy (first-touch of a fresh numpy result array is page-fault bound on one thread).
#include <stdint.h>
#include <string.h>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <algorithm>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>
#include "../../include/rnvp.h"

namespace {

#if defined(__SSE2__)
// The staging buffers are read next by the GPU's DMA engine, not by this core: non-temporal stores keep 12 MB per step out
// of the cores' caches (an upload whose source lines are dirty in 15 L2 caches was measured at 13 GB/s instead of 52).
inline void store4(float* d, const float* s) { _mm_stream_ps(d, _mm_loadu_ps(s)); }
inline void store4(float* d, const double* s) {
  _mm_stream_ps(d, _mm_movelh_ps(_mm_cvtpd_ps(_mm_loadu_pd(s)), _mm_cvtpd_ps(_mm_loadu_pd(s + 2))));
}
#endif

template <typename T>
void gather_range(const T* src, int64_t width, const int64_t* idx, int64_t row0, int64_t r0, int64_t r1, float* dst) {
  constexpr int AHEAD = 16;                      // random rows: prefetch every cache line of the row 16 rows ahead
  const int64_t row_bytes = width * (int64_t)sizeof(T);
#if defined(__SSE2__)
  const bool stream_ok = width % 4 == 0 && ((uintptr_t)dst & 15) == 0;
#endif
  for (int64_t r = r0; r < r1; ++r) {
    if (idx && r + AHEAD < r1) {
      const char* nx = (const char*)(src + idx[r + AHEAD] * width);
      for (int64_t b = 0; b < row_bytes; b += 64) __builtin_prefetch(nx + b);
    }
    const T* s = src + (idx ? idx[r] : row0 + r) * width;
    float* d = dst + r * width;
#if defined(__SSE2__)
    if (stream_ok) {                               // 16-byte chunks with non-temporal stores (see store4)
      for (int64_t j = 0; j < width; j += 4) store4(d + j, s + j);
      continue;
    }
#endif
    for (int64_t j = 0; j < width; ++j) d[j] = (float)s[j];
  }
#if defined(__SSE2__)
  if (stream_ok) _mm_sfence();
#endif
}

// Persistent worker pool (created on first use, one per process): spawning 8-16 std::threads per call costs ~0.3 ms, as
// much as the gather of a 75,776-row batch itself.  run_threads splits [0, n) into contiguous ranges; the caller works too.
class Pool {
 public:
  static Pool& get() { static Pool p; return p; }
  template <typename F>
  void run(int64_t n, int64_t min_per_thread, int threads, F f) {
    int t = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(threads, kMax + 1), n / std::max<int64_t>(min_per_thread, 1)));
    if (t <= 1) { f(0, n); return; }
    std::unique_lock<std::mutex> call(call_mu_);                 // one parallel region at a time
    ensure(t - 1);
    const int64_t per = (n + t - 1) / t;
    {
      std::lock_guard<std::mutex> lk(mu_);
      job_ = [&](int w) { f(std::min(n, (int64_t)(w + 1) * per), std::min(n, (int64_t)(w + 2) * per)); };
      active_ = t - 1; pending_ = t - 1; ++epoch_;
    }
    cv_.notify_all();
    f(0, std::min(n, per));
    std::unique_lock<std::mutex> lk(mu_);
    done_.wait(lk, [&] { return pending_ == 0; });
    job_ = nullptr;
  }

 private:
  static constexpr int kMax = 31;
  Pool() = default;
  ~Pool() {
    { std::lock_guard<std::mutex> lk(mu_); stop_ = true; ++epoch_; }
    cv_.notify_all();
    for (auto& th : workers_) th.join();
  }
  void ensure(int n) {
    while ((int)workers_.size() < n) {
      const int w = (int)workers_.size();
      workers_.emplace_back([this, w] {
        uint64_t seen = 0;
        for (;;) {
          std::function<void(int)> job;
          {
            std::unique_lock<std::mutex> lk(mu_);
            cv_.wait(lk, [&] { return stop_ || epoch_ != seen; });
            if (stop_) return;
            seen = epoch_;
            if (w >= active_) continue;
            job = job_;
          }
          job(w);
          {
            std::lock_guard<std::mutex> lk(mu_);
            if (--pending_ == 0) done_.notify_all();
          }
        }
      });
    }
  }
  std::mutex mu_, call_mu_;
  std::condition_variable cv_, done_;
  std::vector<std::thread> workers_;
  std::function<void(int)> job_;
  int active_ = 0, pending_ = 0;
  uint64_t epoch_ = 0;
  bool stop_ = false;
};

template <typename F>
void run_threads(int64_t n, int64_t min_per_thread, int threads, F f) { Pool::get().run(n, min_per_thread, threads, f); }

}  // namespace

extern "C" {

int rnvp_host_gather_xc(const void* src_x, int x_is_f64, int64_t width_x, const void* src_c, int c_is_f64, int64_t width_c,
                           const int64_t* idx, int64_t row0, int64_t n, float* dst_x, float* dst_c, int threads) {
  if (!src_x || !dst_x || width_x < 1 || n < 0 || row0 < 0 || (src_c && (!dst_c || width_c < 1))) return RNVP_EINVAL;
  auto work = [=](int64_t r0, int64_t r1) {
    if (x_is_f64) gather_range((const double*)src_x, width_x, idx, row0, r0, r1, dst_x);
    else gather_range((const float*)src_x, width_x, idx, row0, r0, r1, dst_x);
    if (src_c) {
      if (c_is_f64) gather_range((const double*)src_c, width_c, idx, row0, r0, r1, dst_c);
      else gather_range((const float*)src_c, width_c, idx, row0, r0, r1, dst_c);
    }
  };
  run_threads(n, std::max<int64_t>(1, 32768 / (width_x + width_c)), threads, work);
  return 0;
}

int rnvp_host_copy(void* dst, const void* src, int64_t bytes, int threads) {
  if (!src || !dst || bytes < 0) return RNVP_EINVAL;
  auto work = [=](int64_t b0, int64_t b1) { memcpy((char*)dst + b0, (const char*)src + b0, (size_t)(b1 - b0)); };
  run_threads(bytes, 1 << 20, threads, work);
  return 0;
}

}  // extern "C"
