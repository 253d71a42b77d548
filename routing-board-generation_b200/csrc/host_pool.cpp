// host_pool.cpp -- host threads of the _host variants' transport layer (plain C++, no CUDA).
//
// rbg_connector_step_host_io moves the observation over the bus as bytes (the codes are <= 3 * RBG_MAX_N) and
// these workers widen them to the int32 the API returns, straight into the caller's buffer, slice by slice while
// the next slices are still in flight.  This is a format conversion of the transport, not part of the env step:
// every value is computed on the GPU.  Non-temporal stores: the widened observation is written once and read by
// somebody else, and a regular store would first read every destination line.
#include <pthread.h>
#include <sched.h>
#include <stdint.h>
#include <stdlib.h>
#include <unistd.h>

#include <atomic>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>
#include <vector>

#if defined(__x86_64__)
#include <immintrin.h>
#endif

namespace rbg {

namespace {

struct Piece {
  const uint8_t *src;
  int32_t *dst;
  size_t n;
  int bits;  // 8: a code per byte; 4: two codes per byte, low nibble first
};

void widen4_scalar(const uint8_t *src, int32_t *dst, size_t n) {
  for (size_t i = 0; i < n; ++i) dst[i] = (src[i >> 1] >> (4 * (i & 1))) & 15;
}

void widen_scalar(const uint8_t *src, int32_t *dst, size_t n) {
  for (size_t i = 0; i < n; ++i) dst[i] = src[i];
}

#if defined(__x86_64__)
__attribute__((target("avx2"))) void widen_avx2(const uint8_t *src, int32_t *dst, size_t n) {
  size_t i = 0;
  while (i < n && (reinterpret_cast<uintptr_t>(dst + i) & 31u)) {  // stream stores want 32-byte aligned lines
    dst[i] = src[i];
    ++i;
  }
  for (; i + 32 <= n; i += 32) {
    const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i));
    const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i + 16));
    _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i), _mm256_cvtepu8_epi32(a));
    _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i + 8), _mm256_cvtepu8_epi32(_mm_srli_si128(a, 8)));
    _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i + 16), _mm256_cvtepu8_epi32(b));
    _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i + 24), _mm256_cvtepu8_epi32(_mm_srli_si128(b, 8)));
  }
  for (; i < n; ++i) dst[i] = src[i];
  _mm_sfence();
}
#endif

#if defined(__x86_64__)
// 16 source bytes -> 32 int32 per iteration; NT: the destination is 32-byte aligned after an EVEN number of scalar outputs
// (the caller checks), so that the vector loop starts on a whole source byte
template <bool NT>
__attribute__((target("avx2"))) void widen4_avx2(const uint8_t *src, int32_t *dst, size_t n) {
  size_t i = 0;
  if (NT)
    while (i < n && (reinterpret_cast<uintptr_t>(dst + i) & 31u)) {
      dst[i] = (src[i >> 1] >> (4 * (i & 1))) & 15;
      ++i;
    }
  const __m128i m = _mm_set1_epi8(15);
  for (; i + 32 <= n; i += 32) {
    const __m128i x = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + (i >> 1)));
    const __m128i lo = _mm_and_si128(x, m), hi = _mm_and_si128(_mm_srli_epi16(x, 4), m);
    const __m128i a = _mm_unpacklo_epi8(lo, hi), b = _mm_unpackhi_epi8(lo, hi);
    const __m256i o0 = _mm256_cvtepu8_epi32(a), o1 = _mm256_cvtepu8_epi32(_mm_srli_si128(a, 8));
    const __m256i o2 = _mm256_cvtepu8_epi32(b), o3 = _mm256_cvtepu8_epi32(_mm_srli_si128(b, 8));
    if (NT) {
      _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i), o0);
      _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i + 8), o1);
      _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i + 16), o2);
      _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i + 24), o3);
    } else {
      _mm256_storeu_si256(reinterpret_cast<__m256i *>(dst + i), o0);
      _mm256_storeu_si256(reinterpret_cast<__m256i *>(dst + i + 8), o1);
      _mm256_storeu_si256(reinterpret_cast<__m256i *>(dst + i + 16), o2);
      _mm256_storeu_si256(reinterpret_cast<__m256i *>(dst + i + 24), o3);
    }
  }
  for (; i < n; ++i) dst[i] = (src[i >> 1] >> (4 * (i & 1))) & 15;
  if (NT) _mm_sfence();
}
#endif

void widen4(const uint8_t *src, int32_t *dst, size_t n) {
#if defined(__x86_64__)
  static const bool avx2 = __builtin_cpu_supports("avx2");
  if (avx2) {
    // outputs to the next 32-byte boundary of dst: odd (a destination at an odd int32 offset) would leave the vector loop
    // in the middle of a source byte: plain unaligned stores then
    const size_t head = ((32u - (reinterpret_cast<uintptr_t>(dst) & 31u)) & 31u) >> 2;
    return (head & 1u) == 0 ? widen4_avx2<true>(src, dst, n) : widen4_avx2<false>(src, dst, n);
  }
#endif
  widen4_scalar(src, dst, n);
}

void widen(const uint8_t *src, int32_t *dst, size_t n) {
#if defined(__x86_64__)
  static const bool avx2 = __builtin_cpu_supports("avx2");
  if (avx2) return widen_avx2(src, dst, n);
#endif
  widen_scalar(src, dst, n);
}

inline void cpu_relax() {
#if defined(__x86_64__)
  _mm_pause();
#endif
}

int usable_cores() {
  cpu_set_t set;
  CPU_ZERO(&set);
  int n = 0;
  if (sched_getaffinity(0, sizeof(set), &set) == 0) n = CPU_COUNT(&set);
  if (n < 1) n = (int)std::thread::hardware_concurrency();
  return n < 1 ? 1 : n;
}

class Pool {
 public:
  Pool() {
    int n = usable_cores();
    // one process per GPU on one host (torchrun exports LOCAL_WORLD_SIZE): the ranks share the cores
    if (const char *e = getenv("LOCAL_WORLD_SIZE")) {
      const int w = atoi(e);
      if (w > 1) n = n / w;
    }
    // The conversion is bound by host memory bandwidth long before all cores stream stores (measured on a 16-vCPU
    // box: 8 threads 1.2-1.6 ms per 65 536-env step, 16 threads 2.3 ms; the caller's thread polls the copy events,
    // and the other hardware thread of a core adds nothing to a stream of stores): half of them to start with, the
    // caller (rbg_connector_step_host_io) tries the other counts on its first calls and keeps the fastest.
    fixed_ = false;
    if (const char *e = getenv("RBG_HOST_THREADS")) {
      const int v = atoi(e);
      if (v >= 1) {
        n = v;
        fixed_ = true;
      }
    }
    if (n < 1) n = 1;
    if (n > 64) n = 64;
    threads_ = n;
    active_ = fixed_ || n < 4 ? n : n / 2;
    for (int i = 0; i < n; ++i) {
      std::thread t([this, i] { run(i); });
      t.detach();  // the pool lives as long as the process (never destroyed: workers may be parked at exit)
    }
  }
  int threads() const { return active_; }
  int max_threads() const { return threads_; }
  bool fixed() const { return fixed_; }
  void set_active(int a) {
    {
      std::lock_guard<std::mutex> lock(mu_);
      active_ = a < 1 ? 1 : (a > threads_ ? threads_ : a);
    }
    park_.notify_all();
    cv_.notify_all();
  }
  void submit(const uint8_t *src, int32_t *dst, size_t n, int bits = 8) {
    if (n == 0) return;
    // pieces of whole 64-byte destination lines, a few per worker so that a slow core does not hold the slice back
    size_t per = (n + (size_t)active_ * 2 - 1) / ((size_t)active_ * 2);
    per = (per + 63) & ~(size_t)63;
    if (per < 16384) per = 16384;
    {
      std::lock_guard<std::mutex> lock(mu_);
      for (size_t off = 0; off < n; off += per) {
        q_.push_back(Piece{src + (bits == 4 ? off >> 1 : off), dst + off, n - off < per ? n - off : per, bits});  // per is a multiple of 64
        ++pending_;
        avail_.fetch_add(1, std::memory_order_release);
      }
    }
    cv_.notify_all();
  }
  void wait() {
    std::unique_lock<std::mutex> lock(mu_);
    done_.wait(lock, [this] { return pending_ == 0; });
  }

 private:
  void run(int idx) {
    for (;;) {
      Piece p;
      {
        // workers beyond the active count sleep on their own condition variable: on the work queue's they would be woken
        // (and go back to sleep) at every slice, which cost the active ones 12 % of the step on a 16-core host
        if (idx >= active_) {
          std::unique_lock<std::mutex> lock(mu_);
          park_.wait(lock, [this, idx] { return idx < active_; });
          continue;
        }
        // a step hands over a slice every ~70 us: poll for a short while before parking on the condition variable
        for (int spin = 0; spin < 4000 && avail_.load(std::memory_order_acquire) == 0; ++spin) cpu_relax();
        std::unique_lock<std::mutex> lock(mu_);
        cv_.wait(lock, [this, idx] { return !q_.empty() || idx >= active_; });
        if (idx >= active_) continue;
        p = q_.front();
        q_.pop_front();
        avail_.fetch_sub(1, std::memory_order_relaxed);
      }
      if (p.bits == 4)
        widen4(p.src, p.dst, p.n);
      else
        widen(p.src, p.dst, p.n);
      {
        std::lock_guard<std::mutex> lock(mu_);
        if (--pending_ == 0) done_.notify_all();
      }
    }
  }
  std::mutex mu_;
  std::condition_variable cv_, done_, park_;
  std::deque<Piece> q_;
  size_t pending_ = 0;
  std::atomic<long> avail_{0};
  int threads_ = 0;
  std::atomic<int> active_{0};
  bool fixed_ = false;
};

Pool &pool() {
  // leaked on purpose (see the constructor); a forked child has the pointer but none of the threads: it gets its own
  static Pool *p = nullptr;
  static pid_t owner = 0;
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  if (!p || owner != getpid()) {
    p = new Pool();
    owner = getpid();
  }
  return *p;
}

}  // namespace

int host_pool_threads() { return pool().threads(); }
int host_pool_max_threads() { return pool().max_threads(); }
bool host_pool_fixed() { return pool().fixed(); }
void host_pool_set_threads(int n) { pool().set_active(n); }
void host_pool_widen(const uint8_t *src, int32_t *dst, size_t n) { pool().submit(src, dst, n); }
void host_pool_widen4(const uint8_t *src, int32_t *dst, size_t n) { pool().submit(src, dst, n, 4); }
void host_pool_wait() { pool().wait(); }

}  // namespace rbg
