// Host side of the device -> host path: the count matrix crosses PCIe in a narrow format
// (uint8 / uint16 with an exact overflow list, or int32) into pinned staging buffers, and these
// multi-threaded routines expand it into the caller's matrix (int32, or the reference's int64:
// prosstt/simulation.py:651 returns the int64 array of scipy's nbinom.rvs) while the GPU samples
// the next chunk.  Pure data movement: no sampling arithmetic runs on the CPU.
//
// Plain C ABI (include/prosstt_b200.h): host pointers, sizes, a thread count.
#include <immintrin.h>
#include <stdint.h>
#include <string.h>
#include <sys/mman.h>
#include <unistd.h>
#include <algorithm>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>
#include "../../include/prosstt_b200.h"

namespace {

int clamp_threads(int threads, int64_t n, int64_t min_per_thread) {
  int hw = (int)std::thread::hardware_concurrency();
  if (hw <= 0) hw = 1;
  if (threads <= 0) threads = hw;
  const int64_t useful = std::max<int64_t>(1, n / std::max<int64_t>(1, min_per_thread));
  return (int)std::max<int64_t>(1, std::min<int64_t>(std::min(threads, 256), useful));
}

// Worker threads that outlive the calls: an expansion runs once per staged chunk (every few
// milliseconds), and starting 15 threads each time costs a visible share of it.  One job at a time
// (callers queue on run_m_); the caller works too.  Never destroyed (threads die with the process); a
// forked child starts its own.
class Pool {
 public:
  static Pool &get() {
    static Pool *pool = nullptr;
    static std::mutex guard;
    std::lock_guard<std::mutex> g(guard);
    if (pool == nullptr || pool->pid_ != getpid()) pool = new Pool();
    return *pool;
  }
  void run(int tasks, const std::function<void(int)> &fn) {
    if (tasks <= 1) { if (tasks == 1) fn(0); return; }
    std::lock_guard<std::mutex> one_job(run_m_);
    std::unique_lock<std::mutex> lk(m_);
    while ((int)th_.size() < tasks - 1) th_.emplace_back([this] { work(); });
    fn_ = &fn; tasks_ = tasks; next_ = 0; done_ = 0;
    cv_.notify_all();
    take(lk);
    done_cv_.wait(lk, [this] { return done_ == tasks_; });
    fn_ = nullptr; tasks_ = 0; next_ = 0;
  }

 private:
  Pool() : pid_(getpid()) {}
  void take(std::unique_lock<std::mutex> &lk) {              // called with m_ held
    while (next_ < tasks_) {
      const int t = next_++;
      lk.unlock();
      (*fn_)(t);
      lk.lock();
      if (++done_ == tasks_) done_cv_.notify_all();
    }
  }
  void work() {
    std::unique_lock<std::mutex> lk(m_);
    for (;;) {
      cv_.wait(lk, [this] { return next_ < tasks_; });
      take(lk);
    }
  }
  std::mutex run_m_, m_;
  std::condition_variable cv_, done_cv_;
  std::vector<std::thread> th_;
  const std::function<void(int)> *fn_ = nullptr;
  int tasks_ = 0, next_ = 0, done_ = 0;
  pid_t pid_;
};

// run fn(lo, hi) over [0, n) cut into `threads` contiguous slices aligned to 64 elements
template <class F>
void parallel_slices(int64_t n, int threads, F fn) {
  if (threads <= 1) { fn((int64_t)0, n); return; }
  const int64_t per = ((n + threads - 1) / threads + 63) & ~(int64_t)63;
  Pool::get().run(threads, [&](int t) {
    const int64_t lo = std::min(n, per * t), hi = std::min(n, per * (t + 1));
    if (lo < hi) fn(lo, hi);
  });
}

template <class S, class D>
__attribute__((target_clones("avx512f", "avx2", "default")))
void widen_slice(const S *__restrict__ src, D *__restrict__ dst, int64_t lo, int64_t hi) {
  for (int64_t i = lo; i < hi; ++i) dst[i] = (D)src[i];
}

// The same expansion with non-temporal (streaming) 64-byte stores: the destination lines are written
// whole without being read first, which halves the memory traffic of a destination that is not in
// cache (a pinned or re-used result matrix: read 1 + write 4 instead of read 1 + read 4 + write 4 bytes
// per uint8 -> int32 count).  AVX-512 only; other CPUs and the unaligned edges take the ordinary loop.
template <class S, class D> struct Expand;
#define PST_EXPAND(S, D, LOAD, CVT, PER)                                                                   \
  template <> struct Expand<S, D> {                                                                        \
    static constexpr int per = PER;                         /* elements per 64-byte store */                \
    __attribute__((target("avx512f,avx512bw,avx512vl"))) static inline void one(const S *s, D *d) {        \
      _mm512_stream_si512(reinterpret_cast<__m512i *>(d), CVT(LOAD(s)));                                   \
    }                                                                                                      \
  };
#define PST_LD128(s) _mm_loadu_si128(reinterpret_cast<const __m128i *>(s))
#define PST_LD256(s) _mm256_loadu_si256(reinterpret_cast<const __m256i *>(s))
#define PST_LD512(s) _mm512_loadu_si512(reinterpret_cast<const void *>(s))
#define PST_LD64(s) _mm_loadl_epi64(reinterpret_cast<const __m128i *>(s))
#define PST_ID(v) (v)
PST_EXPAND(uint8_t, int32_t, PST_LD128, _mm512_cvtepu8_epi32, 16)
PST_EXPAND(uint16_t, int32_t, PST_LD256, _mm512_cvtepu16_epi32, 16)
PST_EXPAND(uint8_t, int64_t, PST_LD64, _mm512_cvtepu8_epi64, 8)
PST_EXPAND(uint16_t, int64_t, PST_LD128, _mm512_cvtepu16_epi64, 8)
PST_EXPAND(int32_t, int64_t, PST_LD256, _mm512_cvtepi32_epi64, 8)
PST_EXPAND(int32_t, int32_t, PST_LD512, PST_ID, 16)
#undef PST_EXPAND

template <class S, class D>
__attribute__((target("avx512f,avx512bw,avx512vl")))
void widen_slice_stream(const S *__restrict__ src, D *__restrict__ dst, int64_t lo, int64_t hi) {
  constexpr int per = Expand<S, D>::per;
  int64_t i = lo;
  while (i < hi && (reinterpret_cast<uintptr_t>(dst + i) & 63u) != 0) { dst[i] = (D)src[i]; ++i; }   // to a 64-byte line
  for (; i + 4 * per <= hi; i += 4 * per) {
    Expand<S, D>::one(src + i, dst + i);
    Expand<S, D>::one(src + i + per, dst + i + per);
    Expand<S, D>::one(src + i + 2 * per, dst + i + 2 * per);
    Expand<S, D>::one(src + i + 3 * per, dst + i + 3 * per);
  }
  for (; i + per <= hi; i += per) Expand<S, D>::one(src + i, dst + i);
  for (; i < hi; ++i) dst[i] = (D)src[i];
  _mm_sfence();                                            // streaming stores are ordered before the join
}

bool cpu_streams() {
  static const bool ok = __builtin_cpu_supports("avx512f") && __builtin_cpu_supports("avx512bw") &&
                         __builtin_cpu_supports("avx512vl");
  return ok;
}

template <class S, class D>
void widen(const void *src, void *dst, int64_t n, int threads, bool stream) {
  const S *s = static_cast<const S *>(src);
  D *d = static_cast<D *>(dst);
  // a destination that is not aligned to its own element size cannot be brought to a 64-byte line
  const bool st = stream && cpu_streams() && (reinterpret_cast<uintptr_t>(dst) % sizeof(D)) == 0;
  parallel_slices(n, clamp_threads(threads, n, 1 << 16), [=](int64_t lo, int64_t hi) {
    if (st) widen_slice_stream<S, D>(s, d, lo, hi);
    else widen_slice<S, D>(s, d, lo, hi);
  });
}

int widen_any(const void *src, int32_t src_bits, void *dst, int32_t dst_bits, int64_t n, int32_t threads, bool stream) {
  if (n < 0 || (n > 0 && (!src || !dst))) return -1;
  if (n == 0) return 0;
  if (src_bits == 8 && dst_bits == 32) widen<uint8_t, int32_t>(src, dst, n, threads, stream);
  else if (src_bits == 16 && dst_bits == 32) widen<uint16_t, int32_t>(src, dst, n, threads, stream);
  else if (src_bits == 8 && dst_bits == 64) widen<uint8_t, int64_t>(src, dst, n, threads, stream);
  else if (src_bits == 16 && dst_bits == 64) widen<uint16_t, int64_t>(src, dst, n, threads, stream);
  else if (src_bits == 32 && dst_bits == 64) widen<int32_t, int64_t>(src, dst, n, threads, stream);
  else if (src_bits == 32 && dst_bits == 32 && stream) widen<int32_t, int32_t>(src, dst, n, threads, true);
  else if (src_bits == 32 && dst_bits == 32) {
    const char *s = static_cast<const char *>(src);
    char *d = static_cast<char *>(dst);
    parallel_slices(n, clamp_threads(threads, n, 1 << 16),
                    [=](int64_t lo, int64_t hi) { memcpy(d + 4 * lo, s + 4 * lo, (size_t)(4 * (hi - lo))); });
  } else {
    return -1;
  }
  return 0;
}

__attribute__((target_clones("avx512f", "avx2", "default")))
uint64_t sum_words(const uint32_t *__restrict__ p, int64_t lo, int64_t hi) {
  uint64_t a = 0;
  for (int64_t i = lo; i < hi; ++i) a += p[i];
  return a;
}

}  // namespace

extern "C" int pst_host_widen(const void *src, int32_t src_bits, void *dst, int32_t dst_bits, int64_t n,
                              int32_t threads) {
  return widen_any(src, src_bits, dst, dst_bits, n, threads, false);
}

// 1 when pst_host_widen_stream really uses non-temporal stores on this CPU (AVX-512), 0 when it falls
// back to ordinary ones: what the choice of the device->host transport rests on.
extern "C" int pst_host_stream_stores(void) { return cpu_streams() ? 1 : 0; }

extern "C" int pst_host_widen_stream(const void *src, int32_t src_bits, void *dst, int32_t dst_bits, int64_t n,
                                     int32_t threads) {
  return widen_any(src, src_bits, dst, dst_bits, n, threads, true);
}

// Ask for transparent huge pages under a freshly allocated (untouched) result buffer: the expansion
// threads take one page fault per 2 MiB instead of one per 4 KiB when they first write it.  Advice only:
// returns 0 when it was given, 1 when the platform does not offer it (nothing changes either way).
extern "C" int pst_host_prepare(void *buffer, int64_t bytes) {
#if defined(MADV_HUGEPAGE)
  if (!buffer || bytes < (int64_t)(4 << 20)) return 1;
  const uintptr_t huge = (uintptr_t)2 << 20;
  const uintptr_t lo = ((uintptr_t)buffer + huge - 1) & ~(huge - 1);
  const uintptr_t hi = ((uintptr_t)buffer + (uintptr_t)bytes) & ~(huge - 1);
  if (hi <= lo) return 1;
  return madvise(reinterpret_cast<void *>(lo), hi - lo, MADV_HUGEPAGE) == 0 ? 0 : 1;
#else
  (void)buffer; (void)bytes;
  return 1;
#endif
}

// dst[index[i] - base] = value[i] for the entries with base <= index[i] < base + n (the exact values of
// the elements that saturated the narrow format); dst holds dst_bits-wide integers.
extern "C" int pst_host_apply_overflow(void *dst, int32_t dst_bits, int64_t base, int64_t n, const int64_t *index,
                                       const int32_t *value, int64_t entries) {
  if (entries < 0 || n < 0 || (entries > 0 && (!dst || !index || !value))) return -1;
  if (dst_bits != 32 && dst_bits != 64) return -1;
  // scattered single-element writes (each one a cache miss in a matrix of gigabytes): a few threads keep
  // more of them in flight; an index listed twice carries the same value, so slices need no ordering
  const int threads = std::min(clamp_threads(0, entries, 1 << 14), 16);
  parallel_slices(entries, threads, [=](int64_t lo, int64_t hi) {
    for (int64_t i = lo; i < hi; ++i) {
      const int64_t at = index[i] - base;
      if (at < 0 || at >= n) continue;
      if (dst_bits == 32) static_cast<int32_t *>(dst)[at] = value[i];
      else static_cast<int64_t *>(dst)[at] = (int64_t)value[i];
    }
  });
  return 0;
}

// Sum of the buffer read as uint32 words (bytes must be a multiple of 4): the cheapest sink that
// still touches every byte; used by the streamed C5 benchmark and as a transfer checksum.
extern "C" uint64_t pst_host_checksum(const void *src, int64_t bytes, int32_t threads) {
  if (!src || bytes <= 0) return 0;
  const int64_t n = bytes / 4;
  const uint32_t *p = static_cast<const uint32_t *>(src);
  const int t = clamp_threads(threads, n, 1 << 18);
  std::vector<uint64_t> part((size_t)t + 1, 0);
  const int64_t per = ((n + t - 1) / t + 63) & ~(int64_t)63;
  parallel_slices(n, t, [&](int64_t lo, int64_t hi) { part[(size_t)(lo / per)] = sum_words(p, lo, hi); });
  uint64_t total = 0;
  for (uint64_t v : part) total += v;
  return total;
}

// zlib's crc32_combine: the CRC-32 of A || B from crc32(A), crc32(B) and |B| (products in GF(2) modulo the
// CRC polynomial, x^(8 |B|) by squaring); the compressed CSR file's members are CRC-ed chunk by chunk on the
// device.
namespace {
uint32_t crc_multmodp(uint32_t a, uint32_t b) {
  uint32_t p = 0;
  for (uint32_t m = 1u << 31; m != 0; m >>= 1) {
    if (a & m) p ^= b;
    b = (b & 1) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
  }
  return p;
}
}  // namespace

extern "C" uint32_t pst_host_crc32_combine(uint32_t crc1, uint32_t crc2, int64_t len2) {
  if (len2 <= 0) return crc1 ^ crc2;
  uint32_t x2n = 1u << 30, p = 1u << 31;             // x^(2^k) for k = 0, and x^0
  for (int k = 0; k < 3; ++k) x2n = crc_multmodp(x2n, x2n);   // x^8: one byte
  for (uint64_t n = (uint64_t)len2; n; n >>= 1) {
    if (n & 1) p = crc_multmodp(x2n, p);
    x2n = crc_multmodp(x2n, x2n);
  }
  return crc_multmodp(p, crc1) ^ crc2;
}
