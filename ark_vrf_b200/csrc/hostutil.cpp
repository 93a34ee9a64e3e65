// Host-side helpers of libavrf_gpu.so that want CPU-specific code (compiled by the host compiler, never by cudafe).
#include "hostutil.h"

#include <string.h>

#if defined(__x86_64__)
#include <immintrin.h>

__attribute__((target("avx2"))) static void copy_nt_avx2(void* dst, const void* src, size_t n) {
  char* d = static_cast<char*>(dst);
  const char* s = static_cast<const char*>(src);
  for (size_t i = 0; i < n; i += 32)
    _mm256_stream_si256(reinterpret_cast<__m256i*>(d + i), _mm256_loadu_si256(reinterpret_cast<const __m256i*>(s + i)));
}

static const bool g_avx2 = __builtin_cpu_supports("avx2");

// One staged proof: its fixed-size fields (32-byte multiples each) and n_ios pairs (128 B each), every destination
// 32-byte aligned.
__attribute__((target("avx2"))) static void stage_proof_avx2(const avrf::StageField* f, size_t nf, uint8_t* dio, const uint8_t* ios,
                                                             size_t io_bytes) {
  for (size_t k = 0; k < nf; k++)
    for (size_t i = 0; i < f[k].bytes; i += 32)
      _mm256_stream_si256(reinterpret_cast<__m256i*>(f[k].dst + i), _mm256_loadu_si256(reinterpret_cast<const __m256i*>(f[k].src + i)));
  for (size_t i = 0; i < io_bytes; i += 32)
    _mm256_stream_si256(reinterpret_cast<__m256i*>(dio + i), _mm256_loadu_si256(reinterpret_cast<const __m256i*>(ios + i)));
}

namespace avrf {
void stage_copy(void* dst, const void* src, size_t n) {
  if (g_avx2 && (n & 31) == 0 && (reinterpret_cast<uintptr_t>(dst) & 31) == 0) copy_nt_avx2(dst, src, n);
  else memcpy(dst, src, n);
}
void stage_proof(const StageField* f, size_t nf, uint8_t* dio, const uint8_t* ios, size_t io_bytes) {
  if (g_avx2) {
    stage_proof_avx2(f, nf, dio, ios, io_bytes);
  } else {
    for (size_t k = 0; k < nf; k++) memcpy(f[k].dst, f[k].src, f[k].bytes);
    if (io_bytes) memcpy(dio, ios, io_bytes);
  }
}
void stage_fence() { _mm_sfence(); }
}  // namespace avrf
#else
namespace avrf {
void stage_copy(void* dst, const void* src, size_t n) { memcpy(dst, src, n); }
void stage_proof(const StageField* f, size_t nf, uint8_t* dio, const uint8_t* ios, size_t io_bytes) {
  for (size_t k = 0; k < nf; k++) memcpy(f[k].dst, f[k].src, f[k].bytes);
  if (io_bytes) memcpy(dio, ios, io_bytes);
}
void stage_fence() {}
}  // namespace avrf
#endif
