// Shared device/host helpers for the fugue_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/fugue_b200.h"

#define FB_NULL_KEY_BITS 0x7FF8000000000000ULL

// ---- error handling (thread-local message, int status) ---------------------
void fb_set_error(const char* fmt, ...);
#define FB_CHECK(cond, ...)                                                    \
  do {                                                                         \
    if (!(cond)) {                                                             \
      fb_set_error(__VA_ARGS__);                                               \
      return 1;                                                                \
    }                                                                          \
  } while (0)
#define FB_CUDA(expr)                                                          \
  do {                                                                         \
    cudaError_t _e = (expr);                                                   \
    if (_e != cudaSuccess) {                                                   \
      fb_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),     \
                   __FILE__, __LINE__);                                        \
      return 2;                                                                \
    }                                                                          \
  } while (0)

struct FbDeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit FbDeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~FbDeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

int fb_sm_count(int dev);

// ---- key description passed by value to kernels -----------------------------
struct FbKeys {
  const void* ptr[FB_MAX_KEYS];
  const uint8_t* valid[FB_MAX_KEYS];
  int32_t width[FB_MAX_KEYS];
  int32_t nkeys;
  int32_t digit_shift;  // < 0: hash mode; >= 0: radix-sort mode, id = (key[0] >> digit_shift) & (num - 1)
};

// Division-free `h % d` for a runtime-invariant 32-bit divisor d >= 1
// (Granlund & Montgomery, "Division by invariant integers using multiplication",
//  unsigned round-up variant with a 65-bit magic split as 2^64 + magic).
struct FbDiv {
  uint64_t magic;
  uint32_t d;
  uint32_t shift;  // l - 1 where l = ceil(log2 d); unused for d == 1
};

static inline FbDiv fb_make_div(uint32_t d) {
  FbDiv r;
  r.d = d;
  r.magic = 0;
  r.shift = 0;
  if (d <= 1) return r;
  uint32_t l = 32 - (uint32_t)__builtin_clz(d - 1);  // ceil(log2 d), 1..32
  unsigned __int128 num = ((unsigned __int128)1 << 64) * (((unsigned __int128)1 << l) - d);
  r.magic = (uint64_t)(num / d) + 1;
  r.shift = l - 1;
  return r;
}

#ifdef __CUDACC__
#define FB_HD __host__ __device__ __forceinline__
#else
#define FB_HD inline
#endif

FB_HD uint64_t fb_mulhi64(uint64_t a, uint64_t b) {
#ifdef __CUDA_ARCH__
  return __umul64hi(a, b);
#else
  return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

// d not a power of two
FB_HD uint32_t fb_fastmod_magic(uint64_t n, const FbDiv& dv) {
  uint64_t q = fb_mulhi64(dv.magic, n);
  uint64_t t = ((n - q) >> 1) + q;
  q = t >> dv.shift;
  return (uint32_t)(n - q * dv.d);
}

FB_HD uint32_t fb_fastmod(uint64_t n, const FbDiv& dv) {
  if ((dv.d & (dv.d - 1)) == 0) return (uint32_t)n & (dv.d - 1);  // power of two (and d == 1)
  return fb_fastmod_magic(n, dv);
}

// pandas _hash_ndarray finaliser (splitmix64)
FB_HD uint64_t fb_fmix64(uint64_t h) {
  h ^= h >> 30;
  h *= 0xBF58476D1CE4E5B9ULL;
  h ^= h >> 27;
  h *= 0x94D049BB133111EBULL;
  h ^= h >> 31;
  return h;
}

#ifdef __CUDACC__
__device__ __forceinline__ uint64_t fb_load_bits(const void* p, int width, int64_t i) {
  switch (width) {
    case 1: return __ldg((const uint8_t*)p + i);
    case 2: return __ldg((const uint16_t*)p + i);
    case 4: return __ldg((const uint32_t*)p + i);
    default: return __ldg((const unsigned long long*)p + i);
  }
}

// pandas combine_hash_arrays over the key tuple of row i
__device__ __forceinline__ uint64_t fb_row_hash(const FbKeys& k, int64_t i) {
  uint64_t out = 0x345678ULL, mult = 1000003ULL;
#pragma unroll 1
  for (int c = 0; c < k.nkeys; ++c) {
    uint64_t b = fb_load_bits(k.ptr[c], k.width[c], i);
    if (k.valid[c] != nullptr && __ldg(k.valid[c] + i) == 0) b = FB_NULL_KEY_BITS;
    out ^= fb_fmix64(b);
    out *= mult;
    mult += (uint64_t)(82520 + 2 * (k.nkeys - c));
  }
  return out + 97531ULL;
}

// single non-null 8-byte key: closed form
__device__ __forceinline__ uint64_t fb_hash_single_u64(uint64_t bits) {
  return ((0x345678ULL ^ fb_fmix64(bits)) * 1000003ULL) + 97531ULL;
}

__device__ __forceinline__ unsigned fb_lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}
#endif
