// Shared helpers for the prompt_tts_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/prompt_tts_b200.h"

typedef __nv_bfloat16 bf16;

void pt_set_error(const char* fmt, ...);

#define PT_REQUIRE(cond, ...)        \
  do {                               \
    if (!(cond)) {                   \
      pt_set_error(__VA_ARGS__);     \
      return PT_EINVAL;              \
    }                                \
  } while (0)

#define PT_CUDA_OK(expr)                                                          \
  do {                                                                            \
    cudaError_t e__ = (expr);                                                     \
    if (e__ != cudaSuccess) {                                                     \
      pt_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__)); \
      return PT_ECUDA;                                                            \
    }                                                                             \
  } while (0)

extern unsigned long long g_pt_launches;  // kernels launched by this library (api.cu)
#define PT_LAUNCH_CHECK()            \
  do {                               \
    ++g_pt_launches;                 \
    PT_CUDA_OK(cudaGetLastError());  \
  } while (0)

// Run `expr` (a cudaFuncSetAttribute call: per-device state) once per device and per call site, thread-safely.  A process-wide
// `static bool` would leave a second device of the same process without its opt-in shared memory.
#define PT_ONCE_PER_DEVICE(expr)                                              \
  do {                                                                        \
    static std::atomic<unsigned long long> done__{0};                         \
    int dev__ = 0;                                                            \
    PT_CUDA_OK(cudaGetDevice(&dev__));                                        \
    const unsigned long long bit__ = 1ull << (dev__ & 63);                    \
    if (!(done__.load(std::memory_order_acquire) & bit__)) {                  \
      PT_CUDA_OK(expr);                                                       \
      done__.fetch_or(bit__, std::memory_order_release);                      \
    }                                                                         \
  } while (0)

extern int g_pt_sm_reserve;  // SMs the persistent kernels leave free (api.cu: pt_set_sm_reserve)
static inline int pt_num_sms_physical() {
  static std::atomic<int> cache[64];
  int dev = 0;
  cudaGetDevice(&dev);
  int n = cache[dev & 63].load(std::memory_order_relaxed);
  if (!n) {
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
    cache[dev & 63].store(n, std::memory_order_relaxed);
  }
  return n;
}
// SM count the persistent grids (GEMM, attention) are sized for
static inline int pt_num_sms() {
  const int n = pt_num_sms_physical() - g_pt_sm_reserve;
  return n > 1 ? n : 1;
}

// Grid of a grid-stride kernel: one block per `per_block` items, at most `waves` blocks per SM
static inline unsigned grid_for(long long items, int per_block, int waves = 8) {
  long long b = (items + per_block - 1) / per_block;
  const long long cap = (long long)pt_num_sms() * waves;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (unsigned)b;
}
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// Sum of `acc` over the block (blockDim.x a multiple of 32), valid in thread 0.  Call it from every thread: it synchronises.
__device__ __forceinline__ float block_sum(float acc) {
  acc = warp_sum(acc);
  __shared__ float sh[32];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  float v = 0.f;
  if (threadIdx.x < 32) {
    v = threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0.f;
    v = warp_sum(v);
  }
  return v;
}

// 8 x bf16 <-> 8 x float through ONE 16-byte access.  The carrier is four plain 32-bit words moved as a uint4: a struct of
// __nv_bfloat162 members is copied member-wise by the compiler (the type is not trivially copyable), which turns every
// "16-byte" access into four 4-byte ones with a 16-byte stride -- four times the load/store instructions and, for stores,
// four partial writes per sector (found with cuobjdump: STG.E x4 instead of STG.E.128 in every kernel using it).
struct __align__(16) bf16x8 {
  uint32_t w[4];
};
__device__ __forceinline__ bf16x8 ld16(const void* p) {
  const uint4 t = *reinterpret_cast<const uint4*>(p);
  bf16x8 r;
  r.w[0] = t.x, r.w[1] = t.y, r.w[2] = t.z, r.w[3] = t.w;
  return r;
}
__device__ __forceinline__ void st16(void* p, const bf16x8& r) { *reinterpret_cast<uint4*>(p) = make_uint4(r.w[0], r.w[1], r.w[2], r.w[3]); }
__device__ __forceinline__ float2 bf2_to_f2(uint32_t w) { return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u)); }
__device__ __forceinline__ uint32_t f2_to_bf2(float lo, float hi) {
  const __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&t);
}
// issue the 16-byte load now (4 registers), convert when the value is needed -- lets a thread keep many loads in flight without
// holding 8 fp32 registers per vector
__device__ __forceinline__ bf16x8 load8raw(const bf16* p) { return ld16(p); }
__device__ __forceinline__ void unpack8(const bf16x8& r, float* f) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = bf2_to_f2(r.w[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
// same values, but the compiler cannot see that (the words pass through a volatile mov): a kernel that converts the same raw
// vector in several phases re-converts it each time instead of keeping the 8 fp32 results alive in registers across phases
__device__ __forceinline__ void unpack8_again(const bf16x8& r, float* f) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    uint32_t w;
    asm volatile("mov.b32 %0, %1;" : "=r"(w) : "r"(r.w[i]));
    const float2 t = bf2_to_f2(w);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ void load8(const bf16* p, float* f) { unpack8(ld16(p), f); }
__device__ __forceinline__ void store8(bf16* p, const float* f) {
  bf16x8 r;
#pragma unroll
  for (int i = 0; i < 4; ++i) r.w[i] = f2_to_bf2(f[2 * i], f[2 * i + 1]);
  st16(p, r);
}

__device__ __forceinline__ float silu_f(float x) { return x / (1.f + __expf(-x)); }
__device__ __forceinline__ float silu_grad_f(float x) {
  float s = 1.f / (1.f + __expf(-x));
  return s * (1.f + x * (1.f - s));
}
