// Common device/host helpers for the Robust U-Net sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/rbunet.h"

typedef __nv_bfloat16 bf16;

// ---------------------------------------------------------------------------------------------
// error handling: never throw / exit across the C ABI; record a message, return a negative code
// ---------------------------------------------------------------------------------------------
void rbu_set_error(const char* fmt, ...);

#define RBU_CHECK_ARG(cond, ...)                                   \
  do {                                                             \
    if (!(cond)) {                                                 \
      rbu_set_error(__VA_ARGS__);                                  \
      return RBU_ERR_INVALID;                                      \
    }                                                              \
  } while (0)

#define RBU_CHECK_CUDA(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      rbu_set_error("%s:%d CUDA error %s: %s", __FILE__, __LINE__, #expr,                 \
                    cudaGetErrorString(_e));                                              \
      return RBU_ERR_CUDA;                                                                \
    }                                                                                     \
  } while (0)

// every kernel launch of the library goes through this macro: it also feeds rbu_launch_count()
#include <atomic>
extern std::atomic<unsigned long long> g_rbu_launches;
#define RBU_CHECK_LAUNCH()                                        \
  do {                                                            \
    g_rbu_launches.fetch_add(1, std::memory_order_relaxed);       \
    RBU_CHECK_CUDA(cudaGetLastError());                           \
  } while (0)

int rbu_num_sms();          // SM count of the CURRENT device (cached per device ordinal)

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device: one bit per device ordinal, set once.
// Usage:  static std::atomic<unsigned long long> done{0};  if (rbu_first_use_on_device(&done)) cudaFuncSetAttribute(...)
bool rbu_first_use_on_device(std::atomic<unsigned long long>* done_mask);

static inline int rbu_cdiv(long a, long b) { return (int)((a + b - 1) / b); }

// grid.x (blocks per image, grid.y = images) of a streaming kernel whose threads keep per-(image, channel) coefficients in
// registers: every block pays a prologue of 24-64 scalar loads per thread before its first 16-byte load, so a thread
// should stream at least `min_iters` x U vectors -- as long as ~3 blocks per SM remain in flight -- and at most ~32
// resident warps per SM over a few waves are useful.  `per_iter` = items one block covers per loop iteration (threads x U).
int rbu_stream_blocks(long items_per_image, int per_iter, int images);

// Deterministic column sums of per-CTA partial rows part[nblk][stride] (backward_ops.cu): out1[k] = sum of column k for
// k < K1, out2[k] = sum of column K1 + k for k < K2 (fixed order, double accumulation).  Long lists are first folded in
// `scratch`, which must hold colsum_scratch_floats(K1 + K2) floats.
size_t colsum_scratch_floats(int K);
int colsum_split(const float* part, int nblk, long stride, int K1, float* out1, int K2, float* out2, float* scratch,
                 cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__

struct __align__(16) bf16x8 {
  __nv_bfloat162 v[4];
};

__device__ __forceinline__ bf16x8 ld_bf16x8(const bf16* p) {
  bf16x8 r;
  *reinterpret_cast<uint4*>(&r) = __ldg(reinterpret_cast<const uint4*>(p));
  return r;
}
// streaming (read-once) variant: do not pollute L1
__device__ __forceinline__ bf16x8 ld_bf16x8_stream(const bf16* p) {
  bf16x8 r;
  uint4 u;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "l"(p));
  *reinterpret_cast<uint4*>(&r) = u;
  return r;
}
// Pull the line behind `p` into L2 without tying up a register (see rb_bwd1_kernel).
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void st_bf16x8(bf16* p, const bf16x8& v) {
  *reinterpret_cast<uint4*>(p) = *reinterpret_cast<const uint4*>(&v);
}
__device__ __forceinline__ void unpack8(const bf16x8& v, float* f) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(v.v[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ bf16x8 pack8(const float* f) {
  bf16x8 r;
#pragma unroll
  for (int i = 0; i < 4; ++i) r.v[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return r;
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

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

#endif  // __CUDACC__
