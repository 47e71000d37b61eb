// Shared helpers for libhgt_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "hgt_b200.h"

#define HGT_SM_COUNT_FALLBACK 148

void hgt_set_error(const char* fmt, ...);
int hgt_sm_count();

#define HGT_CHECK_CUDA(expr)                                                                      \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess) {                                                                      \
      hgt_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));   \
      return 2;                                                                                   \
    }                                                                                             \
  } while (0)

#define HGT_REQUIRE(cond, ...)                                                                    \
  do {                                                                                            \
    if (!(cond)) {                                                                                \
      hgt_set_error(__VA_ARGS__);                                                                 \
      return 1;                                                                                   \
    }                                                                                             \
  } while (0)

extern unsigned long long g_hgt_launches;   // kernels launched by this library (bench.py reports it)
#define HGT_LAUNCH_CHECK()                  \
  do {                                      \
    ++g_hgt_launches;                       \
    HGT_CHECK_CUDA(cudaGetLastError());     \
  } while (0)

static inline size_t hgt_align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

__device__ __forceinline__ float hgt_gelu_erf(float x) {
  // F.gelu default (exact erf form), conv.py:119
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}

// The operand format of every tcgen05 GEMM: x = hi + lo with hi = rn(x), lo = rn(x - hi), both bf16.  Every producer
// splits through these two helpers, so pre-split operands (and sharded runs) round exactly like the GEMM's own split.
__device__ __forceinline__ void hgt_split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}
// Four consecutive values, stored as one 8-byte word into each of hi and lo.
__device__ __forceinline__ void hgt_split_bf16x4(const float (&v)[4], uint2* hi, uint2* lo) {
  __nv_bfloat16 h[4], l[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) hgt_split_bf16(v[j], h[j], l[j]);
  *hi = *reinterpret_cast<uint2*>(h);
  *lo = *reinterpret_cast<uint2*>(l);
}

// ---- ordered reductions (deterministic backward, torch.use_deterministic_algorithms) ------------------------------------
// Partial results of a reduction are written to [chunks, stride] scratch and summed in chunk order, so the bits of the
// result depend only on the problem shape, never on which CTA finished first.
__device__ __forceinline__ float hgt_chunk_sum(const float* part, int chunks, int64_t stride) {
  float s = 0.f;
  for (int c = 0; c < chunks; ++c) s += part[(int64_t)c * stride];
  return s;
}
// One segment of hgt_ordered_sum_launch: dst[dst + i] += sum_{c < chunks} part[part + c * n + i]  (i < n).
struct hgt_sum_seg {
  int64_t part, dst;
  int32_t chunks, pad;
};
// segs: device array of n_segs segments (all of width n).
int hgt_ordered_sum_launch(const float* part, const hgt_sum_seg* segs, int n_segs, int64_t n, float* dst,
                           cudaStream_t st);
