// HGTConv.update epilogue (conv.py:129-133): sigmoid(skip)-gated residual + per-type LayerNorm.
// One warp per node row; the row (d <= 1024 floats) stays in registers between the two LayerNorm passes.
// HBM-bound: reads o and x (2*d*4 B), writes out (d*4 B) per node.
#include <cuda_bf16.h>

#include "common.cuh"

namespace {

constexpr int kMaxPerLane = 32;   // d <= 1024

__global__ void __launch_bounds__(256)
k_update_epilogue(const float* __restrict__ o, const float* __restrict__ x, const int32_t* __restrict__ type_row0,
                  int T, const float* __restrict__ skip, const float* __restrict__ norm_w,
                  const float* __restrict__ norm_b, const float* const* __restrict__ norm_wp,
                  const float* const* __restrict__ norm_bp, const int32_t* __restrict__ perm,
                  const int32_t* __restrict__ type_active, int64_t n_nodes, int d, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (row >= n_nodes) return;
  // node type of this rank: types are contiguous in rank order, T is small
  int t = 0;
  while (t < T && row >= type_row0[t + 1]) ++t;
  if (type_active && t < T && row - type_row0[t] >= type_active[t]) return;   // halo source: no output row
  if (perm && perm[row] < 0) return;             // sharded out_map: -1 = row without an output (e.g. unknown-type halo)
  float* orow = out + (perm ? (int64_t)perm[row] : row) * d;
  if (t >= T) {                                  // type outside [0,T): the reference leaves zeros (conv.py:120)
    for (int c = lane; c < d; c += 32) orow[c] = 0.f;
    return;
  }
  // skip == NULL: plain residual y = o + x (DenseHGTConv, conv.py:261,273)
  const float alpha = skip ? 1.0f / (1.0f + __expf(-skip[t])) : 1.0f;    // torch.sigmoid(self.skip[t]), conv.py:129
  const float beta = skip ? 1.0f - alpha : 1.0f;
  const float* op = o + row * d;
  const float* xp = x + row * d;
  float y[kMaxPerLane];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxPerLane; ++i) {
    int c = lane + i * 32;
    if (c < d) {
      y[i] = op[c] * alpha + xp[c] * beta;                 // conv.py:131,133
      sum += y[i];
    } else {
      y[i] = 0.f;
    }
  }
  if (norm_w == nullptr && norm_wp == nullptr) {
#pragma unroll
    for (int i = 0; i < kMaxPerLane; ++i) {
      int c = lane + i * 32;
      if (c < d) orow[c] = y[i];
    }
    return;
  }
  for (int s = 16; s > 0; s >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, s);
  const float mean = sum / d;
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxPerLane; ++i) {
    int c = lane + i * 32;
    if (c < d) {
      float dlt = y[i] - mean;
      var = fmaf(dlt, dlt, var);
    }
  }
  for (int s = 16; s > 0; s >>= 1) var += __shfl_xor_sync(0xffffffffu, var, s);
  const float rstd = rsqrtf(var / d + 1e-5f);              // nn.LayerNorm eps (conv.py:40)
  const float* w = norm_wp ? norm_wp[t] : norm_w + (int64_t)t * d;
  const float* b = norm_bp ? norm_bp[t] : norm_b + (int64_t)t * d;
#pragma unroll
  for (int i = 0; i < kMaxPerLane; ++i) {
    int c = lane + i * 32;
    if (c < d) orow[c] = (y[i] - mean) * rstd * w[c] + b[c];
  }
}

// The next layer's projection GEMM consumes its input as a bf16 hi/lo split: emit it here instead of re-reading `out`.
__device__ __forceinline__ void split_store(uint2* hi, uint2* lo, int64_t idx, const float4& v) {
  const float f[4] = {v.x, v.y, v.z, v.w};
  hgt_split_bf16x4(f, hi + idx, lo + idx);
}

// Vectorised variant: d % 4 == 0, each lane owns NV float4 chunks (chunk c = lane + 32*i), 128-bit loads/stores.
template <int NV>
__global__ void __launch_bounds__(256)
k_update_epilogue_vec(const float* __restrict__ o, const float* __restrict__ x, const int32_t* __restrict__ type_row0,
                      int T, const float* __restrict__ skip, const float* __restrict__ norm_w,
                      const float* __restrict__ norm_b, const float* const* __restrict__ norm_wp,
                      const float* const* __restrict__ norm_bp, const int32_t* __restrict__ perm,
                      const int32_t* __restrict__ type_active, int64_t n_nodes, int d, float* __restrict__ out,
                      uint2* __restrict__ out_hi, uint2* __restrict__ out_lo) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (row >= n_nodes) return;
  const int nvec = d >> 2;
  if (type_active) {
    // sharded runs: most local rows may be halo sources without an output row — leave before touching their data
    int t0 = 0;
    while (t0 < T && row >= type_row0[t0 + 1]) ++t0;
    if (t0 < T && row - type_row0[t0] >= type_active[t0]) return;
    if (perm && perm[row] < 0) return;
  }
  // issue the row loads first; the (short, warp-uniform) type search overlaps with them
  float4 ov[NV], xv[NV];
  const float4* op = reinterpret_cast<const float4*>(o + row * d);
  const float4* xp = reinterpret_cast<const float4*>(x + row * d);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    if (c < nvec) { ov[i] = __ldcs(op + c); xv[i] = __ldcs(xp + c); }
    else { ov[i] = make_float4(0.f, 0.f, 0.f, 0.f); xv[i] = ov[i]; }
  }
  int t = 0;
  while (t < T && row >= type_row0[t + 1]) ++t;
  if (type_active && t < T && row - type_row0[t] >= type_active[t]) return;
  if (perm && perm[row] < 0) return;             // sharded out_map: -1 = row without an output
  float4* orow = reinterpret_cast<float4*>(out + (perm ? (int64_t)perm[row] : row) * d);
  if (t >= T) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = lane + 32 * i;
      if (c < nvec) {
        orow[c] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (out_hi) split_store(out_hi, out_lo, row * nvec + c, make_float4(0.f, 0.f, 0.f, 0.f));
      }
    }
    return;
  }
  const float alpha = skip ? 1.0f / (1.0f + __expf(-skip[t])) : 1.0f;
  const float beta = skip ? 1.0f - alpha : 1.0f;
  float4 y[NV];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    y[i].x = ov[i].x * alpha + xv[i].x * beta;
    y[i].y = ov[i].y * alpha + xv[i].y * beta;
    y[i].z = ov[i].z * alpha + xv[i].z * beta;
    y[i].w = ov[i].w * alpha + xv[i].w * beta;
    sum += (y[i].x + y[i].y) + (y[i].z + y[i].w);
  }
  if (norm_w == nullptr && norm_wp == nullptr) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = lane + 32 * i;
      if (c < nvec) {
        __stcs(orow + c, y[i]);
        if (out_hi) split_store(out_hi, out_lo, row * nvec + c, y[i]);
      }
    }
    return;
  }
  for (int s = 16; s > 0; s >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, s);
  const float mean = sum / d;
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    if (c < nvec) {
      float a = y[i].x - mean, b = y[i].y - mean, e = y[i].z - mean, f = y[i].w - mean;
      var += (a * a + b * b) + (e * e + f * f);
    }
  }
  for (int s = 16; s > 0; s >>= 1) var += __shfl_xor_sync(0xffffffffu, var, s);
  const float rstd = rsqrtf(var / d + 1e-5f);
  const float4* w = reinterpret_cast<const float4*>(norm_wp ? norm_wp[t] : norm_w + (int64_t)t * d);
  const float4* b = reinterpret_cast<const float4*>(norm_bp ? norm_bp[t] : norm_b + (int64_t)t * d);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    if (c < nvec) {
      const float4 wv = __ldg(w + c), bv = __ldg(b + c);
      float4 r;
      r.x = (y[i].x - mean) * rstd * wv.x + bv.x;
      r.y = (y[i].y - mean) * rstd * wv.y + bv.y;
      r.z = (y[i].z - mean) * rstd * wv.z + bv.z;
      r.w = (y[i].w - mean) * rstd * wv.w + bv.w;
      __stcs(orow + c, r);
      if (out_hi) split_store(out_hi, out_lo, row * nvec + c, r);
    }
  }
}

template <int NV>
void launch_vec(const float* o, const float* x, const int32_t* type_row0, int T, const float* skip,
                const float* norm_w, const float* norm_b, const float* const* norm_wp, const float* const* norm_bp,
                const int32_t* perm, const int32_t* type_active, int64_t n_nodes, int d, float* out, uint2* out_hi,
                uint2* out_lo, cudaStream_t st) {
  const int warps_per_block = 8;
  unsigned grid = (unsigned)((n_nodes + warps_per_block - 1) / warps_per_block);
  k_update_epilogue_vec<NV><<<grid, warps_per_block * 32, 0, st>>>(o, x, type_row0, T, skip, norm_w, norm_b, norm_wp,
                                                                  norm_bp, perm, type_active, n_nodes, d, out, out_hi,
                                                                  out_lo);
}

}  // namespace

int hgt_update_epilogue_impl(const float* o, const float* x, const int32_t* type_row0, int32_t num_types,
                             const float* skip, const float* norm_w, const float* norm_b, const float* const* norm_wp,
                             const float* const* norm_bp, const int32_t* perm, const int32_t* type_active,
                             int64_t n_nodes, int32_t d, float* out, void* out_hi, void* out_lo, cudaStream_t st) {
  HGT_REQUIRE(d >= 1 && d <= 32 * kMaxPerLane, "hgt_update_epilogue: d=%d unsupported (max %d)", d,
              32 * kMaxPerLane);
  HGT_REQUIRE((norm_w == nullptr) == (norm_b == nullptr) && (norm_wp == nullptr) == (norm_bp == nullptr),
              "hgt_update_epilogue: LayerNorm weight and bias must go together");
  if (n_nodes == 0) return 0;
  // with pointer tables the per-type vectors are separate nn.LayerNorm parameters: torch allocations, 16-byte aligned
  const bool aligned = (d % 4 == 0) && ((reinterpret_cast<uintptr_t>(o) | reinterpret_cast<uintptr_t>(x) |
                                        reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(norm_w) |
                                        reinterpret_cast<uintptr_t>(norm_b)) % 16 == 0);
  HGT_REQUIRE((out_hi != nullptr) == (out_lo != nullptr), "hgt_update_epilogue: out_hi/out_lo must go together");
  HGT_REQUIRE(out_hi == nullptr || (aligned && d % 8 == 0 && perm == nullptr && type_active == nullptr),
              "hgt_update_epilogue: the split output needs d %% 8 == 0, 16-byte aligned buffers and identity row order");
  uint2* hi2 = reinterpret_cast<uint2*>(out_hi);
  uint2* lo2 = reinterpret_cast<uint2*>(out_lo);
  if (aligned && d <= 1024) {
    const int nv = (d / 4 + 31) / 32;
    if (nv <= 1) launch_vec<1>(o, x, type_row0, num_types, skip, norm_w, norm_b, norm_wp, norm_bp, perm, type_active, n_nodes, d, out, hi2, lo2, st);
    else if (nv <= 2) launch_vec<2>(o, x, type_row0, num_types, skip, norm_w, norm_b, norm_wp, norm_bp, perm, type_active, n_nodes, d, out, hi2, lo2, st);
    else if (nv <= 4) launch_vec<4>(o, x, type_row0, num_types, skip, norm_w, norm_b, norm_wp, norm_bp, perm, type_active, n_nodes, d, out, hi2, lo2, st);
    else launch_vec<8>(o, x, type_row0, num_types, skip, norm_w, norm_b, norm_wp, norm_bp, perm, type_active, n_nodes, d, out, hi2, lo2, st);
    HGT_LAUNCH_CHECK();
    return 0;
  }
  const int warps_per_block = 8;
  unsigned grid = (unsigned)((n_nodes + warps_per_block - 1) / warps_per_block);
  k_update_epilogue<<<grid, warps_per_block * 32, 0, st>>>(o, x, type_row0, num_types, skip, norm_w, norm_b, norm_wp,
                                                           norm_bp, perm, type_active, n_nodes, d, out);
  HGT_LAUNCH_CHECK();
  return 0;
}

extern "C" int hgt_update_epilogue(const float* o, const float* x, const int32_t* type_row0, int32_t num_types,
                                   const float* skip, const float* norm_w, const float* norm_b,
                                   const int32_t* perm, const int32_t* type_active, int64_t n_nodes, int32_t d,
                                   float* out, void* out_hi, void* out_lo, void* stream_) {
  return hgt_update_epilogue_impl(o, x, type_row0, num_types, skip, norm_w, norm_b, nullptr, nullptr, perm,
                                  type_active, n_nodes, d, out, out_hi, out_lo, (cudaStream_t)stream_);
}
