// Backward of the typed (per-node-type) linear layers — hgt_typed_linear_bwd.
//
// Forward (linear.cu / linear_tc.cu):  out[cblock c of group g][m, n] = sum_k A[a_row0_g + m, k] * W[w_row0_g + c*width + n, k] + b
// Backward, for the same group / column-block tables:
//   dA[a_row0_g + m, k]            = sum_c sum_n dOut_c[m, n] * W[w_row0_g + c*width + n, k]      ("dX":  K = n_cblocks * width)
//   dW[w_row0_g + c*width + n, k] += sum_m dOut_c[m, n] * A[a_row0_g + m, k]                      ("dW":  K = rows of the group)
//   db[w_row0_g + c*width + n]    += sum_m dOut_c[m, n]
// The reference gets these from autograd over per-edge nn.Linear calls (conv.py:96-104,125; OAG/train_paper_field.py:249).
//
// Tensor-core path (tcgen05, sm_100a): the same split-bf16 x3 scheme as the forward (x = hi + lo, three bf16 products
// in one fp32 TMEM accumulator):
//   k_act_split / k_split_colsum   fp32 -> bf16 hi/lo (optionally gelu first); the dOut split pass also produces db
//   k_lin_dx_tc   one 128 x BN tile of dA per CTA; K runs over (column block, 64-wide k-block); A operand = dOut tiles
//                 (K-major), B operand = W^T (a transposed, zero-padded bf16 split of the small weight matrix);
//                 epilogue: optional `+= dA`, optional `* gelu'(aux)` (the gelu in front of the a_linears, conv.py:119)
//   k_lin_dw_tc   dW tile [128 of width] x [BN of K_in] per CTA, reduction over a chunk of the group's rows; both operands
//                 are MN-major (the reduction index is the row index): TMA boxes {64 columns, 64 rows}, SWIZZLE_128B,
//                 tcgen05 MN-major descriptors; partial tiles are added with red.global.add.v4.f32
// Every (group, column block) gets its own tensor map (tight row extents => rows past the group are zero-filled by TMA, so the
// reduction never sees a neighbour's rows); the maps live in the workspace (global memory).
// SIMT fp32 path for shapes the tensor cores cannot take (width % 8, K % 16, overlapping groups such as the RTE tables).
#include <cuda.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <utility>
#include <vector>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace {

using namespace tcp;

constexpr int kMaxGroups = 64;
constexpr int BK = 64;                  // 64 bf16 = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int BW_THREADS = 192;         // warp 0: TMA, warp 1: MMA + TMEM, warps 2-5: epilogue
constexpr uint32_t ATOM_BYTES = 64 * 128;   // one {64 x 64} bf16 TMA box

// Tensor maps are read from global memory (written by a host copy earlier on the stream): acquire them for the TMA proxy.
__device__ __forceinline__ void map_acquire(const CUtensorMap* m) {
  asm volatile("fence.proxy.tensormap::generic.acquire.gpu [%0], 128;" ::"l"(m) : "memory");
}

__device__ __forceinline__ float gelu_grad(float x) {
  // d/dx [0.5 x (1 + erf(x / sqrt 2))]
  return 0.5f * (1.0f + erff(x * 0.70710678118654752440f)) + x * 0.39894228040143267794f * __expf(-0.5f * x * x);
}

// ---- fp32 [rows, K] (row stride ld) -> act(x) as fp32 and/or the bf16 hi/lo split [rows, Kp] -------------------------
__global__ void k_act_split(const float* __restrict__ in, int64_t ld, int64_t rows, int K, int Kp, int act,
                            float* __restrict__ out_f32, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  const int vec_per_row = Kp / 4;
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= rows * vec_per_row) return;
  const int64_t r = i / vec_per_row;
  const int c = (int)(i - r * vec_per_row) * 4;
  float v[4];
  const float* src = in + r * ld + c;
  if (c + 3 < K && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
    const float4 t = *reinterpret_cast<const float4*>(src);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = (c + j < K) ? src[j] : 0.f;
  }
  if (act == 1) {
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = hgt_gelu_erf(v[j]);
  }
  if (out_f32) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (c + j < K) out_f32[r * K + c + j] = v[j];
  }
  if (hi) hgt_split_bf16x4(v, reinterpret_cast<uint2*>(hi + r * Kp + c), reinterpret_cast<uint2*>(lo + r * Kp + c));
}

// ---- W [w_rows, K] -> W^T split, block-padded:  WT[k, blk*wpad + n] = W[blk*width + n, k], zero for n >= width ----------
__global__ void k_wt_split(const float* __restrict__ W, int64_t w_rows, int K, int width, int wpad, int64_t wt_cols,
                           __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)K * wt_cols) return;
  const int k = (int)(i / wt_cols);
  const int64_t col = i - (int64_t)k * wt_cols;
  const int64_t blk = col / wpad;
  const int n = (int)(col - blk * wpad);
  float v = 0.f;
  const int64_t wr = blk * width + n;
  if (n < width && wr < w_rows) v = W[wr * K + k];
  hgt_split_bf16(v, hi[i], lo[i]);
}

// ---- dOut split pass + bias gradient ---------------------------------------------------------------------------------
struct GcTask {            // one (group, column block)
  int64_t out_off, ld, rows, a_row0;
  int32_t w_row;           // first W row of this column block
  int32_t has_bias;
  int32_t first_unit;      // scheduling prefix (meaning depends on the kernel)
  int32_t n_chunks;
  int32_t map_dout;        // index of the dOut hi map (lo = +1)
  int32_t map_x;           // index of the group's A hi map (lo = +1)
  int32_t group, wt_col0;  // wt_col0: first column of this block inside W^T
};

// One CTA = one task x SPLIT_ROWS rows.  Thread (cx, ry): float4 column cx*4, rows ry, ry+RY, ...; column sums are reduced
// across ry in shared memory and added to db with one atomic per column and CTA.
constexpr int SPLIT_ROWS = 256;
__global__ void __launch_bounds__(256)
k_split_colsum(const float* __restrict__ dout, const GcTask* __restrict__ tasks, int n_tasks, int width,
               __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, float* __restrict__ db) {
  __shared__ float red[256 * 4];
  int unit = blockIdx.x, t = 0;
  while (t + 1 < n_tasks && unit >= tasks[t + 1].first_unit) ++t;
  const GcTask tk = tasks[t];
  const int64_t r0 = (int64_t)(unit - tk.first_unit) * SPLIT_ROWS;
  const int64_t r1 = min(tk.rows, r0 + SPLIT_ROWS);
  const int vecs = width / 4;                       // width % 4 == 0 on this path
  const int cxn = min(vecs, 256);                   // threads along columns
  const int ryn = 256 / cxn;
  const int cx = threadIdx.x % cxn, ry = threadIdx.x / cxn;
  for (int base = 0; base < vecs; base += cxn) {              // uniform trip count (barriers inside)
    const int c0 = base + cx;
    float s[4] = {0.f, 0.f, 0.f, 0.f};
    if (ry < ryn && c0 < vecs) {
      for (int64_t r = r0 + ry; r < r1; r += ryn) {
        const int64_t off = tk.out_off + r * tk.ld + c0 * 4;
        const float4 v4 = *reinterpret_cast<const float4*>(dout + off);
        const float v[4] = {v4.x, v4.y, v4.z, v4.w};
        hgt_split_bf16x4(v, reinterpret_cast<uint2*>(hi + off), reinterpret_cast<uint2*>(lo + off));
#pragma unroll
        for (int j = 0; j < 4; ++j) s[j] += v[j];
      }
    }
    if (db && tk.has_bias) {
#pragma unroll
      for (int j = 0; j < 4; ++j) red[threadIdx.x * 4 + j] = s[j];
      __syncthreads();
      if (ry == 0 && c0 < vecs) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float a = 0.f;
          for (int y = 0; y < ryn; ++y) a += red[(y * cxn + cx) * 4 + j];
          atomicAdd(db + tk.w_row + c0 * 4 + j, a);
        }
      }
      __syncthreads();
    }
  }
}

// ---- dX: dA tile = sum over (column block, k-block) of dOut tile x W^T tile --------------------------------------------
struct DxSched {
  int32_t first_tile[kMaxGroups + 1];
  int32_t n_tiles_n;
  int32_t bn_box;            // rows of the W^T TMA box (n-tile width in shared memory)
};

__global__ void __launch_bounds__(BW_THREADS, 1)
k_lin_dx_tc(const CUtensorMap* __restrict__ maps, int map_wt, const GcTask* __restrict__ tasks,
            const int32_t* __restrict__ group_task0, const hgt_lin_group* __restrict__ groups, int n_groups, int K_in,
            int width, float* __restrict__ dA, int accumulate, const float* __restrict__ gelu_aux, DxSched sc) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = smem_dyn + ((1024u - (s_u32(smem_dyn) & 1023u)) & 1023u);
  constexpr int STAGES = 2;
  const uint32_t a_bytes = 128 * BK * 2;                       // 16 KB (two 64-row boxes)
  const uint32_t b_bytes = (uint32_t)sc.bn_box * BK * 2;
  const uint32_t stage_bytes = 2 * a_bytes + 2 * b_bytes;      // A_hi, A_lo, B_hi, B_lo
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)STAGES * stage_bytes);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int tile = blockIdx.x, g = 0;
  while (g + 1 < n_groups && tile >= sc.first_tile[g + 1]) ++g;
  const hgt_lin_group grp = groups[g];
  const int local = tile - sc.first_tile[g];
  const int mt = local / sc.n_tiles_n, nt = local - mt * sc.n_tiles_n;
  const int64_t m0 = (int64_t)mt * 128;
  const int n0 = nt * 256;
  const int bn = min(256, K_in - n0);                           // multiple of 16
  const int kb_per_c = (width + BK - 1) / BK;
  const int total_iters = grp.n_cblocks * kb_per_c;
  const int task0 = group_task0[g];

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(s_u32(&full_bar[s]), 1);
      mbar_init(s_u32(&empty_bar[s]), 1);
    }
    mbar_init(s_u32(tmem_full_bar), 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc<1>(s_u32(tmem_ptr_smem), 256u);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    if (lane == 0) {
      const CUtensorMap* m_wt_hi = maps + map_wt;
      const CUtensorMap* m_wt_lo = maps + map_wt + 1;
      map_acquire(m_wt_hi);
      map_acquire(m_wt_lo);
      for (int c = 0; c < grp.n_cblocks; ++c) {
        map_acquire(maps + tasks[task0 + c].map_dout);
        map_acquire(maps + tasks[task0 + c].map_dout + 1);
      }
      for (int it = 0; it < total_iters; ++it) {
        const int s = it % STAGES;
        const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
        mbar_wait(s_u32(&empty_bar[s]), ph ^ 1u);
        const int c = it / kb_per_c, kb = it - c * kb_per_c;
        const GcTask tk = tasks[task0 + c];
        const CUtensorMap* m_hi = maps + tk.map_dout;
        const CUtensorMap* m_lo = m_hi + 1;
        const uint32_t bar = s_u32(&full_bar[s]);
        const uint32_t sa = s_u32(smem + (size_t)s * stage_bytes);
        mbar_expect_tx(bar, stage_bytes);
        tma_load_2d(sa, m_hi, kb * BK, (int)m0, bar);
        tma_load_2d(sa + ATOM_BYTES, m_hi, kb * BK, (int)m0 + 64, bar);
        tma_load_2d(sa + a_bytes, m_lo, kb * BK, (int)m0, bar);
        tma_load_2d(sa + a_bytes + ATOM_BYTES, m_lo, kb * BK, (int)m0 + 64, bar);
        tma_load_2d(sa + 2 * a_bytes, m_wt_hi, tk.wt_col0 + kb * BK, n0, bar);
        tma_load_2d(sa + 2 * a_bytes + b_bytes, m_wt_lo, tk.wt_col0 + kb * BK, n0, bar);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = idesc_bf16(128, bn, false, false);
      for (int it = 0; it < total_iters; ++it) {
        const int s = it % STAGES;
        const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
        mbar_wait(s_u32(&full_bar[s]), ph);
        tc_fence_after();
        const uint32_t sa = s_u32(smem + (size_t)s * stage_bytes);
        const uint64_t a_hi = desc_k_sw128(sa), a_lo = desc_k_sw128(sa + a_bytes);
        const uint64_t b_hi = desc_k_sw128(sa + 2 * a_bytes), b_lo = desc_k_sw128(sa + 2 * a_bytes + b_bytes);
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) {
          const uint64_t o = (uint64_t)(2 * k);                 // +32 bytes inside the swizzle row
          umma_bf16_ss(tmem_base, a_hi + o, b_hi + o, idesc, (it > 0 || k > 0) ? 1u : 0u);
          umma_bf16_ss(tmem_base, a_hi + o, b_lo + o, idesc, 1u);
          umma_bf16_ss(tmem_base, a_lo + o, b_hi + o, idesc, 1u);
        }
        umma_commit(s_u32(&empty_bar[s]));
      }
      umma_commit(s_u32(tmem_full_bar));
    }
  } else {
    const int lg = warp & 3;                                     // TMEM lane quarter this warp may read
    const int row = lg * 32 + lane;
    mbar_wait(s_u32(tmem_full_bar), 0);
    tc_fence_after();
    const bool row_ok = total_iters > 0 && m0 + row < grp.m;
    const int64_t grow = grp.a_row0 + m0 + row;
    float* orow = dA + grow * K_in + n0;
    const float* xrow = gelu_aux ? gelu_aux + grow * K_in + n0 : nullptr;
    for (int c = 0; c < bn; c += 16) {
      uint32_t r[16];
      tmem_ld16(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)c, r);
      tmem_ld_wait();
      if (row_ok) {
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          float4 v = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]),
                                 __uint_as_float(r[j + 3]));
          if (xrow) {
            const float4 x = *reinterpret_cast<const float4*>(xrow + c + j);
            v.x *= gelu_grad(x.x); v.y *= gelu_grad(x.y); v.z *= gelu_grad(x.z); v.w *= gelu_grad(x.w);
          }
          if (accumulate) {
            const float4 o = *reinterpret_cast<const float4*>(orow + c + j);
            v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
          }
          *reinterpret_cast<float4*>(orow + c + j) = v;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tmem_dealloc<1>(tmem_base, 256u);
  }
}

// ---- dW: [128 rows of the column block] x [BN columns of K_in] += dOut_c^T A over a chunk of rows ---------------------
__global__ void __launch_bounds__(BW_THREADS, 1)
k_lin_dw_tc(const CUtensorMap* __restrict__ maps, const GcTask* __restrict__ tasks, int n_tasks, int K_in, int width,
            int m_tiles, int n_tiles, int chunk_rows, float* __restrict__ dW) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = smem_dyn + ((1024u - (s_u32(smem_dyn) & 1023u)) & 1023u);
  constexpr int STAGES = 2;
  const uint32_t a_bytes = 2 * ATOM_BYTES;                      // dOut: 128 columns = 2 atoms of {64 cols x 64 rows}
  const int n_atoms = min(4, (K_in + 63) / 64);
  const uint32_t b_bytes = (uint32_t)n_atoms * ATOM_BYTES;      // A: up to 256 columns
  const uint32_t stage_bytes = 2 * a_bytes + 2 * b_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)STAGES * stage_bytes);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int unit = blockIdx.x, t = 0;
  while (t + 1 < n_tasks && unit >= tasks[t + 1].first_unit) ++t;
  const GcTask tk = tasks[t];
  int local = unit - tk.first_unit;
  const int chunk = local / (m_tiles * n_tiles);
  local -= chunk * m_tiles * n_tiles;
  const int mt = local / n_tiles, nt = local - mt * n_tiles;
  const int n0 = nt * 256;
  const int bn = min(256, K_in - n0);                            // multiple of 16
  const int atoms_here = (bn + 63) / 64;
  const int64_t r0 = (int64_t)chunk * chunk_rows;
  const int64_t r1 = min(tk.rows, r0 + chunk_rows);
  const int total_iters = (int)((r1 - r0 + BK - 1) / BK);

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(s_u32(&full_bar[s]), 1);
      mbar_init(s_u32(&empty_bar[s]), 1);
    }
    mbar_init(s_u32(tmem_full_bar), 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc<1>(s_u32(tmem_ptr_smem), 256u);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    if (lane == 0) {
      const CUtensorMap* d_hi = maps + tk.map_dout;
      const CUtensorMap* d_lo = d_hi + 1;
      const CUtensorMap* x_hi = maps + tk.map_x;
      const CUtensorMap* x_lo = x_hi + 1;
      map_acquire(d_hi); map_acquire(d_lo); map_acquire(x_hi); map_acquire(x_lo);
      const uint32_t tx = 2 * a_bytes + 2 * (uint32_t)atoms_here * ATOM_BYTES;
      for (int it = 0; it < total_iters; ++it) {
        const int s = it % STAGES;
        const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
        mbar_wait(s_u32(&empty_bar[s]), ph ^ 1u);
        const int row = (int)(r0 + (int64_t)it * BK);
        const uint32_t bar = s_u32(&full_bar[s]);
        const uint32_t sa = s_u32(smem + (size_t)s * stage_bytes);
        mbar_expect_tx(bar, tx);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          tma_load_2d(sa + j * ATOM_BYTES, d_hi, mt * 128 + j * 64, row, bar);
          tma_load_2d(sa + a_bytes + j * ATOM_BYTES, d_lo, mt * 128 + j * 64, row, bar);
        }
        for (int j = 0; j < atoms_here; ++j) {
          tma_load_2d(sa + 2 * a_bytes + j * ATOM_BYTES, x_hi, n0 + j * 64, row, bar);
          tma_load_2d(sa + 2 * a_bytes + b_bytes + j * ATOM_BYTES, x_lo, n0 + j * 64, row, bar);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = idesc_bf16(128, bn, true, true);
      for (int it = 0; it < total_iters; ++it) {
        const int s = it % STAGES;
        const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
        mbar_wait(s_u32(&full_bar[s]), ph);
        tc_fence_after();
        const uint32_t sa = s_u32(smem + (size_t)s * stage_bytes);
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) {
          const uint32_t ko = (uint32_t)k * UMMA_K * 128;          // 16 k-rows of 128 bytes
          const uint64_t a_hi = desc_mn_sw128(sa + ko, ATOM_BYTES);
          const uint64_t a_lo = desc_mn_sw128(sa + a_bytes + ko, ATOM_BYTES);
          const uint64_t b_hi = desc_mn_sw128(sa + 2 * a_bytes + ko, ATOM_BYTES);
          const uint64_t b_lo = desc_mn_sw128(sa + 2 * a_bytes + b_bytes + ko, ATOM_BYTES);
          umma_bf16_ss(tmem_base, a_hi, b_hi, idesc, (it > 0 || k > 0) ? 1u : 0u);
          umma_bf16_ss(tmem_base, a_hi, b_lo, idesc, 1u);
          umma_bf16_ss(tmem_base, a_lo, b_hi, idesc, 1u);
        }
        umma_commit(s_u32(&empty_bar[s]));
      }
      umma_commit(s_u32(tmem_full_bar));
    }
  } else {
    const int lg = warp & 3;
    const int row = lg * 32 + lane;                                // row of the dW tile = column of the dOut block
    mbar_wait(s_u32(tmem_full_bar), 0);
    tc_fence_after();
    const bool row_ok = total_iters > 0 && mt * 128 + row < width;
    float* wrow = dW + ((int64_t)tk.w_row + mt * 128 + row) * K_in + n0;
    for (int c = 0; c < bn; c += 16) {
      uint32_t r[16];
      tmem_ld16(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)c, r);
      tmem_ld_wait();
      if (row_ok) {
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(wrow + c + j), "f"(__uint_as_float(r[j])),
                       "f"(__uint_as_float(r[j + 1])), "f"(__uint_as_float(r[j + 2])), "f"(__uint_as_float(r[j + 3]))
                       : "memory");
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tmem_dealloc<1>(tmem_base, 256u);
  }
}

// ---- SIMT fp32 fallbacks ------------------------------------------------------------------------------------------------
// dA[a_row0 + m, k] (+)= sum_c sum_n dOut_c[m, n] * W[w_row + n, k].  One thread per (m, k); atomicAdd because groups may
// share A rows (the RTE tables: every <type, relation> pair projects the same 240-row table).
__global__ void k_lin_dx_simt(const float* __restrict__ dout, const float* __restrict__ W, const GcTask* __restrict__ tasks,
                              const int32_t* __restrict__ group_task0, const hgt_lin_group* __restrict__ groups,
                              int n_groups, const int64_t* __restrict__ group_first, int K_in, int width,
                              const float* __restrict__ gelu_aux, float* __restrict__ dA) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int g = 0;
  while (g + 1 < n_groups && i >= group_first[g + 1]) ++g;
  if (i >= group_first[n_groups]) return;
  const hgt_lin_group grp = groups[g];
  const int64_t li = i - group_first[g];
  const int64_t m = li / K_in;
  const int k = (int)(li - m * K_in);
  float acc = 0.f;
  for (int c = 0; c < grp.n_cblocks; ++c) {
    const GcTask tk = tasks[group_task0[g] + c];
    const float* drow = dout + tk.out_off + m * tk.ld;
    const float* wcol = W + (int64_t)tk.w_row * K_in + k;
    for (int n = 0; n < width; ++n) acc = fmaf(drow[n], wcol[(int64_t)n * K_in], acc);
  }
  const int64_t o = (grp.a_row0 + m) * K_in + k;
  if (gelu_aux) acc *= gelu_grad(gelu_aux[o]);
  atomicAdd(dA + o, acc);
}

// dW[w_row + n, k] += sum_m dOut_c[m, n] * A[a_row0 + m, k];  db[w_row + n] += sum_m dOut_c[m, n].
// One CTA = one task x (32 n) x (32 k) x a chunk of rows; 256 threads, 4 outputs each.
constexpr int DW_SIMT_ROWS = 2048;
__global__ void __launch_bounds__(256)
k_lin_dw_simt(const float* __restrict__ dout, const float* __restrict__ A, int64_t lda, const GcTask* __restrict__ tasks,
              int n_tasks, int K_in, int width, int n_tiles, int k_tiles, float* __restrict__ dW, float* __restrict__ db) {
  __shared__ float sd[32][33], sa[32][33];
  int unit = blockIdx.x, t = 0;
  while (t + 1 < n_tasks && unit >= tasks[t + 1].first_unit) ++t;
  const GcTask tk = tasks[t];
  int local = unit - tk.first_unit;
  const int chunk = local / (n_tiles * k_tiles);
  local -= chunk * n_tiles * k_tiles;
  const int ntile = local / k_tiles, ktile = local - ntile * k_tiles;
  const int n0 = ntile * 32, k0 = ktile * 32;
  const int64_t r0 = (int64_t)chunk * DW_SIMT_ROWS, r1 = min(tk.rows, r0 + DW_SIMT_ROWS);
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;       // ty: 0..7
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  float bsum = 0.f;
  for (int64_t rb = r0; rb < r1; rb += 32) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int rr = ty + 8 * j;
      const int64_t r = rb + rr;
      float dv = 0.f, av = 0.f;
      if (r < r1) {
        if (n0 + tx < width) dv = dout[tk.out_off + r * tk.ld + n0 + tx];
        if (k0 + tx < K_in) av = A[(tk.a_row0 + r) * lda + k0 + tx];
      }
      sd[rr][tx] = dv;
      sa[rr][tx] = av;
    }
    __syncthreads();
#pragma unroll 8
    for (int rr = 0; rr < 32; ++rr) {
      const float a = sa[rr][tx];
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[j] = fmaf(sd[rr][ty + 8 * j], a, acc[j]);
    }
    if (ktile == 0 && ty == 0) {
      for (int rr = 0; rr < 32; ++rr) bsum += sd[rr][tx];
    }
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int n = n0 + ty + 8 * j;
    if (n < width && k0 + tx < K_in) atomicAdd(dW + ((int64_t)tk.w_row + n) * K_in + k0 + tx, acc[j]);
  }
  if (db && tk.has_bias && ktile == 0 && ty == 0 && n0 + tx < width) atomicAdd(db + tk.w_row + n0 + tx, bsum);
}

// ---- host helpers ---------------------------------------------------------------------------------------------------------
struct BwdLayout {
  bool tc;
  int Kp, wpad;
  int64_t a_rows, w_rows, wt_cols;
  int n_tasks;
  size_t off_maps, off_tasks, off_gt0, off_gfirst, off_dhi, off_dlo, off_ahi, off_alo, off_wthi, off_wtlo, total;
};

bool groups_overlap(const hgt_lin_group* h, int n) {
  for (int i = 0; i < n; ++i)
    for (int j = i + 1; j < n; ++j) {
      if (h[i].m == 0 || h[j].m == 0) continue;
      if (h[i].a_row0 < h[j].a_row0 + h[j].m && h[j].a_row0 < h[i].a_row0 + h[i].m) return true;
    }
  return false;
}

bool bwd_tc_ok(const hgt_lin_group* h_groups, int n_groups, const hgt_lin_cblock* h_cb, int K, int width, int64_t lda) {
  if (width % 8 || K % 16 || K < 64 || width < 16 || lda != K) return false;
  if (groups_overlap(h_groups, n_groups)) return false;
  int64_t rows = 0;
  for (int g = 0; g < n_groups; ++g) {
    rows += h_groups[g].m;
    for (int c = 0; c < h_groups[g].n_cblocks; ++c) {
      const hgt_lin_cblock& cb = h_cb[h_groups[g].cb_first + c];
      if (cb.out_off % 8 || cb.ld % 8) return false;
    }
  }
  return rows >= 512;                      // tiny problems (RTE tables, unit tests at c1 size) stay on the SIMT kernels
}

BwdLayout bwd_layout(const hgt_lin_group* h_groups, int n_groups, const hgt_lin_cblock* h_cb, int K, int width,
                     int64_t lda, int64_t dout_elems, bool have_dsplit, bool have_asplit, int impl) {
  BwdLayout L{};
  L.tc = impl == 2 || (impl == 0 && bwd_tc_ok(h_groups, n_groups, h_cb, K, width, lda));
  L.Kp = K;
  L.wpad = (width + BK - 1) / BK * BK;
  L.a_rows = 0;
  L.w_rows = 0;
  L.n_tasks = 0;
  for (int g = 0; g < n_groups; ++g) {
    L.a_rows = std::max<int64_t>(L.a_rows, h_groups[g].a_row0 + h_groups[g].m);
    L.w_rows = std::max<int64_t>(L.w_rows, (int64_t)h_groups[g].w_row0 + (int64_t)h_groups[g].n_cblocks * width);
    L.n_tasks += h_groups[g].n_cblocks;
  }
  L.wt_cols = (L.w_rows + width - 1) / width * L.wpad;
  size_t p = 0;
  auto take = [&](size_t bytes) { size_t o = p; p += hgt_align_up(bytes, 256); return o; };
  L.off_maps = take((size_t)(2 * L.n_tasks + 2 * n_groups + 2) * sizeof(CUtensorMap));
  L.off_tasks = take((size_t)std::max(L.n_tasks, 1) * sizeof(GcTask));
  L.off_gt0 = take((size_t)(n_groups + 1) * sizeof(int32_t));
  L.off_gfirst = take((size_t)(n_groups + 1) * sizeof(int64_t));
  if (L.tc) {
    L.off_dhi = take(have_dsplit ? 0 : (size_t)dout_elems * 2);
    L.off_dlo = take(have_dsplit ? 0 : (size_t)dout_elems * 2);
    L.off_ahi = take(have_asplit ? 0 : (size_t)L.a_rows * L.Kp * 2);
    L.off_alo = take(have_asplit ? 0 : (size_t)L.a_rows * L.Kp * 2);
    L.off_wthi = take((size_t)K * L.wt_cols * 2);
    L.off_wtlo = take((size_t)K * L.wt_cols * 2);
  }
  L.total = p + 256;
  return L;
}

}  // namespace

// k_act_split over [rows, K] into split rows of pitch Kp (a multiple of 4, >= K); also the forward GEMM's operand split.
int hgt_act_split_launch(const float* in, int64_t ld, int64_t rows, int K, int Kp, int act, float* out_f32,
                         __nv_bfloat16* hi, __nv_bfloat16* lo, cudaStream_t st) {
  if (rows == 0) return 0;
  const int64_t n = rows * (Kp / 4);
  k_act_split<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(in, ld, rows, K, Kp, act, out_f32, hi, lo);
  HGT_LAUNCH_CHECK();
  return 0;
}

extern "C" int hgt_act_split(const float* in, int64_t ld, int64_t rows, int32_t K, int32_t act, float* out_f32,
                             void* hi, void* lo, void* stream_) {
  HGT_REQUIRE(in && (out_f32 || (hi && lo)), "hgt_act_split: NULL argument");
  HGT_REQUIRE(act == 0 || act == 1, "hgt_act_split: act=%d (0 = identity, 1 = gelu)", act);
  HGT_REQUIRE(!hi || K % 8 == 0, "hgt_act_split: the bf16 split needs K %% 8 == 0 (K=%d)", K);
  return hgt_act_split_launch(in, ld, rows, K, (K + 3) / 4 * 4, act, out_f32, reinterpret_cast<__nv_bfloat16*>(hi),
                              reinterpret_cast<__nv_bfloat16*>(lo), (cudaStream_t)stream_);
}

extern "C" int hgt_typed_linear_bwd_workspace_bytes(const hgt_lin_group* h_groups, int32_t n_groups,
                                                    const hgt_lin_cblock* h_cblocks, int32_t K, int32_t cb_width,
                                                    int64_t lda, int64_t dout_elems, int32_t have_dout_split,
                                                    int32_t have_a_split, int32_t impl, size_t* out_bytes) {
  HGT_REQUIRE(out_bytes && (n_groups == 0 || (h_groups && h_cblocks)), "hgt_typed_linear_bwd_workspace_bytes: NULL argument");
  HGT_REQUIRE(n_groups >= 0 && n_groups <= kMaxGroups, "hgt_typed_linear_bwd: n_groups=%d exceeds %d", n_groups, kMaxGroups);
  *out_bytes = bwd_layout(h_groups, n_groups, h_cblocks, K, cb_width, lda, dout_elems, have_dout_split != 0,
                          have_a_split != 0, impl).total;
  return 0;
}

extern "C" int hgt_typed_linear_bwd(const float* dout, const void* dout_hi, const void* dout_lo, int64_t dout_elems,
                                    const float* A, int64_t lda, const void* a_hi_in, const void* a_lo_in,
                                    const float* W, int32_t K, int32_t cb_width, const hgt_lin_group* groups,
                                    const hgt_lin_group* h_groups, int32_t n_groups, const hgt_lin_cblock* h_cblocks,
                                    float* dA, int32_t accumulate_dA, const float* gelu_aux, float* dW, float* db,
                                    int32_t impl, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HGT_REQUIRE(n_groups >= 0 && n_groups <= kMaxGroups, "hgt_typed_linear_bwd: n_groups=%d exceeds %d", n_groups, kMaxGroups);
  HGT_REQUIRE(K > 0 && cb_width > 0 && W, "hgt_typed_linear_bwd: K=%d cb_width=%d", K, cb_width);
  if (n_groups == 0) return 0;
  HGT_REQUIRE(groups && h_groups && h_cblocks, "hgt_typed_linear_bwd: NULL group tables");
  const bool have_dsplit = dout_hi && dout_lo, have_asplit = a_hi_in && a_lo_in;
  HGT_REQUIRE(dout || have_dsplit, "hgt_typed_linear_bwd: neither dout nor its bf16 split given");
  const BwdLayout L = bwd_layout(h_groups, n_groups, h_cblocks, K, cb_width, lda, dout_elems, have_dsplit, have_asplit, impl);
  HGT_REQUIRE(workspace && workspace_bytes >= L.total, "hgt_typed_linear_bwd: workspace too small (%zu < %zu)",
              workspace_bytes, L.total);
  if (L.tc)
    HGT_REQUIRE(cb_width % 8 == 0 && K % 16 == 0 && K >= 64 && lda == K && !groups_overlap(h_groups, n_groups),
                "hgt_typed_linear_bwd: tensor-core path does not support K=%d cb_width=%d lda=%lld (or overlapping groups)",
                K, cb_width, (long long)lda);
  else
    HGT_REQUIRE(dout && (A || !dW), "hgt_typed_linear_bwd: the SIMT path needs fp32 dout and A");
  char* base = reinterpret_cast<char*>(hgt_align_up(reinterpret_cast<size_t>(workspace), 256));

  // ---- task table (one entry per group x column block) ----
  std::vector<GcTask> tasks(std::max(L.n_tasks, 1));
  std::vector<int32_t> gt0(n_groups + 1);
  std::vector<int64_t> gfirst(n_groups + 1);
  int nt = 0;
  int64_t elems = 0;
  for (int g = 0; g < n_groups; ++g) {
    gt0[g] = nt;
    gfirst[g] = elems;
    elems += h_groups[g].m * K;
    HGT_REQUIRE(h_groups[g].w_row0 % cb_width == 0, "hgt_typed_linear_bwd: w_row0=%d is not a multiple of cb_width=%d",
                h_groups[g].w_row0, cb_width);
    for (int c = 0; c < h_groups[g].n_cblocks; ++c, ++nt) {
      const hgt_lin_cblock& cb = h_cblocks[h_groups[g].cb_first + c];
      GcTask& t = tasks[nt];
      t.out_off = cb.out_off;
      t.ld = cb.ld;
      t.rows = h_groups[g].m;
      t.a_row0 = h_groups[g].a_row0;
      t.w_row = h_groups[g].w_row0 + c * cb_width;
      t.has_bias = h_groups[g].has_bias;
      t.first_unit = 0;
      t.n_chunks = 0;
      t.map_dout = 2 * nt;
      t.map_x = 2 * L.n_tasks + 2 * g;
      t.group = g;
      t.wt_col0 = (t.w_row / cb_width) * L.wpad;
      HGT_REQUIRE(dout_elems <= 0 || h_groups[g].m == 0 ||
                      cb.out_off + (h_groups[g].m - 1) * cb.ld + cb_width <= dout_elems,
                  "hgt_typed_linear_bwd: column block %d of group %d exceeds dout_elems", c, g);
    }
  }
  gt0[n_groups] = nt;
  gfirst[n_groups] = elems;
  GcTask* d_tasks = reinterpret_cast<GcTask*>(base + L.off_tasks);
  int32_t* d_gt0 = reinterpret_cast<int32_t*>(base + L.off_gt0);
  int64_t* d_gfirst = reinterpret_cast<int64_t*>(base + L.off_gfirst);
  auto upload_tasks = [&]() -> int {
    HGT_CHECK_CUDA(cudaMemcpyAsync(d_tasks, tasks.data(), (size_t)nt * sizeof(GcTask), cudaMemcpyHostToDevice, st));
    return 0;
  };
  HGT_CHECK_CUDA(cudaMemcpyAsync(d_gt0, gt0.data(), gt0.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  HGT_CHECK_CUDA(cudaMemcpyAsync(d_gfirst, gfirst.data(), gfirst.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  int rc;

  if (!L.tc) {
    // ---------------- SIMT fp32 path ----------------
    if (dA) {
      if (!accumulate_dA) HGT_CHECK_CUDA(cudaMemsetAsync(dA, 0, (size_t)L.a_rows * K * sizeof(float), st));
      if ((rc = upload_tasks())) return rc;
      if (elems > 0) {
        k_lin_dx_simt<<<(unsigned)((elems + 255) / 256), 256, 0, st>>>(dout, W, d_tasks, d_gt0, groups, n_groups, d_gfirst, K,
                                                                       cb_width, gelu_aux, dA);
        HGT_LAUNCH_CHECK();
      }
    }
    if (dW) {
      const int n_tiles = (cb_width + 31) / 32, k_tiles = (K + 31) / 32;
      int64_t units = 0;
      for (int t = 0; t < nt; ++t) {
        tasks[t].first_unit = (int32_t)units;
        tasks[t].n_chunks = (int32_t)((tasks[t].rows + DW_SIMT_ROWS - 1) / DW_SIMT_ROWS);
        units += (int64_t)tasks[t].n_chunks * n_tiles * k_tiles;
        HGT_REQUIRE(units < 2147483647ll, "hgt_typed_linear_bwd: too many units");
      }
      if ((rc = upload_tasks())) return rc;
      if (units > 0) {
        k_lin_dw_simt<<<(unsigned)units, 256, 0, st>>>(dout, A, lda, d_tasks, nt, K, cb_width, n_tiles, k_tiles, dW, db);
        HGT_LAUNCH_CHECK();
      }
    }
    return 0;
  }

  // ---------------- tensor-core path ----------------
  __nv_bfloat16* d_hi = have_dsplit ? reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(dout_hi))
                                    : reinterpret_cast<__nv_bfloat16*>(base + L.off_dhi);
  __nv_bfloat16* d_lo = have_dsplit ? reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(dout_lo))
                                    : reinterpret_cast<__nv_bfloat16*>(base + L.off_dlo);
  __nv_bfloat16* a_hi = have_asplit ? reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(a_hi_in))
                                    : reinterpret_cast<__nv_bfloat16*>(base + L.off_ahi);
  __nv_bfloat16* a_lo = have_asplit ? reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(a_lo_in))
                                    : reinterpret_cast<__nv_bfloat16*>(base + L.off_alo);
  __nv_bfloat16* wt_hi = reinterpret_cast<__nv_bfloat16*>(base + L.off_wthi);
  __nv_bfloat16* wt_lo = reinterpret_cast<__nv_bfloat16*>(base + L.off_wtlo);

  // 1. dOut split (+ db) unless the producer already split it
  if (!have_dsplit) {
    int64_t units = 0;
    for (int t = 0; t < nt; ++t) {
      tasks[t].first_unit = (int32_t)units;
      units += (tasks[t].rows + SPLIT_ROWS - 1) / SPLIT_ROWS;
      HGT_REQUIRE(units < 2147483647ll, "hgt_typed_linear_bwd: too many units");
    }
    if ((rc = upload_tasks())) return rc;
    if (units > 0) {
      k_split_colsum<<<(unsigned)units, 256, 0, st>>>(dout, d_tasks, nt, cb_width, d_hi, d_lo, db);
      HGT_LAUNCH_CHECK();
    }
  }
  // 2. A split (dW needs it) unless saved by the forward
  if (dW && !have_asplit && L.a_rows > 0) {
    HGT_REQUIRE(A, "hgt_typed_linear_bwd: dW needs A or its bf16 split");
    if ((rc = hgt_act_split_launch(A, lda, L.a_rows, K, K, 0, nullptr, a_hi, a_lo, st))) return rc;
  }
  // 3. W^T split (dX)
  if (dA) {
    const int64_t n = (int64_t)K * L.wt_cols;
    k_wt_split<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(W, L.w_rows, K, cb_width, L.wpad, L.wt_cols, wt_hi, wt_lo);
    HGT_LAUNCH_CHECK();
  }
  // 4. tensor maps: per task dOut hi/lo {cols = width, rows = m}; per group A hi/lo {cols = K, rows = m}; W^T hi/lo
  std::vector<CUtensorMap> maps(2 * nt + 2 * n_groups + 2);
  for (int t = 0; t < nt; ++t) {
    const int64_t off = tasks[t].out_off, rows = tasks[t].rows, ld = tasks[t].ld;
    if ((rc = hgt_make_tma_map_bf16(&maps[2 * t], d_hi + off, rows, cb_width, ld, 64))) return rc;
    if ((rc = hgt_make_tma_map_bf16(&maps[2 * t + 1], d_lo + off, rows, cb_width, ld, 64))) return rc;
  }
  for (int g = 0; g < n_groups; ++g) {
    const int64_t off = h_groups[g].a_row0 * K, rows = h_groups[g].m;
    if ((rc = hgt_make_tma_map_bf16(&maps[2 * nt + 2 * g], a_hi + off, rows, K, K, 64))) return rc;
    if ((rc = hgt_make_tma_map_bf16(&maps[2 * nt + 2 * g + 1], a_lo + off, rows, K, K, 64))) return rc;
  }
  const int map_wt = 2 * nt + 2 * n_groups;
  const int bn_box = K >= 256 ? 256 : K;
  if ((rc = hgt_make_tma_map_bf16(&maps[map_wt], wt_hi, K, L.wt_cols, L.wt_cols, bn_box))) return rc;
  if ((rc = hgt_make_tma_map_bf16(&maps[map_wt + 1], wt_lo, K, L.wt_cols, L.wt_cols, bn_box))) return rc;
  CUtensorMap* d_maps = reinterpret_cast<CUtensorMap*>(base + L.off_maps);
  HGT_CHECK_CUDA(cudaMemcpyAsync(d_maps, maps.data(), maps.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice, st));

  // 5. dX
  if (dA) {
    // rows that no group covers keep a zero gradient
    if (!accumulate_dA) {
      std::vector<std::pair<int64_t, int64_t>> iv;
      for (int g = 0; g < n_groups; ++g)
        if (h_groups[g].m > 0) iv.emplace_back(h_groups[g].a_row0, h_groups[g].a_row0 + h_groups[g].m);
      std::sort(iv.begin(), iv.end());
      int64_t pos = 0;
      for (auto& p : iv) {
        if (p.first > pos) HGT_CHECK_CUDA(cudaMemsetAsync(dA + pos * K, 0, (size_t)(p.first - pos) * K * sizeof(float), st));
        pos = std::max(pos, p.second);
      }
    }
    DxSched sc;
    sc.n_tiles_n = (K + 255) / 256;
    sc.bn_box = bn_box;
    int64_t total = 0;
    for (int g = 0; g < n_groups; ++g) {
      sc.first_tile[g] = (int32_t)total;
      total += (h_groups[g].m + 127) / 128 * sc.n_tiles_n;
      HGT_REQUIRE(total < 2147483647ll, "hgt_typed_linear_bwd: too many tiles");
    }
    sc.first_tile[n_groups] = (int32_t)total;
    if (total > 0) {
      const size_t smem = 1024 + 2 * (size_t)(2 * 128 * BK * 2 + 2 * bn_box * BK * 2) + 8 * 8 + 16;
      HGT_CHECK_CUDA(cudaFuncSetAttribute(k_lin_dx_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      // the task table for dX only needs map indices / wt_col0 (already set); first_unit is unused here
      if (have_dsplit && (rc = upload_tasks())) return rc;
      k_lin_dx_tc<<<(unsigned)total, BW_THREADS, smem, st>>>(d_maps, map_wt, d_tasks, d_gt0, groups, n_groups, K, cb_width,
                                                             dA, accumulate_dA, gelu_aux, sc);
      HGT_LAUNCH_CHECK();
    }
  }
  // 6. dW
  if (dW) {
    const int m_tiles = (cb_width + 127) / 128, n_tiles = (K + 255) / 256;
    // chunk the reduction so that the grid has a few waves of CTAs
    int64_t work = 0;
    for (int t = 0; t < nt; ++t) work += tasks[t].rows * m_tiles * n_tiles;
    int64_t chunk = work / (4 * (int64_t)hgt_sm_count());
    chunk = (chunk + BK - 1) / BK * BK;
    if (chunk < 1024) chunk = 1024;
    if (chunk > 32768) chunk = 32768;
    int64_t units = 0;
    for (int t = 0; t < nt; ++t) {
      tasks[t].first_unit = (int32_t)units;
      tasks[t].n_chunks = (int32_t)((tasks[t].rows + chunk - 1) / chunk);
      units += (int64_t)tasks[t].n_chunks * m_tiles * n_tiles;
      HGT_REQUIRE(units < 2147483647ll, "hgt_typed_linear_bwd: too many units");
    }
    // the split / dX kernels enqueued above read the previous version of the table: stream order keeps them apart
    GcTask* d_tasks2 = d_tasks;
    HGT_CHECK_CUDA(cudaMemcpyAsync(d_tasks2, tasks.data(), (size_t)nt * sizeof(GcTask), cudaMemcpyHostToDevice, st));
    if (units > 0) {
      const int n_atoms = std::min(4, (K + 63) / 64);
      const size_t smem = 1024 + 2 * (size_t)(2 * 2 * ATOM_BYTES + 2 * n_atoms * ATOM_BYTES) + 8 * 8 + 16;
      HGT_CHECK_CUDA(cudaFuncSetAttribute(k_lin_dw_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      k_lin_dw_tc<<<(unsigned)units, BW_THREADS, smem, st>>>(d_maps, d_tasks2, nt, K, cb_width, m_tiles, n_tiles, (int)chunk,
                                                             dW);
      HGT_LAUNCH_CHECK();
    }
  }
  return 0;
}
