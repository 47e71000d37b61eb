// Fused HGT edge kernel (forward): for every destination i, over its in-edges e = (j -r-> i)
//     s[e,h]  = <Q[i,h,:], K'[j,r,h,:] (+ K'R[pair,dt,h,:])>              (conv.py:96-99, folded)
//     att[e,h] = exp(s - max_i) / (sum_i exp(s - max_i) + 1e-16)            (PyG softmax, conv.py:108)
//     agg[i]  = sum_e att[e,h] * V'[j,r,h,:] (+ V'R[pair,dt,h,:])           (conv.py:109-111 + scatter-add)
// in ONE pass over a destination-sorted CSR with an online (running max / running sum) softmax.
//
// Work decomposition: a warp owns a tile = a run of consecutive destinations (or a piece of one hub
// destination).  Inside the warp, lane = (head h, sub-lane) with LPH = 32/HP lanes per head
// (HP = n_heads rounded up to a power of two); each lane keeps NCH chunks of VEC floats of its head's
// slice of Q / K' / V' / acc in registers, so the per-head dot product is a log2(LPH)-step shuffle
// reduction of a single value and the softmax state (m, l) is per lane.
//
// Two data paths for the per-edge [K'|V'] row (2*d floats, contiguous):
//   variant 1 (LDG)  : vector loads straight into registers, EDGE_UNROLL rows in flight per warp.
//   variant 2 (TMA)  : cp.async.bulk (1-D bulk tensor copy, SASS UBLKCP) into a per-warp shared-memory
//                      ring with mbarrier transaction counting; the warp issues STAGES rows ahead.
// Roofline: HBM-bound; algorithmic bytes per edge = 2*d*4 (row) + 4 (kv_row) [+4 rte_row, +2*d*4 from L2]
// and per destination d*4 (Q) + d*4 (agg) + 4 (row_ptr).
//
// The tables may also be bf16 (hgt_edge_forward_bf16kv, inference): both variants take the row element type as a
// template parameter, lanes widen the row to fp32 as they load it, and everything after the load is the fp32 code.
// A bf16 row halves the per-edge bytes: 2*d*2 + 4.
#include <cuda_bf16.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace {

using namespace tcp;

constexpr int kWarpsPerCta = 16;
constexpr int kCtaThreads = kWarpsPerCta * 32;

struct EdgeParams {
  const float* q;
  const void* kv;            // [rows+1, 2d] of the kernel's row type (float or __nv_bfloat16)
  const void* kvr;           // same type; nullptr when !use_RTE
  const int32_t* row_ptr;
  const int32_t* kv_row;
  const int32_t* rte_row;
  const int32_t* csr_eid;
  const int32_t* tiles;
  int32_t n_tiles;           // exact count, or an upper bound when d_counts is given
  const int32_t* d_counts;   // optional device {n_tiles, n_split, n_hubs} written by hgt_plan_tiles (sync-free plans)
  const int32_t* type_row0;  // optional (with type_active): [T+2] row prefix per type
  const int32_t* type_active;// optional [T]: rows past type_active[t] inside type t are halo sources without an output
  int32_t T;
  int32_t d, H, DK, LPH, lph_shift;
  int32_t apply_gelu;
  float* agg_out;            // nullptr when only the split bf16 copy is wanted
  __nv_bfloat16* g_hi;       // optional: result as bf16 hi/lo split (operand of the tcgen05 a_linear GEMM)
  __nv_bfloat16* g_lo;
  float* att_out;            // nullptr unless requested
  float* stats_out;          // nullptr unless requested
  float* partial;            // [n_split][2*H + d]
  int32_t* tile_counter;
  int32_t stages;            // TMA variant
};

// sharded runs: destination `dst` lies past the active (owned) prefix of its node type
__device__ __forceinline__ bool dst_inactive(const EdgeParams& p, int dst) {
  int t = 0;
  while (t < p.T && dst >= p.type_row0[t + 1]) ++t;
  return t < p.T && dst - p.type_row0[t] >= p.type_active[t];
}

template <int VEC> struct VecT;
template <> struct VecT<1> { using type = float; };
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<4> { using type = float4; };

template <int VEC>
__device__ __forceinline__ void load_vec(float (&dst)[VEC], const float* p) {
  using V = typename VecT<VEC>::type;
  V v = *reinterpret_cast<const V*>(p);
  const float* f = reinterpret_cast<const float*>(&v);
#pragma unroll
  for (int i = 0; i < VEC; ++i) dst[i] = f[i];
}
template <int VEC>
__device__ __forceinline__ void load_vec_nc(float (&dst)[VEC], const float* p) {
  // streaming gather: read-only path, do not allocate in L1
  if constexpr (VEC == 4) {
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(dst[0]), "=f"(dst[1]), "=f"(dst[2]), "=f"(dst[3]) : "l"(p));
  } else if constexpr (VEC == 2) {
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(dst[0]), "=f"(dst[1]) : "l"(p));
  } else {
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(dst[0]) : "l"(p));
  }
}
// bf16 -> fp32 is exact: the bf16 bits are the upper half of the fp32 word
__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }

// VEC consecutive row elements, widened to fp32: load_row (cached; also shared memory) and load_row_nc (streaming gather)
template <int VEC>
__device__ __forceinline__ void load_row(float (&dst)[VEC], const float* p) { load_vec<VEC>(dst, p); }
template <int VEC>
__device__ __forceinline__ void load_row_nc(float (&dst)[VEC], const float* p) { load_vec_nc<VEC>(dst, p); }
template <int VEC>
__device__ __forceinline__ void widen_bf16(float (&dst)[VEC], const uint32_t* w) {
  if constexpr (VEC == 1) {
    dst[0] = bf16_lo(w[0]);
  } else {
#pragma unroll
    for (int i = 0; i < VEC / 2; ++i) { dst[2 * i] = bf16_lo(w[i]); dst[2 * i + 1] = bf16_hi(w[i]); }
  }
}
template <int VEC>
__device__ __forceinline__ void load_row(float (&dst)[VEC], const __nv_bfloat16* p) {
  uint32_t w[(VEC + 1) / 2];
  if constexpr (VEC == 4) {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    w[0] = u.x; w[1] = u.y;
  } else if constexpr (VEC == 2) {
    w[0] = *reinterpret_cast<const uint32_t*>(p);
  } else {
    w[0] = *reinterpret_cast<const unsigned short*>(p);
  }
  widen_bf16<VEC>(dst, w);
}
template <int VEC>
__device__ __forceinline__ void load_row_nc(float (&dst)[VEC], const __nv_bfloat16* p) {
  uint32_t w[(VEC + 1) / 2];
  if constexpr (VEC == 4) {
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(w[0]), "=r"(w[1]) : "l"(p));
  } else if constexpr (VEC == 2) {
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(w[0]) : "l"(p));
  } else {
    unsigned short h;
    asm volatile("ld.global.nc.L1::no_allocate.u16 %0, [%1];" : "=h"(h) : "l"(p));
    w[0] = h;
  }
  widen_bf16<VEC>(dst, w);
}

template <int VEC>
__device__ __forceinline__ void store_vec(float* p, const float (&src)[VEC]) {
  using V = typename VecT<VEC>::type;
  V v;
  float* f = reinterpret_cast<float*>(&v);
#pragma unroll
  for (int i = 0; i < VEC; ++i) f[i] = src[i];
  *reinterpret_cast<V*>(p) = v;
}

template <int VEC>
__device__ __forceinline__ void store_split_bf16(__nv_bfloat16* hi, __nv_bfloat16* lo, const float (&src)[VEC]) {
  __nv_bfloat16 h[VEC], l[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) hgt_split_bf16(src[i], h[i], l[i]);
  if constexpr (VEC == 4) {
    *reinterpret_cast<uint2*>(hi) = *reinterpret_cast<uint2*>(h);
    *reinterpret_cast<uint2*>(lo) = *reinterpret_cast<uint2*>(l);
  } else if constexpr (VEC == 2) {
    *reinterpret_cast<uint32_t*>(hi) = *reinterpret_cast<uint32_t*>(h);
    *reinterpret_cast<uint32_t*>(lo) = *reinterpret_cast<uint32_t*>(l);
  } else {
    hi[0] = h[0];
    lo[0] = l[0];
  }
}

__device__ __forceinline__ float head_reduce(float v, int lph) {
  // lanes of one head are an aligned group of `lph` (power of two) consecutive lanes
  for (int o = lph >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Per-lane softmax/accumulator state for the current destination.
template <int VEC, int NCH>
struct LaneState {
  float m, l;
  float acc[NCH][VEC];
  __device__ __forceinline__ void reset() {
    m = -INFINITY;
    l = 0.f;
#pragma unroll
    for (int t = 0; t < NCH; ++t)
#pragma unroll
      for (int v = 0; v < VEC; ++v) acc[t][v] = 0.f;
  }
};

// Element offset of chunk t of this lane inside a d-float row, or -1 when the chunk is padding.
struct LaneMap {
  int h, sub, lph, dk, base;
  bool head_ok;
  __device__ __forceinline__ LaneMap(const EdgeParams& p, int lane) {
    lph = p.LPH;
    h = lane >> p.lph_shift;
    sub = lane & (lph - 1);
    dk = p.DK;
    head_ok = h < p.H;
    base = h * dk;
  }
  template <int VEC>
  __device__ __forceinline__ int off(int t) const {
    int o = (sub + t * lph) * VEC;
    return (head_ok && o < dk) ? base + o : -1;
  }
};

template <int VEC, int NCH>
__device__ __forceinline__ void finalize_destination(const EdgeParams& p, const LaneMap& lm, int lane, int dst,
                                                      LaneState<VEC, NCH>& st, int seg_begin, int seg_end,
                                                      bool split_piece, int pslot) {
  if (split_piece) {
    // un-normalised partial result of a hub piece; merged by k_merge_partials
    float* w = p.partial + (int64_t)pslot * (2 * p.H + p.d);
    if (lm.head_ok && lm.sub == 0) { w[lm.h] = st.m; w[p.H + lm.h] = st.l; }
#pragma unroll
    for (int t = 0; t < NCH; ++t) {
      int o = lm.off<VEC>(t);
      if (o >= 0) store_vec<VEC>(w + 2 * p.H + o, st.acc[t]);
    }
    return;
  }
  const float inv = 1.0f / (st.l + 1e-16f);                  // PyG softmax denominator, conv.py:108
  float* orow = p.agg_out + (int64_t)dst * p.d;
#pragma unroll
  for (int t = 0; t < NCH; ++t) {
    int o = lm.off<VEC>(t);
    if (o >= 0) {
      float r[VEC];
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        float x = st.acc[t][v] * inv;
        r[v] = p.apply_gelu ? hgt_gelu_erf(x) : x;
      }
      if (p.agg_out) store_vec<VEC>(orow + o, r);
      if (p.g_hi) store_split_bf16<VEC>(p.g_hi + (int64_t)dst * p.d + o, p.g_lo + (int64_t)dst * p.d + o, r);
    }
  }
  if (p.stats_out && lm.head_ok && lm.sub == 0) {
    p.stats_out[(int64_t)dst * 2 * p.H + lm.h] = st.m;
    p.stats_out[(int64_t)dst * 2 * p.H + p.H + lm.h] = st.l;
  }
  if (p.att_out && lm.head_ok && lm.sub == 0) {
    // second pass over this lane's own raw scores (written by this same thread during the main pass)
    for (int c = seg_begin; c < seg_end; ++c) {
      float* a = p.att_out + (int64_t)p.csr_eid[c] * p.H + lm.h;
      *a = __expf(*a - st.m) * inv;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// variant 1: direct register gather
// ------------------------------------------------------------------------------------------------
template <typename KvT, int VEC, int NCH>
__global__ void __launch_bounds__(kCtaThreads, 1)
k_edge_fwd_ldg(EdgeParams p) {
  // rows in flight per warp: bounded by the register budget (2 * U * NCH * VEC floats of staging)
  constexpr int EDGE_UNROLL = (NCH * VEC >= 32) ? 1 : (NCH * VEC >= 16 ? 2 : 4);
  const int lane = threadIdx.x & 31;
  const LaneMap lm(p, lane);
  const bool rte = p.kvr != nullptr;
  const KvT* kv = static_cast<const KvT*>(p.kv);
  const KvT* kvr = static_cast<const KvT*>(p.kvr);
  const int64_t row_stride = 2 * (int64_t)p.d;
  int offs[NCH];
#pragma unroll
  for (int t = 0; t < NCH; ++t) offs[t] = lm.off<VEC>(t);

  const int n_tiles = p.d_counts ? p.d_counts[0] : p.n_tiles;
  for (;;) {
    int tile = 0;
    if (lane == 0) tile = atomicAdd(p.tile_counter, 1);
    tile = __shfl_sync(0xffffffffu, tile, 0);
    if (tile >= n_tiles) break;
    const int4 tl = reinterpret_cast<const int4*>(p.tiles)[tile];
    const bool split = tl.y < 0;
    const int d_begin = tl.x, d_end = split ? tl.x + 1 : tl.y;
    int seg_begin = tl.z;
    for (int dst = d_begin; dst < d_end; ++dst) {
      const int seg_end = split ? tl.w : p.row_ptr[dst + 1];
      if (p.type_active && seg_end == seg_begin && dst_inactive(p, dst)) continue;   // halo row: no output wanted
      LaneState<VEC, NCH> st;
      st.reset();
      if (seg_end > seg_begin) {
        float q[NCH][VEC];
        const float* qrow = p.q + (int64_t)dst * p.d;
#pragma unroll
        for (int t = 0; t < NCH; ++t) {
          if (offs[t] >= 0) load_vec<VEC>(q[t], qrow + offs[t]);
          else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) q[t][v] = 0.f;
          }
        }
        for (int c0 = seg_begin; c0 < seg_end; c0 += EDGE_UNROLL) {
          float kk[EDGE_UNROLL][NCH][VEC], vv[EDGE_UNROLL][NCH][VEC];
          int nb = min(EDGE_UNROLL, seg_end - c0);
#pragma unroll
          for (int u = 0; u < EDGE_UNROLL; ++u) {
            if (u < nb) {
              const KvT* row = kv + (int64_t)p.kv_row[c0 + u] * row_stride;
#pragma unroll
              for (int t = 0; t < NCH; ++t) {
                if (offs[t] >= 0) {
                  load_row_nc<VEC>(kk[u][t], row + offs[t]);
                  load_row_nc<VEC>(vv[u][t], row + p.d + offs[t]);
                } else {
#pragma unroll
                  for (int v = 0; v < VEC; ++v) { kk[u][t][v] = 0.f; vv[u][t][v] = 0.f; }
                }
              }
            }
          }
          if (rte) {
#pragma unroll
            for (int u = 0; u < EDGE_UNROLL; ++u) {
              if (u < nb) {
                const KvT* row = kvr + (int64_t)p.rte_row[c0 + u] * row_stride;
#pragma unroll
                for (int t = 0; t < NCH; ++t) {
                  if (offs[t] >= 0) {
                    float a[VEC], b[VEC];
                    load_row<VEC>(a, row + offs[t]);
                    load_row<VEC>(b, row + p.d + offs[t]);
#pragma unroll
                    for (int v = 0; v < VEC; ++v) { kk[u][t][v] += a[v]; vv[u][t][v] += b[v]; }
                  }
                }
              }
            }
          }
          float s[EDGE_UNROLL];
          float bmax = -INFINITY;
#pragma unroll
          for (int u = 0; u < EDGE_UNROLL; ++u) {
            float part = 0.f;
            if (u < nb) {
#pragma unroll
              for (int t = 0; t < NCH; ++t)
#pragma unroll
                for (int v = 0; v < VEC; ++v) part = fmaf(q[t][v], kk[u][t][v], part);
            }
            s[u] = head_reduce(part, lm.lph);
            if (u < nb) bmax = fmaxf(bmax, s[u]);
          }
          if (p.att_out && lm.head_ok && lm.sub == 0) {
#pragma unroll
            for (int u = 0; u < EDGE_UNROLL; ++u)
              if (u < nb) p.att_out[(int64_t)p.csr_eid[c0 + u] * p.H + lm.h] = s[u];
          }
          const float m_new = fmaxf(st.m, bmax);
          const float scale = __expf(st.m - m_new);
          float pw[EDGE_UNROLL];
          float psum = 0.f;
#pragma unroll
          for (int u = 0; u < EDGE_UNROLL; ++u) {
            pw[u] = (u < nb) ? __expf(s[u] - m_new) : 0.f;
            psum += pw[u];
          }
          st.l = st.l * scale + psum;
          st.m = m_new;
#pragma unroll
          for (int t = 0; t < NCH; ++t)
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
              float a = st.acc[t][v] * scale;
#pragma unroll
              for (int u = 0; u < EDGE_UNROLL; ++u)
                if (u < nb) a = fmaf(pw[u], vv[u][t][v], a);
              st.acc[t][v] = a;
            }
        }
      }
      finalize_destination<VEC, NCH>(p, lm, lane, dst, st, seg_begin, seg_end, split, split ? -tl.y - 1 : 0);
      seg_begin = seg_end;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// variant 2: bulk async copy (TMA engine) -> per-warp shared-memory ring
// ------------------------------------------------------------------------------------------------
template <typename KvT, int VEC, int NCH>
__global__ void __launch_bounds__(kCtaThreads, (VEC * NCH <= 4) ? 2 : 1)   // narrow rows (d_k <= 16): two CTAs per SM
k_edge_fwd_tma(EdgeParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const LaneMap lm(p, lane);
  const bool rte = p.kvr != nullptr;
  const int S = p.stages;
  const KvT* kv = static_cast<const KvT*>(p.kv);
  const KvT* kvr = static_cast<const KvT*>(p.kvr);
  const uint32_t row_bytes = 2u * (uint32_t)p.d * (uint32_t)sizeof(KvT);
  const uint32_t slot_bytes = rte ? 2u * row_bytes : row_bytes;
  const int64_t row_stride = 2 * (int64_t)p.d;
  // layout: [warps][S][slot_bytes] rows, then [warps][S] mbarriers
  unsigned char* ring = smem_raw + (size_t)warp * S * slot_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + (size_t)kWarpsPerCta * S * slot_bytes) + warp * S;
  if (lane == 0) {
    for (int s = 0; s < S; ++s) mbar_init(s_u32(&bars[s]), 1);
    fence_mbar_init();
  }
  __syncwarp();
  int offs[NCH];
#pragma unroll
  for (int t = 0; t < NCH; ++t) offs[t] = lm.off<VEC>(t);

  uint32_t it = 0;   // rows consumed so far by this warp (slot = it % S, parity = (it / S) & 1)

  const int n_tiles = p.d_counts ? p.d_counts[0] : p.n_tiles;
  for (;;) {
    int tile = 0;
    if (lane == 0) tile = atomicAdd(p.tile_counter, 1);
    tile = __shfl_sync(0xffffffffu, tile, 0);
    if (tile >= n_tiles) break;
    const int4 tl = reinterpret_cast<const int4*>(p.tiles)[tile];
    const bool split = tl.y < 0;
    const int d_begin = tl.x, d_end = split ? tl.x + 1 : tl.y;
    const int e0 = tl.z;
    const int e1 = tl.w;
    // index batches: lane holds kv_row[ibase + lane]; two batches give a 32..64 edge look-ahead window
    int ibase = e0;
    int idxA = (ibase + lane < e1) ? p.kv_row[ibase + lane] : 0;
    int idxB = (ibase + 32 + lane < e1) ? p.kv_row[ibase + 32 + lane] : 0;
    int ridxA = 0, ridxB = 0;
    if (rte) {
      ridxA = (ibase + lane < e1) ? p.rte_row[ibase + lane] : 0;
      ridxB = (ibase + 32 + lane < e1) ? p.rte_row[ibase + 32 + lane] : 0;
    }
    uint32_t issue_it = it;
    auto issue = [&](int c) {
      // all lanes participate in the shuffles; lane 0 arms the barrier and launches the copies
      while (c - ibase >= 32) {
        ibase += 32;
        idxA = idxB;
        idxB = (ibase + 32 + lane < e1) ? p.kv_row[ibase + 32 + lane] : 0;
        if (rte) {
          ridxA = ridxB;
          ridxB = (ibase + 32 + lane < e1) ? p.rte_row[ibase + 32 + lane] : 0;
        }
      }
      const int row = __shfl_sync(0xffffffffu, idxA, c - ibase);
      const int rrow = rte ? __shfl_sync(0xffffffffu, ridxA, c - ibase) : 0;
      const uint32_t slot = issue_it % S;
      if (lane == 0) {
        const uint32_t bar = s_u32(&bars[slot]);
        const uint32_t dst = s_u32(ring + (size_t)slot * slot_bytes);
        mbar_expect_tx(bar, slot_bytes);
        bulk_g2s(dst, kv + (int64_t)row * row_stride, row_bytes, bar);
        if (rte) bulk_g2s(dst + row_bytes, kvr + (int64_t)rrow * row_stride, row_bytes, bar);
      }
      ++issue_it;
    };
    const int n_pro = min(S, e1 - e0);
    for (int i = 0; i < n_pro; ++i) issue(e0 + i);

    int seg_begin = e0;
    for (int dst = d_begin; dst < d_end; ++dst) {
      const int seg_end = split ? e1 : p.row_ptr[dst + 1];
      if (p.type_active && seg_end == seg_begin && dst_inactive(p, dst)) continue;   // halo row: no output wanted
      LaneState<VEC, NCH> st;
      st.reset();
      if (seg_end > seg_begin) {
        float q[NCH][VEC];
        const float* qrow = p.q + (int64_t)dst * p.d;
#pragma unroll
        for (int t = 0; t < NCH; ++t) {
          if (offs[t] >= 0) load_vec<VEC>(q[t], qrow + offs[t]);
          else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) q[t][v] = 0.f;
          }
        }
        for (int c = seg_begin; c < seg_end; ++c) {
          const uint32_t slot = it % S;
          mbar_wait(s_u32(&bars[slot]), (it / S) & 1u);
          const KvT* srow = reinterpret_cast<const KvT*>(ring + (size_t)slot * slot_bytes);
          float kk[NCH][VEC], vv[NCH][VEC];
          float part = 0.f;
#pragma unroll
          for (int t = 0; t < NCH; ++t) {
            if (offs[t] >= 0) {
              load_row<VEC>(kk[t], srow + offs[t]);
              load_row<VEC>(vv[t], srow + p.d + offs[t]);
              if (rte) {
                float a[VEC], b[VEC];
                load_row<VEC>(a, srow + row_stride + offs[t]);
                load_row<VEC>(b, srow + row_stride + p.d + offs[t]);
#pragma unroll
                for (int v = 0; v < VEC; ++v) { kk[t][v] += a[v]; vv[t][v] += b[v]; }
              }
#pragma unroll
              for (int v = 0; v < VEC; ++v) part = fmaf(q[t][v], kk[t][v], part);
            } else {
#pragma unroll
              for (int v = 0; v < VEC; ++v) vv[t][v] = 0.f;
            }
          }
          ++it;
          __syncwarp();                                   // every lane has read the slot
          if (c + S < e1) issue(c + S);                   // refill it (row c+S maps to the same slot)
          const float s = head_reduce(part, lm.lph);
          if (p.att_out && lm.head_ok && lm.sub == 0) p.att_out[(int64_t)p.csr_eid[c] * p.H + lm.h] = s;
          const float m_new = fmaxf(st.m, s);
          const float scale = __expf(st.m - m_new);
          const float pw = __expf(s - m_new);
          st.l = st.l * scale + pw;
          st.m = m_new;
#pragma unroll
          for (int t = 0; t < NCH; ++t)
#pragma unroll
            for (int v = 0; v < VEC; ++v) st.acc[t][v] = fmaf(pw, vv[t][v], st.acc[t][v] * scale);
        }
      }
      finalize_destination<VEC, NCH>(p, lm, lane, dst, st, seg_begin, seg_end, split, split ? -tl.y - 1 : 0);
      seg_begin = seg_end;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// merge of hub pieces: one 1024-thread CTA per hub (hub list from hgt_plan_tiles).  The (max, sum, acc)
// partials of a hub's pieces are combined with the usual log-sum-exp rescaling; pieces are spread over the
// 32 warps so a hub cut into thousands of pieces (power-law graphs) still merges in microseconds.
// ------------------------------------------------------------------------------------------------
constexpr int kMergeThreads = 1024;

__global__ void __launch_bounds__(kMergeThreads)
k_merge_partials(EdgeParams p, const int32_t* __restrict__ hubs, int n_hubs_host) {
  const int n_hubs = p.d_counts ? p.d_counts[2] : n_hubs_host;
  __shared__ float s_M[32], s_L[32], s_inv[32];
  __shared__ float s_red[32][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int stride = 2 * p.H + p.d;
  for (int hb = blockIdx.x; hb < n_hubs; hb += gridDim.x) {
    const int dst = hubs[4 * hb], slot0 = hubs[4 * hb + 1], pieces = hubs[4 * hb + 2];
    const float* part = p.partial + (int64_t)slot0 * stride;
    // per head: M = max_k m_k, then L = sum_k l_k * exp(m_k - M)
    for (int h = warp; h < p.H; h += 32) {
      float mx = -INFINITY;
      for (int k = lane; k < pieces; k += 32) mx = fmaxf(mx, part[(int64_t)k * stride + h]);
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      float l = 0.f;
      for (int k = lane; k < pieces; k += 32) {
        const float* w = part + (int64_t)k * stride;
        l += w[p.H + h] * __expf(w[h] - mx);
      }
      for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
      if (lane == 0) { s_M[h] = mx; s_L[h] = l; s_inv[h] = 1.0f / (l + 1e-16f); }
    }
    __syncthreads();
    // columns in chunks of 32; warp w accumulates the pieces k = w, w+32, ...
    for (int c0 = 0; c0 < p.d; c0 += 32) {
      const int c = c0 + lane;
      float a = 0.f;
      if (c < p.d) {
        const int h = c / p.DK;
        const float M = s_M[h];
        for (int k = warp; k < pieces; k += 32) {
          const float* w = part + (int64_t)k * stride;
          a = fmaf(w[2 * p.H + c], __expf(w[h] - M), a);
        }
      }
      s_red[warp][lane] = a;
      __syncthreads();
      if (warp == 0 && c < p.d) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < 32; ++w) t += s_red[w][lane];
        t *= s_inv[c / p.DK];
        t = p.apply_gelu ? hgt_gelu_erf(t) : t;
        if (p.agg_out) p.agg_out[(int64_t)dst * p.d + c] = t;
        if (p.g_hi) hgt_split_bf16(t, p.g_hi[(int64_t)dst * p.d + c], p.g_lo[(int64_t)dst * p.d + c]);
      }
      __syncthreads();
    }
    if (p.stats_out && threadIdx.x < p.H) {
      p.stats_out[(int64_t)dst * 2 * p.H + threadIdx.x] = s_M[threadIdx.x];
      p.stats_out[(int64_t)dst * 2 * p.H + p.H + threadIdx.x] = s_L[threadIdx.x];
    }
    if (p.att_out) {
      const int seg_begin = p.row_ptr[dst], seg_end = p.row_ptr[dst + 1];
      const int64_t n = (int64_t)(seg_end - seg_begin) * p.H;
      for (int64_t i = threadIdx.x; i < n; i += kMergeThreads) {
        const int c = seg_begin + (int)(i / p.H), h = (int)(i % p.H);
        float* a = p.att_out + (int64_t)p.csr_eid[c] * p.H + h;
        *a = __expf(*a - s_M[h]) * s_inv[h];
      }
    }
    __syncthreads();
  }
}

template <typename KvT, int VEC, int NCH>
int launch_variant(const EdgeParams& p, int variant, int grid, size_t smem, cudaStream_t st) {
  if (variant == 1) {
    k_edge_fwd_ldg<KvT, VEC, NCH><<<grid, kCtaThreads, 0, st>>>(p);
  } else {
    static size_t configured = 0;            // per instantiation: raise the dynamic shared-memory limit once, not per launch
    if (smem > configured) {
      HGT_CHECK_CUDA(cudaFuncSetAttribute(k_edge_fwd_tma<KvT, VEC, NCH>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)smem));
      configured = smem;
    }
    k_edge_fwd_tma<KvT, VEC, NCH><<<grid, kCtaThreads, smem, st>>>(p);
  }
  HGT_LAUNCH_CHECK();
  return 0;
}

template <typename KvT, int VEC>
int dispatch_nch(const EdgeParams& p, int nch, int variant, int grid, size_t smem, cudaStream_t st) {
  switch (nch) {
    case 1: return launch_variant<KvT, VEC, 1>(p, variant, grid, smem, st);
    case 2: return launch_variant<KvT, VEC, 2>(p, variant, grid, smem, st);
    case 4: return launch_variant<KvT, VEC, 4>(p, variant, grid, smem, st);
    case 8: return launch_variant<KvT, VEC, 8>(p, variant, grid, smem, st);
  }
  hgt_set_error("hgt_edge_forward: internal: unsupported chunk count %d", nch);
  return 1;
}

}  // namespace

extern "C" int hgt_edge_workspace_bytes(int32_t n_split_tiles, int32_t d, int32_t n_heads, size_t* out_bytes) {
  HGT_REQUIRE(out_bytes, "hgt_edge_workspace_bytes: out_bytes is NULL");
  *out_bytes = 256 + sizeof(float) * (size_t)(n_split_tiles > 0 ? n_split_tiles : 0) * (2 * (size_t)n_heads + d);
  return 0;
}


// Shared host side of hgt_edge_forward (fp32 tables) and hgt_edge_forward_bf16kv (bf16 tables).
template <typename KvT>
static int edge_forward(const char* fn, const float* q, const void* kv, const void* kvr, const int32_t* row_ptr,
                        const int32_t* kv_row, const int32_t* rte_row, const int32_t* csr_eid, const int32_t* tiles,
                        int32_t n_tiles, int32_t n_split_tiles, const int32_t* hubs, int32_t n_hubs, int64_t n_nodes,
                        int32_t d, int32_t n_heads, int32_t apply_gelu, float* agg_out, float* att_out,
                        float* stats_out, void* g_hi, void* g_lo, void* workspace, size_t workspace_bytes,
                        int32_t variant, const int32_t* d_tile_counts, const int32_t* type_row0, int32_t num_types,
                        const int32_t* type_active, cudaStream_t st) {
  HGT_REQUIRE(n_heads >= 1 && n_heads <= 32, "%s: n_heads=%d unsupported (1..32)", fn, n_heads);
  HGT_REQUIRE(d % n_heads == 0, "%s: d=%d not divisible by n_heads=%d", fn, d, n_heads);
  HGT_REQUIRE((kvr != nullptr) == (rte_row != nullptr), "%s: kvr and rte_row must go together", fn);
  HGT_REQUIRE((g_hi != nullptr) == (g_lo != nullptr) && (agg_out != nullptr || g_hi != nullptr),
              "%s: need agg_out and/or the (g_hi, g_lo) pair", fn);
  HGT_REQUIRE(g_hi == nullptr || d % 8 == 0, "%s: split output needs d %% 8 == 0 (d=%d)", fn, d);
  size_t need = 0;
  hgt_edge_workspace_bytes(n_split_tiles, d, n_heads, &need);
  HGT_REQUIRE(workspace_bytes >= need, "%s: workspace too small (%zu < %zu)", fn, workspace_bytes, need);
  if (n_nodes == 0 || n_tiles == 0) return 0;

  EdgeParams p;
  p.q = q; p.kv = kv; p.kvr = kvr; p.row_ptr = row_ptr; p.kv_row = kv_row; p.rte_row = rte_row;
  p.csr_eid = csr_eid; p.tiles = tiles; p.n_tiles = n_tiles; p.d_counts = d_tile_counts; p.d = d;
  p.type_row0 = type_row0; p.type_active = (type_row0 && num_types > 0) ? type_active : nullptr; p.T = num_types; p.H = n_heads; p.DK = d / n_heads;
  int hp = 1, shift = 5;
  while (hp < n_heads) hp <<= 1;
  p.LPH = 32 / hp;
  for (shift = 0; (1 << shift) < p.LPH; ++shift) {}
  p.lph_shift = shift;
  p.apply_gelu = apply_gelu;
  p.agg_out = agg_out; p.att_out = att_out; p.stats_out = stats_out;
  p.g_hi = reinterpret_cast<__nv_bfloat16*>(g_hi); p.g_lo = reinterpret_cast<__nv_bfloat16*>(g_lo);
  p.tile_counter = reinterpret_cast<int32_t*>(workspace);
  p.partial = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + 256);

  // lane mapping: VEC floats per chunk, NCH chunks per lane
  int vec = 1;
  for (int v : {4, 2}) {
    if (p.DK % v == 0 && p.DK / v >= p.LPH) { vec = v; break; }
  }
  int chunks = (p.DK + vec * p.LPH - 1) / (vec * p.LPH);
  int nch = 1;
  while (nch < chunks) nch <<= 1;
  HGT_REQUIRE(nch <= 8, "%s: head width d_k=%d with %d heads needs %d chunks per lane (max 8)", fn, p.DK, n_heads,
              chunks);

  const int sms = hgt_sm_count();
  int grid = sms;
  size_t smem = 0;
  const size_t row_bytes = 2 * (size_t)d * sizeof(KvT);
  const size_t slot_bytes = kvr ? 2 * row_bytes : row_bytes;
  if (variant == 0) variant = 2;
  // narrow rows (one float4 per lane): the kernel is bound by per-destination latency, not by bytes in flight, so two
  // CTAs share an SM (32 warps) with half the ring each
  const bool two_ctas = vec * nch <= 4;
  if (variant == 2) {
    const size_t budget = two_ctas ? 100 * 1024 : 200 * 1024;
    int stages = (int)(budget / (kWarpsPerCta * slot_bytes));
    if (stages > 8) stages = 8;   // also for bf16 rows: a cap of 16 measured no faster (DESIGN.md 4.1)
    if (stages < 2 || row_bytes % 16 != 0) variant = 1;     // rows too wide / misaligned for the ring
    else {
      p.stages = stages;
      smem = (size_t)kWarpsPerCta * stages * (slot_bytes + 8);
    }
  }
  HGT_REQUIRE(variant == 1 || variant == 2, "%s: unknown variant %d", fn, variant);
  // persistent grid: one CTA per SM, never more CTAs than tiles/warps
  if (two_ctas && variant == 2) grid = 2 * sms;
  int max_ctas = (n_tiles + kWarpsPerCta - 1) / kWarpsPerCta;
  if (grid > max_ctas) grid = max_ctas;
  HGT_CHECK_CUDA(cudaMemsetAsync(p.tile_counter, 0, sizeof(int32_t), st));
  int rc;
  if (vec == 4) rc = dispatch_nch<KvT, 4>(p, nch, variant, grid, smem, st);
  else if (vec == 2) rc = dispatch_nch<KvT, 2>(p, nch, variant, grid, smem, st);
  else rc = dispatch_nch<KvT, 1>(p, nch, variant, grid, smem, st);
  if (rc) return rc;
  if (n_split_tiles > 0) {
    HGT_REQUIRE(hubs != nullptr && n_hubs > 0, "%s: split tiles present but no hub list given", fn);
    k_merge_partials<<<n_hubs < 4 * sms ? n_hubs : 4 * sms, kMergeThreads, 0, st>>>(p, hubs, n_hubs);
    HGT_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" int hgt_edge_forward(const float* q, const float* kv, const float* kvr, const int32_t* row_ptr,
                                const int32_t* kv_row, const int32_t* rte_row, const int32_t* csr_eid,
                                const int32_t* tiles, int32_t n_tiles, int32_t n_split_tiles, const int32_t* hubs,
                                int32_t n_hubs, int64_t n_nodes,
                                int64_t n_edges, int32_t d, int32_t n_heads, int32_t apply_gelu, float* agg_out,
                                float* att_out, float* stats_out, void* g_hi, void* g_lo, void* workspace,
                                size_t workspace_bytes, int32_t variant, const int32_t* d_tile_counts,
                                const int32_t* type_row0, int32_t num_types, const int32_t* type_active,
                                void* stream_) {
  (void)n_edges;
  return edge_forward<float>("hgt_edge_forward", q, kv, kvr, row_ptr, kv_row, rte_row, csr_eid, tiles, n_tiles,
                             n_split_tiles, hubs, n_hubs, n_nodes, d, n_heads, apply_gelu, agg_out, att_out, stats_out,
                             g_hi, g_lo, workspace, workspace_bytes, variant, d_tile_counts, type_row0, num_types,
                             type_active, (cudaStream_t)stream_);
}

extern "C" int hgt_edge_forward_bf16kv(const float* q, const void* kv, const void* kvr, const int32_t* row_ptr,
                                       const int32_t* kv_row, const int32_t* rte_row, const int32_t* csr_eid,
                                       const int32_t* tiles, int32_t n_tiles, int32_t n_split_tiles,
                                       const int32_t* hubs, int32_t n_hubs, int64_t n_nodes, int64_t n_edges, int32_t d,
                                       int32_t n_heads, int32_t apply_gelu, float* agg_out, float* att_out,
                                       float* stats_out, void* g_hi, void* g_lo, void* workspace,
                                       size_t workspace_bytes, int32_t variant, const int32_t* d_tile_counts,
                                       const int32_t* type_row0, int32_t num_types, const int32_t* type_active,
                                       void* stream_) {
  (void)n_edges;
  return edge_forward<__nv_bfloat16>("hgt_edge_forward_bf16kv", q, kv, kvr, row_ptr, kv_row, rte_row, csr_eid, tiles,
                                     n_tiles, n_split_tiles, hubs, n_hubs, n_nodes, d, n_heads, apply_gelu, agg_out,
                                     att_out, stats_out, g_hi, g_lo, workspace, workspace_bytes, variant,
                                     d_tile_counts, type_row0, num_types, type_active, (cudaStream_t)stream_);
}
