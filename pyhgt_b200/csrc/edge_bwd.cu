// Backward of the fused HGT edge kernel (see edge.cu for the forward and the lane mapping).
//
// Forward per destination i and head h:  s_e = <q_i, k_e>,  p_e = exp(s_e - m_i) / (l_i + 1e-16),
//                                         agg_i = sum_e p_e v_e            (k_e / v_e include the RTE rows)
// Given dagg_i:   dv_e = p_e * dagg_i          dp_e = <dagg_i, v_e>          D_i = <dagg_i, agg_i> (= sum_e p_e dp_e)
//                 ds_e = p_e * (dp_e - D_i)    dq_i = sum_e ds_e k_e         dk_e = ds_e * q_i
// One pass over the destination-sorted CSR; p is recomputed from the saved per-(destination, head) (m, l).
// dq is owned by the destination's warp (atomics only for split hub pieces); dk / dv are scattered into the
// [K'|V'] gradient table (and the RTE gradient table) with vector fp32 reductions (red.global.add.v4.f32):
// many edges share a <source, relation> row.  The trailing all-zero row collects the gradient of edges that
// matched no triple and is discarded by the caller.
//
// Deterministic variant (hgt_edge_backward_det, torch.use_deterministic_algorithms): no floating-point atomics.
//   destination pass  the same walk over the destination tiles computes dq and D_i = <dagg_i, agg_i> [N, H] only;
//                     hub pieces write partial dq rows, merged in piece order.
//   source pass       walks a second index that groups the CSR positions by [K'|V'] row (hgt_plan_group_by, tiles by
//                     hgt_plan_tiles over its segments): a warp owns a row, loads it once, gathers q_i, dagg_i, (m, l)
//                     and D_i of every out-edge and writes the row's gradient once (zero rows included, so no memset).
//                     Hub rows are split into pieces, merged in piece order.  The RTE table gradient is the same pass
//                     over a grouping by RTE row.
#include "common.cuh"

namespace {

constexpr int kWarps = 8;

struct BwdParams {
  const float* q;
  const float* kv;
  const float* kvr;
  const float* agg;
  const float* dagg;
  const float* stats;        // [N, 2H] (m, l)
  const int32_t* row_ptr;
  const int32_t* kv_row;
  const int32_t* rte_row;
  const int32_t* tiles;
  int32_t n_tiles;
  const int32_t* d_counts;   // optional device {n_tiles, ...} (sync-free plans): n_tiles is then an upper bound
  int32_t d, H, DK, LPH, lph_shift;
  float* dq;                 // [N, d]   zero-initialised by hgt_edge_backward
  float* dkv;                // [rows+1, 2d] zero-initialised
  float* dkvr;               // [P*240+1, 2d] zero-initialised or nullptr
  int32_t* tile_counter;
  float* D;                  // deterministic destination pass: [N, H] <dagg, agg>
  float* dq_part;            // deterministic destination pass: [n_split, d] partial dq of hub pieces
};

template <int VEC>
__device__ __forceinline__ void ld_vec(float (&dst)[VEC], const float* p) {
  if constexpr (VEC == 4) {
    float4 t = *reinterpret_cast<const float4*>(p);
    dst[0] = t.x; dst[1] = t.y; dst[2] = t.z; dst[3] = t.w;
  } else if constexpr (VEC == 2) {
    float2 t = *reinterpret_cast<const float2*>(p);
    dst[0] = t.x; dst[1] = t.y;
  } else {
    dst[0] = *p;
  }
}
template <int VEC>
__device__ __forceinline__ void red_add_vec(float* p, const float (&v)[VEC]) {
  if constexpr (VEC == 4) {
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3])
                 : "memory");
  } else if constexpr (VEC == 2) {
    asm volatile("red.global.add.v2.f32 [%0], {%1,%2};" ::"l"(p), "f"(v[0]), "f"(v[1]) : "memory");
  } else {
    asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v[0]) : "memory");
  }
}
__device__ __forceinline__ float head_sum(float v, int lph) {
  for (int o = lph >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int VEC, int NCH, bool DET>
__device__ __forceinline__ void edge_bwd_body(const BwdParams& p) {
  const int lane = threadIdx.x & 31;
  const int lph = p.LPH;
  const int h = lane >> p.lph_shift;
  const int sub = lane & (lph - 1);
  const bool head_ok = h < p.H;
  int offs[NCH];
#pragma unroll
  for (int t = 0; t < NCH; ++t) {
    int o = (sub + t * lph) * VEC;
    offs[t] = (head_ok && o < p.DK) ? h * p.DK + o : -1;
  }
  const int64_t row_stride = 2 * (int64_t)p.d;
  const bool rte = p.kvr != nullptr;

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
      if (seg_end > seg_begin) {
        float q[NCH][VEC], da[NCH][VEC], dq[NCH][VEC];
        float dpart = 0.f;
#pragma unroll
        for (int t = 0; t < NCH; ++t) {
          if (offs[t] >= 0) {
            float ag[VEC];
            ld_vec<VEC>(q[t], p.q + (int64_t)dst * p.d + offs[t]);
            ld_vec<VEC>(da[t], p.dagg + (int64_t)dst * p.d + offs[t]);
            ld_vec<VEC>(ag, p.agg + (int64_t)dst * p.d + offs[t]);
#pragma unroll
            for (int v = 0; v < VEC; ++v) dpart = fmaf(da[t][v], ag[v], dpart);
          } else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) { q[t][v] = 0.f; da[t][v] = 0.f; }
          }
#pragma unroll
          for (int v = 0; v < VEC; ++v) dq[t][v] = 0.f;
        }
        const float D = head_sum(dpart, lph);
        if (DET && head_ok && sub == 0 && (!split || seg_begin == p.row_ptr[dst])) p.D[(int64_t)dst * p.H + h] = D;
        float m = 0.f, inv_l = 0.f;
        if (head_ok) {
          m = p.stats[(int64_t)dst * 2 * p.H + h];
          inv_l = 1.0f / (p.stats[(int64_t)dst * 2 * p.H + p.H + h] + 1e-16f);
        }
        for (int c = seg_begin; c < seg_end; ++c) {
          const int64_t row = p.kv_row[c];
          const int64_t rrow = rte ? p.rte_row[c] : 0;
          const float* kvp = p.kv + row * row_stride;
          float kk[NCH][VEC], vv[NCH][VEC];
          float spart = 0.f, dppart = 0.f;
#pragma unroll
          for (int t = 0; t < NCH; ++t) {
            if (offs[t] >= 0) {
              ld_vec<VEC>(kk[t], kvp + offs[t]);
              ld_vec<VEC>(vv[t], kvp + p.d + offs[t]);
              if (rte) {
                float a[VEC], b[VEC];
                ld_vec<VEC>(a, p.kvr + rrow * row_stride + offs[t]);
                ld_vec<VEC>(b, p.kvr + rrow * row_stride + p.d + offs[t]);
#pragma unroll
                for (int v = 0; v < VEC; ++v) { kk[t][v] += a[v]; vv[t][v] += b[v]; }
              }
#pragma unroll
              for (int v = 0; v < VEC; ++v) {
                spart = fmaf(q[t][v], kk[t][v], spart);
                dppart = fmaf(da[t][v], vv[t][v], dppart);
              }
            }
          }
          const float s = head_sum(spart, lph);
          const float dp = head_sum(dppart, lph);
          const float pe = __expf(s - m) * inv_l;
          const float ds = pe * (dp - D);
          float* gk = p.dkv + row * row_stride;
#pragma unroll
          for (int t = 0; t < NCH; ++t) {
            if (offs[t] >= 0) {
              float gkv[VEC], gvv[VEC];
#pragma unroll
              for (int v = 0; v < VEC; ++v) {
                dq[t][v] = fmaf(ds, kk[t][v], dq[t][v]);
                gkv[v] = ds * q[t][v];
                gvv[v] = pe * da[t][v];
              }
              if (!DET) {
                red_add_vec<VEC>(gk + offs[t], gkv);
                red_add_vec<VEC>(gk + p.d + offs[t], gvv);
                if (rte) {
                  red_add_vec<VEC>(p.dkvr + rrow * row_stride + offs[t], gkv);
                  red_add_vec<VEC>(p.dkvr + rrow * row_stride + p.d + offs[t], gvv);
                }
              }
            }
          }
        }
        float* gq = (DET && split) ? p.dq_part + (int64_t)(-tl.y - 1) * p.d : p.dq + (int64_t)dst * p.d;
#pragma unroll
        for (int t = 0; t < NCH; ++t) {
          if (offs[t] >= 0) {
            if (!DET && split) red_add_vec<VEC>(gq + offs[t], dq[t]);
            else {
#pragma unroll
              for (int v = 0; v < VEC; ++v) gq[offs[t] + v] = dq[t][v];
            }
          }
        }
      } else if (DET) {
        // no in-edges: a zero dq row (the deterministic path does not zero-fill dq)
        float* gq = p.dq + (int64_t)dst * p.d;
#pragma unroll
        for (int t = 0; t < NCH; ++t)
          if (offs[t] >= 0) {
#pragma unroll
            for (int v = 0; v < VEC; ++v) gq[offs[t] + v] = 0.f;
          }
      }
      seg_begin = seg_end;
    }
  }
}

template <int VEC, int NCH>
__global__ void __launch_bounds__(kWarps * 32)
k_edge_bwd(BwdParams p) {
  edge_bwd_body<VEC, NCH, false>(p);
}
template <int VEC, int NCH>
__global__ void __launch_bounds__(kWarps * 32)
k_det_edge_dst(BwdParams p) {
  edge_bwd_body<VEC, NCH, true>(p);
}

// ---- deterministic source-major pass ------------------------------------------------------------------------------------
// For each row `key` of an owned table (the [K'|V'] table, or the RTE table) and each CSR position c = pos[j],
// j in [ptr[key], ptr[key+1]) (the edges reading that row, in CSR order):
//   k_e = own[key].K + other[other_idx[c]].K,  v_e likewise   (other: the table the edge adds to it, or none)
//   grad[key] = sum_e [ds_e * q_i | p_e * dagg_i]             (i = csr_dst[c]; p_e, ds_e recomputed as in k_edge_bwd)
struct SrcParams {
  const float* q;
  const float* dagg;
  const float* stats;        // [N, 2H] (m, l)
  const float* D;            // [N, H]
  const float* own;          // [keys, 2d]
  const float* other;        // [*, 2d] or nullptr
  const int32_t* other_idx;  // [E] by CSR position, or nullptr
  const int32_t* csr_dst;    // [E]
  const int32_t* ptr;        // [keys+1]
  const int32_t* pos;        // [E]
  const int32_t* tiles;
  int32_t n_tiles;
  const int32_t* d_counts;
  int32_t d, H, DK, LPH, lph_shift;
  float* out;                // [keys, 2d]: every row written
  float* part;               // [n_split, 2d] partial rows of hub pieces
  int32_t* tile_counter;
};

template <int VEC, int NCH>
__global__ void __launch_bounds__(kWarps * 32)
k_det_edge_src(SrcParams p) {
  const int lane = threadIdx.x & 31;
  const int lph = p.LPH;
  const int h = lane >> p.lph_shift;
  const int sub = lane & (lph - 1);
  const bool head_ok = h < p.H;
  int offs[NCH];
#pragma unroll
  for (int t = 0; t < NCH; ++t) {
    int o = (sub + t * lph) * VEC;
    offs[t] = (head_ok && o < p.DK) ? h * p.DK + o : -1;
  }
  const int64_t row_stride = 2 * (int64_t)p.d;
  const bool has_other = p.other != nullptr;
  const int n_tiles = p.d_counts ? p.d_counts[0] : p.n_tiles;
  for (;;) {
    int tile = 0;
    if (lane == 0) tile = atomicAdd(p.tile_counter, 1);
    tile = __shfl_sync(0xffffffffu, tile, 0);
    if (tile >= n_tiles) break;
    const int4 tl = reinterpret_cast<const int4*>(p.tiles)[tile];
    const bool split = tl.y < 0;
    const int k_begin = tl.x, k_end = split ? tl.x + 1 : tl.y;
    int seg_begin = tl.z;
    for (int key = k_begin; key < k_end; ++key) {
      const int seg_end = split ? tl.w : p.ptr[key + 1];
      float ok[NCH][VEC], ov[NCH][VEC], gk[NCH][VEC], gv[NCH][VEC];
      const float* own = p.own + (int64_t)key * row_stride;
#pragma unroll
      for (int t = 0; t < NCH; ++t) {
        if (offs[t] >= 0 && seg_end > seg_begin) {
          ld_vec<VEC>(ok[t], own + offs[t]);
          ld_vec<VEC>(ov[t], own + p.d + offs[t]);
        } else {
#pragma unroll
          for (int v = 0; v < VEC; ++v) { ok[t][v] = 0.f; ov[t][v] = 0.f; }
        }
#pragma unroll
        for (int v = 0; v < VEC; ++v) { gk[t][v] = 0.f; gv[t][v] = 0.f; }
      }
      for (int j = seg_begin; j < seg_end; ++j) {
        const int c = p.pos[j];
        const int64_t i = p.csr_dst[c];
        const float* orow = has_other ? p.other + (int64_t)p.other_idx[c] * row_stride : nullptr;
        float q[NCH][VEC], da[NCH][VEC], kk[NCH][VEC], vv[NCH][VEC];
        float spart = 0.f, dppart = 0.f;
#pragma unroll
        for (int t = 0; t < NCH; ++t) {
          if (offs[t] >= 0) {
            ld_vec<VEC>(q[t], p.q + i * p.d + offs[t]);
            ld_vec<VEC>(da[t], p.dagg + i * p.d + offs[t]);
#pragma unroll
            for (int v = 0; v < VEC; ++v) { kk[t][v] = ok[t][v]; vv[t][v] = ov[t][v]; }
            if (has_other) {
              float a[VEC], b[VEC];
              ld_vec<VEC>(a, orow + offs[t]);
              ld_vec<VEC>(b, orow + p.d + offs[t]);
#pragma unroll
              for (int v = 0; v < VEC; ++v) { kk[t][v] += a[v]; vv[t][v] += b[v]; }
            }
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
              spart = fmaf(q[t][v], kk[t][v], spart);
              dppart = fmaf(da[t][v], vv[t][v], dppart);
            }
          }
        }
        const float s = head_sum(spart, lph);
        const float dp = head_sum(dppart, lph);
        float m = 0.f, inv_l = 0.f, D = 0.f;
        if (head_ok) {
          m = p.stats[i * 2 * p.H + h];
          inv_l = 1.0f / (p.stats[i * 2 * p.H + p.H + h] + 1e-16f);
          D = p.D[i * p.H + h];
        }
        const float pe = __expf(s - m) * inv_l;
        const float ds = pe * (dp - D);
#pragma unroll
        for (int t = 0; t < NCH; ++t) {
          if (offs[t] >= 0) {
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
              gk[t][v] = fmaf(ds, q[t][v], gk[t][v]);
              gv[t][v] = fmaf(pe, da[t][v], gv[t][v]);
            }
          }
        }
      }
      float* g = split ? p.part + (int64_t)(-tl.y - 1) * row_stride : p.out + (int64_t)key * row_stride;
#pragma unroll
      for (int t = 0; t < NCH; ++t) {
        if (offs[t] >= 0) {
#pragma unroll
          for (int v = 0; v < VEC; ++v) {
            g[offs[t] + v] = gk[t][v];
            g[p.d + offs[t] + v] = gv[t][v];
          }
        }
      }
      seg_begin = seg_end;
    }
  }
}

// Hub pieces: out[key] = sum of the pieces' partial rows in piece order (hubs: {key, first slot, pieces, 0}).
__global__ void k_det_merge_pieces(const float* __restrict__ part, int64_t width, const int32_t* __restrict__ hubs,
                                   int n_hubs_host, const int32_t* __restrict__ d_counts, float* __restrict__ out) {
  const int n_hubs = d_counts ? d_counts[2] : n_hubs_host;
  for (int hb = blockIdx.x; hb < n_hubs; hb += gridDim.x) {
    const int64_t key = hubs[4 * hb], slot0 = hubs[4 * hb + 1];
    const int pieces = hubs[4 * hb + 2];
    for (int64_t j = threadIdx.x; j < width; j += blockDim.x)
      out[key * width + j] = hgt_chunk_sum(part + slot0 * width + j, pieces, width);
  }
}

template <int VEC>
int dispatch(const BwdParams& p, int nch, int grid, cudaStream_t st) {
  switch (nch) {
    case 1: k_edge_bwd<VEC, 1><<<grid, kWarps * 32, 0, st>>>(p); break;
    case 2: k_edge_bwd<VEC, 2><<<grid, kWarps * 32, 0, st>>>(p); break;
    case 4: k_edge_bwd<VEC, 4><<<grid, kWarps * 32, 0, st>>>(p); break;
    case 8: k_edge_bwd<VEC, 8><<<grid, kWarps * 32, 0, st>>>(p); break;
    default: hgt_set_error("hgt_edge_backward: unsupported chunk count %d", nch); return 1;
  }
  HGT_LAUNCH_CHECK();
  return 0;
}

struct LaneMap {
  int LPH, lph_shift, vec, nch;
};
LaneMap lane_map(int d, int n_heads) {
  LaneMap m;
  const int DK = d / n_heads;
  int hp = 1;
  while (hp < n_heads) hp <<= 1;
  m.LPH = 32 / hp;
  m.lph_shift = 0;
  while ((1 << m.lph_shift) < m.LPH) ++m.lph_shift;
  m.vec = 1;
  for (int v : {4, 2})
    if (DK % v == 0 && DK / v >= m.LPH) { m.vec = v; break; }
  const int chunks = (DK + m.vec * m.LPH - 1) / (m.vec * m.LPH);
  m.nch = 1;
  while (m.nch < chunks) m.nch <<= 1;
  return m;
}

template <int VEC, int NCH>
void launch_det(const BwdParams& bp, const SrcParams* sp, int grid, cudaStream_t st) {
  if (sp) k_det_edge_src<VEC, NCH><<<grid, kWarps * 32, 0, st>>>(*sp);
  else k_det_edge_dst<VEC, NCH><<<grid, kWarps * 32, 0, st>>>(bp);
}
int dispatch_det(const LaneMap& lm, const BwdParams& bp, const SrcParams* sp, int n_tiles, cudaStream_t st) {
  int grid = hgt_sm_count() * 4;
  const int max_ctas = (n_tiles + kWarps - 1) / kWarps;
  if (grid > max_ctas) grid = max_ctas;
  if (grid == 0) return 0;
#define HGT_DET_NCH(V)                                          \
  switch (lm.nch) {                                             \
    case 1: launch_det<V, 1>(bp, sp, grid, st); break;          \
    case 2: launch_det<V, 2>(bp, sp, grid, st); break;          \
    case 4: launch_det<V, 4>(bp, sp, grid, st); break;          \
    default: launch_det<V, 8>(bp, sp, grid, st); break;         \
  }
  if (lm.vec == 4) { HGT_DET_NCH(4) }
  else if (lm.vec == 2) { HGT_DET_NCH(2) }
  else { HGT_DET_NCH(1) }
#undef HGT_DET_NCH
  HGT_LAUNCH_CHECK();
  return 0;
}

int merge_pieces(const float* part, int64_t width, const hgt_tile_set& ts, float* out, cudaStream_t st) {
  if (ts.n_hubs <= 0) return 0;
  const int grid = ts.n_hubs < 4 * hgt_sm_count() ? ts.n_hubs : 4 * hgt_sm_count();
  k_det_merge_pieces<<<grid, 256, 0, st>>>(part, width, ts.hubs, ts.n_hubs, ts.d_counts, out);
  HGT_LAUNCH_CHECK();
  return 0;
}

struct DetLayout {
  size_t off_D, off_dq_part, off_kv_part, off_rte_part, total;
};
DetLayout det_layout(int64_t n_nodes, int32_t d, int32_t n_heads, const hgt_tile_set* dst, const hgt_tile_set* src,
                     const hgt_tile_set* rte) {
  DetLayout L;
  size_t p = 256;                                    // three tile counters
  auto take = [&](size_t bytes) { size_t o = p; p += hgt_align_up(bytes, 256); return o; };
  auto split_of = [](const hgt_tile_set* t) { return (size_t)(t && t->n_split > 0 ? t->n_split : 0); };
  L.off_D = take((size_t)n_nodes * n_heads * sizeof(float));
  L.off_dq_part = take(split_of(dst) * d * sizeof(float));
  L.off_kv_part = take(split_of(src) * 2 * d * sizeof(float));
  L.off_rte_part = take(split_of(rte) * 2 * d * sizeof(float));
  L.total = p + 256;                                 // slack for aligning the caller's base pointer
  return L;
}

}  // namespace

extern "C" int hgt_edge_backward_det_workspace_bytes(int64_t n_nodes, int32_t d, int32_t n_heads,
                                                     const hgt_tile_set* dst, const hgt_tile_set* src,
                                                     const hgt_tile_set* rte, size_t* out_bytes) {
  HGT_REQUIRE(out_bytes && n_nodes >= 0 && n_heads >= 1, "hgt_edge_backward_det_workspace_bytes: bad argument");
  *out_bytes = det_layout(n_nodes, d, n_heads, dst, src, rte).total;
  return 0;
}

extern "C" int hgt_edge_backward_det(const float* q, const float* kv, const float* kvr, const float* agg,
                                     const float* dagg, const float* stats, const int32_t* kv_row,
                                     const int32_t* rte_row, const int32_t* csr_dst, const hgt_tile_set* dst,
                                     const hgt_tile_set* src, const hgt_tile_set* rte, int64_t n_nodes, int32_t d,
                                     int32_t n_heads, float* dq, float* dkv, float* dkvr, void* workspace,
                                     size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HGT_REQUIRE(n_heads >= 1 && n_heads <= 32 && d % n_heads == 0, "hgt_edge_backward_det: bad d=%d / n_heads=%d", d,
              n_heads);
  HGT_REQUIRE(dst && src && dst->ptr && src->ptr && src->pos && csr_dst && kv_row,
              "hgt_edge_backward_det: NULL index argument");
  HGT_REQUIRE((kvr != nullptr) == (rte_row != nullptr) && (kvr != nullptr) == (dkvr != nullptr) &&
                  (kvr != nullptr) == (rte != nullptr && rte->ptr != nullptr && rte->pos != nullptr),
              "hgt_edge_backward_det: kvr, rte_row, dkvr and the RTE index must go together");
  const DetLayout L = det_layout(n_nodes, d, n_heads, dst, src, rte);
  HGT_REQUIRE(workspace && workspace_bytes >= L.total, "hgt_edge_backward_det: workspace too small (%zu < %zu)",
              workspace_bytes, L.total);
  const LaneMap lm = lane_map(d, n_heads);
  HGT_REQUIRE(lm.nch <= 8, "hgt_edge_backward_det: head width d_k=%d needs more than 8 chunks per lane", d / n_heads);
  char* base = reinterpret_cast<char*>(hgt_align_up(reinterpret_cast<size_t>(workspace), 256));
  int32_t* counters = reinterpret_cast<int32_t*>(base);
  HGT_CHECK_CUDA(cudaMemsetAsync(counters, 0, 3 * sizeof(int32_t), st));
  int rc;

  // 1. destination pass: dq and D
  BwdParams bp{};
  bp.q = q; bp.kv = kv; bp.kvr = kvr; bp.agg = agg; bp.dagg = dagg; bp.stats = stats; bp.row_ptr = dst->ptr;
  bp.kv_row = kv_row; bp.rte_row = rte_row; bp.tiles = dst->tiles; bp.n_tiles = dst->n_tiles; bp.d_counts = dst->d_counts;
  bp.d = d; bp.H = n_heads; bp.DK = d / n_heads; bp.LPH = lm.LPH; bp.lph_shift = lm.lph_shift;
  bp.dq = dq; bp.tile_counter = counters;
  bp.D = reinterpret_cast<float*>(base + L.off_D);
  bp.dq_part = reinterpret_cast<float*>(base + L.off_dq_part);
  if (n_nodes > 0 && dst->n_tiles > 0) {
    if ((rc = dispatch_det(lm, bp, nullptr, dst->n_tiles, st))) return rc;
    if ((rc = merge_pieces(bp.dq_part, d, *dst, dq, st))) return rc;
  }

  // 2. source passes: the [K'|V'] table, then the RTE table
  for (int pass = 0; pass < (kvr ? 2 : 1); ++pass) {
    const hgt_tile_set& ts = pass == 0 ? *src : *rte;
    SrcParams sp{};
    sp.q = q; sp.dagg = dagg; sp.stats = stats; sp.D = bp.D;
    sp.own = pass == 0 ? kv : kvr;
    sp.other = pass == 0 ? kvr : kv;
    sp.other_idx = pass == 0 ? rte_row : kv_row;
    sp.csr_dst = csr_dst; sp.ptr = ts.ptr; sp.pos = ts.pos; sp.tiles = ts.tiles; sp.n_tiles = ts.n_tiles;
    sp.d_counts = ts.d_counts;
    sp.d = d; sp.H = n_heads; sp.DK = d / n_heads; sp.LPH = lm.LPH; sp.lph_shift = lm.lph_shift;
    sp.out = pass == 0 ? dkv : dkvr;
    sp.part = reinterpret_cast<float*>(base + (pass == 0 ? L.off_kv_part : L.off_rte_part));
    sp.tile_counter = counters + 1 + pass;
    if (ts.n_tiles > 0) {
      if ((rc = dispatch_det(lm, bp, &sp, ts.n_tiles, st))) return rc;
      if ((rc = merge_pieces(sp.part, 2 * (int64_t)d, ts, sp.out, st))) return rc;
    }
  }
  return 0;
}

extern "C" int hgt_edge_backward(const float* q, const float* kv, const float* kvr, const float* agg,
                                 const float* dagg, const float* stats, const int32_t* row_ptr,
                                 const int32_t* kv_row, const int32_t* rte_row, const int32_t* tiles, int32_t n_tiles,
                                 int64_t n_nodes, int32_t d, int32_t n_heads, int64_t kv_rows_total,
                                 int64_t kvr_rows_total, float* dq, float* dkv, float* dkvr,
                                 void* workspace, size_t workspace_bytes, const int32_t* d_tile_counts, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HGT_REQUIRE(n_heads >= 1 && n_heads <= 32 && d % n_heads == 0, "hgt_edge_backward: bad d=%d / n_heads=%d", d, n_heads);
  HGT_REQUIRE((kvr != nullptr) == (rte_row != nullptr) && (kvr != nullptr) == (dkvr != nullptr),
              "hgt_edge_backward: kvr, rte_row and dkvr must go together");
  HGT_REQUIRE(workspace && workspace_bytes >= 256, "hgt_edge_backward: workspace too small");
  // the kernel accumulates (dk / dv of a <source, relation> row come from many edges): this call owns the initialisation
  if (n_nodes > 0) HGT_CHECK_CUDA(cudaMemsetAsync(dq, 0, (size_t)n_nodes * d * sizeof(float), st));
  if (kv_rows_total > 0) HGT_CHECK_CUDA(cudaMemsetAsync(dkv, 0, (size_t)kv_rows_total * 2 * d * sizeof(float), st));
  if (dkvr && kvr_rows_total > 0)
    HGT_CHECK_CUDA(cudaMemsetAsync(dkvr, 0, (size_t)kvr_rows_total * 2 * d * sizeof(float), st));
  if (n_nodes == 0 || n_tiles == 0) return 0;
  BwdParams p;
  p.q = q; p.kv = kv; p.kvr = kvr; p.agg = agg; p.dagg = dagg; p.stats = stats; p.row_ptr = row_ptr;
  p.kv_row = kv_row; p.rte_row = rte_row; p.tiles = tiles; p.n_tiles = n_tiles; p.d_counts = d_tile_counts; p.d = d; p.H = n_heads;
  p.DK = d / n_heads;
  int hp = 1;
  while (hp < n_heads) hp <<= 1;
  p.LPH = 32 / hp;
  int shift = 0;
  while ((1 << shift) < p.LPH) ++shift;
  p.lph_shift = shift;
  p.dq = dq; p.dkv = dkv; p.dkvr = dkvr;
  p.tile_counter = reinterpret_cast<int32_t*>(workspace);
  int vec = 1;
  for (int v : {4, 2})
    if (p.DK % v == 0 && p.DK / v >= p.LPH) { vec = v; break; }
  int chunks = (p.DK + vec * p.LPH - 1) / (vec * p.LPH), nch = 1;
  while (nch < chunks) nch <<= 1;
  HGT_REQUIRE(nch <= 8, "hgt_edge_backward: head width d_k=%d needs %d chunks per lane (max 8)", p.DK, chunks);
  HGT_CHECK_CUDA(cudaMemsetAsync(p.tile_counter, 0, sizeof(int32_t), st));
  int grid = hgt_sm_count() * 4;
  int max_ctas = (n_tiles + kWarps - 1) / kWarps;
  if (grid > max_ctas) grid = max_ctas;
  if (vec == 4) return dispatch<4>(p, nch, grid, st);
  if (vec == 2) return dispatch<2>(p, nch, grid, st);
  return dispatch<1>(p, nch, grid, st);
}
