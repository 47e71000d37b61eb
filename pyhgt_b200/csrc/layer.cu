// One C-ABI call for a whole HGTConv forward (inference): gather (if the node types are not pre-sorted) ->
// weight fold -> typed projections (+ RTE tables) -> fused edge kernel -> typed a_linear -> gated skip + LayerNorm.
// The caller hands over the plan arrays, the parameter pointer tables and ONE workspace; everything is enqueued on
// the given stream without any host synchronisation.  This is what a non-Python host binds for the layer
// (reference boundary: HGTConv.forward, pyHGT/conv.py:56-134); the Python class uses it too, so that a layer costs
// one ctypes call instead of a dozen (the reference's sampled-subgraph batches are launch/host-bound).
// With kv_bf16 the [K'|V'] and K'R/V'R tables are written and gathered as bf16 (inference mode, see the header).
#include "common.cuh"

int hgt_update_epilogue_impl(const float* o, const float* x, const int32_t* type_row0, int32_t num_types,
                             const float* skip, const float* norm_w, const float* norm_b, const float* const* norm_wp,
                             const float* const* norm_bp, const int32_t* perm, const int32_t* type_active,
                             int64_t n_nodes, int32_t d, float* out, void* out_hi, void* out_lo, cudaStream_t st);
bool hgt_typed_linear_tc_supported(int64_t lda, int32_t K, int32_t cb_width);

namespace {

struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* b) : base(reinterpret_cast<char*>(b)) {}
  template <typename T>
  T* take(size_t count) {
    size_t o = off;
    off += hgt_align_up(count * sizeof(T), 256);
    return base ? reinterpret_cast<T*>(base + o) : nullptr;
  }
  void* take_bytes(size_t bytes) { return take<char>(bytes); }
};

struct Layout {
  float *x_sorted, *w_cat, *b_cat, *proj, *rt, *kvr, *g_act, *wa_cat, *ba_cat, *o;
  void *kv16, *kvr16;                                      // kv_bf16: the bf16 tables (else NULL)
  void *g_hi, *g_lo, *ws_proj, *ws_edge, *ws_upd;
  size_t ws_proj_bytes, ws_edge_bytes, ws_upd_bytes, total;
  bool fuse_split, presplit_x;
};

int plan_layout(const hgt_conv_args* a, void* base, Layout* L) {
  Carver c(base);
  const int64_t N = a->n_nodes;
  const int d = a->d_out, din = a->d_in;
  const bool tc_upd = a->linear_impl != 1 && hgt_typed_linear_tc_supported(d, d, d);
  L->fuse_split = tc_upd;                                  // edge kernel writes gelu(agg) as the bf16 hi/lo split
  L->presplit_x = a->x_hi != nullptr && a->x_lo != nullptr && a->perm == nullptr && a->linear_impl != 1 &&
                  hgt_typed_linear_tc_supported(din, din, d);
  L->x_sorted = a->perm ? c.take<float>((size_t)N * din) : nullptr;
  L->w_cat = c.take<float>((size_t)(a->cat_rows > 0 ? a->cat_rows : 1) * din);
  L->b_cat = c.take<float>((size_t)(a->cat_rows > 0 ? a->cat_rows : 1));
  L->proj = c.take<float>((size_t)a->proj_elems);
  L->kv16 = a->kv_bf16 ? c.take<__nv_bfloat16>(((size_t)a->kv_rows + 1) * 2 * d) : nullptr;
  int rc;
  if (L->presplit_x)
    rc = hgt_typed_linear_presplit_workspace_bytes(a->h_proj_groups, a->n_proj_groups, din, d, &L->ws_proj_bytes);
  else
    rc = hgt_typed_linear_workspace_bytes(a->h_proj_groups, a->n_proj_groups, din, d, a->linear_impl, &L->ws_proj_bytes);
  if (rc) return rc;
  L->ws_proj = c.take_bytes(L->ws_proj_bytes + 256);
  L->rt = L->kvr = nullptr;
  L->kvr16 = nullptr;
  if (a->use_rte) {
    L->rt = c.take<float>((size_t)HGT_RTE_MAX_LEN * din);
    const size_t kvr_elems = ((size_t)a->n_pairs * HGT_RTE_MAX_LEN + 1) * 2 * d;
    if (a->kv_bf16)
      L->kvr16 = c.take<__nv_bfloat16>(kvr_elems);
    else
      L->kvr = c.take<float>(kvr_elems);
  }
  if ((rc = hgt_edge_workspace_bytes(a->n_split, d, a->n_heads, &L->ws_edge_bytes))) return rc;
  L->ws_edge = c.take_bytes(L->ws_edge_bytes);
  L->g_act = nullptr;
  L->g_hi = L->g_lo = nullptr;
  if (L->fuse_split) {
    L->g_hi = c.take_bytes((size_t)N * d * 2);
    L->g_lo = c.take_bytes((size_t)N * d * 2);
  } else {
    L->g_act = c.take<float>((size_t)N * d);
  }
  L->wa_cat = c.take<float>((size_t)a->num_types * d * d);
  L->ba_cat = c.take<float>((size_t)a->num_types * d);
  if (L->fuse_split)
    rc = hgt_typed_linear_presplit_workspace_bytes(a->h_upd_groups, a->n_upd_groups, d, d, &L->ws_upd_bytes);
  else
    rc = hgt_typed_linear_workspace_bytes(a->h_upd_groups, a->n_upd_groups, d, d, a->linear_impl, &L->ws_upd_bytes);
  if (rc) return rc;
  L->ws_upd = c.take_bytes(L->ws_upd_bytes + 256);
  L->o = c.take<float>((size_t)N * d);
  L->total = c.off + 256;
  return 0;
}

}  // namespace

extern "C" uint64_t hgt_conv_args_size(void) { return sizeof(hgt_conv_args); }

extern "C" int hgt_conv_workspace_bytes(const hgt_conv_args* a, size_t* out_bytes) {
  HGT_REQUIRE(a && out_bytes, "hgt_conv_workspace_bytes: NULL argument");
  Layout L;
  int rc = plan_layout(a, nullptr, &L);
  if (rc) return rc;
  *out_bytes = L.total;
  return 0;
}

extern "C" int hgt_conv_forward(const hgt_conv_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  HGT_REQUIRE(a && workspace, "hgt_conv_forward: NULL argument");
  HGT_REQUIRE(a->d_in == a->d_out, "hgt_conv_forward: in_dim must equal out_dim (conv.py:131)");
  HGT_REQUIRE(!a->use_rte || a->rte_row, "hgt_conv_forward: use_rte needs rte_row");
  cudaStream_t st = (cudaStream_t)stream;
  Layout L;
  void* base = reinterpret_cast<void*>(hgt_align_up(reinterpret_cast<size_t>(workspace), 256));
  int rc = plan_layout(a, base, &L);
  if (rc) return rc;
  HGT_REQUIRE(workspace_bytes >= L.total, "hgt_conv_forward: workspace too small (%zu < %zu)", workspace_bytes, L.total);
  const int64_t N = a->n_nodes;
  const int d = a->d_out, din = a->d_in, T = a->num_types, P = a->n_pairs;
  const bool bf16 = a->kv_bf16 != 0;
  HGT_REQUIRE(!bf16 || (a->n_q_groups >= 0 && a->n_q_groups <= a->n_proj_groups),
              "hgt_conv_forward: n_q_groups=%d outside [0, n_proj_groups=%d]", a->n_q_groups, a->n_proj_groups);
  if (bf16) {
    // the bf16 layout: Q groups (one column block each) first, then [K'|V'] groups (an even number of blocks each).
    // An fp32-layout table (Q and K'/V' blocks in one group, an odd count) would write bf16 rows at fp32 offsets.
    for (int g = 0; g < a->n_proj_groups; ++g) {
      const int nc = a->h_proj_groups[g].n_cblocks;
      HGT_REQUIRE(g < a->n_q_groups ? nc == 1 : nc % 2 == 0,
                  "hgt_conv_forward: kv_bf16 needs the Q groups (1 column block) first and then the [K'|V'] groups "
                  "(an even number of blocks); group %d has %d blocks with n_q_groups=%d", g, nc, a->n_q_groups);
    }
  }
  if (N == 0) return 0;

  const float* x_sorted = a->x;
  if (a->perm) {
    if ((rc = hgt_gather_rows(a->x, a->perm, N, din, L.x_sorted, stream))) return rc;
    x_sorted = L.x_sorted;
  }
  if ((rc = hgt_fold_weights(a->wq, a->bq, a->wk, a->bk, a->wv, a->bv, a->relation_att, a->relation_msg,
                             a->relation_pri, T, a->num_relations, a->n_heads, din, d, P, a->pair_type, a->pair_rel,
                             a->cat_row0, a->q_row0, L.w_cat, L.b_cat, stream)))
    return rc;
  // trailing all-zero [K'|V'] row (edges that match no <s,t,r> triple)
  if (bf16)
    HGT_CHECK_CUDA(cudaMemsetAsync(reinterpret_cast<__nv_bfloat16*>(L.kv16) + a->kv_rows * 2 * (int64_t)d, 0,
                                   sizeof(__nv_bfloat16) * 2 * d, st));
  else
    HGT_CHECK_CUDA(cudaMemsetAsync(L.proj + a->kv_off + a->kv_rows * 2 * (int64_t)d, 0, sizeof(float) * 2 * d, st));
  // fp32 groups (all of them, or the leading Q groups with bf16 tables), then the bf16 [K'|V'] groups
  const int n_f32 = bf16 ? a->n_q_groups : a->n_proj_groups;
  const int n_kv16 = a->n_proj_groups - n_f32;
  const hgt_lin_group* kv_groups = a->proj_groups + n_f32;
  const hgt_lin_group* h_kv_groups = a->h_proj_groups + n_f32;
  bool presplit = L.presplit_x;
  const void *x_hi = a->x_hi, *x_lo = a->x_lo;
  if (bf16 && !presplit && L.fuse_split) {
    // two tensor-core GEMMs over the same x: split it once, into the g_hi / g_lo buffers (the edge kernel fills them
    // only after the projection); the presplit GEMM rounds exactly like the GEMM's own split
    if ((rc = hgt_act_split(x_sorted, din, N, din, 0, nullptr, L.g_hi, L.g_lo, stream))) return rc;
    presplit = true;
    x_hi = L.g_hi;
    x_lo = L.g_lo;
  }
  if (presplit)
    rc = hgt_typed_linear_presplit(x_hi, x_lo, L.w_cat, L.b_cat, din, d, a->proj_groups, a->h_proj_groups,
                                   n_f32, a->proj_cblocks, L.proj, L.ws_proj, L.ws_proj_bytes + 256, stream);
  else
    rc = hgt_typed_linear(x_sorted, din, L.w_cat, L.b_cat, din, d, a->proj_groups, a->h_proj_groups, n_f32,
                          a->proj_cblocks, L.proj, a->linear_impl, L.ws_proj, L.ws_proj_bytes + 256, stream);
  if (rc) return rc;
  if (bf16 && n_kv16 > 0) {
    if (presplit)
      rc = hgt_typed_linear_presplit_bf16(x_hi, x_lo, L.w_cat, L.b_cat, din, d, kv_groups, h_kv_groups, n_kv16,
                                          a->proj_cblocks, L.kv16, L.ws_proj, L.ws_proj_bytes + 256, stream);
    else
      rc = hgt_typed_linear_bf16(x_sorted, din, L.w_cat, L.b_cat, din, d, kv_groups, h_kv_groups, n_kv16,
                                 a->proj_cblocks, L.kv16, a->linear_impl, L.ws_proj, L.ws_proj_bytes + 256, stream);
    if (rc) return rc;
  }
  if (a->use_rte) {
    if ((rc = hgt_typed_linear(a->emb_weight, din, a->emb_lin_w, a->emb_lin_b, din, din, a->rt_groups, a->h_rt_groups, 1,
                               a->rt_cblocks, L.rt, 1, nullptr, 0, stream)))
      return rc;
    const int64_t zero_row = (int64_t)P * HGT_RTE_MAX_LEN * 2 * d;
    if (bf16) {
      HGT_CHECK_CUDA(cudaMemsetAsync(reinterpret_cast<__nv_bfloat16*>(L.kvr16) + zero_row, 0,
                                     sizeof(__nv_bfloat16) * 2 * d, st));
      rc = hgt_typed_linear_bf16(L.rt, din, L.w_cat, nullptr, din, d, a->rte_groups, a->h_rte_groups, a->n_rte_groups,
                                 a->rte_cblocks, L.kvr16, 1, nullptr, 0, stream);
    } else {
      HGT_CHECK_CUDA(cudaMemsetAsync(L.kvr + zero_row, 0, sizeof(float) * 2 * d, st));
      rc = hgt_typed_linear(L.rt, din, L.w_cat, nullptr, din, d, a->rte_groups, a->h_rte_groups, a->n_rte_groups,
                            a->rte_cblocks, L.kvr, 1, nullptr, 0, stream);
    }
    if (rc) return rc;
  }
  if (bf16)
    rc = hgt_edge_forward_bf16kv(L.proj + a->q_off, L.kv16, L.kvr16, a->row_ptr, a->kv_row,
                                 a->use_rte ? a->rte_row : nullptr, a->csr_eid, a->tiles, a->n_tiles, a->n_split,
                                 a->hubs, a->n_hubs, N, a->n_edges, d, a->n_heads, 1, L.g_act, a->att, nullptr, L.g_hi,
                                 L.g_lo, L.ws_edge, L.ws_edge_bytes, a->edge_variant, a->d_tile_counts, a->type_row0, T,
                                 a->type_active, stream);
  else
    rc = hgt_edge_forward(L.proj + a->q_off, L.proj + a->kv_off, L.kvr, a->row_ptr, a->kv_row,
                          a->use_rte ? a->rte_row : nullptr, a->csr_eid, a->tiles, a->n_tiles, a->n_split, a->hubs,
                          a->n_hubs, N, a->n_edges, d, a->n_heads, 1, L.g_act, a->att, nullptr, L.g_hi, L.g_lo,
                          L.ws_edge, L.ws_edge_bytes, a->edge_variant, a->d_tile_counts, a->type_row0, T,
                          a->type_active, stream);
  if (rc) return rc;
  if ((rc = hgt_concat_linears(a->wa, a->ba, T, d, d, L.wa_cat, L.ba_cat, stream))) return rc;
  if (L.fuse_split)
    rc = hgt_typed_linear_presplit(L.g_hi, L.g_lo, L.wa_cat, L.ba_cat, d, d, a->upd_groups, a->h_upd_groups,
                                   a->n_upd_groups, a->upd_cblocks, L.o, L.ws_upd, L.ws_upd_bytes + 256, stream);
  else
    rc = hgt_typed_linear(L.g_act, d, L.wa_cat, L.ba_cat, d, d, a->upd_groups, a->h_upd_groups, a->n_upd_groups,
                          a->upd_cblocks, L.o, a->linear_impl, L.ws_upd, L.ws_upd_bytes + 256, stream);
  if (rc) return rc;
  const int32_t* perm_out = a->out_map ? a->out_map : a->perm;
  return hgt_update_epilogue_impl(L.o, x_sorted, a->type_row0, T, a->skip, nullptr, nullptr,
                                  a->use_norm ? a->norm_w : nullptr, a->use_norm ? a->norm_b : nullptr, perm_out,
                                  a->type_active, N, d, a->out, a->out_hi, a->out_lo, st);
}
