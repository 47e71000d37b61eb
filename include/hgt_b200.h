/* hgt_b200.h — C ABI of libhgt_b200.so: the B200 (sm_100a) implementation of pyHGT's HGTConv
 * message-passing hot path.
 *
 * Boundary being replaced (reference = acbull/pyHGT, paths relative to the reference root):
 *   pyHGT/conv.py:56-58    HGTConv.forward -> MessagePassing.propagate
 *   pyHGT/conv.py:60-111   HGTConv.message  (typed Q/K/V projections, relation_att / relation_msg,
 *                                           relation_pri, torch_geometric.utils.softmax by target)
 *   pyHGT/conv.py:114-134  HGTConv.update   (gelu, typed a_linear, sigmoid(skip) gate, LayerNorm)
 *   pyHGT/conv.py:283-299  RelTemporalEncoding
 *   third-party: torch_geometric 1.3.2 propagate/softmax, torch_scatter 1.3.2 scatter_add/max
 * The reference has no FFI of its own (pure Python); the Python class pyhgt_b200.HGTConv binds these
 * entry points with ctypes (see INTEGRATION.md for the stub a pyHGT maintainer would add).
 *
 * Conventions
 *   - Every function returns 0 on success, non-zero on error; hgt_last_error() then returns a
 *     thread-local, NUL-terminated description.  Nothing throws across the boundary.
 *   - All pointers are DEVICE pointers unless the parameter name starts with `h_`.
 *   - The caller owns every buffer (inputs, outputs, workspaces).  The library never allocates or frees
 *     device memory and never synchronises the stream unless the function's comment says so.
 *   - `stream` is a cudaStream_t passed as void* (so the header needs no CUDA include).
 *   - Internal node order ("rank order"): nodes sorted stably by node type.  rank[n] is the position of
 *     original node n, perm[k] the original id at position k.  All tables (Q, KV, agg) are in rank order.
 */
#ifndef HGT_B200_H
#define HGT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HGT_RTE_MAX_LEN 240 /* RelTemporalEncoding max_len, conv.py:287 */

const char* hgt_last_error(void);
int hgt_abi_version(void);
/* Number of CUDA kernels this library has launched so far in this process (diagnostics / bench.py). */
uint64_t hgt_kernel_launches(void);

/* ------------------------------------------------------------------------------------------------
 * Graph ingest: int64 COO (the tensors pyHGT/data.py:251-256 `to_torch` emits) -> plan arrays.
 * Replaces PyG propagate's per-layer index_select gathers and the T*T*R boolean triple masks
 * (conv.py:71-84) with one destination-sorted CSR built once per graph.
 * ---------------------------------------------------------------------------------------------- */

/* Bytes of scratch needed by hgt_plan_nodes / hgt_plan_edges_sort / hgt_plan_tiles. */
int hgt_plan_workspace_bytes(int64_t n_nodes, int64_t n_edges, size_t* out_bytes);

/* Stable sort of nodes by type.  rank/perm: [N] int32.  type_count: [T+1] int32 (bucket T collects nodes
 * whose type is outside [0,T): the reference leaves their output rows zero, conv.py:120-124).
 * sorted_flag[0] = 1 if node_type was already non-decreasing (then rank = perm = identity). */
int hgt_plan_nodes(const int64_t* node_type, int64_t n_nodes, int32_t num_types,
                   int32_t* rank, int32_t* perm, int32_t* type_count, int32_t* sorted_flag,
                   void* workspace, size_t workspace_bytes, void* stream);

/* Sort edges by destination rank (stable in original edge order).
 *   edge_index [2,E] int64 row-major (row 0 = source j, row 1 = target i; data.py:245,254)
 *   row_ptr [N+1] int32, csr_eid [E] int32 (CSR position -> original edge id),
 *   presence [T*R] int32: 1 where some valid edge has <source_type, relation> (the "pairs"),
 *   flags [4] int32: flags[0] != 0 => an endpoint id was outside [0,N). */
int hgt_plan_edges_sort(const int64_t* edge_index, const int64_t* edge_type, const int64_t* node_type,
                        const int32_t* rank, int64_t n_nodes, int64_t n_edges,
                        int32_t num_types, int32_t num_relations,
                        int32_t* row_ptr, int32_t* csr_eid, int32_t* presence, int32_t* flags,
                        void* workspace, size_t workspace_bytes, void* stream);

/* Per-CSR-edge gather indices.
 *   pair_of [T*R] int32: pair id of <source_type, relation> or -1;  pair_row0 [P] int32: first KV-table
 *   row of each pair;  type_row0 [T+1] int32: first rank of each type;  zero_row: index of the all-zero
 *   KV row used for edges that match no triple (score 0, message 0: conv.py:68-69).
 *   kv_row [E] int32;  rte_row [E] int32 (pair*240 + dt, or zero_rte_row) — pass NULL when edge_time is
 *   NULL.  flags[1] != 0 => an edge_time was outside [0,240) (nn.Embedding would raise, conv.py:299). */
int hgt_plan_edges_fill(const int64_t* edge_index, const int64_t* edge_type, const int64_t* edge_time,
                        const int64_t* node_type, const int32_t* rank, const int32_t* csr_eid,
                        int64_t n_nodes, int64_t n_edges, int32_t num_types, int32_t num_relations,
                        const int32_t* pair_of, const int32_t* pair_row0, const int32_t* type_row0,
                        int32_t zero_row, int32_t zero_rte_row,
                        int32_t* kv_row, int32_t* rte_row, int32_t* flags, void* stream);

/* Balanced work tiles for the edge kernel: consecutive destination ranks are grouped until a tile holds
 * about `target_edges` edges; a destination with more than `split_edges` in-edges is cut into several
 * tiles whose partial (max, sum, acc) are merged afterwards.
 *   tiles [max_tiles,4] int32 = {dst_begin, dst_end, edge_begin, edge_end}; for a split destination
 *   the second field is -(partial_slot+1) < 0 and [edge_begin, edge_end) is a sub-range of its segment.
 *   hubs [max_hubs,4] int32 = {dst, first partial slot, pieces, 0} for every split destination;
 *   n_tiles [3] int32 = {number of tiles, number of split (partial) tiles, number of hubs}.
 * Synchronises the stream (returns the counts to the host through h_n_tiles[3]) — unless h_n_tiles is NULL: then
 * nothing is read back or synchronised, the counts stay in d_n_tiles (pass it to the edge kernels as d_tile_counts)
 * and the caller sizes with the bounds  max_tiles >= (2E+N)/(2*target_edges) + 3*(E/split_edges) + 16,
 * max_hubs >= E/split_edges + 1,  split pieces <= 2*(E/split_edges) + 1. */
int hgt_plan_tiles(const int32_t* row_ptr, int64_t n_nodes, int64_t n_edges,
                   int32_t target_edges, int32_t split_edges,
                   int32_t* tiles, int64_t max_tiles, int32_t* hubs, int64_t max_hubs,
                   int32_t* d_n_tiles, int32_t* h_n_tiles,
                   void* workspace, size_t workspace_bytes, void* stream);

/* out[k,:] = in[perm[k],:]  (rows of `width` floats); used only when node_type is not pre-sorted. */
int hgt_gather_rows(const float* in, const int32_t* perm, int64_t n_rows, int32_t width,
                    float* out, void* stream);

/* Multi-GPU halo exchange fused into one kernel: out[i,:] = peer[src_rank[i]][src_row[i],:], where
 * peer_ptrs_dev is the DEVICE address of an array of world_size device pointers to every rank's [rows,width]
 * feature buffer (NVLink peer mappings, e.g. torch symmetric memory `buffer_ptrs_dev`); `row_base` is added to every
 * src_row (double-buffered publish areas inside one symmetric allocation).  The caller orders the ranks: publish ->
 * barrier -> pull; with two publish areas used alternately that ONE barrier per exchange also guarantees that nobody
 * still reads the area about to be overwritten.  width % 4 == 0. */
int hgt_halo_pull(uint64_t peer_ptrs_dev, const int32_t* src_rank, const int32_t* src_row, int64_t n_rows,
                  int32_t width, int64_t row_base, float* out, void* stream);
/* Same pull fused with the operand conversion of the projection GEMM: every row is written as the bf16 hi/lo split
 * (hi/lo [n_rows, width], the A operand of hgt_typed_linear_presplit) while it crosses NVLink; the fp32 copy is kept
 * only for rows owned by `self_rank` (the update epilogue's skip connection reads those).  width % 8 == 0.
 * `order` (NULL = 0..n_rows-1): the sequence in which the rows are processed; a sequence that cycles through the owners
 * (and starts at a different owner on every rank) keeps every NVLink source evenly loaded. */
int hgt_halo_pull_split(uint64_t peer_ptrs_dev, const int32_t* src_rank, const int32_t* src_row,
                        const int32_t* order, int64_t n_rows, int32_t width, int32_t self_rank, int64_t row_base,
                        float* out_f32, void* hi, void* lo, void* stream);

/* Push variant of the fused exchange (experimental): the OWNER converts its rows and stores the bf16 hi/lo split straight
 * into the consumers' operand buffers (posted NVLink writes).  Item i: row push_src[i] of x_own [rows, width] -> row
 * row_base + push_dst[i] of rank push_peer[i]'s hi / lo buffers (hi_ptrs_dev / lo_ptrs_dev: DEVICE arrays of world_size
 * device pointers, peer mappings); items addressed to self_rank also write the fp32 row into x_local_f32.  The caller
 * orders the ranks (push -> barrier -> consume; two destination areas used alternately).  width % 8 == 0. */
int hgt_halo_push_split(const float* x_own, const int32_t* push_peer, const int32_t* push_src, const int32_t* push_dst,
                        int64_t n_items, int32_t width, int32_t self_rank, int64_t row_base, uint64_t hi_ptrs_dev,
                        uint64_t lo_ptrs_dev, float* x_local_f32, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Typed (per-node-type) linear layers — "per-type linear dispatch" (conv.py:73-77,96-97,103,125).
 * ---------------------------------------------------------------------------------------------- */

typedef struct {
  int64_t a_row0;    /* first row of A used by this group                                   */
  int64_t m;         /* rows in this group (nodes of this type; 240 for the RTE tables)      */
  int32_t w_row0;    /* first row of the concatenated weight matrix W [sum n_out, K]         */
  int32_t n_cblocks; /* output column blocks of width `cb_width` each                        */
  int32_t cb_first;  /* index of this group's first entry in the column-block table          */
  int32_t has_bias;
} hgt_lin_group;

typedef struct {
  int64_t out_off;   /* element offset of (group row 0, column 0 of this block) from `out`   */
  int64_t ld;        /* elements between consecutive rows of this block's destination        */
} hgt_lin_cblock;

/* Fold the relation matrices into per-<source type, relation> weights (SURVEY.md §8 a4):
 *   W_cat rows for type t: [ W_q^t ; for each pair p=(t,r): K'_p ; V'_p ]  with
 *   K'_p[h*dk+c,:] = pri[r,h]/sqrt(dk) * sum_a att[r,h,a,c] * W_k^t[h*dk+a,:]   (conv.py:97-99)
 *   V'_p[h*dk+c,:] =                     sum_a msg[r,h,a,c] * W_v^t[h*dk+a,:]   (conv.py:103-104)
 * and the same for the biases.  wq/wk/wv/bq/bk/bv are DEVICE arrays of T device pointers (one
 * nn.Linear per type, conv.py:34-38).  pair_type/pair_rel: [P] int32; cat_row0: [P] int32 first W_cat
 * row of the pair's K' block (V' follows at +d_out); q_row0: [T] int32 first W_cat row of W_q^t. */
int hgt_fold_weights(const float* const* wq, const float* const* bq,
                     const float* const* wk, const float* const* bk,
                     const float* const* wv, const float* const* bv,
                     const float* relation_att, const float* relation_msg, const float* relation_pri,
                     int32_t num_types, int32_t num_relations, int32_t n_heads, int32_t d_in, int32_t d_out,
                     int32_t n_pairs, const int32_t* pair_type, const int32_t* pair_rel,
                     const int32_t* cat_row0, const int32_t* q_row0,
                     float* w_cat, float* b_cat, void* stream);

/* Concatenate T per-type [rows,cols] matrices (and [rows] biases) into one: w_cat [T*rows, cols]. */
int hgt_concat_linears(const float* const* w, const float* const* b, int32_t num_types,
                       int32_t rows, int32_t cols, float* w_cat, float* b_cat, void* stream);

/* RelTemporalEncoding (conv.py:299) needs no entry point of its own: RT = emb.weight @ lin.weight^T + lin.bias
 * [240,d] is one hgt_typed_linear call, and its projection through every pair's K'/V' weights another. */

/* out[cblock c of group g][m, n] = sum_k A[a_row0_g + m, k] * W[w_row0_g + c*cb_width + n, k] (+ bias).
 * fp32 in / fp32 out.  `impl`: 0 = auto, 1 = SIMT fp32 FMA kernel, 2 = tcgen05 split-bf16 tensor-core
 * kernel (three bf16 products of a hi/lo operand split accumulated in one fp32 TMEM accumulator: accurate
 * to ~1e-5 relative; needs cb_width % 16 == 0 and K >= 64, workspace for the split operands).
 * groups/cblocks are DEVICE arrays; h_groups is the same table on the host (used to size the grid; no
 * device read-back). */
int hgt_typed_linear_workspace_bytes(const hgt_lin_group* h_groups, int32_t n_groups, int32_t K,
                                     int32_t cb_width, int32_t impl, size_t* out_bytes);
int hgt_typed_linear(const float* A, int64_t lda, const float* W, const float* bias, int32_t K,
                     int32_t cb_width, const hgt_lin_group* groups, const hgt_lin_group* h_groups,
                     int32_t n_groups, const hgt_lin_cblock* cblocks, float* out, int32_t impl,
                     void* workspace, size_t workspace_bytes, void* stream);
/* Same product on the tensor-core kernel with the A operand already split by its producer: a_hi / a_lo are bf16
 * [rows, K] (K % 8 == 0, row stride K).  Saves the split pass over A (workspace: W split only). */
int hgt_typed_linear_presplit_workspace_bytes(const hgt_lin_group* h_groups, int32_t n_groups, int32_t K,
                                              int32_t cb_width, size_t* out_bytes);
int hgt_typed_linear_presplit(const void* a_hi, const void* a_lo, const float* W, const float* bias, int32_t K,
                              int32_t cb_width, const hgt_lin_group* groups, const hgt_lin_group* h_groups,
                              int32_t n_groups, const hgt_lin_cblock* cblocks, float* out,
                              void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused edge kernel: gather -> relation-specific score -> softmax by destination -> weighted sum
 * (conv.py:99,108-111 + PyG scatter-add), one pass over the destination-sorted CSR.
 * ---------------------------------------------------------------------------------------------- */

/*  q       [N, d]        rank order, Q[i] = W_q^{type(i)} x_i + b
 *  kv      [rows+1, 2d]  row = [K' | V'] of <source node, relation>; last row all zero
 *  kvr     [P*240+1, 2d] RTE contribution per <pair, dt> (NULL when !use_RTE); last row all zero
 *  tiles / hubs from hgt_plan_tiles;  partial workspace: n_split * (2*H + d) floats
 *  agg_out [N, d]  gelu(sum_e att[e] * V'[e]) if apply_gelu else the raw sum   (conv.py:119)
 *  att_out [E, H]  softmax weights in ORIGINAL edge order (conv.py:108 `self.att`) or NULL
 *  stats_out [N, 2H] per-destination (max, sum) per head, or NULL (kept for the backward pass)
 *  g_hi / g_lo [N, d] bf16 or NULL: the same result as a bf16 hi/lo split (x = hi + lo to ~2^-17), i.e. the
 *           pre-split A operand of hgt_typed_linear_presplit; agg_out may then be NULL.  Needs d % 8 == 0.
 *  variant: 0 = auto, 1 = direct register gather (LDG), 2 = bulk-async-copy shared-memory ring (TMA)
 *  d_tile_counts: NULL, or the device counts {n_tiles, n_split, n_hubs} hgt_plan_tiles wrote in its sync-free mode; then
 *           n_tiles / n_split_tiles / n_hubs are the UPPER BOUNDS the arrays were sized with and the kernels read the
 *           true counts from the device (no host read-back between plan build and layer).
 *  type_row0 [T+2] / type_active [T]: NULL, or (sharded runs) the same tables hgt_update_epilogue takes: destinations
 *           past the active prefix of their type are halo sources — they have no in-edges and no output row is written. */
int hgt_edge_workspace_bytes(int32_t n_split_tiles, int32_t d, int32_t n_heads, size_t* out_bytes);
int hgt_edge_forward(const float* q, const float* kv, const float* kvr,
                     const int32_t* row_ptr, const int32_t* kv_row, const int32_t* rte_row,
                     const int32_t* csr_eid, const int32_t* tiles, int32_t n_tiles, int32_t n_split_tiles,
                     const int32_t* hubs, int32_t n_hubs,
                     int64_t n_nodes, int64_t n_edges, int32_t d, int32_t n_heads, int32_t apply_gelu,
                     float* agg_out, float* att_out, float* stats_out, void* g_hi, void* g_lo,
                     void* workspace, size_t workspace_bytes, int32_t variant, const int32_t* d_tile_counts,
                     const int32_t* type_row0, int32_t num_types, const int32_t* type_active, void* stream);

/* Backward of hgt_edge_forward (training; the reference differentiates the same ops with autograd,
 * OAG/train_paper_field.py:249).  Inputs: the forward's q / kv / kvr tables, its un-activated output
 * `agg` (apply_gelu = 0), the saved per-destination softmax statistics `stats` [N,2H] and the incoming
 * gradient `dagg` [N,d].  Outputs (ZERO-INITIALISED BY THIS CALL, on the stream): dq [N,d],
 * dkv [kv_rows_total, 2d] (gradient of the [K'|V'] table; kv_rows_total counts the trailing all-zero row, whose
 * gradient is to be discarded), dkvr [kvr_rows_total, 2d] or NULL.  workspace: >= 256 bytes. */
int hgt_edge_backward(const float* q, const float* kv, const float* kvr, const float* agg, const float* dagg,
                      const float* stats, const int32_t* row_ptr, const int32_t* kv_row, const int32_t* rte_row,
                      const int32_t* tiles, int32_t n_tiles, int64_t n_nodes, int32_t d, int32_t n_heads,
                      int64_t kv_rows_total, int64_t kvr_rows_total,
                      float* dq, float* dkv, float* dkvr, void* workspace, size_t workspace_bytes,
                      const int32_t* d_tile_counts, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Deterministic backward (the path pyhgt_b200 takes under torch.use_deterministic_algorithms(True)).
 * Same results as the default backward up to the order of floating-point sums, but every sum runs in an order fixed
 * by the problem shape: no floating-point atomics, and no partitioning that depends on the card.  Two runs on the same
 * inputs give the same bits.  Each *_det call takes its non-det sibling's arguments plus a workspace sized by its
 * *_workspace_bytes query; none allocates or synchronises.
 * ---------------------------------------------------------------------------------------------- */

/* Stable group-by: ptr [n_keys+1] = exclusive prefix of the key histogram; pos [n] = the positions i of key[i] grouped
 * by key, increasing inside each group (stable radix sort).  Keys must lie in [0, n_keys). */
int hgt_plan_group_by_workspace_bytes(int64_t n, int32_t n_keys, size_t* out_bytes);
int hgt_plan_group_by(const int32_t* key, int64_t n, int32_t n_keys, int32_t* ptr, int32_t* pos, void* workspace,
                      size_t workspace_bytes, void* stream);
/* csr_dst [n_edges]: the destination (rank) of every position of the destination-sorted CSR row_ptr [n_nodes+1]. */
int hgt_plan_csr_dst(const int32_t* row_ptr, int64_t n_nodes, int64_t n_edges, int32_t* csr_dst, void* stream);

/* One edge index for the deterministic edge backward: segments ptr [n_keys+1] over the CSR positions pos (pos NULL:
 * the positions themselves, i.e. the destination CSR), cut into tiles / hubs by hgt_plan_tiles over ptr.  n_tiles,
 * n_split, n_hubs: exact counts, or with d_counts (hgt_plan_tiles' sync-free mode) the bounds the arrays were sized with. */
typedef struct {
  const int32_t* ptr;
  const int32_t* pos;
  const int32_t* tiles;
  const int32_t* hubs;
  const int32_t* d_counts;
  int32_t n_tiles, n_split, n_hubs, reserved;
} hgt_tile_set;

/* Deterministic hgt_edge_backward.  dst: the destination CSR (row_ptr, tiles / hubs of the forward); src: the CSR
 * positions grouped by kv_row (n_keys = kv_rows_total, trailing zero row included); rte: grouped by rte_row
 * (n_keys = P*240+1), or NULL without RTE.  csr_dst from hgt_plan_csr_dst.  Every row of dq [N,d], dkv [kv_rows_total,2d]
 * and dkvr [P*240+1,2d] is written (rows without edges as zeros): no zero-initialisation is needed. */
int hgt_edge_backward_det_workspace_bytes(int64_t n_nodes, int32_t d, int32_t n_heads, const hgt_tile_set* dst,
                                          const hgt_tile_set* src, const hgt_tile_set* rte, size_t* out_bytes);
int hgt_edge_backward_det(const float* q, const float* kv, const float* kvr, const float* agg, const float* dagg,
                          const float* stats, const int32_t* kv_row, const int32_t* rte_row, const int32_t* csr_dst,
                          const hgt_tile_set* dst, const hgt_tile_set* src, const hgt_tile_set* rte, int64_t n_nodes,
                          int32_t d, int32_t n_heads, float* dq, float* dkv, float* dkvr, void* workspace,
                          size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Backward of the typed linears (training path).  For the group / column-block tables of the forward call:
 *   dA[a_row0_g + m, k]             = sum_c sum_n dOut_c[m, n] * W[w_row0_g + c*cb_width + n, k]   (* gelu'(gelu_aux) if given)
 *   dW[w_row0_g + c*cb_width + n,k] += sum_m dOut_c[m, n] * A[a_row0_g + m, k]
 *   db[w_row0_g + c*cb_width + n]   += sum_m dOut_c[m, n]           (groups with has_bias)
 * dout has the layout of the forward's `out` (flat buffer addressed through the column-block table, dout_elems
 * elements).  dW / db are ACCUMULATED INTO (several groups may share W rows: the caller zero-initialises them once per
 * step); dA is written (rows BETWEEN / BEFORE the groups that no group covers are zeroed; rows past the last group are the
 * caller's) unless accumulate_dA != 0, in which case the product is added to its current content.  dA / dW / db may each be NULL to skip that product.
 * Tensor-core path (impl 0 = auto, 2 = force): tcgen05 split-bf16 x3 like the forward; takes the operands either as
 * fp32 (split here; the dout split pass also yields db) or already split by their producers (dout_hi/lo in dout's
 * layout; a_hi/a_lo [rows, K] as left by hgt_act_split in the forward) — with a pre-split dout, db is NOT computed.
 * impl 1 = fp32 SIMT kernels (any shape; also chosen automatically for cb_width % 8, K % 16, K < 64, overlapping groups
 * such as the RTE tables, or tiny problems).  h_cblocks: HOST copy of the column-block table. */
int hgt_typed_linear_bwd_workspace_bytes(const hgt_lin_group* h_groups, int32_t n_groups, const hgt_lin_cblock* h_cblocks,
                                         int32_t K, int32_t cb_width, int64_t lda, int64_t dout_elems,
                                         int32_t have_dout_split, int32_t have_a_split, int32_t impl, size_t* out_bytes);
int hgt_typed_linear_bwd(const float* dout, const void* dout_hi, const void* dout_lo, int64_t dout_elems,
                         const float* A, int64_t lda, const void* a_hi, const void* a_lo,
                         const float* W, int32_t K, int32_t cb_width, const hgt_lin_group* groups,
                         const hgt_lin_group* h_groups, int32_t n_groups, const hgt_lin_cblock* h_cblocks,
                         float* dA, int32_t accumulate_dA, const float* gelu_aux, float* dW, float* db,
                         int32_t impl, void* workspace, size_t workspace_bytes, void* stream);

/* Deterministic hgt_typed_linear_bwd (same arguments and semantics): partial dW / db tiles go to the workspace and are
 * summed in chunk order; the SIMT dA walks overlapping groups in group order. */
int hgt_typed_linear_bwd_det_workspace_bytes(const hgt_lin_group* h_groups, int32_t n_groups,
                                             const hgt_lin_cblock* h_cblocks, int32_t K, int32_t cb_width, int64_t lda,
                                             int64_t dout_elems, int32_t have_dout_split, int32_t have_a_split,
                                             int32_t impl, size_t* out_bytes);
int hgt_typed_linear_bwd_det(const float* dout, const void* dout_hi, const void* dout_lo, int64_t dout_elems,
                             const float* A, int64_t lda, const void* a_hi, const void* a_lo,
                             const float* W, int32_t K, int32_t cb_width, const hgt_lin_group* groups,
                             const hgt_lin_group* h_groups, int32_t n_groups, const hgt_lin_cblock* h_cblocks,
                             float* dA, int32_t accumulate_dA, const float* gelu_aux, float* dW, float* db,
                             int32_t impl, void* workspace, size_t workspace_bytes, void* stream);

/* act(in) as fp32 (out_f32 [rows, K], or NULL) and/or as the bf16 hi/lo operand split (hi/lo [rows, K], or NULL; needs
 * K % 8 == 0).  act: 0 = identity, 1 = exact-erf gelu (conv.py:119).  The training forward keeps the split for the
 * backward pass (it is the A operand of the dW product). */
int hgt_act_split(const float* in, int64_t ld, int64_t rows, int32_t K, int32_t act, float* out_f32,
                  void* hi, void* lo, void* stream);

/* Backward of hgt_update_epilogue (conv.py:129-133).  dout [N,d] in ORIGINAL node order (perm as in the forward);
 * o / x [N,d] rank order (the forward's inputs); norm_w [T,d] or NULL.  Outputs: d_o, d_x [N,d] rank order (rows of
 * out-of-range type get zeros), d_skip [T], d_norm_w / d_norm_b [T,d] (zero-initialised by this call).
 * skip == NULL: residual mode (y = o + x), d_skip is not touched.  type_active as in the forward: rows past
 * type_active[t] get zero gradients and their (never computed) `o` rows are not read. */
int hgt_update_backward(const float* dout, const float* o, const float* x, const int32_t* type_row0, int32_t num_types,
                        const float* skip, const float* norm_w, const int32_t* perm, const int32_t* type_active,
                        int64_t n_nodes, int32_t d,
                        float* d_o, float* d_x, float* d_skip, float* d_norm_w, float* d_norm_b, void* stream);
/* Deterministic hgt_update_backward: per-warp partial sums of d skip / d norm in the workspace, summed in row order. */
int hgt_update_backward_det_workspace_bytes(int64_t n_nodes, int32_t num_types, int32_t d, size_t* out_bytes);
int hgt_update_backward_det(const float* dout, const float* o, const float* x, const int32_t* type_row0,
                            int32_t num_types, const float* skip, const float* norm_w, const int32_t* perm,
                            const int32_t* type_active, int64_t n_nodes, int32_t d, float* d_o, float* d_x,
                            float* d_skip, float* d_norm_w, float* d_norm_b, void* workspace, size_t workspace_bytes,
                            void* stream);

/* Backward of hgt_fold_weights for the K'/V' blocks: from d W_cat / d b_cat to the gradients of k_linears / v_linears
 * (stacked [T, d_out, d_in] / [T, d_out]) and relation_att / relation_msg [R,H,dk,dk], relation_pri [R,H]; all outputs
 * are zero-initialised by this call.  (The W_q rows of W_cat are plain copies: their gradient is the matching slice.) */
int hgt_fold_backward(const float* d_w_cat, const float* d_b_cat, const float* const* wk, const float* const* bk,
                      const float* const* wv, const float* const* bv, const float* relation_att,
                      const float* relation_msg, const float* relation_pri, int32_t num_types, int32_t num_relations,
                      int32_t n_heads, int32_t d_in, int32_t d_out, int32_t n_pairs, const int32_t* pair_type,
                      const int32_t* pair_rel, const int32_t* cat_row0, float* d_wk, float* d_bk, float* d_wv,
                      float* d_bv, float* d_att, float* d_msg, float* d_pri, void* stream);
/* Deterministic hgt_fold_backward: each type (relation) sums its pairs in pair order. */
int hgt_fold_backward_det_workspace_bytes(int32_t num_relations, int32_t n_heads, int32_t d_out, size_t* out_bytes);
int hgt_fold_backward_det(const float* d_w_cat, const float* d_b_cat, const float* const* wk, const float* const* bk,
                          const float* const* wv, const float* const* bv, const float* relation_att,
                          const float* relation_msg, const float* relation_pri, int32_t num_types,
                          int32_t num_relations, int32_t n_heads, int32_t d_in, int32_t d_out, int32_t n_pairs,
                          const int32_t* pair_type, const int32_t* pair_rel, const int32_t* cat_row0, float* d_wk,
                          float* d_bk, float* d_wv, float* d_bv, float* d_att, float* d_msg, float* d_pri,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Update epilogue (conv.py:129-133): y = o*sigmoid(skip[t]) + x*(1-sigmoid(skip[t])); LayerNorm_t(y)
 * (eps 1e-5, affine) iff use_norm; rows of out-of-range type are written as zeros (conv.py:120).
 * skip == NULL selects the plain residual y = o + x of DenseHGTConv (conv.py:261,273).
 *   o [N,d] rank order (a_linear output, after dropout if training);  x [N,d] rank order;
 *   type_row0 [T+2] int32 prefix of type_count;  norm_w/norm_b [T,d] or NULL;  perm NULL if identity;
 *   type_active [T] int32 or NULL: when given, only the first type_active[t] rows of type t are written
 *   (sharded runs: the remaining rows are halo sources that need no output);
 *   out [N,d] in ORIGINAL node order;
 *   out_hi / out_lo [N,d] bf16 or NULL: `out` again as the bf16 hi/lo split that the NEXT layer's projection GEMM
 *   consumes (hgt_typed_linear_presplit) — only with perm == NULL, type_active == NULL, d % 8 == 0.
 * ---------------------------------------------------------------------------------------------- */
int hgt_update_epilogue(const float* o, const float* x, const int32_t* type_row0, int32_t num_types,
                        const float* skip, const float* norm_w, const float* norm_b,
                        const int32_t* perm, const int32_t* type_active, int64_t n_nodes, int32_t d,
                        float* out, void* out_hi, void* out_lo, void* stream);


/* ------------------------------------------------------------------------------------------------
 * Whole layer in one call (inference): HGTConv.forward, pyHGT/conv.py:56-134.
 * Every pointer below is a DEVICE pointer except the h_* tables (host copies of the typed-linear group tables, used
 * only to size grids).  Parameter pointer tables (wq ... norm_b) are device arrays of num_types device pointers, one
 * per nn.Linear / nn.LayerNorm of the module (conv.py:34-40).  The plan arrays come from hgt_plan_*; the typed-linear
 * tables are the ones hgt_typed_linear takes (projection: Q + [K'|V'] blocks; rte: K'R/V'R tables; rt: the single
 * 240 x d group of RelTemporalEncoding.lin; upd: a_linears).  Nothing is allocated or synchronised.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  /* sizes and switches */
  int64_t n_nodes, n_edges, kv_rows, cat_rows, q_off, kv_off, proj_elems;
  int32_t num_types, num_relations, n_heads, d_in, d_out, n_pairs;
  int32_t use_rte, use_norm, edge_variant, linear_impl;
  int32_t n_tiles, n_split, n_hubs;
  int32_t n_proj_groups, n_rte_groups, n_upd_groups;
  /* plan (hgt_plan_*) */
  const int32_t* perm;        /* NULL when node_type is already sorted */
  const int32_t* type_row0;   /* [T+2] */
  const int32_t* type_active; /* [T] or NULL (sharded runs) */
  const int32_t* out_map;     /* [N] or NULL: rank-order row -> output row (sharded runs) */
  const int32_t* row_ptr;
  const int32_t* kv_row;
  const int32_t* rte_row;     /* NULL when !use_rte */
  const int32_t* csr_eid;
  const int32_t* tiles;
  const int32_t* hubs;
  const int32_t* d_tile_counts; /* NULL, or device {n_tiles, n_split, n_hubs}: n_tiles/n_split/n_hubs above are bounds */
  const int32_t* pair_type;
  const int32_t* pair_rel;
  const int32_t* cat_row0;
  const int32_t* q_row0;
  /* typed-linear tables */
  const hgt_lin_group* proj_groups; const hgt_lin_group* h_proj_groups; const hgt_lin_cblock* proj_cblocks;
  const hgt_lin_group* rte_groups;  const hgt_lin_group* h_rte_groups;  const hgt_lin_cblock* rte_cblocks;
  const hgt_lin_group* rt_groups;   const hgt_lin_group* h_rt_groups;   const hgt_lin_cblock* rt_cblocks;
  const hgt_lin_group* upd_groups;  const hgt_lin_group* h_upd_groups;  const hgt_lin_cblock* upd_cblocks;
  /* parameters */
  const float* const* wq; const float* const* bq;
  const float* const* wk; const float* const* bk;
  const float* const* wv; const float* const* bv;
  const float* const* wa; const float* const* ba;
  const float* const* norm_w; const float* const* norm_b;   /* NULL when !use_norm */
  const float* relation_att; const float* relation_msg; const float* relation_pri; const float* skip;
  const float* emb_weight; const float* emb_lin_w; const float* emb_lin_b;   /* NULL when !use_rte */
  /* data */
  const float* x;             /* [N, d_in] in original node order */
  const void* x_hi; const void* x_lo;   /* optional: x already split to bf16 hi/lo (rank order == original order) */
  float* out;                 /* [N or out rows, d_out] */
  float* att;                 /* [E, H] or NULL */
  void* out_hi; void* out_lo; /* optional: out again as the bf16 hi/lo split for the next layer */
} hgt_conv_args;

uint64_t hgt_conv_args_size(void);   /* sizeof(hgt_conv_args): lets a foreign-language binding check its struct layout */
int hgt_conv_workspace_bytes(const hgt_conv_args* args, size_t* out_bytes);
int hgt_conv_forward(const hgt_conv_args* args, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * HOST helper of HGSampling (pyHGT/data.py:123-130; pyhgt_b200/sampler.py): every pointer is a HOST pointer, nothing
 * touches the GPU.  Applies the sampled neighbours of one <target type, source type, relation> adjacency slice to the
 * budget of the source type (flat arrays over node ids; `stamp` reproduces the reference dict's insertion order).
 * Returns the number of budget entries added / updated, -1 if an id lies outside [0, n). */
int64_t hgt_sampler_budget_update(const int64_t* h_ids, const int64_t* h_times, int64_t n_sampled, int64_t target_time,
                                  int64_t no_time, int64_t max_time, int64_t n, const uint8_t* h_in_layer,
                                  uint8_t* h_in_budget, double* h_score, int64_t* h_budget_time, int64_t* h_stamp,
                                  int64_t* h_stamp_counter, int32_t* h_touched_layer);

/* One <target type, source type, relation> adjacency of the frozen graph in CSR form (host arrays; rows in the
 * reference dict's insertion order) and the layer_data / budget of one node type as flat arrays over node ids. */
typedef struct {
  const int64_t* row_of; int64_t n_row_of;   /* target id -> CSR row, -1 = no adjacency */
  const int64_t* ptr; const int64_t* nbr; const int64_t* time;
  int32_t src_state;                         /* index of the source type's hgt_sampler_state */
  int32_t skip;                              /* 1 for the 'self' relation (data.py:116) */
} hgt_sampler_block;
typedef struct {
  int64_t n;
  uint8_t* in_layer; uint8_t* in_budget; double* score; int64_t* b_time; int64_t* stamp;
  int64_t* log; int64_t log_len;             /* ids in budget-insertion order (capacity n) */
  int64_t layer_seq; int64_t budget_seq;     /* first-touch numbers of layer_data[type] / budget[type], -1 = untouched */
} hgt_sampler_state;
/* add_budget (pyHGT/data.py:108-130) for a batch of target nodes of one type, target-major, blocks in dict order; the
 * uniform draws are made by the caller (numpy's global RNG, same order) and passed as positions.  0 = ok. */
int64_t hgt_sampler_add_budget(const int64_t* h_target_ids, const int64_t* h_target_times, int64_t n_targets,
                               const hgt_sampler_block* h_blocks, int32_t n_blocks, hgt_sampler_state* h_states,
                               int32_t n_states, int64_t sampled_number, const int64_t* h_draw_off,
                               const int64_t* h_draw_pos, int64_t no_time, int64_t max_time, int64_t* h_counters);

#ifdef __cplusplus
}
#endif
#endif /* HGT_B200_H */
