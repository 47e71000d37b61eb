// Typed (per-node-type) linear layers of HGTConv: weight folding (relation_att / relation_msg /
// relation_pri into the K/V projections, SURVEY.md §8 a4) and the grouped GEMM front end.
// This file holds the fp32 SIMT kernel (impl 1); the tcgen05 tensor-core kernel (impl 2) lives in
// linear_tc.cu and is dispatched from hgt_typed_linear below.
#include "common.cuh"

int hgt_typed_linear_tc(const float* A, int64_t lda, const float* W, const float* bias, int32_t K,
                        int32_t cb_width, const hgt_lin_group* groups, const hgt_lin_group* h_groups,
                        int32_t n_groups, const hgt_lin_cblock* cblocks, float* out, void* workspace,
                        size_t workspace_bytes, cudaStream_t st);
int hgt_typed_linear_tc(const float* A, int64_t lda, const float* W, const float* bias, int32_t K,
                        int32_t cb_width, const hgt_lin_group* groups, const hgt_lin_group* h_groups,
                        int32_t n_groups, const hgt_lin_cblock* cblocks, __nv_bfloat16* out, void* workspace,
                        size_t workspace_bytes, cudaStream_t st);
bool hgt_typed_linear_tc_supported(int64_t lda, int32_t K, int32_t cb_width);
size_t hgt_typed_linear_tc_workspace(const hgt_lin_group* h_groups, int32_t n_groups, int32_t K, int32_t cb_width);

namespace {

constexpr int kMaxGroups = 64;

// ---- weight folding ----------------------------------------------------------------------------
// One thread per element of a K' or V' block (column index d_in is the bias).
__global__ void k_fold_pairs(const float* const* __restrict__ wk, const float* const* __restrict__ bk,
                             const float* const* __restrict__ wv, const float* const* __restrict__ bv,
                             const float* __restrict__ rel_att, const float* __restrict__ rel_msg,
                             const float* __restrict__ rel_pri, int H, int d_in, int d_out, int n_pairs,
                             const int32_t* __restrict__ pair_type, const int32_t* __restrict__ pair_rel,
                             const int32_t* __restrict__ cat_row0, float* __restrict__ w_cat,
                             float* __restrict__ b_cat) {
  const int dk = d_out / H;
  const int64_t per_block = (int64_t)d_out * (d_in + 1);
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= per_block * 2 * n_pairs) return;
  int p = (int)(i / (2 * per_block));
  int64_t rem = i - (int64_t)p * 2 * per_block;
  int which = (int)(rem / per_block);          // 0 = K', 1 = V'
  rem -= which * per_block;
  int row = (int)(rem / (d_in + 1));
  int col = (int)(rem - (int64_t)row * (d_in + 1));
  int h = row / dk, c = row - h * dk;
  int t = pair_type[p], r = pair_rel[p];
  const float* rel = (which ? rel_msg : rel_att) + ((int64_t)(r * H + h) * dk) * dk;   // [a][c]
  const float* w = which ? wv[t] : wk[t];
  const float* b = which ? bv[t] : bk[t];
  float acc = 0.f;
  if (col < d_in) {
    for (int a = 0; a < dk; ++a) acc = fmaf(rel[a * dk + c], w[(int64_t)(h * dk + a) * d_in + col], acc);
  } else {
    for (int a = 0; a < dk; ++a) acc = fmaf(rel[a * dk + c], b[h * dk + a], acc);
  }
  if (!which) acc *= rel_pri[r * H + h] * rsqrtf((float)dk);   // conv.py:99
  int64_t out_row = (int64_t)cat_row0[p] + which * d_out + row;
  if (col < d_in) w_cat[out_row * d_in + col] = acc;
  else b_cat[out_row] = acc;
}

__global__ void k_copy_linears(const float* const* __restrict__ w, const float* const* __restrict__ b, int T,
                               int rows, int cols, const int32_t* __restrict__ row0,
                               float* __restrict__ w_cat, float* __restrict__ b_cat) {
  const int64_t per = (int64_t)rows * (cols + 1);
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= per * T) return;
  int t = (int)(i / per);
  int64_t rem = i - (int64_t)t * per;
  int row = (int)(rem / (cols + 1));
  int col = (int)(rem - (int64_t)row * (cols + 1));
  int64_t out_row = (row0 ? (int64_t)row0[t] : (int64_t)t * rows) + row;
  if (col < cols) w_cat[out_row * cols + col] = w[t][(int64_t)row * cols + col];
  else b_cat[out_row] = b[t][row];
}

// ---- fp32 SIMT grouped GEMM --------------------------------------------------------------------
constexpr int BM = 128, BN = 64, BK = 16, GEMM_THREADS = 256;
constexpr int LDA_S = BM + 4, LDW_S = BN + 4;

struct TilePrefix {
  int32_t first_tile[kMaxGroups + 1];
  int32_t n_tiles_n;   // n-tiles per column block
};

template <typename OutT>
__global__ void __launch_bounds__(GEMM_THREADS)
k_typed_linear_simt(const float* __restrict__ A, int64_t lda, const float* __restrict__ W,
                    const float* __restrict__ bias, int K, int cb_width,
                    const hgt_lin_group* __restrict__ groups, int n_groups,
                    const hgt_lin_cblock* __restrict__ cblocks, OutT* __restrict__ out, TilePrefix tp) {
  __shared__ __align__(16) float As[BK][LDA_S];
  __shared__ __align__(16) float Ws[BK][LDW_S];
  int tile = blockIdx.x;
  int g = 0;
  while (g + 1 < n_groups && tile >= tp.first_tile[g + 1]) ++g;
  const hgt_lin_group grp = groups[g];
  int local = tile - tp.first_tile[g];
  const int per_m = grp.n_cblocks * tp.n_tiles_n;
  const int mt = local / per_m;
  local -= mt * per_m;
  const int cb = local / tp.n_tiles_n;
  const int nt = local - cb * tp.n_tiles_n;
  const hgt_lin_cblock cblk = cblocks[grp.cb_first + cb];

  const int64_t m0 = (int64_t)mt * BM;                      // row within group
  const int n0 = nt * BN;                                    // column within the block
  const int64_t w_row0 = (int64_t)grp.w_row0 + (int64_t)cb * cb_width + n0;
  const int rows_here = (int)min((int64_t)BM, grp.m - m0);
  const int cols_here = min(BN, cb_width - n0);

  const int tid = threadIdx.x;
  const int tm = tid / 16, tn = tid % 16;
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const float* Ag = A + (grp.a_row0 + m0) * lda;
  const float* Wg = W + w_row0 * (int64_t)K;

  for (int k0 = 0; k0 < K; k0 += BK) {
    // A tile: 128 rows x 16 k  (8 elements per thread), W tile: 64 rows x 16 k (4 per thread)
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      int idx = tid + it * GEMM_THREADS;       // 0..2047
      int r = idx / BK, kk = idx % BK;
      float v = 0.f;
      if (r < rows_here && k0 + kk < K) v = Ag[(int64_t)r * lda + k0 + kk];
      As[kk][r] = v;
    }
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      int idx = tid + it * GEMM_THREADS;       // 0..1023
      int r = idx / BK, kk = idx % BK;
      float v = 0.f;
      if (r < cols_here && k0 + kk < K) v = Wg[(int64_t)r * K + k0 + kk];
      Ws[kk][r] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float4 a0 = *reinterpret_cast<const float4*>(&As[kk][tm * 8]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[kk][tm * 8 + 4]);
      float4 b0 = *reinterpret_cast<const float4*>(&Ws[kk][tn * 4]);
      float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float b[4] = {b0.x, b0.y, b0.z, b0.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  float bj[4] = {0.f, 0.f, 0.f, 0.f};
  if (grp.has_bias && bias) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (tn * 4 + j < cols_here) bj[j] = bias[w_row0 + tn * 4 + j];
  }
  OutT* Og = out + cblk.out_off + m0 * cblk.ld + n0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int r = tm * 8 + i;
    if (r >= rows_here) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int c = tn * 4 + j;
      if (c < cols_here) hgt_store_out(Og + (int64_t)r * cblk.ld + c, acc[i][j] + bj[j]);
    }
  }
}

// hgt_typed_linear for either output type: the fp32 and the bf16 entry points share dispatch, kernels and accumulation
// order, so the bf16 result is the fp32 result rounded to nearest even.
template <typename OutT>
int typed_linear(const float* A, int64_t lda, const float* W, const float* bias, int32_t K, int32_t cb_width,
                 const hgt_lin_group* groups, const hgt_lin_group* h_groups, int32_t n_groups,
                 const hgt_lin_cblock* cblocks, OutT* out, int32_t impl, void* workspace, size_t workspace_bytes,
                 cudaStream_t st) {
  HGT_REQUIRE(n_groups >= 0, "hgt_typed_linear: n_groups=%d", n_groups);
  HGT_REQUIRE(K > 0 && cb_width > 0, "hgt_typed_linear: K=%d cb_width=%d", K, cb_width);
  if (n_groups == 0) return 0;
  if (n_groups > kMaxGroups) {
    // schemas with many <type, relation> pairs: the per-launch tile prefix holds kMaxGroups entries, so launch in
    // chunks (same stream, same workspace: launches are ordered)
    for (int g0 = 0; g0 < n_groups; g0 += kMaxGroups) {
      const int n = n_groups - g0 < kMaxGroups ? n_groups - g0 : kMaxGroups;
      int rc = typed_linear<OutT>(A, lda, W, bias, K, cb_width, groups + g0, h_groups + g0, n, cblocks, out, impl,
                                  workspace, workspace_bytes, st);
      if (rc) return rc;
    }
    return 0;
  }
  if (impl == 0) impl = hgt_typed_linear_tc_supported(lda, K, cb_width) ? 2 : 1;
  if (impl == 2) {
    HGT_REQUIRE(hgt_typed_linear_tc_supported(lda, K, cb_width),
                "hgt_typed_linear: tensor-core kernel does not support lda=%lld K=%d cb_width=%d",
                (long long)lda, K, cb_width);
    return hgt_typed_linear_tc(A, lda, W, bias, K, cb_width, groups, h_groups, n_groups, cblocks, out, workspace,
                               workspace_bytes, st);
  }
  HGT_REQUIRE(impl == 1, "hgt_typed_linear: unknown impl %d", impl);
  TilePrefix tp;
  tp.n_tiles_n = (cb_width + BN - 1) / BN;
  int64_t total = 0;
  for (int g = 0; g < n_groups; ++g) {
    tp.first_tile[g] = (int32_t)total;
    int64_t mt = (h_groups[g].m + BM - 1) / BM;
    total += mt * h_groups[g].n_cblocks * tp.n_tiles_n;
    HGT_REQUIRE(total < 2147483647ll, "hgt_typed_linear: too many tiles");
  }
  tp.first_tile[n_groups] = (int32_t)total;
  if (total == 0) return 0;
  k_typed_linear_simt<OutT><<<(unsigned)total, GEMM_THREADS, 0, st>>>(A, lda, W, bias, K, cb_width, groups, n_groups,
                                                                      cblocks, out, tp);
  HGT_LAUNCH_CHECK();
  return 0;
}

}  // namespace

extern "C" int hgt_fold_weights(const float* const* wq, const float* const* bq, const float* const* wk,
                                const float* const* bk, const float* const* wv, const float* const* bv,
                                const float* relation_att, const float* relation_msg, const float* relation_pri,
                                int32_t num_types, int32_t num_relations, int32_t n_heads, int32_t d_in,
                                int32_t d_out, int32_t n_pairs, const int32_t* pair_type, const int32_t* pair_rel,
                                const int32_t* cat_row0, const int32_t* q_row0, float* w_cat, float* b_cat,
                                void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HGT_REQUIRE(n_heads > 0 && d_out % n_heads == 0, "hgt_fold_weights: d_out=%d not divisible by n_heads=%d",
              d_out, n_heads);
  (void)num_relations;
  {
    int64_t total = (int64_t)num_types * d_out * (d_in + 1);
    k_copy_linears<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(wq, bq, num_types, d_out, d_in, q_row0,
                                                                    w_cat, b_cat);
    HGT_LAUNCH_CHECK();
  }
  if (n_pairs > 0) {
    int64_t total = (int64_t)n_pairs * 2 * d_out * (d_in + 1);
    k_fold_pairs<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(wk, bk, wv, bv, relation_att, relation_msg,
                                                                  relation_pri, n_heads, d_in, d_out, n_pairs,
                                                                  pair_type, pair_rel, cat_row0, w_cat, b_cat);
    HGT_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" int hgt_concat_linears(const float* const* w, const float* const* b, int32_t num_types, int32_t rows,
                                  int32_t cols, float* w_cat, float* b_cat, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  int64_t total = (int64_t)num_types * rows * (cols + 1);
  if (total == 0) return 0;
  k_copy_linears<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(w, b, num_types, rows, cols, nullptr, w_cat,
                                                                  b_cat);
  HGT_LAUNCH_CHECK();
  return 0;
}

extern "C" int hgt_typed_linear_workspace_bytes(const hgt_lin_group* h_groups, int32_t n_groups, int32_t K,
                                                int32_t cb_width, int32_t impl, size_t* out_bytes) {
  HGT_REQUIRE(out_bytes && (h_groups || n_groups == 0), "hgt_typed_linear_workspace_bytes: NULL argument");
  if (impl == 0) impl = hgt_typed_linear_tc_supported(K, K, cb_width) ? 2 : 1;
  *out_bytes = (impl == 2 && n_groups > 0) ? hgt_typed_linear_tc_workspace(h_groups, n_groups, K, cb_width) : 0;
  return 0;
}

extern "C" int hgt_typed_linear(const float* A, int64_t lda, const float* W, const float* bias, int32_t K,
                                int32_t cb_width, const hgt_lin_group* groups, const hgt_lin_group* h_groups,
                                int32_t n_groups, const hgt_lin_cblock* cblocks, float* out, int32_t impl,
                                void* workspace, size_t workspace_bytes, void* stream_) {
  return typed_linear<float>(A, lda, W, bias, K, cb_width, groups, h_groups, n_groups, cblocks, out, impl, workspace,
                             workspace_bytes, (cudaStream_t)stream_);
}

extern "C" int hgt_typed_linear_bf16_workspace_bytes(const hgt_lin_group* h_groups, int32_t n_groups, int32_t K,
                                                     int32_t cb_width, int32_t impl, size_t* out_bytes) {
  // every path stores bf16 straight from its epilogue: the same workspace as the fp32 output
  return hgt_typed_linear_workspace_bytes(h_groups, n_groups, K, cb_width, impl, out_bytes);
}

extern "C" int hgt_typed_linear_bf16(const float* A, int64_t lda, const float* W, const float* bias, int32_t K,
                                     int32_t cb_width, const hgt_lin_group* groups, const hgt_lin_group* h_groups,
                                     int32_t n_groups, const hgt_lin_cblock* cblocks, void* out, int32_t impl,
                                     void* workspace, size_t workspace_bytes, void* stream_) {
  return typed_linear<__nv_bfloat16>(A, lda, W, bias, K, cb_width, groups, h_groups, n_groups, cblocks,
                                     reinterpret_cast<__nv_bfloat16*>(out), impl, workspace, workspace_bytes,
                                     (cudaStream_t)stream_);
}
