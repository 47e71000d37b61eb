// Backward of the small stages around the typed GEMMs (training path; the reference differentiates the same ops with
// autograd, OAG/train_paper_field.py:249):
//   hgt_update_backward   gated skip + LayerNorm (conv.py:129-133)  -> d o, d x, d skip, d norm.{weight,bias}
//   hgt_fold_backward     relation fold into the typed K/V weights (conv.py:97-99,103-104; hgt_fold_weights)
//                         -> d k_linears / v_linears (weight, bias), d relation_att / relation_msg / relation_pri
#include "common.cuh"

namespace {

// One warp per node row, ROWS_PER_WARP consecutive rows per warp; lane owns columns lane, lane+32, ...
// Forward:  y = o*a + x*(1-a),  a = sigmoid(skip[t]);   out = LayerNorm_t(y) = (y-mean)*rstd*w + b   (iff use_norm)
// Backward: dyh = dout*w;  dy = rstd*(dyh - mean(dyh) - yh*mean(dyh*yh));  do = a*dy;  dx = (1-a)*dy;
//           d a = sum dy*(o-x);  d skip[t] += d a * a*(1-a);  d w += dout*yh;  d b += dout.
constexpr int UB_WARPS = 8;
constexpr int UB_ROWS_PER_WARP = 16;

// DET: no atomics; warp w writes its per-type sums [d nw | d nb | d a] to part[(w + t) * (2d + 1)] (a warp's rows span
// consecutive types, so w + t is unique per (warp, type) and the slots of one type are contiguous in warp order), and
// k_det_update_reduce sums them in warp order.
template <int NPL, bool DET>
__device__ __forceinline__ void update_bwd_body(const float* __restrict__ dout, const float* __restrict__ o,
                                                const float* __restrict__ x, const int32_t* __restrict__ type_row0,
                                                int T, const float* __restrict__ skip, const float* __restrict__ norm_w,
                                                const int32_t* __restrict__ perm, const int32_t* __restrict__ type_active,
                                                int64_t n_nodes, int d, float* __restrict__ d_o, float* __restrict__ d_x,
                                                float* __restrict__ d_skip, float* __restrict__ d_nw,
                                                float* __restrict__ d_nb, float* __restrict__ part) {
  extern __shared__ float s_red[];                  // [2*d + 1] block-level partial sums (uniform-type blocks)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t block_row0 = (int64_t)blockIdx.x * UB_WARPS * UB_ROWS_PER_WARP;
  const int64_t block_row1 = min(n_nodes, block_row0 + UB_WARPS * UB_ROWS_PER_WARP);
  auto type_of = [&](int64_t row) {
    int t = 0;
    while (t < T && row >= type_row0[t + 1]) ++t;
    return t;
  };
  const int t_first = type_of(block_row0), t_last = type_of(block_row1 - 1);
  const bool uniform = !DET && t_first == t_last;
  if (!DET) {
    for (int i = threadIdx.x; i < 2 * d + 1; i += blockDim.x) s_red[i] = 0.f;
    __syncthreads();
  }

  float acc_w[NPL], acc_b[NPL];
  float acc_a = 0.f;
#pragma unroll
  for (int i = 0; i < NPL; ++i) acc_w[i] = acc_b[i] = 0.f;
  int cur_t = -1;
  auto flush = [&](int t) {
    if (t < 0 || t >= T) return;
    float da = 0.f;
    if (skip) {
      const float a = 1.0f / (1.0f + __expf(-skip[t]));
      da = acc_a;
      for (int s = 16; s > 0; s >>= 1) da += __shfl_xor_sync(0xffffffffu, da, s);
      da *= a * (1.0f - a);
    }
    if (DET) {
      float* w = part + ((int64_t)blockIdx.x * UB_WARPS + warp + t) * (2 * d + 1);
#pragma unroll
      for (int i = 0; i < NPL; ++i) {
        const int c = lane + 32 * i;
        if (c < d) { w[c] = acc_w[i]; w[d + c] = acc_b[i]; }
      }
      if (lane == 0) w[2 * d] = da;
    } else if (uniform) {
      if (lane == 0 && skip) atomicAdd(&s_red[2 * d], da);
      if (norm_w) {
#pragma unroll
        for (int i = 0; i < NPL; ++i) {
          const int c = lane + 32 * i;
          if (c < d) { atomicAdd(&s_red[c], acc_w[i]); atomicAdd(&s_red[d + c], acc_b[i]); }
        }
      }
    } else {
      if (lane == 0 && skip) atomicAdd(d_skip + t, da);
      if (norm_w) {
#pragma unroll
        for (int i = 0; i < NPL; ++i) {
          const int c = lane + 32 * i;
          if (c < d) { atomicAdd(d_nw + (int64_t)t * d + c, acc_w[i]); atomicAdd(d_nb + (int64_t)t * d + c, acc_b[i]); }
        }
      }
    }
    acc_a = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) acc_w[i] = acc_b[i] = 0.f;
  };

  const int64_t w_row0 = block_row0 + (int64_t)warp * UB_ROWS_PER_WARP;
  for (int rr = 0; rr < UB_ROWS_PER_WARP; ++rr) {
    const int64_t row = w_row0 + rr;
    if (row >= n_nodes) break;
    const int t = type_of(row);
    if (t != cur_t) { flush(cur_t); cur_t = t; }
    float* dorow = d_o + row * d;
    float* dxrow = d_x + row * d;
    // unknown type: the forward wrote zeros (conv.py:120); rows past type_active[t] (sharded runs: halo sources) had no
    // output row at all: neither contributes a gradient, and their `o` rows were never computed
    if (t >= T || (type_active && row - type_row0[t] >= type_active[t])) {
#pragma unroll
      for (int i = 0; i < NPL; ++i) {
        const int c = lane + 32 * i;
        if (c < d) { dorow[c] = 0.f; dxrow[c] = 0.f; }
      }
      continue;
    }
    const float a = skip ? 1.0f / (1.0f + __expf(-skip[t])) : 1.0f;
    const float b1 = skip ? 1.0f - a : 1.0f;
    const float* gr = dout + (perm ? (int64_t)perm[row] : row) * d;
    const float* orow = o + row * d;
    const float* xrow = x + row * d;
    float y[NPL], g[NPL], df[NPL];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      if (c < d) {
        const float ov = orow[c], xv = xrow[c];
        g[i] = gr[c];
        df[i] = ov - xv;
        y[i] = ov * a + xv * b1;
        sum += y[i];
      } else {
        g[i] = df[i] = y[i] = 0.f;
      }
    }
    if (norm_w) {
      for (int s = 16; s > 0; s >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, s);
      const float mean = sum / d;
      float var = 0.f;
#pragma unroll
      for (int i = 0; i < NPL; ++i) {
        const int c = lane + 32 * i;
        if (c < d) { const float dl = y[i] - mean; var = fmaf(dl, dl, var); }
      }
      for (int s = 16; s > 0; s >>= 1) var += __shfl_xor_sync(0xffffffffu, var, s);
      const float rstd = rsqrtf(var / d + 1e-5f);
      const float* w = norm_w + (int64_t)t * d;
      float m1 = 0.f, m2 = 0.f;
#pragma unroll
      for (int i = 0; i < NPL; ++i) {
        const int c = lane + 32 * i;
        if (c < d) {
          const float yh = (y[i] - mean) * rstd;
          acc_w[i] = fmaf(g[i], yh, acc_w[i]);
          acc_b[i] += g[i];
          const float dyh = g[i] * w[c];
          y[i] = yh;
          g[i] = dyh;
          m1 += dyh;
          m2 = fmaf(dyh, yh, m2);
        }
      }
      for (int s = 16; s > 0; s >>= 1) {
        m1 += __shfl_xor_sync(0xffffffffu, m1, s);
        m2 += __shfl_xor_sync(0xffffffffu, m2, s);
      }
      m1 /= d;
      m2 /= d;
#pragma unroll
      for (int i = 0; i < NPL; ++i) g[i] = rstd * (g[i] - m1 - y[i] * m2);      // g := dy
    }
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = lane + 32 * i;
      if (c < d) {
        dorow[c] = a * g[i];
        dxrow[c] = b1 * g[i];
        acc_a = fmaf(g[i], df[i], acc_a);
      }
    }
  }
  flush(cur_t);
  if (!DET && uniform) {
    __syncthreads();
    if (t_first < T) {
      if (norm_w) {
        for (int i = threadIdx.x; i < d; i += blockDim.x) {
          atomicAdd(d_nw + (int64_t)t_first * d + i, s_red[i]);
          atomicAdd(d_nb + (int64_t)t_first * d + i, s_red[d + i]);
        }
      }
      if (threadIdx.x == 0 && skip) atomicAdd(d_skip + t_first, s_red[2 * d]);
    }
  }
}

template <int NPL>
__global__ void __launch_bounds__(UB_WARPS * 32)
k_update_bwd(const float* __restrict__ dout, const float* __restrict__ o, const float* __restrict__ x,
             const int32_t* __restrict__ type_row0, int T, const float* __restrict__ skip,
             const float* __restrict__ norm_w, const int32_t* __restrict__ perm,
             const int32_t* __restrict__ type_active, int64_t n_nodes, int d,
             float* __restrict__ d_o, float* __restrict__ d_x, float* __restrict__ d_skip, float* __restrict__ d_nw,
             float* __restrict__ d_nb) {
  update_bwd_body<NPL, false>(dout, o, x, type_row0, T, skip, norm_w, perm, type_active, n_nodes, d, d_o, d_x, d_skip,
                              d_nw, d_nb, nullptr);
}
template <int NPL>
__global__ void __launch_bounds__(UB_WARPS * 32)
k_det_update_bwd(const float* __restrict__ dout, const float* __restrict__ o, const float* __restrict__ x,
                 const int32_t* __restrict__ type_row0, int T, const float* __restrict__ skip,
                 const float* __restrict__ norm_w, const int32_t* __restrict__ perm,
                 const int32_t* __restrict__ type_active, int64_t n_nodes, int d, float* __restrict__ d_o,
                 float* __restrict__ d_x, float* __restrict__ part) {
  update_bwd_body<NPL, true>(dout, o, x, type_row0, T, skip, norm_w, perm, type_active, n_nodes, d, d_o, d_x, nullptr,
                             nullptr, nullptr, part);
}

// One thread per (type t, column j of [d nw | d nb | d a]): sums the slots of the warps holding rows of t, in warp order.
__global__ void k_det_update_reduce(const float* __restrict__ part, const int32_t* __restrict__ type_row0, int T, int d,
                                    const float* __restrict__ skip, float* __restrict__ d_skip,
                                    float* __restrict__ d_nw, float* __restrict__ d_nb) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int W = 2 * d + 1;
  if (i >= (int64_t)T * W) return;
  const int t = (int)(i / W), j = (int)(i - (int64_t)t * W);
  const int64_t r0 = type_row0[t], r1 = type_row0[t + 1];
  float s = 0.f;
  if (r1 > r0) {
    const int64_t w0 = r0 / UB_ROWS_PER_WARP, w1 = (r1 - 1) / UB_ROWS_PER_WARP;
    s = hgt_chunk_sum(part + (w0 + t) * W + j, (int)(w1 - w0 + 1), W);
  }
  if (j < d) { if (d_nw) d_nw[(int64_t)t * d + j] = s; }
  else if (j < 2 * d) { if (d_nb) d_nb[(int64_t)t * d + j - d] = s; }
  else if (skip) d_skip[t] = s;
}

// ---- fold backward -----------------------------------------------------------------------------------------------------
// Forward (linear.cu k_fold_pairs):  W'[p,which][h*dk+c, col] = s * sum_a rel[r,h,a,c] * W[t][h*dk+a, col]  (col = d_in: bias)
// with rel = relation_att, s = pri[r,h]/sqrt(dk) for K' (which 0) and rel = relation_msg, s = 1 for V' (which 1).
// (a) d W[t][h*dk+a, col] += s * sum_c rel[a,c] * G[h*dk+c, col]           one thread per (p, which, row h*dk+a, col)
__device__ __forceinline__ float fold_w_term(const float* __restrict__ g_w, const float* __restrict__ g_b,
                                             const float* __restrict__ rel_att, const float* __restrict__ rel_msg,
                                             const float* __restrict__ rel_pri, int H, int dk, int d_in, int d_out,
                                             int r, int cat_row0, int which, int row, int col) {
  const int h = row / dk, a = row - h * dk;
  const float* rel = (which ? rel_msg : rel_att) + ((int64_t)(r * H + h) * dk) * dk;   // [a][c]
  const int64_t g_row0 = (int64_t)cat_row0 + which * d_out + h * dk;
  float acc = 0.f;
  if (col < d_in) {
    for (int c = 0; c < dk; ++c) acc = fmaf(rel[a * dk + c], g_w[(g_row0 + c) * d_in + col], acc);
  } else {
    for (int c = 0; c < dk; ++c) acc = fmaf(rel[a * dk + c], g_b[g_row0 + c], acc);
  }
  if (!which) acc *= rel_pri[r * H + h] * rsqrtf((float)dk);
  return acc;
}
__global__ void k_fold_bwd_w(const float* __restrict__ g_w, const float* __restrict__ g_b,
                             const float* __restrict__ rel_att, const float* __restrict__ rel_msg,
                             const float* __restrict__ rel_pri, int H, int d_in, int d_out, int n_pairs,
                             const int32_t* __restrict__ pair_type, const int32_t* __restrict__ pair_rel,
                             const int32_t* __restrict__ cat_row0, float* __restrict__ d_wk, float* __restrict__ d_bk,
                             float* __restrict__ d_wv, float* __restrict__ d_bv) {
  const int dk = d_out / H;
  const int64_t per_block = (int64_t)d_out * (d_in + 1);
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= per_block * 2 * n_pairs) return;
  const int p = (int)(i / (2 * per_block));
  int64_t rem = i - (int64_t)p * 2 * per_block;
  const int which = (int)(rem / per_block);
  rem -= which * per_block;
  const int row = (int)(rem / (d_in + 1));
  const int col = (int)(rem - (int64_t)row * (d_in + 1));
  const int t = pair_type[p];
  const float acc = fold_w_term(g_w, g_b, rel_att, rel_msg, rel_pri, H, dk, d_in, d_out, pair_rel[p], cat_row0[p], which,
                                row, col);
  if (col < d_in) atomicAdd((which ? d_wv : d_wk) + ((int64_t)t * d_out + row) * d_in + col, acc);
  else atomicAdd((which ? d_bv : d_bk) + (int64_t)t * d_out + row, acc);
}
// Deterministic variant: one thread per (type, which, row, col) walks the pairs of its type in pair order and stores once.
__global__ void k_det_fold_w(const float* __restrict__ g_w, const float* __restrict__ g_b,
                             const float* __restrict__ rel_att, const float* __restrict__ rel_msg,
                             const float* __restrict__ rel_pri, int T, int H, int d_in, int d_out, int n_pairs,
                             const int32_t* __restrict__ pair_type, const int32_t* __restrict__ pair_rel,
                             const int32_t* __restrict__ cat_row0, float* __restrict__ d_wk, float* __restrict__ d_bk,
                             float* __restrict__ d_wv, float* __restrict__ d_bv) {
  const int dk = d_out / H;
  const int64_t per_block = (int64_t)d_out * (d_in + 1);
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= per_block * 2 * T) return;
  const int t = (int)(i / (2 * per_block));
  int64_t rem = i - (int64_t)t * 2 * per_block;
  const int which = (int)(rem / per_block);
  rem -= which * per_block;
  const int row = (int)(rem / (d_in + 1));
  const int col = (int)(rem - (int64_t)row * (d_in + 1));
  float acc = 0.f;
  for (int p = 0; p < n_pairs; ++p)
    if (pair_type[p] == t)
      acc += fold_w_term(g_w, g_b, rel_att, rel_msg, rel_pri, H, dk, d_in, d_out, pair_rel[p], cat_row0[p], which, row, col);
  if (col < d_in) (which ? d_wv : d_wk)[((int64_t)t * d_out + row) * d_in + col] = acc;
  else (which ? d_bv : d_bk)[(int64_t)t * d_out + row] = acc;
}

// (b) val[a,c] = sum_col W[t][h*dk+a, col] * G[h*dk+c, col]  (bias column included);
//     d rel[r,h,a,c] += s * val;   d pri[r,h] += sum_{a,c} att[a,c] * val / sqrt(dk)   (K' only)
// One warp per (p, which, h, a, c); lanes split the columns.
__device__ __forceinline__ float fold_rel_term(const float* __restrict__ g_w, const float* __restrict__ g_b,
                                               const float* const* __restrict__ wk, const float* const* __restrict__ bk,
                                               const float* const* __restrict__ wv, const float* const* __restrict__ bv,
                                               int d_in, int d_out, int dk, int t, int cat_row0, int which, int h, int a,
                                               int c, int lane) {
  const float* w = (which ? wv[t] : wk[t]) + (int64_t)(h * dk + a) * d_in;
  const int64_t g_row = (int64_t)cat_row0 + which * d_out + h * dk + c;
  const float* g = g_w + g_row * d_in;
  float val = 0.f;
  for (int col = lane; col < d_in; col += 32) val = fmaf(w[col], g[col], val);
  if (lane == 0) val = fmaf((which ? bv[t] : bk[t])[h * dk + a], g_b[g_row], val);
  for (int s = 16; s > 0; s >>= 1) val += __shfl_xor_sync(0xffffffffu, val, s);
  return val;
}
__global__ void k_fold_bwd_rel(const float* __restrict__ g_w, const float* __restrict__ g_b,
                               const float* const* __restrict__ wk, const float* const* __restrict__ bk,
                               const float* const* __restrict__ wv, const float* const* __restrict__ bv,
                               const float* __restrict__ rel_att, const float* __restrict__ rel_pri, int H, int d_in,
                               int d_out, int n_pairs, const int32_t* __restrict__ pair_type,
                               const int32_t* __restrict__ pair_rel, const int32_t* __restrict__ cat_row0,
                               float* __restrict__ d_att, float* __restrict__ d_msg, float* __restrict__ d_pri) {
  const int dk = d_out / H;
  const int lane = threadIdx.x & 31;
  const int64_t wid = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t per_pair = (int64_t)2 * H * dk * dk;
  if (wid >= per_pair * n_pairs) return;
  const int p = (int)(wid / per_pair);
  int64_t rem = wid - (int64_t)p * per_pair;
  const int which = (int)(rem / ((int64_t)H * dk * dk));
  rem -= (int64_t)which * H * dk * dk;
  const int h = (int)(rem / (dk * dk));
  rem -= (int64_t)h * dk * dk;
  const int a = (int)(rem / dk), c = (int)(rem - (int64_t)a * dk);
  const int r = pair_rel[p];
  const float val = fold_rel_term(g_w, g_b, wk, bk, wv, bv, d_in, d_out, dk, pair_type[p], cat_row0[p], which, h, a, c,
                                  lane);
  if (lane == 0) {
    const int64_t ridx = ((int64_t)(r * H + h) * dk + a) * dk + c;
    if (which) {
      atomicAdd(d_msg + ridx, val);
    } else {
      const float inv = rsqrtf((float)dk);
      atomicAdd(d_att + ridx, val * rel_pri[r * H + h] * inv);
      atomicAdd(d_pri + r * H + h, val * rel_att[ridx] * inv);
    }
  }
}

// Deterministic variant: one warp per (relation, which, h, a, c) walks the pairs of its relation in pair order.  d pri
// needs a further sum over (a, c): each warp stores its term to pri_part[a * dk + c][r * H + h], and the caller sums
// those dk * dk chunks in order.
__global__ void k_det_fold_rel(const float* __restrict__ g_w, const float* __restrict__ g_b,
                               const float* const* __restrict__ wk, const float* const* __restrict__ bk,
                               const float* const* __restrict__ wv, const float* const* __restrict__ bv,
                               const float* __restrict__ rel_att, const float* __restrict__ rel_pri, int R, int H,
                               int d_in, int d_out, int n_pairs, const int32_t* __restrict__ pair_type,
                               const int32_t* __restrict__ pair_rel, const int32_t* __restrict__ cat_row0,
                               float* __restrict__ d_att, float* __restrict__ d_msg, float* __restrict__ pri_part) {
  const int dk = d_out / H;
  const int lane = threadIdx.x & 31;
  const int64_t wid = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t per_rel = (int64_t)2 * H * dk * dk;
  if (wid >= per_rel * R) return;
  const int r = (int)(wid / per_rel);
  int64_t rem = wid - (int64_t)r * per_rel;
  const int which = (int)(rem / ((int64_t)H * dk * dk));
  rem -= (int64_t)which * H * dk * dk;
  const int h = (int)(rem / (dk * dk));
  rem -= (int64_t)h * dk * dk;
  const int a = (int)(rem / dk), c = (int)(rem - (int64_t)a * dk);
  float sum = 0.f;
  for (int p = 0; p < n_pairs; ++p)
    if (pair_rel[p] == r)
      sum += fold_rel_term(g_w, g_b, wk, bk, wv, bv, d_in, d_out, dk, pair_type[p], cat_row0[p], which, h, a, c, lane);
  if (lane == 0) {
    const int64_t ridx = ((int64_t)(r * H + h) * dk + a) * dk + c;
    if (which) {
      d_msg[ridx] = sum;
    } else {
      const float inv = rsqrtf((float)dk);
      d_att[ridx] = sum * rel_pri[r * H + h] * inv;
      pri_part[((int64_t)a * dk + c) * R * H + r * H + h] = sum * rel_att[ridx] * inv;
    }
  }
}

template <int NPL>
void launch_update_bwd(const float* dout, const float* o, const float* x, const int32_t* type_row0, int T,
                       const float* skip, const float* norm_w, const int32_t* perm, const int32_t* type_active,
                       int64_t n, int d, float* d_o,
                       float* d_x, float* d_skip, float* d_nw, float* d_nb, cudaStream_t st) {
  const int rows_per_block = UB_WARPS * UB_ROWS_PER_WARP;
  const unsigned grid = (unsigned)((n + rows_per_block - 1) / rows_per_block);
  k_update_bwd<NPL><<<grid, UB_WARPS * 32, (2 * d + 1) * sizeof(float), st>>>(dout, o, x, type_row0, T, skip, norm_w, perm,
                                                                             type_active, n, d, d_o, d_x, d_skip, d_nw,
                                                                             d_nb);
}
template <int NPL>
void launch_det_update_bwd(const float* dout, const float* o, const float* x, const int32_t* type_row0, int T,
                           const float* skip, const float* norm_w, const int32_t* perm, const int32_t* type_active,
                           int64_t n, int d, float* d_o, float* d_x, float* part, cudaStream_t st) {
  const int rows_per_block = UB_WARPS * UB_ROWS_PER_WARP;
  const unsigned grid = (unsigned)((n + rows_per_block - 1) / rows_per_block);
  k_det_update_bwd<NPL><<<grid, UB_WARPS * 32, 0, st>>>(dout, o, x, type_row0, T, skip, norm_w, perm, type_active, n, d,
                                                        d_o, d_x, part);
}

}  // namespace

extern "C" int hgt_update_backward(const float* dout, const float* o, const float* x, const int32_t* type_row0,
                                   int32_t num_types, const float* skip, const float* norm_w, const int32_t* perm,
                                   const int32_t* type_active, int64_t n_nodes, int32_t d, float* d_o, float* d_x, float* d_skip, float* d_norm_w,
                                   float* d_norm_b, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HGT_REQUIRE(dout && o && x && type_row0 && d_o && d_x && (d_skip || !skip), "hgt_update_backward: NULL argument");
  HGT_REQUIRE(d >= 1 && d <= 1024, "hgt_update_backward: d=%d unsupported (max 1024)", d);
  HGT_REQUIRE(!norm_w || (d_norm_w && d_norm_b), "hgt_update_backward: LayerNorm gradients need output buffers");
  if (skip) HGT_CHECK_CUDA(cudaMemsetAsync(d_skip, 0, (size_t)num_types * sizeof(float), st));
  if (norm_w) {
    HGT_CHECK_CUDA(cudaMemsetAsync(d_norm_w, 0, (size_t)num_types * d * sizeof(float), st));
    HGT_CHECK_CUDA(cudaMemsetAsync(d_norm_b, 0, (size_t)num_types * d * sizeof(float), st));
  }
  if (n_nodes == 0) return 0;
  const int npl = (d + 31) / 32;
#define HGT_UB(N) launch_update_bwd<N>(dout, o, x, type_row0, num_types, skip, norm_w, perm, type_active, n_nodes, d, d_o, d_x, d_skip, \
                                       d_norm_w, d_norm_b, st)
  if (npl <= 2) HGT_UB(2);
  else if (npl <= 4) HGT_UB(4);
  else if (npl <= 8) HGT_UB(8);
  else if (npl <= 16) HGT_UB(16);
  else HGT_UB(32);
#undef HGT_UB
  HGT_LAUNCH_CHECK();
  return 0;
}

extern "C" int hgt_fold_backward(const float* d_w_cat, const float* d_b_cat, const float* const* wk,
                                 const float* const* bk, const float* const* wv, const float* const* bv,
                                 const float* relation_att, const float* relation_msg, const float* relation_pri,
                                 int32_t num_types, int32_t num_relations, int32_t n_heads, int32_t d_in, int32_t d_out,
                                 int32_t n_pairs, const int32_t* pair_type, const int32_t* pair_rel,
                                 const int32_t* cat_row0, float* d_wk, float* d_bk, float* d_wv, float* d_bv,
                                 float* d_att, float* d_msg, float* d_pri, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HGT_REQUIRE(n_heads > 0 && d_out % n_heads == 0, "hgt_fold_backward: d_out=%d not divisible by n_heads=%d", d_out, n_heads);
  HGT_REQUIRE(d_wk && d_bk && d_wv && d_bv && d_att && d_msg && d_pri, "hgt_fold_backward: NULL output");
  const int dk = d_out / n_heads;
  const size_t wbytes = (size_t)num_types * d_out * d_in * sizeof(float), bbytes = (size_t)num_types * d_out * sizeof(float);
  const size_t rbytes = (size_t)num_relations * n_heads * dk * dk * sizeof(float);
  HGT_CHECK_CUDA(cudaMemsetAsync(d_wk, 0, wbytes, st));
  HGT_CHECK_CUDA(cudaMemsetAsync(d_wv, 0, wbytes, st));
  HGT_CHECK_CUDA(cudaMemsetAsync(d_bk, 0, bbytes, st));
  HGT_CHECK_CUDA(cudaMemsetAsync(d_bv, 0, bbytes, st));
  HGT_CHECK_CUDA(cudaMemsetAsync(d_att, 0, rbytes, st));
  HGT_CHECK_CUDA(cudaMemsetAsync(d_msg, 0, rbytes, st));
  HGT_CHECK_CUDA(cudaMemsetAsync(d_pri, 0, (size_t)num_relations * n_heads * sizeof(float), st));
  if (n_pairs == 0) return 0;
  HGT_REQUIRE(d_w_cat && d_b_cat && wk && bk && wv && bv, "hgt_fold_backward: NULL input");
  {
    const int64_t total = (int64_t)n_pairs * 2 * d_out * (d_in + 1);
    k_fold_bwd_w<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_w_cat, d_b_cat, relation_att, relation_msg,
                                                                  relation_pri, n_heads, d_in, d_out, n_pairs, pair_type,
                                                                  pair_rel, cat_row0, d_wk, d_bk, d_wv, d_bv);
    HGT_LAUNCH_CHECK();
  }
  {
    const int64_t warps = (int64_t)n_pairs * 2 * n_heads * dk * dk;
    k_fold_bwd_rel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(d_w_cat, d_b_cat, wk, bk, wv, bv, relation_att,
                                                                        relation_pri, n_heads, d_in, d_out, n_pairs,
                                                                        pair_type, pair_rel, cat_row0, d_att, d_msg, d_pri);
    HGT_LAUNCH_CHECK();
  }
  return 0;
}

// Partial sums of the deterministic update backward: one [2d + 1] slot per (warp, type it touches).
static size_t update_det_part_floats(int64_t n_nodes, int32_t num_types, int32_t d) {
  const int64_t warps = (n_nodes + UB_WARPS * UB_ROWS_PER_WARP - 1) / (UB_WARPS * UB_ROWS_PER_WARP) * UB_WARPS;
  return (size_t)(warps + num_types) * (2 * (size_t)d + 1);
}

extern "C" int hgt_update_backward_det_workspace_bytes(int64_t n_nodes, int32_t num_types, int32_t d,
                                                       size_t* out_bytes) {
  HGT_REQUIRE(out_bytes && n_nodes >= 0 && num_types >= 1 && d >= 1, "hgt_update_backward_det_workspace_bytes: bad argument");
  *out_bytes = update_det_part_floats(n_nodes, num_types, d) * sizeof(float) + 256;
  return 0;
}

extern "C" int hgt_update_backward_det(const float* dout, const float* o, const float* x, const int32_t* type_row0,
                                       int32_t num_types, const float* skip, const float* norm_w, const int32_t* perm,
                                       const int32_t* type_active, int64_t n_nodes, int32_t d, float* d_o, float* d_x,
                                       float* d_skip, float* d_norm_w, float* d_norm_b, void* workspace,
                                       size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HGT_REQUIRE(dout && o && x && type_row0 && d_o && d_x && (d_skip || !skip), "hgt_update_backward_det: NULL argument");
  HGT_REQUIRE(d >= 1 && d <= 1024, "hgt_update_backward_det: d=%d unsupported (max 1024)", d);
  HGT_REQUIRE(num_types >= 1, "hgt_update_backward_det: num_types=%d", num_types);
  HGT_REQUIRE(!norm_w || (d_norm_w && d_norm_b), "hgt_update_backward_det: LayerNorm gradients need output buffers");
  size_t need = 0;
  hgt_update_backward_det_workspace_bytes(n_nodes, num_types, d, &need);
  HGT_REQUIRE(workspace && workspace_bytes >= need, "hgt_update_backward_det: workspace too small (%zu < %zu)",
              workspace_bytes, need);
  float* part = reinterpret_cast<float*>(hgt_align_up(reinterpret_cast<size_t>(workspace), 256));
  if (n_nodes > 0) {
    const int npl = (d + 31) / 32;
#define HGT_UB(N) launch_det_update_bwd<N>(dout, o, x, type_row0, num_types, skip, norm_w, perm, type_active, n_nodes, d, \
                                           d_o, d_x, part, st)
    if (npl <= 2) HGT_UB(2);
    else if (npl <= 4) HGT_UB(4);
    else if (npl <= 8) HGT_UB(8);
    else if (npl <= 16) HGT_UB(16);
    else HGT_UB(32);
#undef HGT_UB
    HGT_LAUNCH_CHECK();
  }
  // every (type, column) is written, also for types without rows
  const int64_t total = (int64_t)num_types * (2 * d + 1);
  k_det_update_reduce<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(part, type_row0, num_types, d, skip, d_skip,
                                                                      norm_w ? d_norm_w : nullptr,
                                                                      norm_w ? d_norm_b : nullptr);
  HGT_LAUNCH_CHECK();
  return 0;
}

extern "C" int hgt_fold_backward_det_workspace_bytes(int32_t num_relations, int32_t n_heads, int32_t d_out,
                                                     size_t* out_bytes) {
  HGT_REQUIRE(out_bytes && n_heads > 0 && d_out % n_heads == 0 && num_relations >= 0,
              "hgt_fold_backward_det_workspace_bytes: bad argument");
  const size_t dk = d_out / n_heads;
  *out_bytes = 256 + hgt_align_up((size_t)num_relations * n_heads * dk * dk * sizeof(float), 256) + sizeof(hgt_sum_seg);
  return 0;
}

extern "C" int hgt_fold_backward_det(const float* d_w_cat, const float* d_b_cat, const float* const* wk,
                                     const float* const* bk, const float* const* wv, const float* const* bv,
                                     const float* relation_att, const float* relation_msg, const float* relation_pri,
                                     int32_t num_types, int32_t num_relations, int32_t n_heads, int32_t d_in,
                                     int32_t d_out, int32_t n_pairs, const int32_t* pair_type, const int32_t* pair_rel,
                                     const int32_t* cat_row0, float* d_wk, float* d_bk, float* d_wv, float* d_bv,
                                     float* d_att, float* d_msg, float* d_pri, void* workspace, size_t workspace_bytes,
                                     void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HGT_REQUIRE(n_heads > 0 && d_out % n_heads == 0, "hgt_fold_backward_det: d_out=%d not divisible by n_heads=%d", d_out,
              n_heads);
  HGT_REQUIRE(d_wk && d_bk && d_wv && d_bv && d_att && d_msg && d_pri, "hgt_fold_backward_det: NULL output");
  HGT_REQUIRE(n_pairs == 0 || (d_w_cat && d_b_cat && wk && bk && wv && bv), "hgt_fold_backward_det: NULL input");
  size_t need = 0;
  hgt_fold_backward_det_workspace_bytes(num_relations, n_heads, d_out, &need);
  HGT_REQUIRE(workspace && workspace_bytes >= need, "hgt_fold_backward_det: workspace too small (%zu < %zu)",
              workspace_bytes, need);
  const int dk = d_out / n_heads;
  char* base = reinterpret_cast<char*>(hgt_align_up(reinterpret_cast<size_t>(workspace), 256));
  float* pri_part = reinterpret_cast<float*>(base);
  hgt_sum_seg* d_seg = reinterpret_cast<hgt_sum_seg*>(
      base + hgt_align_up((size_t)num_relations * n_heads * dk * dk * sizeof(float), 256));
  HGT_CHECK_CUDA(cudaMemsetAsync(d_pri, 0, (size_t)num_relations * n_heads * sizeof(float), st));
  {
    const int64_t total = (int64_t)num_types * 2 * d_out * (d_in + 1);
    if (total > 0) {
      k_det_fold_w<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_w_cat, d_b_cat, relation_att, relation_msg,
                                                                    relation_pri, num_types, n_heads, d_in, d_out,
                                                                    n_pairs, pair_type, pair_rel, cat_row0, d_wk, d_bk,
                                                                    d_wv, d_bv);
      HGT_LAUNCH_CHECK();
    }
  }
  const int64_t warps = (int64_t)num_relations * 2 * n_heads * dk * dk;
  if (warps == 0) return 0;
  k_det_fold_rel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(d_w_cat, d_b_cat, wk, bk, wv, bv, relation_att,
                                                                      relation_pri, num_relations, n_heads, d_in, d_out,
                                                                      n_pairs, pair_type, pair_rel, cat_row0, d_att,
                                                                      d_msg, pri_part);
  HGT_LAUNCH_CHECK();
  const hgt_sum_seg seg{0, 0, dk * dk, 0};
  HGT_CHECK_CUDA(cudaMemcpyAsync(d_seg, &seg, sizeof(seg), cudaMemcpyHostToDevice, st));
  return hgt_ordered_sum_launch(pri_part, d_seg, 1, (int64_t)num_relations * n_heads, d_pri, st);
}
