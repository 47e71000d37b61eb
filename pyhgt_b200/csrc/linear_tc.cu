// Typed linear layers on the 5th-generation tensor cores (tcgen05) with fp32-grade accuracy.
//
// fp32 operands are split into two bf16 terms, x = x_hi + x_lo (|x - x_hi - x_lo| <= 2^-17 |x|), and
//     A*W^T  ~=  A_hi*W_hi^T + A_hi*W_lo^T + A_lo*W_hi^T            (dropped term ~2^-18)
// is accumulated in ONE fp32 TMEM accumulator by running three bf16 passes over K inside the same
// tile: 3 tensor-core products at the bf16 rate instead of an fp32 FMA GEMM, error ~1e-5 relative —
// far inside the 1e-3 parity bar, where a single bf16 or tf32 product would not be.
//
// Three kernels share the TMA / UMMA / TMEM plumbing below (all: SWIZZLE_128B K-major operands, fp32 accumulate in TMEM):
//   k_typed_linear_tc3  (default when the column block is a multiple of 256): CTA PAIR, cta_group::2, W-stationary,
//                       persistent; 256 x 256 pair tile, double-buffered TMEM accumulator, 8-warp transposing epilogue.
//   k_typed_linear_tc2  same design on one CTA (n-tile = widest divisor of the column block whose resident W fits).
//   k_typed_linear_tc   one 128 x BN tile per CTA, both operands streamed (fallback for very wide K).
// Output tiles follow the same group / column-block tables as the SIMT kernel in linear.cu.
#include <cuda.h>
#include <cuda_bf16.h>

#include <type_traits>

#include "common.cuh"
#include "tc_ptx.cuh"

int hgt_act_split_launch(const float* in, int64_t ld, int64_t rows, int K, int Kp, int act, float* out_f32,
                         __nv_bfloat16* hi, __nv_bfloat16* lo, cudaStream_t st);

namespace {

using namespace tcp;

constexpr int kMaxGroups = 64;
constexpr int TC_BM = 128;
constexpr int TC_BK = 64;              // 64 bf16 = 128 bytes = one SWIZZLE_128B row
constexpr int TC_THREADS = 192;
constexpr int UMMA_K = 16;

// Two fp32 values rounded to nearest even as a packed bf16 pair (first value at the lower address).
__device__ __forceinline__ uint32_t bf16x2_bits(float a, float b) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}

struct TcTilePrefix {
  int32_t first_tile[kMaxGroups + 1];
  int32_t n_tiles_n;
};

// ---- the GEMM -------------------------------------------------------------------------------------
template <typename OutT>
__global__ void __launch_bounds__(TC_THREADS, 2)
k_typed_linear_tc(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                  const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                  const float* __restrict__ bias, int Kp, int cb_width, int BN, int stages, int tmem_cols,
                  const hgt_lin_group* __restrict__ groups, int n_groups,
                  const hgt_lin_cblock* __restrict__ cblocks, OutT* __restrict__ out, TcTilePrefix tp) {
  extern __shared__ unsigned char smem_dyn[];
  // carve: [stages][A 16 KB | B BN*128 B] (1024-aligned), then barriers, tmem pointer, bias tile
  unsigned char* smem = smem_dyn + ((1024u - (s_u32(smem_dyn) & 1023u)) & 1023u);   // keeps the shared address space
  const uint32_t a_bytes = TC_BM * TC_BK * 2;
  const uint32_t b_bytes = (uint32_t)BN * TC_BK * 2;
  const uint32_t b_bytes_al = (b_bytes + 1023) & ~1023u;
  const uint32_t stage_bytes = a_bytes + b_bytes_al;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)stages * stage_bytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + stages;
  uint64_t* tmem_full_bar = bars + 2 * stages;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * stages + 1);
  float* s_bias = reinterpret_cast<float*>(tmem_ptr_smem + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // ---- tile decode ----
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
  const int64_t m0 = (int64_t)mt * TC_BM;
  const int n0 = nt * BN;
  const int a_row = (int)(grp.a_row0 + m0);
  const int w_row = grp.w_row0 + cb * cb_width + n0;
  const int rows_here = (int)min((int64_t)TC_BM, grp.m - m0);
  const int k_blocks = (Kp + TC_BK - 1) / TC_BK;
  const int total_iters = 3 * k_blocks;

  if (warp == 0 && lane == 0) {
    prefetch_map(&map_a_hi);
    prefetch_map(&map_a_lo);
    prefetch_map(&map_w_hi);
    prefetch_map(&map_w_lo);
    for (int s = 0; s < stages; ++s) {
      mbar_init(s_u32(&full_bar[s]), 1);
      mbar_init(s_u32(&empty_bar[s]), 1);
    }
    mbar_init(s_u32(tmem_full_bar), 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc<1>(s_u32(tmem_ptr_smem), (uint32_t)tmem_cols);
  }
  if (warp >= 2) {
    for (int c = threadIdx.x - 64; c < BN; c += TC_THREADS - 64)
      s_bias[c] = (grp.has_bias && bias) ? bias[w_row + c] : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer =====
      for (int it = 0; it < total_iters; ++it) {
        const int s = it % stages;
        const uint32_t ph = (uint32_t)(it / stages) & 1u;
        mbar_wait(s_u32(&empty_bar[s]), ph ^ 1u);
        const int pass = it / k_blocks;                    // 0: hi*hi, 1: hi*lo, 2: lo*hi
        const int kb = it - pass * k_blocks;
        const CUtensorMap* ma = (pass == 2) ? &map_a_lo : &map_a_hi;
        const CUtensorMap* mw = (pass == 1) ? &map_w_lo : &map_w_hi;
        const uint32_t bar = s_u32(&full_bar[s]);
        const uint32_t sa = s_u32(smem + (size_t)s * stage_bytes);
        mbar_expect_tx(bar, a_bytes + b_bytes);
        tma_load_2d(sa, ma, kb * TC_BK, a_row, bar);
        tma_load_2d(sa + a_bytes, mw, kb * TC_BK, w_row, bar);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===== MMA issuer =====
      const uint32_t idesc = idesc_bf16(TC_BM, BN, false, false);
      for (int it = 0; it < total_iters; ++it) {
        const int s = it % stages;
        const uint32_t ph = (uint32_t)(it / stages) & 1u;
        mbar_wait(s_u32(&full_bar[s]), ph);
        tc_fence_after();
        const uint32_t sa = s_u32(smem + (size_t)s * stage_bytes);
        const uint64_t da = desc_k_sw128(sa);
        const uint64_t db = desc_k_sw128(sa + a_bytes);
#pragma unroll
        for (int k = 0; k < TC_BK / UMMA_K; ++k) {
          // advance 16 bf16 = 32 bytes inside the 128-byte swizzle row: +2 in the (addr >> 4) field
          umma_bf16_ss(tmem_base, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (it > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(s_u32(&empty_bar[s]));                  // frees the smem slot when these MMAs retire
      }
      umma_commit(s_u32(tmem_full_bar));                    // accumulator complete
    }
  } else {
    // ===== epilogue warps: TMEM lane group = warp % 4 =====
    const int lg = warp & 3;
    const int row = lg * 32 + lane;
    mbar_wait(s_u32(tmem_full_bar), 0);
    tc_fence_after();
    OutT* orow = out + cblk.out_off + (m0 + row) * cblk.ld + n0;
    const bool row_ok = row < rows_here;
    for (int c = 0; c < BN; c += 16) {
      uint32_t r[16];
      tmem_ld16(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)c, r);
      tmem_ld_wait();
      if (row_ok) {
        if constexpr (std::is_same<OutT, float>::value) {
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            float4 v;
            v.x = __uint_as_float(r[j + 0]) + s_bias[c + j + 0];
            v.y = __uint_as_float(r[j + 1]) + s_bias[c + j + 1];
            v.z = __uint_as_float(r[j + 2]) + s_bias[c + j + 2];
            v.w = __uint_as_float(r[j + 3]) + s_bias[c + j + 3];
            *reinterpret_cast<float4*>(orow + c + j) = v;
          }
        } else {
          // bf16 row: 16 values = two 16-byte stores
          uint32_t w[8];
#pragma unroll
          for (int j = 0; j < 8; ++j)
            w[j] = bf16x2_bits(__uint_as_float(r[2 * j]) + s_bias[c + 2 * j],
                               __uint_as_float(r[2 * j + 1]) + s_bias[c + 2 * j + 1]);
          *reinterpret_cast<uint4*>(orow + c) = make_uint4(w[0], w[1], w[2], w[3]);
          *reinterpret_cast<uint4*>(orow + c + 8) = make_uint4(w[4], w[5], w[6], w[7]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tmem_dealloc<1>(tmem_base, (uint32_t)tmem_cols);
  }
}


// ---- W-stationary persistent GEMM (default) -------------------------------------------------------
// A "unit" = one column task (group, column block, n-tile of BN columns) x a chunk of up to TC2_MCH m-tiles.
// The CTA keeps the column task's W_hi / W_lo tiles (all K) resident in shared memory, streams the A_hi / A_lo
// k-blocks of successive m-tiles through a ring, and issues per k-block the three products
// A_hi*W_hi + A_hi*W_lo + A_lo*W_hi into a double-buffered TMEM accumulator, so the epilogue of m-tile i
// overlaps the MMAs of m-tile i+1.  Units are ordered m-chunk-major so that CTAs running concurrently read the
// same A rows from L2 with different W.  L2->SM traffic per output tile drops from 384 KB (tile-per-CTA kernel
// below) to 128 KB (+ W amortised over the chunk).
constexpr int TC2_MCH = 8;                     // m-tiles (tc3: 256-row pair steps) per unit
constexpr int TC2_STAGE_CAP = 8;               // A ring stages at most

// Epilogue of one accumulator tile, shared by the persistent kernels.  8 epilogue warps: warp e (0..7) reads TMEM
// lane quarter (warp id % 4) and the 16-column chunks c0 = 16*(e/4), +32, ...  TMEM hands each lane one ROW, so the
// chunk is transposed through a per-warp staging buffer and written with 4 lanes per 64 contiguous bytes of a row
// (full 32-byte sectors).  All shared-memory reads are issued before the dependent adds / predicated stores.
constexpr int TC2_EPI_WARPS = 8;
constexpr int TC2_THREADS = 64 + 32 * TC2_EPI_WARPS;
// The staging region is sized for rows of 20 floats, although the swizzled drain below uses 16 of them: its size enters
// the shared-memory budget and with it the A-ring stage counts of both persistent kernels.
constexpr int TC2_STG_LD = 20;
constexpr int TC2_STAGE_BYTES = TC2_EPI_WARPS * 32 * TC2_STG_LD * 4;

// The drain is software-pipelined: the TMEM load of chunk i+1 is in flight while chunk i goes through the staging
// buffer and out to global memory (two named register buffers), and the staging buffer is swizzled so that neither side
// has bank conflicts.  Measured at C2 together with the .cta-scope pair barriers: projection 3.90 -> 3.81 ms against the
// round-1 drain; a drain straight from registers without the transpose ran at the same speed
// (profiles/r02_gemm_epilogue_ab.md); see DESIGN.md section 9 for what was ruled out as the limiter.
template <typename OutT>
__device__ __forceinline__ void tc_epi_chunk(const uint32_t (&r)[16], int c0, float* stg, const float* s_bias,
                                             OutT* out_tile, int64_t ld, int64_t rows_left, int lane) {
  // staging rows of 64 bytes, the 16-byte piece j of row r kept at position j ^ ((r >> 1) & 3): the row-per-lane writes
  // and the 4-lanes-per-row reads both touch every bank once per quarter warp (no conflicts, 4 wavefronts per access)
  const int sub = lane & 3, rsel = lane >> 2;
  const int wsw = (lane >> 1) & 3;
#pragma unroll
  for (int j = 0; j < 4; ++j)
    *reinterpret_cast<uint4*>(stg + lane * 16 + ((j ^ wsw) << 2)) =
        make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
  __syncwarp();
  if constexpr (std::is_same<OutT, float>::value) {
    const float4 b = *reinterpret_cast<const float4*>(s_bias + c0 + sub * 4);
    const int rsw = (sub ^ ((rsel >> 1) & 3)) << 2;                   // (8k + rsel) >> 1 & 3 == rsel >> 1 & 3
    float4 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = *reinterpret_cast<const float4*>(stg + (8 * k + rsel) * 16 + rsw);
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int rr = 8 * k + rsel;
      if (rr < rows_left) {
        float4 w = v[k];
        w.x += b.x; w.y += b.y; w.z += b.z; w.w += b.w;
        *reinterpret_cast<float4*>(out_tile + (int64_t)rr * ld + c0 + sub * 4) = w;
      }
    }
  } else {
    // bf16 rows: the 16 columns of a row are 32 bytes, two lanes of 8 values (one 16-byte store each), 16 rows per
    // pass.  Lane (row rh, half h) reads pieces 2h and 2h+1 of its staging row; the swizzle keeps each quarter warp on
    // distinct banks.
    const int h = lane & 1, rh = lane >> 1;
    const int sw = (rh >> 1) & 3;                                      // (16k + rh) >> 1 & 3 == rh >> 1 & 3
    const float4 b0 = *reinterpret_cast<const float4*>(s_bias + c0 + h * 8);
    const float4 b1 = *reinterpret_cast<const float4*>(s_bias + c0 + h * 8 + 4);
    float4 v[2][2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const float* srow = stg + (16 * k + rh) * 16;
      v[k][0] = *reinterpret_cast<const float4*>(srow + (((2 * h) ^ sw) << 2));
      v[k][1] = *reinterpret_cast<const float4*>(srow + (((2 * h + 1) ^ sw) << 2));
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int rr = 16 * k + rh;
      if (rr < rows_left) {
        const uint4 w = make_uint4(bf16x2_bits(v[k][0].x + b0.x, v[k][0].y + b0.y),
                                   bf16x2_bits(v[k][0].z + b0.z, v[k][0].w + b0.w),
                                   bf16x2_bits(v[k][1].x + b1.x, v[k][1].y + b1.y),
                                   bf16x2_bits(v[k][1].z + b1.z, v[k][1].w + b1.w));
        *reinterpret_cast<uint4*>(out_tile + (int64_t)rr * ld + c0 + h * 8) = w;
      }
    }
  }
}

template <typename OutT>
__device__ __forceinline__ void tc_epilogue_tile_pf(uint32_t t_row, int n_cols, int chunk0, float* stg,
                                                    const float* s_bias, OutT* out_tile, int64_t ld,
                                                    int64_t rows_left, int lane) {
  uint32_t ra[16], rb[16];
  int c0 = 16 * chunk0;
  if (c0 >= n_cols) return;
  tmem_ld16(t_row + (uint32_t)c0, ra);
  for (; c0 < n_cols; c0 += 64) {
    const bool has_b = c0 + 32 < n_cols;
    tmem_ld_wait();                                                    // ra has landed
    if (has_b) tmem_ld16(t_row + (uint32_t)(c0 + 32), rb);
    tc_epi_chunk(ra, c0, stg, s_bias, out_tile, ld, rows_left, lane);
    if (!has_b) break;
    tmem_ld_wait();                                                    // rb has landed
    if (c0 + 64 < n_cols) tmem_ld16(t_row + (uint32_t)(c0 + 64), ra);
    tc_epi_chunk(rb, c0 + 32, stg, s_bias, out_tile, ld, rows_left, lane);
  }
}

struct Tc2Sched {
  int32_t first_unit[kMaxGroups + 1];
  int32_t n_tiles_n;
};

template <typename OutT>
__global__ void __launch_bounds__(TC2_THREADS, 1)
k_typed_linear_tc2(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                   const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                   const float* __restrict__ bias, int Kp, int cb_width, int BN, int stages, int tmem_cols,
                   const hgt_lin_group* __restrict__ groups, int n_groups,
                   const hgt_lin_cblock* __restrict__ cblocks, OutT* __restrict__ out, Tc2Sched sc) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = smem_dyn + ((1024u - (s_u32(smem_dyn) & 1023u)) & 1023u);   // keeps the shared address space
  const int k_blocks = (Kp + TC_BK - 1) / TC_BK;
  const uint32_t a_bytes = TC_BM * TC_BK * 2;                       // one A tile (hi or lo)
  const uint32_t b_bytes = (uint32_t)BN * TC_BK * 2;                // one W tile (hi or lo)
  const uint32_t b_bytes_al = (b_bytes + 1023) & ~1023u;
  const uint32_t w_region = (uint32_t)k_blocks * 2 * b_bytes_al;    // resident W
  const uint32_t a_stage = a_bytes;                                 // one tile per stage: A_hi(kb), A_lo(kb), A_hi(kb+1), ...
  unsigned char* w_smem = smem;
  unsigned char* a_smem = smem + w_region;
  uint64_t* bars = reinterpret_cast<uint64_t*>(a_smem + (size_t)stages * a_stage);
  uint64_t* a_full = bars;
  uint64_t* a_empty = bars + stages;
  uint64_t* w_full = bars + 2 * stages;
  uint64_t* w_empty = w_full + 1;
  uint64_t* t_full = w_empty + 1;       // [2]
  uint64_t* t_empty = t_full + 2;       // [2]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(t_empty + 2);
  float* s_bias = reinterpret_cast<float*>(tmem_ptr_smem + 4);        // 16-byte aligned: the barrier block is 16*(stages+3) B
  float* s_stage = s_bias + ((BN + 3) & ~3);                          // [4 warps][32][TC2_STG_LD] epilogue transpose

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_units = sc.first_unit[n_groups];

  if (warp == 0 && lane == 0) {
    prefetch_map(&map_a_hi);
    prefetch_map(&map_a_lo);
    prefetch_map(&map_w_hi);
    prefetch_map(&map_w_lo);
    for (int s = 0; s < stages; ++s) {
      mbar_init(s_u32(&a_full[s]), 1);
      mbar_init(s_u32(&a_empty[s]), 1);
    }
    mbar_init(s_u32(w_full), 1);
    mbar_init(s_u32(w_empty), 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(s_u32(&t_full[b]), 1);
      mbar_init(s_u32(&t_empty[b]), TC2_EPI_WARPS);                  // one arrival per epilogue warp
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc<1>(s_u32(tmem_ptr_smem), (uint32_t)tmem_cols);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  // unit decode shared by all roles
  struct Unit { int64_t m_first; int n_mt; int a_row0; int w_row; int64_t m_rows; int64_t out_off; int64_t ld; int n0;
                int has_bias; };
  auto decode = [&](int u, Unit& un) {
    int g = 0;
    while (g + 1 < n_groups && u >= sc.first_unit[g + 1]) ++g;
    const hgt_lin_group grp = groups[g];
    int local = u - sc.first_unit[g];
    const int ncol = grp.n_cblocks * sc.n_tiles_n;
    const int chunk = local / ncol;
    const int col = local - chunk * ncol;
    const int cb = col / sc.n_tiles_n;
    const int nt = col - cb * sc.n_tiles_n;
    const hgt_lin_cblock cblk = cblocks[grp.cb_first + cb];
    const int64_t mt_total = (grp.m + TC_BM - 1) / TC_BM;
    un.m_first = (int64_t)chunk * TC2_MCH;
    un.n_mt = (int)min((int64_t)TC2_MCH, mt_total - un.m_first);
    un.a_row0 = (int)grp.a_row0;
    un.m_rows = grp.m;
    un.n0 = nt * BN;
    un.w_row = grp.w_row0 + cb * cb_width + un.n0;
    un.out_off = cblk.out_off;
    un.ld = cblk.ld;
    un.has_bias = grp.has_bias;
  };

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer =====
      uint32_t a_it = 0, unit_it = 0;
      for (int u = blockIdx.x; u < total_units; u += gridDim.x, ++unit_it) {
        Unit un;
        decode(u, un);
        mbar_wait(s_u32(w_empty), (unit_it & 1u) ^ 1u);               // previous unit's MMAs are done with W
        mbar_expect_tx(s_u32(w_full), (uint32_t)k_blocks * 2 * b_bytes);
        for (int kb = 0; kb < k_blocks; ++kb) {
          tma_load_2d(s_u32(w_smem + (size_t)(2 * kb) * b_bytes_al), &map_w_hi, kb * TC_BK, un.w_row, s_u32(w_full));
          tma_load_2d(s_u32(w_smem + (size_t)(2 * kb + 1) * b_bytes_al), &map_w_lo, kb * TC_BK, un.w_row, s_u32(w_full));
        }
        for (int mt = 0; mt < un.n_mt; ++mt) {
          const int a_row = un.a_row0 + (int)((un.m_first + mt) * TC_BM);
          for (int j = 0; j < 2 * k_blocks; ++j, ++a_it) {
            const int s = a_it % stages;
            mbar_wait(s_u32(&a_empty[s]), ((a_it / stages) & 1u) ^ 1u);
            const uint32_t bar = s_u32(&a_full[s]);
            mbar_expect_tx(bar, a_bytes);
            tma_load_2d(s_u32(a_smem + (size_t)s * a_stage), (j & 1) ? &map_a_lo : &map_a_hi, (j >> 1) * TC_BK, a_row, bar);
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===== MMA issuer =====
      const uint32_t idesc = idesc_bf16(TC_BM, BN, false, false);
      uint32_t a_it = 0, unit_it = 0, acc_it = 0;
      for (int u = blockIdx.x; u < total_units; u += gridDim.x, ++unit_it) {
        Unit un;
        decode(u, un);
        mbar_wait(s_u32(w_full), unit_it & 1u);
        for (int mt = 0; mt < un.n_mt; ++mt, ++acc_it) {
          const uint32_t buf = acc_it & 1u;
          mbar_wait(s_u32(&t_empty[buf]), ((acc_it >> 1) & 1u) ^ 1u);  // epilogue drained this accumulator
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + buf * (uint32_t)BN;
          for (int j = 0; j < 2 * k_blocks; ++j, ++a_it) {
            const int s = a_it % stages;
            const int kb = j >> 1;
            mbar_wait(s_u32(&a_full[s]), (a_it / stages) & 1u);
            tc_fence_after();
            const uint64_t d_a = desc_k_sw128(s_u32(a_smem + (size_t)s * a_stage));
            const uint64_t d_whi = desc_k_sw128(s_u32(w_smem + (size_t)(2 * kb) * b_bytes_al));
            if (!(j & 1)) {
              // A_hi(kb): A_hi*W_hi + A_hi*W_lo
              const uint64_t d_wlo = desc_k_sw128(s_u32(w_smem + (size_t)(2 * kb + 1) * b_bytes_al));
#pragma unroll
              for (int k = 0; k < TC_BK / UMMA_K; ++k) {
                const uint64_t o = (uint64_t)(2 * k);
                umma_bf16_ss(tmem_d, d_a + o, d_whi + o, idesc, (j > 0 || k > 0) ? 1u : 0u);
                umma_bf16_ss(tmem_d, d_a + o, d_wlo + o, idesc, 1u);
              }
            } else {
              // A_lo(kb): A_lo*W_hi
#pragma unroll
              for (int k = 0; k < TC_BK / UMMA_K; ++k) {
                const uint64_t o = (uint64_t)(2 * k);
                umma_bf16_ss(tmem_d, d_a + o, d_whi + o, idesc, 1u);
              }
            }
            umma_commit(s_u32(&a_empty[s]));
          }
          umma_commit(s_u32(&t_full[buf]));
        }
        umma_commit(s_u32(w_empty));
      }
    }
  } else {
    // ===== epilogue warps (8) =====
    const int lg = warp & 3;
    const int e = warp - 2;
    const int et = threadIdx.x - 64;
    float* stg = s_stage + (size_t)e * (32 * TC2_STG_LD);
    uint32_t acc_it = 0;
    for (int u = blockIdx.x; u < total_units; u += gridDim.x) {
      Unit un;
      decode(u, un);
      asm volatile("bar.sync 1, 256;" ::: "memory");               // previous unit's bias reads are finished
      for (int c = et; c < BN; c += 32 * TC2_EPI_WARPS) s_bias[c] = (un.has_bias && bias) ? bias[un.w_row + c] : 0.f;
      asm volatile("bar.sync 1, 256;" ::: "memory");
      for (int mt = 0; mt < un.n_mt; ++mt, ++acc_it) {
        const uint32_t buf = acc_it & 1u;
        mbar_wait(s_u32(&t_full[buf]), (acc_it >> 1) & 1u);
        tc_fence_after();
        const int64_t m0 = (un.m_first + mt) * TC_BM + lg * 32;
        tc_epilogue_tile_pf(tmem_base + ((uint32_t)(lg * 32) << 16) + buf * (uint32_t)BN, BN, e >> 2, stg, s_bias,
                            out + un.out_off + m0 * un.ld + un.n0, un.ld, un.m_rows - m0, lane);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(s_u32(&t_empty[buf]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tmem_dealloc<1>(tmem_base, (uint32_t)tmem_cols);
  }
}


// ---- 2-CTA (cta_group::2) W-stationary persistent GEMM -------------------------------------------
// A CTA pair (cluster of 2, same TPC) computes a 256 x 256 tile per step: each CTA owns 128 rows of A / of the
// accumulator and keeps HALF of the column task's W (128 of the 256 columns, all K, hi + lo) resident; the
// tcgen05.mma.cta_group::2 instruction issued by the leader reads both halves of W from the two CTAs' shared
// memory.  Each A byte streamed from L2 now feeds a 256-column product, so the A stream needs half the
// bandwidth / in-flight bytes of the single-CTA kernel above (which it could not sustain: TMA-latency-bound at
// ~45 % tensor-pipe utilisation).
// Barrier protocol: a_full / w_full live in the LEADER (both CTAs' TMA loads complete_tx there through the
// peer-bit-masked address, the leader's producer posts expect_tx for both); a_empty / w_empty / t_full are
// per-CTA and signalled by multicast tcgen05.commit; t_empty lives in the leader and collects the 8 epilogue
// warps of the pair.
template <typename OutT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC2_THREADS, 1)
k_typed_linear_tc3(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                   const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                   const float* __restrict__ bias, int Kp, int cb_width, int stages,
                   const hgt_lin_group* __restrict__ groups, int n_groups,
                   const hgt_lin_cblock* __restrict__ cblocks, OutT* __restrict__ out, Tc2Sched sc) {
  constexpr int BNH = 128;              // W columns resident per CTA
  constexpr int BNP = 256;              // columns per pair step
  constexpr int BMP = 256;              // rows per pair step
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = smem_dyn + ((1024u - (s_u32(smem_dyn) & 1023u)) & 1023u);
  const int k_blocks = (Kp + TC_BK - 1) / TC_BK;
  const uint32_t a_bytes = TC_BM * TC_BK * 2;
  const uint32_t b_bytes = (uint32_t)BNH * TC_BK * 2;               // 16 KB
  const uint32_t w_region = (uint32_t)k_blocks * 2 * b_bytes;
  unsigned char* w_smem = smem;
  unsigned char* a_smem = smem + w_region;
  uint64_t* bars = reinterpret_cast<uint64_t*>(a_smem + (size_t)stages * a_bytes);
  uint64_t* a_full = bars;
  uint64_t* a_empty = bars + stages;
  uint64_t* w_full = bars + 2 * stages;
  uint64_t* w_empty = w_full + 1;
  uint64_t* t_full = w_empty + 1;       // [2]
  uint64_t* t_empty = t_full + 2;       // [2]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(t_empty + 2);
  float* s_bias = reinterpret_cast<float*>(tmem_ptr_smem + 4);
  float* s_stage = s_bias + BNP;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta = cluster_ctarank();
  const bool leader = cta == 0;
  const int pair_id = blockIdx.x >> 1;
  const int n_pairs = gridDim.x >> 1;
  const int total_units = sc.first_unit[n_groups];

  if (warp == 0 && lane == 0) {
    prefetch_map(&map_a_hi);
    prefetch_map(&map_a_lo);
    prefetch_map(&map_w_hi);
    prefetch_map(&map_w_lo);
    for (int s = 0; s < stages; ++s) {
      mbar_init(s_u32(&a_full[s]), 1);
      mbar_init(s_u32(&a_empty[s]), 1);
    }
    mbar_init(s_u32(w_full), 1);
    mbar_init(s_u32(w_empty), 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(s_u32(&t_full[b]), 1);
      mbar_init(s_u32(&t_empty[b]), 2 * TC2_EPI_WARPS);              // epilogue warps of both CTAs (used in the leader)
    }
    fence_mbar_init();
  }
  __syncthreads();
  cluster_sync_all();                                                // both CTAs' barriers exist before any remote arrive
  if (warp == 1) {
    tmem_alloc<2>(s_u32(tmem_ptr_smem), 512u);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  struct Unit { int64_t pm_first; int n_pm; int a_row0; int w_row; int64_t m_rows; int64_t out_off; int64_t ld; int n0;
                int has_bias; };
  auto decode = [&](int u, Unit& un) {
    int g = 0;
    while (g + 1 < n_groups && u >= sc.first_unit[g + 1]) ++g;
    const hgt_lin_group grp = groups[g];
    int local = u - sc.first_unit[g];
    const int ncol = grp.n_cblocks * sc.n_tiles_n;
    const int chunk = local / ncol;
    const int col = local - chunk * ncol;
    const int cb = col / sc.n_tiles_n;
    const int nt = col - cb * sc.n_tiles_n;
    const hgt_lin_cblock cblk = cblocks[grp.cb_first + cb];
    const int64_t pm_total = (grp.m + BMP - 1) / BMP;
    un.pm_first = (int64_t)chunk * TC2_MCH;
    un.n_pm = (int)min((int64_t)TC2_MCH, pm_total - un.pm_first);
    un.a_row0 = (int)grp.a_row0;
    un.m_rows = grp.m;
    un.n0 = nt * BNP;
    un.w_row = grp.w_row0 + cb * cb_width + un.n0;
    un.out_off = cblk.out_off;
    un.ld = cblk.ld;
    un.has_bias = grp.has_bias;
  };

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer (both CTAs) =====
      uint32_t a_it = 0, unit_it = 0;
      for (int u = pair_id; u < total_units; u += n_pairs, ++unit_it) {
        Unit un;
        decode(u, un);
        mbar_wait(s_u32(w_empty), (unit_it & 1u) ^ 1u);
        if (leader) mbar_expect_tx(s_u32(w_full), 2u * (uint32_t)k_blocks * 2 * b_bytes);
        const int w_row = un.w_row + (int)cta * BNH;
        for (int kb = 0; kb < k_blocks; ++kb) {
          tma_load_2d_2sm(s_u32(w_smem + (size_t)(2 * kb) * b_bytes), &map_w_hi, kb * TC_BK, w_row, s_u32(w_full));
          tma_load_2d_2sm(s_u32(w_smem + (size_t)(2 * kb + 1) * b_bytes), &map_w_lo, kb * TC_BK, w_row, s_u32(w_full));
        }
        for (int pm = 0; pm < un.n_pm; ++pm) {
          const int a_row = un.a_row0 + (int)((un.pm_first + pm) * BMP) + (int)cta * TC_BM;
          for (int j = 0; j < 2 * k_blocks; ++j, ++a_it) {
            const int s = a_it % stages;
            mbar_wait(s_u32(&a_empty[s]), ((a_it / stages) & 1u) ^ 1u);
            const uint32_t bar = s_u32(&a_full[s]);
            if (leader) mbar_expect_tx(bar, 2u * a_bytes);
            tma_load_2d_2sm(s_u32(a_smem + (size_t)s * a_bytes), (j & 1) ? &map_a_lo : &map_a_hi, (j >> 1) * TC_BK,
                            a_row, bar);
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && leader) {
      // ===== MMA issuer (leader CTA only) =====
      const uint32_t idesc = idesc_bf16(BMP, BNP, false, false);
      uint32_t a_it = 0, unit_it = 0, acc_it = 0;
      for (int u = pair_id; u < total_units; u += n_pairs, ++unit_it) {
        Unit un;
        decode(u, un);
        mbar_wait(s_u32(w_full), unit_it & 1u);
        for (int pm = 0; pm < un.n_pm; ++pm, ++acc_it) {
          const uint32_t buf = acc_it & 1u;
          mbar_wait(s_u32(&t_empty[buf]), ((acc_it >> 1) & 1u) ^ 1u);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + buf * (uint32_t)BNP;
          for (int j = 0; j < 2 * k_blocks; ++j, ++a_it) {
            const int s = a_it % stages;
            const int kb = j >> 1;
            mbar_wait(s_u32(&a_full[s]), (a_it / stages) & 1u);
            tc_fence_after();
            const uint64_t d_a = desc_k_sw128(s_u32(a_smem + (size_t)s * a_bytes));
            const uint64_t d_whi = desc_k_sw128(s_u32(w_smem + (size_t)(2 * kb) * b_bytes));
            if (!(j & 1)) {
              const uint64_t d_wlo = desc_k_sw128(s_u32(w_smem + (size_t)(2 * kb + 1) * b_bytes));
#pragma unroll
              for (int k = 0; k < TC_BK / UMMA_K; ++k) {
                const uint64_t o = (uint64_t)(2 * k);
                umma_bf16_ss_2sm(tmem_d, d_a + o, d_whi + o, idesc, (j > 0 || k > 0) ? 1u : 0u);
                umma_bf16_ss_2sm(tmem_d, d_a + o, d_wlo + o, idesc, 1u);
              }
            } else {
#pragma unroll
              for (int k = 0; k < TC_BK / UMMA_K; ++k) {
                const uint64_t o = (uint64_t)(2 * k);
                umma_bf16_ss_2sm(tmem_d, d_a + o, d_whi + o, idesc, 1u);
              }
            }
            umma_commit_2sm(s_u32(&a_empty[s]));
          }
          umma_commit_2sm(s_u32(&t_full[buf]));
        }
        umma_commit_2sm(s_u32(w_empty));
      }
    }
  } else {
    // ===== epilogue warps (8 per CTA): own 128 rows x 256 columns =====
    const int lg = warp & 3;
    const int e = warp - 2;
    const int et = threadIdx.x - 64;
    float* stg = s_stage + (size_t)e * (32 * TC2_STG_LD);
    uint32_t acc_it = 0;
    for (int u = pair_id; u < total_units; u += n_pairs) {
      Unit un;
      decode(u, un);
      asm volatile("bar.sync 1, 256;" ::: "memory");
      for (int c = et; c < BNP; c += 32 * TC2_EPI_WARPS) s_bias[c] = (un.has_bias && bias) ? bias[un.w_row + c] : 0.f;
      asm volatile("bar.sync 1, 256;" ::: "memory");
      for (int pm = 0; pm < un.n_pm; ++pm, ++acc_it) {
        const uint32_t buf = acc_it & 1u;
        mbar_wait(s_u32(&t_full[buf]), (acc_it >> 1) & 1u);
        tc_fence_after();
        const int64_t m0 = (un.pm_first + pm) * BMP + (int64_t)cta * TC_BM + lg * 32;
        tc_epilogue_tile_pf(tmem_base + ((uint32_t)(lg * 32) << 16) + buf * (uint32_t)BNP, BNP, e >> 2, stg, s_bias,
                            out + un.out_off + m0 * un.ld + un.n0, un.ld, un.m_rows - m0, lane);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cta(s_u32(&t_empty[buf]), 0);      // the leader's barrier collects both CTAs
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                                // peer may still be reading our W through the MMA
  if (warp == 1) {
    tmem_dealloc<2>(tmem_base, 512u);
  }
}

// ---- host side ------------------------------------------------------------------------------------
// operand [rows, Kp] bf16, box {TC_BK columns, box_rows rows}
int make_map(CUtensorMap* m, const void* base, int64_t rows, int Kp, int box_rows) {
  return hgt_make_tma_map_bf16(m, base, rows, Kp, Kp, box_rows);
}

int pick_bn(int cb_width) {
  for (int bn = 128; bn >= 16; bn -= 16)
    if (cb_width % bn == 0) return bn;
  return 0;
}

void extents(const hgt_lin_group* h_groups, int n_groups, int cb_width, int64_t* a_rows, int64_t* w_rows) {
  *a_rows = 0;
  *w_rows = 0;
  for (int g = 0; g < n_groups; ++g) {
    int64_t a = h_groups[g].a_row0 + h_groups[g].m;
    int64_t w = (int64_t)h_groups[g].w_row0 + (int64_t)h_groups[g].n_cblocks * cb_width;
    if (a > *a_rows) *a_rows = a;
    if (w > *w_rows) *w_rows = w;
  }
}

// Unit prefix of the persistent kernels: per group, chunks of TC2_MCH steps of `step_rows` rows x column tasks.
int tc2_schedule(const hgt_lin_group* h_groups, int n_groups, int step_rows, int n_tiles_n, Tc2Sched* sc,
                 int64_t* units) {
  sc->n_tiles_n = n_tiles_n;
  int64_t u = 0;
  for (int g = 0; g < n_groups; ++g) {
    sc->first_unit[g] = (int32_t)u;
    const int64_t steps = (h_groups[g].m + step_rows - 1) / step_rows;
    u += (steps + TC2_MCH - 1) / TC2_MCH * h_groups[g].n_cblocks * n_tiles_n;
    HGT_REQUIRE(u < 2147483647ll, "hgt_typed_linear(tc): too many units");
  }
  sc->first_unit[n_groups] = (int32_t)u;
  *units = u;
  return 0;
}

}  // namespace

bool hgt_typed_linear_tc_supported(int64_t lda, int32_t K, int32_t cb_width) {
  (void)lda;
  return cb_width % 16 == 0 && pick_bn(cb_width) > 0 && K >= TC_BK;
}

size_t hgt_typed_linear_tc_workspace(const hgt_lin_group* h_groups, int32_t n_groups, int32_t K, int32_t cb_width) {
  int64_t a_rows, w_rows;
  extents(h_groups, n_groups, cb_width, &a_rows, &w_rows);
  const int Kp = (K + 7) / 8 * 8;
  return 4 * 256 + 2 * hgt_align_up((size_t)a_rows * Kp * 2, 256) + 2 * hgt_align_up((size_t)w_rows * Kp * 2, 256);
}

template <typename OutT>
static int tc_run(const float* A, int64_t lda, const __nv_bfloat16* a_hi_in, const __nv_bfloat16* a_lo_in,
                  const float* W, const float* bias, int32_t K, int32_t cb_width, const hgt_lin_group* groups,
                  const hgt_lin_group* h_groups, int32_t n_groups, const hgt_lin_cblock* cblocks, OutT* out,
                  void* workspace, size_t workspace_bytes, cudaStream_t st);

int hgt_typed_linear_tc(const float* A, int64_t lda, const float* W, const float* bias, int32_t K, int32_t cb_width,
                        const hgt_lin_group* groups, const hgt_lin_group* h_groups, int32_t n_groups,
                        const hgt_lin_cblock* cblocks, float* out, void* workspace, size_t workspace_bytes,
                        cudaStream_t st) {
  return tc_run(A, lda, nullptr, nullptr, W, bias, K, cb_width, groups, h_groups, n_groups, cblocks, out, workspace,
                workspace_bytes, st);
}
int hgt_typed_linear_tc(const float* A, int64_t lda, const float* W, const float* bias, int32_t K, int32_t cb_width,
                        const hgt_lin_group* groups, const hgt_lin_group* h_groups, int32_t n_groups,
                        const hgt_lin_cblock* cblocks, __nv_bfloat16* out, void* workspace, size_t workspace_bytes,
                        cudaStream_t st) {
  return tc_run(A, lda, nullptr, nullptr, W, bias, K, cb_width, groups, h_groups, n_groups, cblocks, out, workspace,
                workspace_bytes, st);
}

extern "C" int hgt_typed_linear_presplit_workspace_bytes(const hgt_lin_group* h_groups, int32_t n_groups, int32_t K,
                                                         int32_t cb_width, size_t* out_bytes) {
  HGT_REQUIRE(out_bytes && (h_groups || n_groups == 0), "hgt_typed_linear_presplit_workspace_bytes: NULL argument");
  *out_bytes = n_groups > 0 ? hgt_typed_linear_tc_workspace(h_groups, n_groups, K, cb_width) : 0;
  return 0;
}

template <typename OutT>
static int presplit(const void* a_hi, const void* a_lo, const float* W, const float* bias, int32_t K, int32_t cb_width,
                    const hgt_lin_group* groups, const hgt_lin_group* h_groups, int32_t n_groups,
                    const hgt_lin_cblock* cblocks, OutT* out, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  HGT_REQUIRE(a_hi && a_lo, "hgt_typed_linear_presplit: NULL operand");
  HGT_REQUIRE(K % 8 == 0 && hgt_typed_linear_tc_supported(K, K, cb_width),
              "hgt_typed_linear_presplit: unsupported shape K=%d cb_width=%d", K, cb_width);
  if (n_groups == 0) return 0;
  if (n_groups > kMaxGroups) {                               // see hgt_typed_linear: chunked launches
    for (int g0 = 0; g0 < n_groups; g0 += kMaxGroups) {
      const int n = n_groups - g0 < kMaxGroups ? n_groups - g0 : kMaxGroups;
      int rc = presplit(a_hi, a_lo, W, bias, K, cb_width, groups + g0, h_groups + g0, n, cblocks, out, workspace,
                        workspace_bytes, st);
      if (rc) return rc;
    }
    return 0;
  }
  return tc_run(nullptr, 0, reinterpret_cast<const __nv_bfloat16*>(a_hi), reinterpret_cast<const __nv_bfloat16*>(a_lo),
                W, bias, K, cb_width, groups, h_groups, n_groups, cblocks, out, workspace, workspace_bytes, st);
}

extern "C" int hgt_typed_linear_presplit(const void* a_hi, const void* a_lo, const float* W, const float* bias,
                                         int32_t K, int32_t cb_width, const hgt_lin_group* groups,
                                         const hgt_lin_group* h_groups, int32_t n_groups,
                                         const hgt_lin_cblock* cblocks, float* out, void* workspace,
                                         size_t workspace_bytes, void* stream_) {
  return presplit(a_hi, a_lo, W, bias, K, cb_width, groups, h_groups, n_groups, cblocks, out, workspace,
                  workspace_bytes, (cudaStream_t)stream_);
}

extern "C" int hgt_typed_linear_presplit_bf16_workspace_bytes(const hgt_lin_group* h_groups, int32_t n_groups,
                                                              int32_t K, int32_t cb_width, size_t* out_bytes) {
  return hgt_typed_linear_presplit_workspace_bytes(h_groups, n_groups, K, cb_width, out_bytes);
}

extern "C" int hgt_typed_linear_presplit_bf16(const void* a_hi, const void* a_lo, const float* W, const float* bias,
                                              int32_t K, int32_t cb_width, const hgt_lin_group* groups,
                                              const hgt_lin_group* h_groups, int32_t n_groups,
                                              const hgt_lin_cblock* cblocks, void* out, void* workspace,
                                              size_t workspace_bytes, void* stream_) {
  return presplit(a_hi, a_lo, W, bias, K, cb_width, groups, h_groups, n_groups, cblocks,
                  reinterpret_cast<__nv_bfloat16*>(out), workspace, workspace_bytes, (cudaStream_t)stream_);
}

template <typename OutT>
static int tc_run(const float* A, int64_t lda, const __nv_bfloat16* a_hi_in, const __nv_bfloat16* a_lo_in,
                  const float* W, const float* bias, int32_t K, int32_t cb_width, const hgt_lin_group* groups,
                  const hgt_lin_group* h_groups, int32_t n_groups, const hgt_lin_cblock* cblocks, OutT* out,
                  void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const int BN = pick_bn(cb_width);
  HGT_REQUIRE(BN > 0, "hgt_typed_linear(tc): cb_width=%d has no multiple-of-16 tile", cb_width);
  const int Kp = (K + 7) / 8 * 8;
  int64_t a_rows, w_rows;
  extents(h_groups, n_groups, cb_width, &a_rows, &w_rows);
  size_t need = hgt_typed_linear_tc_workspace(h_groups, n_groups, K, cb_width);
  HGT_REQUIRE(workspace && workspace_bytes >= need, "hgt_typed_linear(tc): workspace too small (%zu < %zu)",
              workspace_bytes, need);
  char* p = reinterpret_cast<char*>(hgt_align_up(reinterpret_cast<size_t>(workspace), 256));
  __nv_bfloat16* a_hi = reinterpret_cast<__nv_bfloat16*>(p); p += hgt_align_up((size_t)a_rows * Kp * 2, 256);
  __nv_bfloat16* a_lo = reinterpret_cast<__nv_bfloat16*>(p); p += hgt_align_up((size_t)a_rows * Kp * 2, 256);
  __nv_bfloat16* w_hi = reinterpret_cast<__nv_bfloat16*>(p); p += hgt_align_up((size_t)w_rows * Kp * 2, 256);
  __nv_bfloat16* w_lo = reinterpret_cast<__nv_bfloat16*>(p);
  int rc;
  if (a_hi_in) {
    a_hi = const_cast<__nv_bfloat16*>(a_hi_in);              // split by the producer (e.g. the edge kernel)
    a_lo = const_cast<__nv_bfloat16*>(a_lo_in);
  } else if ((rc = hgt_act_split_launch(A, lda, a_rows, K, Kp, 0, nullptr, a_hi, a_lo, st))) {
    return rc;
  }
  if ((rc = hgt_act_split_launch(W, K, w_rows, K, Kp, 0, nullptr, w_hi, w_lo, st))) return rc;
  CUtensorMap m_a_hi, m_a_lo, m_w_hi, m_w_lo;
  if ((rc = make_map(&m_a_hi, a_hi, a_rows, Kp, TC_BM))) return rc;
  if ((rc = make_map(&m_a_lo, a_lo, a_rows, Kp, TC_BM))) return rc;

  const int k_blocks = (Kp + TC_BK - 1) / TC_BK;
  const size_t a_stage = (size_t)TC_BM * TC_BK * 2;
  if (cb_width % 256 == 0) {
    // ---- 2-CTA kernel: 128 W columns resident per CTA, pair tile 256 x 256 ----
    const size_t w_region = (size_t)k_blocks * 2 * 128 * TC_BK * 2;
    const size_t misc = 1024 + 256 + 256 * 4 + 64 + TC2_STAGE_BYTES + 1024;
    if (w_region + misc + 4 * a_stage <= 227 * 1024) {
      const int stages = min((int)((227 * 1024 - w_region - misc) / a_stage), TC2_STAGE_CAP);
      Tc2Sched sc;
      int64_t units;
      if ((rc = tc2_schedule(h_groups, n_groups, 256, cb_width / 256, &sc, &units))) return rc;
      if (units == 0) return 0;
      if ((rc = make_map(&m_w_hi, w_hi, w_rows, Kp, 128))) return rc;
      if ((rc = make_map(&m_w_lo, w_lo, w_rows, Kp, 128))) return rc;
      size_t smem = 1024 + w_region + (size_t)stages * a_stage + (2 * stages + 6) * 8 + 16 + 256 * 4 + 64 +
                    TC2_STAGE_BYTES;
      int pairs = hgt_sm_count() / 2;
      if (pairs > units) pairs = (int)units;
      HGT_CHECK_CUDA(cudaFuncSetAttribute(k_typed_linear_tc3<OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)smem));
      k_typed_linear_tc3<OutT><<<2 * pairs, TC2_THREADS, smem, st>>>(m_a_hi, m_a_lo, m_w_hi, m_w_lo, bias, Kp, cb_width,
                                                               stages, groups, n_groups, cblocks, out, sc);
      HGT_LAUNCH_CHECK();
      return 0;
    }
  }
  // ---- W-stationary persistent kernel ----
  // widest n-tile whose resident W (all K, hi + lo) still leaves room for >= 4 A stages of 16 KB
  for (int bn = 128; bn >= 16; bn -= 16) {
    if (cb_width % bn) continue;
    const size_t w_region = (size_t)k_blocks * 2 * (((size_t)bn * TC_BK * 2 + 1023) & ~(size_t)1023);
    const size_t misc = 1024 + 256 + (size_t)bn * 4 + 64 + TC2_STAGE_BYTES + 1024;
    if (w_region + misc + 4 * a_stage > 227 * 1024) continue;
    const int stages = min((int)((227 * 1024 - w_region - misc) / a_stage), TC2_STAGE_CAP);
    Tc2Sched sc;
    int64_t units;
    if ((rc = tc2_schedule(h_groups, n_groups, TC_BM, cb_width / bn, &sc, &units))) return rc;
    if (units == 0) return 0;
    if ((rc = make_map(&m_w_hi, w_hi, w_rows, Kp, bn))) return rc;
    if ((rc = make_map(&m_w_lo, w_lo, w_rows, Kp, bn))) return rc;
    int tmem_cols = 32;
    while (tmem_cols < 2 * bn) tmem_cols <<= 1;
    size_t smem = 1024 + w_region + (size_t)stages * a_stage + (2 * stages + 6) * 8 + 16 + (size_t)bn * 4 + 64 +
                  TC2_STAGE_BYTES;
    HGT_CHECK_CUDA(cudaFuncSetAttribute(k_typed_linear_tc2<OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)smem));
    int grid = hgt_sm_count();
    if (grid > units) grid = (int)units;
    k_typed_linear_tc2<OutT><<<grid, TC2_THREADS, smem, st>>>(m_a_hi, m_a_lo, m_w_hi, m_w_lo, bias, Kp, cb_width, bn,
                                                        stages, tmem_cols, groups, n_groups, cblocks, out, sc);
    HGT_LAUNCH_CHECK();
    return 0;
  }
  // ---- one tile per CTA: no resident W fits (Kp > 2240, i.e. more than 35 k-blocks even at n-tile 16) ----
  TcTilePrefix tp;
  tp.n_tiles_n = cb_width / BN;
  int64_t total = 0;
  for (int g = 0; g < n_groups; ++g) {
    tp.first_tile[g] = (int32_t)total;
    total += (h_groups[g].m + TC_BM - 1) / TC_BM * h_groups[g].n_cblocks * tp.n_tiles_n;
    HGT_REQUIRE(total < 2147483647ll, "hgt_typed_linear(tc): too many tiles");
  }
  tp.first_tile[n_groups] = (int32_t)total;
  if (total == 0) return 0;
  if ((rc = make_map(&m_w_hi, w_hi, w_rows, Kp, BN))) return rc;
  if ((rc = make_map(&m_w_lo, w_lo, w_rows, Kp, BN))) return rc;

  const uint32_t a_bytes = TC_BM * TC_BK * 2;
  const uint32_t b_bytes_al = ((uint32_t)BN * TC_BK * 2 + 1023) & ~1023u;
  const uint32_t stage_bytes = a_bytes + b_bytes_al;
  int stages = (int)((100 * 1024) / stage_bytes);
  if (stages > 6) stages = 6;
  if (stages < 2) stages = 2;
  int tmem_cols = 32;
  while (tmem_cols < BN) tmem_cols <<= 1;
  size_t smem = 1024 + (size_t)stages * stage_bytes + (2 * stages + 1) * 8 + 16 + (size_t)BN * 4 + 64;
  HGT_CHECK_CUDA(cudaFuncSetAttribute(k_typed_linear_tc<OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_typed_linear_tc<OutT><<<(unsigned)total, TC_THREADS, smem, st>>>(m_a_hi, m_a_lo, m_w_hi, m_w_lo, bias, Kp, cb_width,
                                                               BN, stages, tmem_cols, groups, n_groups, cblocks, out,
                                                               tp);
  HGT_LAUNCH_CHECK();
  return 0;
}
