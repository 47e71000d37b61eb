// Graph ingest for the HGTConv hot path: int64 COO (pyHGT/data.py:251-256) -> type-sorted node order,
// destination-sorted CSR, per-edge gather rows, balanced work tiles.  Runs once per graph; the sort
// and scans use CUB device primitives (CUDA toolkit), everything else is hand-written.
#include "common.cuh"

#include <cuda_bf16.h>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

namespace {

constexpr int kThreads = 256;

inline int bits_for(int64_t n) {
  int b = 1;
  while ((int64_t(1) << b) < n && b < 31) ++b;
  return b;
}

struct PlanScratch {
  int32_t* keys_in;
  int32_t* keys_out;
  int32_t* vals_in;
  int32_t* counts;   // [N+1]
  int64_t* packed;   // [N+1] (tile planning)
  void* cub_tmp;
  size_t cub_bytes;
};

size_t cub_sort_bytes(int64_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const int32_t*)nullptr, (int32_t*)nullptr,
                                  (const int32_t*)nullptr, (int32_t*)nullptr, (int)n, 0, 32);
  return bytes;
}
size_t cub_scan_bytes(int64_t n) {
  size_t b1 = 0, b2 = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, b1, (const int32_t*)nullptr, (int32_t*)nullptr, (int)n);
  cub::DeviceScan::ExclusiveSum(nullptr, b2, (const int64_t*)nullptr, (int64_t*)nullptr, (int)n);
  return b1 > b2 ? b1 : b2;
}

size_t carve(PlanScratch& s, void* base, int64_t n_nodes, int64_t n_edges) {
  int64_t m = n_nodes > n_edges ? n_nodes : n_edges;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off += hgt_align_up(bytes, 256);
    return base ? (char*)base + o : (char*)nullptr;
  };
  s.keys_in = (int32_t*)take(sizeof(int32_t) * (m + 1));
  s.keys_out = (int32_t*)take(sizeof(int32_t) * (m + 1));
  s.vals_in = (int32_t*)take(sizeof(int32_t) * (m + 1));
  s.counts = (int32_t*)take(sizeof(int32_t) * (n_nodes + 2));
  s.packed = (int64_t*)take(sizeof(int64_t) * (n_nodes + 2));
  size_t a = cub_sort_bytes(m + 1), b = cub_scan_bytes(n_nodes + 2);
  s.cub_bytes = a > b ? a : b;
  s.cub_tmp = take(s.cub_bytes);
  return off;
}

// ---- nodes -------------------------------------------------------------------------------------
__global__ void k_node_keys(const int64_t* __restrict__ node_type, int64_t n, int T,
                            int32_t* __restrict__ keys, int32_t* __restrict__ vals,
                            int32_t* __restrict__ type_count, int32_t* __restrict__ sorted_flag) {
  extern __shared__ int32_t hist[];
  for (int i = threadIdx.x; i <= T; i += blockDim.x) hist[i] = 0;
  __syncthreads();
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) {
    int64_t t = node_type[i];
    int32_t k = (t >= 0 && t < T) ? (int32_t)t : T;
    keys[i] = k;
    vals[i] = (int32_t)i;
    atomicAdd(&hist[k], 1);
    if (i + 1 < n) {
      int64_t t2 = node_type[i + 1];
      int32_t k2 = (t2 >= 0 && t2 < T) ? (int32_t)t2 : T;
      if (k2 < k) *sorted_flag = 0;
    }
  }
  __syncthreads();
  for (int j = threadIdx.x; j <= T; j += blockDim.x)
    if (hist[j]) atomicAdd(&type_count[j], hist[j]);
}

__global__ void k_inverse_perm(const int32_t* __restrict__ perm, int64_t n, int32_t* __restrict__ rank) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) rank[perm[i]] = (int32_t)i;
}

// ---- edges -------------------------------------------------------------------------------------
__global__ void k_edge_keys(const int64_t* __restrict__ edge_index, const int64_t* __restrict__ edge_type,
                            const int64_t* __restrict__ node_type, const int32_t* __restrict__ rank,
                            int64_t N, int64_t E, int T, int R, int32_t* __restrict__ keys,
                            int32_t* __restrict__ vals, int32_t* __restrict__ counts,
                            int32_t* __restrict__ presence, int32_t* __restrict__ flags) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int32_t key = -1;                                  // -1: no histogram contribution (past the end / invalid endpoint)
  if (e < E) {
    int64_t src = edge_index[e], dst = edge_index[E + e];
    vals[e] = (int32_t)e;
    if (src < 0 || src >= N || dst < 0 || dst >= N) {
      flags[0] = 1;
      keys[e] = 0;
    } else {
      key = rank[dst];
      keys[e] = key;
      int64_t s = node_type[src], t = node_type[dst], r = edge_type[e];
      if (s >= 0 && s < T && t >= 0 && t < T && r >= 0 && r < R) presence[s * R + r] = 1;
    }
  }
  // in-degree histogram, aggregated per warp: to_torch hands the edges over in <target type, ...> blocks and real graphs
  // have hub destinations, so neighbouring edges often share a destination — one atomic per distinct key and warp
  // instead of one per edge (power-law C5: 5.2 ms -> contention-free)
  const unsigned same = __match_any_sync(0xffffffffu, key);
  if (key >= 0 && (int)(threadIdx.x & 31) == __ffs(same) - 1) atomicAdd(&counts[key], __popc(same));
}

__global__ void k_edge_fill(const int64_t* __restrict__ edge_index, const int64_t* __restrict__ edge_type,
                            const int64_t* __restrict__ edge_time, const int64_t* __restrict__ node_type,
                            const int32_t* __restrict__ rank, const int32_t* __restrict__ csr_eid,
                            int64_t N, int64_t E, int T, int R, const int32_t* __restrict__ pair_of,
                            const int32_t* __restrict__ pair_row0, const int32_t* __restrict__ type_row0,
                            int32_t zero_row, int32_t zero_rte_row, int32_t* __restrict__ kv_row,
                            int32_t* __restrict__ rte_row, int32_t* __restrict__ flags) {
  int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c >= E) return;
  int64_t e = csr_eid[c];
  int64_t src = edge_index[e], dst = edge_index[E + e];
  int32_t row = zero_row, rrow = zero_rte_row;
  if (src >= 0 && src < N && dst >= 0 && dst < N) {
    int64_t s = node_type[src], t = node_type[dst], r = edge_type[e];
    if (s >= 0 && s < T && t >= 0 && t < T && r >= 0 && r < R) {
      int32_t p = pair_of[s * R + r];
      if (p >= 0) {
        row = pair_row0[p] + (rank[src] - type_row0[s]);
        if (edge_time) {
          int64_t dt = edge_time[e];
          if (dt < 0 || dt >= HGT_RTE_MAX_LEN) {
            flags[1] = 1;   // nn.Embedding would raise (conv.py:299)
            dt = 0;
          }
          rrow = p * HGT_RTE_MAX_LEN + (int32_t)dt;
        }
      }
    }
  }
  kv_row[c] = row;
  if (rte_row) rte_row[c] = rrow;
}

// ---- work tiles --------------------------------------------------------------------------------
// cost(k) = 2*deg(k) + 1 (an edge reads a 2d-float KV row, every destination writes a d-float row).
// A destination starts a tile when its cost prefix enters a new bucket of `tc` units; a hub
// (deg > split) gets ceil(deg/split) tiles of its own.
__device__ __forceinline__ bool tile_starts_at(const int32_t* row_ptr, int64_t k, int tc, int split) {
  if (k == 0) return true;
  int32_t deg_prev = row_ptr[k] - row_ptr[k - 1];
  if (deg_prev > split) return true;                       // first destination after a hub
  int64_t c1 = 2 * (int64_t)row_ptr[k] + k, c0 = 2 * (int64_t)row_ptr[k - 1] + (k - 1);
  return (c1 / tc) != (c0 / tc);
}

__global__ void k_tile_emit_counts(const int32_t* __restrict__ row_ptr, int64_t N, int tc, int split,
                                   int64_t* __restrict__ packed) {
  int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k > N) return;
  if (k == N) { packed[k] = 0; return; }
  int32_t deg = row_ptr[k + 1] - row_ptr[k];
  int64_t emit, emit_split;
  if (deg > split) {
    emit = (deg + split - 1) / split;
    emit_split = emit;
  } else {
    emit = tile_starts_at(row_ptr, k, tc, split) ? 1 : 0;
    emit_split = 0;
  }
  packed[k] = (emit << 32) | emit_split;
}

__global__ void k_tile_write(const int32_t* __restrict__ row_ptr, int64_t N, int tc, int split,
                             const int64_t* __restrict__ packed_scan, int32_t* __restrict__ tiles,
                             int64_t max_tiles, int32_t* __restrict__ n_tiles, int32_t* __restrict__ hubs,
                             int64_t max_hubs) {
  int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k > N) return;
  int64_t slot = packed_scan[k] >> 32, pslot = packed_scan[k] & 0xffffffffll;
  if (k == N) { n_tiles[0] = (int32_t)slot; n_tiles[1] = (int32_t)pslot; return; }
  int32_t b = row_ptr[k], deg = row_ptr[k + 1] - b;
  if (deg > split) {
    int pieces = (deg + split - 1) / split;
    int per = (deg + pieces - 1) / pieces;
    int hidx = atomicAdd(&n_tiles[2], 1);                  // hub list order is arbitrary; each hub merges alone
    if (hidx < max_hubs) {
      hubs[4 * hidx + 0] = (int32_t)k; hubs[4 * hidx + 1] = (int32_t)pslot; hubs[4 * hidx + 2] = pieces;
      hubs[4 * hidx + 3] = 0;
    }
    for (int i = 0; i < pieces; ++i) {
      if (slot + i >= max_tiles) return;
      int32_t* t = tiles + 4 * (slot + i);
      int32_t eb = b + i * per, ee = min(b + deg, eb + per);
      t[0] = (int32_t)k; t[1] = -(int32_t)(pslot + i) - 1; t[2] = eb; t[3] = ee;
    }
  } else if (tile_starts_at(row_ptr, k, tc, split)) {
    if (slot >= max_tiles) return;
    int32_t* t = tiles + 4 * slot;
    t[0] = (int32_t)k; t[1] = 0; t[2] = b; t[3] = 0;     // end fields patched by k_tile_close
  }
}

__global__ void k_tile_close(const int32_t* __restrict__ row_ptr, int64_t N, int32_t* __restrict__ tiles,
                             const int32_t* __restrict__ n_tiles) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int nt = n_tiles[0];
  if (i >= nt) return;
  int32_t* t = tiles + 4 * i;
  if (t[1] < 0) return;                                   // hub piece: complete
  int32_t dend = (i + 1 < nt) ? tiles[4 * (i + 1)] : (int32_t)N;
  t[1] = dend;
  t[3] = row_ptr[dend];
}

__global__ void k_gather_rows(const float4* __restrict__ in, const int32_t* __restrict__ perm, int64_t n_rows,
                              int vec_per_row, float4* __restrict__ out) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t total = n_rows * vec_per_row;
  if (i >= total) return;
  int64_t r = i / vec_per_row;
  int c = (int)(i - r * vec_per_row);
  out[i] = in[(int64_t)perm[r] * vec_per_row + c];
}
__global__ void k_gather_rows_scalar(const float* __restrict__ in, const int32_t* __restrict__ perm,
                                     int64_t n_rows, int width, float* __restrict__ out) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t total = n_rows * width;
  if (i >= total) return;
  int64_t r = i / width;
  int c = (int)(i - r * width);
  out[i] = in[(int64_t)perm[r] * width + c];
}

// Fused halo exchange: one warp per destination row pulls it from the owner's HBM (NVLink peer mapping).
__global__ void k_halo_pull(const float* const* __restrict__ peers, const int32_t* __restrict__ src_rank,
                            const int32_t* __restrict__ src_row, int64_t n_rows, int vec_per_row, int64_t row_base,
                            float4* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp; r < n_rows; r += n_warps) {
    const float4* src = reinterpret_cast<const float4*>(peers[src_rank[r]]) + (row_base + src_row[r]) * vec_per_row;
    float4* dst = out + r * vec_per_row;
    for (int c = lane; c < vec_per_row; c += 32) {
      float4 v;
      asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                   : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(src + c));
      dst[c] = v;
    }
  }
}

// Pull + convert: the halo rows are only ever consumed as the bf16 hi/lo operand split of the projection GEMM, so the
// conversion is done while the row crosses NVLink; fp32 is kept only for the rows this rank owns (skip connection).
template <int VPL>   // float4 chunks per lane and row (row = 32 * VPL float4 at most)
__global__ void __launch_bounds__(256)
k_halo_pull_split(const float* const* __restrict__ peers, const int32_t* __restrict__ src_rank,
                  const int32_t* __restrict__ src_row, const int32_t* __restrict__ order, int64_t n_rows,
                  int vec_per_row, int self_rank, int64_t row_base, float4* __restrict__ out_f32,
                  uint2* __restrict__ hi, uint2* __restrict__ lo) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  constexpr int RB = (VPL <= 2) ? 4 : (VPL <= 4 ? 2 : 1);   // rows per pass: every load of RB rows is in flight before the
                                                            // first conversion, so NVLink round trips overlap
  for (int64_t r0 = warp * RB; r0 < n_rows; r0 += n_warps * RB) {
    float4 v[RB][VPL];
    int owner[RB];
#pragma unroll
    int64_t rows[RB];
#pragma unroll
    for (int b = 0; b < RB; ++b) {
      // `order` staggers the peers: consecutive work items cycle through all owners, so every NVLink source is read by
      // all ranks at an even rate instead of everybody draining owner 0 first
      rows[b] = (r0 + b < n_rows) ? (order ? (int64_t)order[r0 + b] : r0 + b) : -1;
    }
#pragma unroll
    for (int b = 0; b < RB; ++b) {
      const int64_t r = rows[b];
      owner[b] = -1;
      if (r >= 0) {
        owner[b] = src_rank[r];
        const float4* src = reinterpret_cast<const float4*>(peers[owner[b]]) + (row_base + src_row[r]) * vec_per_row;
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
          const int c = lane + 32 * i;
          if (c < vec_per_row)
            asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                         : "=f"(v[b][i].x), "=f"(v[b][i].y), "=f"(v[b][i].z), "=f"(v[b][i].w) : "l"(src + c));
        }
      }
    }
#pragma unroll
    for (int b = 0; b < RB; ++b) {
      const int64_t r = rows[b];
      if (r < 0) continue;
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        const int c = lane + 32 * i;
        if (c < vec_per_row) {
          if (owner[b] == self_rank) out_f32[r * vec_per_row + c] = v[b][i];
          const float f[4] = {v[b][i].x, v[b][i].y, v[b][i].z, v[b][i].w};
          hgt_split_bf16x4(f, &hi[r * vec_per_row + c], &lo[r * vec_per_row + c]);
        }
      }
    }
  }
}

// Push variant of the same exchange (experimental, halo_mode="push"): every OWNER converts its rows once and stores the bf16
// hi/lo split straight into the consumers' symmetric operand buffers — posted NVLink writes instead of reads.  Work item i:
// row push_src[i] of x_own goes to row push_dst[i] (+ row_base) of rank push_peer[i]'s buffers; the items addressed to
// self_rank also keep the fp32 copy the skip connection needs.  The caller interleaves / staggers the peers in the item order.
template <int VPL>
__global__ void __launch_bounds__(256)
k_halo_push_split(const float4* __restrict__ x_own, const int32_t* __restrict__ push_peer,
                  const int32_t* __restrict__ push_src, const int32_t* __restrict__ push_dst, int64_t n_items,
                  int vec_per_row, int self_rank, int64_t row_base, uint2* const* __restrict__ hi_peers,
                  uint2* const* __restrict__ lo_peers, float4* __restrict__ x_local_f32) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp; i < n_items; i += n_warps) {
    const int peer = push_peer[i];
    const float4* src = x_own + (int64_t)push_src[i] * vec_per_row;
    const int64_t drow = (int64_t)push_dst[i];
    uint2* hi = hi_peers[peer] + (row_base + drow) * vec_per_row;
    uint2* lo = lo_peers[peer] + (row_base + drow) * vec_per_row;
    float4 v[VPL];
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
      const int c = lane + 32 * k;
      if (c < vec_per_row) v[k] = __ldg(src + c);
    }
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
      const int c = lane + 32 * k;
      if (c < vec_per_row) {
        if (peer == self_rank) x_local_f32[drow * vec_per_row + c] = v[k];
        const float f[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
        hgt_split_bf16x4(f, hi + c, lo + c);
      }
    }
  }
}

inline unsigned blocks_for(int64_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

}  // namespace

extern "C" int hgt_plan_workspace_bytes(int64_t n_nodes, int64_t n_edges, size_t* out_bytes) {
  HGT_REQUIRE(out_bytes, "hgt_plan_workspace_bytes: out_bytes is NULL");
  HGT_REQUIRE(n_nodes >= 0 && n_edges >= 0 && n_nodes < 2147483000ll && n_edges < 2147483000ll,
              "hgt_plan_workspace_bytes: n_nodes=%lld / n_edges=%lld outside the int32 index range",
              (long long)n_nodes, (long long)n_edges);
  PlanScratch s;
  *out_bytes = carve(s, nullptr, n_nodes, n_edges) + 256;
  return 0;
}

extern "C" int hgt_plan_nodes(const int64_t* node_type, int64_t n_nodes, int32_t num_types,
                              int32_t* rank, int32_t* perm, int32_t* type_count, int32_t* sorted_flag,
                              void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HGT_REQUIRE(num_types >= 1 && num_types <= 4096, "hgt_plan_nodes: num_types=%d unsupported", num_types);
  PlanScratch s;
  size_t need = carve(s, workspace, n_nodes, 0);
  HGT_REQUIRE(workspace_bytes >= need, "hgt_plan_nodes: workspace too small (%zu < %zu)", workspace_bytes, need);
  HGT_CHECK_CUDA(cudaMemsetAsync(type_count, 0, sizeof(int32_t) * (num_types + 1), st));
  int32_t one = 1;
  HGT_CHECK_CUDA(cudaMemcpyAsync(sorted_flag, &one, sizeof(int32_t), cudaMemcpyHostToDevice, st));
  if (n_nodes == 0) return 0;
  k_node_keys<<<blocks_for(n_nodes), kThreads, sizeof(int32_t) * (num_types + 1), st>>>(
      node_type, n_nodes, num_types, s.keys_in, s.vals_in, type_count, sorted_flag);
  HGT_LAUNCH_CHECK();
  size_t tmp = s.cub_bytes;
  HGT_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(s.cub_tmp, tmp, (const int32_t*)s.keys_in, s.keys_out,
                                                 (const int32_t*)s.vals_in, perm, (int)n_nodes, 0,
                                                 bits_for(num_types + 1), st));
  k_inverse_perm<<<blocks_for(n_nodes), kThreads, 0, st>>>(perm, n_nodes, rank);
  HGT_LAUNCH_CHECK();
  return 0;
}

extern "C" int hgt_plan_edges_sort(const int64_t* edge_index, const int64_t* edge_type, const int64_t* node_type,
                                   const int32_t* rank, int64_t n_nodes, int64_t n_edges,
                                   int32_t num_types, int32_t num_relations, int32_t* row_ptr,
                                   int32_t* csr_eid, int32_t* presence, int32_t* flags, void* workspace,
                                   size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  PlanScratch s;
  size_t need = carve(s, workspace, n_nodes, n_edges);
  HGT_REQUIRE(workspace_bytes >= need, "hgt_plan_edges_sort: workspace too small (%zu < %zu)", workspace_bytes, need);
  HGT_CHECK_CUDA(cudaMemsetAsync(s.counts, 0, sizeof(int32_t) * (n_nodes + 1), st));
  HGT_CHECK_CUDA(cudaMemsetAsync(presence, 0, sizeof(int32_t) * num_types * num_relations, st));
  HGT_CHECK_CUDA(cudaMemsetAsync(flags, 0, sizeof(int32_t) * 4, st));
  if (n_edges > 0) {
    k_edge_keys<<<blocks_for(n_edges), kThreads, 0, st>>>(edge_index, edge_type, node_type, rank, n_nodes,
                                                          n_edges, num_types, num_relations, s.keys_in,
                                                          s.vals_in, s.counts, presence, flags);
    HGT_LAUNCH_CHECK();
  }
  size_t tmp = s.cub_bytes;
  HGT_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(s.cub_tmp, tmp, (const int32_t*)s.counts, row_ptr,
                                               (int)(n_nodes + 1), st));
  if (n_edges > 0) {
    tmp = s.cub_bytes;
    HGT_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(s.cub_tmp, tmp, (const int32_t*)s.keys_in, s.keys_out,
                                                   (const int32_t*)s.vals_in, csr_eid, (int)n_edges, 0,
                                                   bits_for(n_nodes > 1 ? n_nodes : 2), st));
  }
  return 0;
}

extern "C" int hgt_plan_edges_fill(const int64_t* edge_index, const int64_t* edge_type, const int64_t* edge_time,
                                   const int64_t* node_type, const int32_t* rank, const int32_t* csr_eid,
                                   int64_t n_nodes, int64_t n_edges, int32_t num_types, int32_t num_relations,
                                   const int32_t* pair_of, const int32_t* pair_row0, const int32_t* type_row0,
                                   int32_t zero_row, int32_t zero_rte_row, int32_t* kv_row, int32_t* rte_row,
                                   int32_t* flags, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (n_edges == 0) return 0;
  HGT_REQUIRE((edge_time != nullptr) == (rte_row != nullptr),
              "hgt_plan_edges_fill: edge_time and rte_row must both be given or both be NULL");
  k_edge_fill<<<blocks_for(n_edges), kThreads, 0, st>>>(edge_index, edge_type, edge_time, node_type, rank,
                                                        csr_eid, n_nodes, n_edges, num_types, num_relations,
                                                        pair_of, pair_row0, type_row0, zero_row, zero_rte_row,
                                                        kv_row, rte_row, flags);
  HGT_LAUNCH_CHECK();
  return 0;
}

extern "C" int hgt_plan_tiles(const int32_t* row_ptr, int64_t n_nodes, int64_t n_edges, int32_t target_edges,
                              int32_t split_edges, int32_t* tiles, int64_t max_tiles, int32_t* hubs,
                              int64_t max_hubs, int32_t* d_n_tiles, int32_t* h_n_tiles, void* workspace,
                              size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HGT_REQUIRE(target_edges >= 1 && split_edges >= 1, "hgt_plan_tiles: bad tile parameters");
  if (h_n_tiles) h_n_tiles[0] = h_n_tiles[1] = h_n_tiles[2] = 0;
  HGT_CHECK_CUDA(cudaMemsetAsync(d_n_tiles, 0, 3 * sizeof(int32_t), st));
  if (n_nodes == 0) return 0;
  int tc = 2 * target_edges;
  PlanScratch s;
  size_t need = carve(s, workspace, n_nodes, n_edges);
  HGT_REQUIRE(workspace_bytes >= need, "hgt_plan_tiles: workspace too small (%zu < %zu)", workspace_bytes, need);
  int64_t* packed = s.packed;
  void* tmp = s.cub_tmp;
  size_t tmp_bytes = s.cub_bytes;
  k_tile_emit_counts<<<blocks_for(n_nodes + 1), kThreads, 0, st>>>(row_ptr, n_nodes, tc, split_edges, packed);
  HGT_LAUNCH_CHECK();
  HGT_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, (const int64_t*)packed, packed,
                                               (int)(n_nodes + 1), st));
  k_tile_write<<<blocks_for(n_nodes + 1), kThreads, 0, st>>>(row_ptr, n_nodes, tc, split_edges, packed, tiles,
                                                             max_tiles, d_n_tiles, hubs, max_hubs);
  HGT_LAUNCH_CHECK();
  if (h_n_tiles == nullptr) {
    // sync-free mode: the counts stay on the device (the edge kernels read them through d_tile_counts); tile slots past
    // max_tiles are never written (k_tile_write clamps), so callers size max_tiles / max_hubs with the documented bounds
    if (max_tiles > 0) {
      k_tile_close<<<blocks_for(max_tiles), kThreads, 0, st>>>(row_ptr, n_nodes, tiles, d_n_tiles);
      HGT_LAUNCH_CHECK();
    }
    return 0;
  }
  HGT_CHECK_CUDA(cudaMemcpyAsync(h_n_tiles, d_n_tiles, 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  HGT_CHECK_CUDA(cudaStreamSynchronize(st));
  HGT_REQUIRE(h_n_tiles[0] <= max_tiles, "hgt_plan_tiles: %d tiles exceed max_tiles=%lld", h_n_tiles[0],
              (long long)max_tiles);
  HGT_REQUIRE(h_n_tiles[2] <= max_hubs, "hgt_plan_tiles: %d hubs exceed max_hubs=%lld", h_n_tiles[2],
              (long long)max_hubs);
  if (h_n_tiles[0] > 0) {
    k_tile_close<<<blocks_for(h_n_tiles[0]), kThreads, 0, st>>>(row_ptr, n_nodes, tiles, d_n_tiles);
    HGT_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" int hgt_gather_rows(const float* in, const int32_t* perm, int64_t n_rows, int32_t width, float* out,
                               void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (n_rows == 0) return 0;
  if (width % 4 == 0 && ((uintptr_t)in % 16 == 0) && ((uintptr_t)out % 16 == 0)) {
    k_gather_rows<<<blocks_for(n_rows * (width / 4)), kThreads, 0, st>>>((const float4*)in, perm, n_rows,
                                                                         width / 4, (float4*)out);
  } else {
    k_gather_rows_scalar<<<blocks_for(n_rows * width), kThreads, 0, st>>>(in, perm, n_rows, width, out);
  }
  HGT_LAUNCH_CHECK();
  return 0;
}

extern "C" int hgt_halo_pull(uint64_t peer_ptrs_dev, const int32_t* src_rank, const int32_t* src_row, int64_t n_rows,
                             int32_t width, int64_t row_base, float* out, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HGT_REQUIRE(width % 4 == 0, "hgt_halo_pull: row width %d must be a multiple of 4 floats", width);
  if (n_rows == 0) return 0;
  const int warps_per_block = 8;
  int64_t blocks = (n_rows + warps_per_block - 1) / warps_per_block;
  int64_t cap = (int64_t)hgt_sm_count() * 16;
  if (blocks > cap) blocks = cap;
  k_halo_pull<<<(unsigned)blocks, warps_per_block * 32, 0, st>>>(reinterpret_cast<const float* const*>(peer_ptrs_dev),
                                                                 src_rank, src_row, n_rows, width / 4, row_base,
                                                                 reinterpret_cast<float4*>(out));
  HGT_LAUNCH_CHECK();
  return 0;
}

extern "C" int hgt_halo_pull_split(uint64_t peer_ptrs_dev, const int32_t* src_rank, const int32_t* src_row,
                                   const int32_t* order, int64_t n_rows, int32_t width, int32_t self_rank,
                                   int64_t row_base, float* out_f32, void* hi, void* lo, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HGT_REQUIRE(width % 8 == 0, "hgt_halo_pull_split: row width %d must be a multiple of 8 floats", width);
  HGT_REQUIRE(out_f32 && hi && lo, "hgt_halo_pull_split: NULL output");
  if (n_rows == 0) return 0;
  const int warps_per_block = 8;
  int64_t blocks = (n_rows + warps_per_block - 1) / warps_per_block;
  int64_t cap = (int64_t)hgt_sm_count() * 16;
  if (blocks > cap) blocks = cap;
  const int vpr = width / 4;
  HGT_REQUIRE(vpr <= 256, "hgt_halo_pull_split: rows of more than 1024 floats are not supported (width=%d)", width);
  auto pf = reinterpret_cast<const float* const*>(peer_ptrs_dev);
  auto o4 = reinterpret_cast<float4*>(out_f32);
  auto h2 = reinterpret_cast<uint2*>(hi);
  auto l2 = reinterpret_cast<uint2*>(lo);
  const unsigned g = (unsigned)blocks, t = warps_per_block * 32;
  if (vpr <= 32) k_halo_pull_split<1><<<g, t, 0, st>>>(pf, src_rank, src_row, order, n_rows, vpr, self_rank, row_base, o4, h2, l2);
  else if (vpr <= 64) k_halo_pull_split<2><<<g, t, 0, st>>>(pf, src_rank, src_row, order, n_rows, vpr, self_rank, row_base, o4, h2, l2);
  else if (vpr <= 128) k_halo_pull_split<4><<<g, t, 0, st>>>(pf, src_rank, src_row, order, n_rows, vpr, self_rank, row_base, o4, h2, l2);
  else k_halo_pull_split<8><<<g, t, 0, st>>>(pf, src_rank, src_row, order, n_rows, vpr, self_rank, row_base, o4, h2, l2);
  HGT_LAUNCH_CHECK();
  return 0;
}

extern "C" int hgt_halo_push_split(const float* x_own, const int32_t* push_peer, const int32_t* push_src,
                                   const int32_t* push_dst, int64_t n_items, int32_t width, int32_t self_rank,
                                   int64_t row_base, uint64_t hi_ptrs_dev, uint64_t lo_ptrs_dev, float* x_local_f32,
                                   void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HGT_REQUIRE(width % 8 == 0 && width / 4 <= 256, "hgt_halo_push_split: row width %d must be a multiple of 8, at most 1024", width);
  HGT_REQUIRE(x_own && push_peer && push_src && push_dst && hi_ptrs_dev && lo_ptrs_dev && x_local_f32,
              "hgt_halo_push_split: NULL argument");
  if (n_items == 0) return 0;
  const int vpr = width / 4;
  int64_t blocks = (n_items + 7) / 8;
  const int64_t cap = (int64_t)hgt_sm_count() * 8;
  if (blocks > cap) blocks = cap;
  auto xo = reinterpret_cast<const float4*>(x_own);
  auto hp = reinterpret_cast<uint2* const*>(hi_ptrs_dev);
  auto lp = reinterpret_cast<uint2* const*>(lo_ptrs_dev);
  auto xl = reinterpret_cast<float4*>(x_local_f32);
  const unsigned g = (unsigned)blocks;
  if (vpr <= 32) k_halo_push_split<1><<<g, 256, 0, st>>>(xo, push_peer, push_src, push_dst, n_items, vpr, self_rank, row_base, hp, lp, xl);
  else if (vpr <= 64) k_halo_push_split<2><<<g, 256, 0, st>>>(xo, push_peer, push_src, push_dst, n_items, vpr, self_rank, row_base, hp, lp, xl);
  else if (vpr <= 128) k_halo_push_split<4><<<g, 256, 0, st>>>(xo, push_peer, push_src, push_dst, n_items, vpr, self_rank, row_base, hp, lp, xl);
  else k_halo_push_split<8><<<g, 256, 0, st>>>(xo, push_peer, push_src, push_dst, n_items, vpr, self_rank, row_base, hp, lp, xl);
  HGT_LAUNCH_CHECK();
  return 0;
}
