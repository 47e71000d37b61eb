// Error channel + small utilities shared by every translation unit of libhgt_b200.so.
#include "common.cuh"
#include "tc_ptx.cuh"

#include <string.h>

static thread_local char g_err[1024] = "";

void hgt_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int hgt_sm_count() {
  static int cached = 0;
  if (cached) return cached;
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
    n = HGT_SM_COUNT_FALLBACK;
  cached = n;
  return n;
}

// The driver entry point is looked up through the runtime, so the library does not link libcuda.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

int hgt_make_tma_map_bf16(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  HGT_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)(rows > 0 ? rows : 1)};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {64u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  HGT_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld ld=%lld box_rows=%d", (int)r,
              (long long)rows, (long long)cols, (long long)ld, box_rows);
  return 0;
}

unsigned long long g_hgt_launches = 0;

extern "C" uint64_t hgt_kernel_launches(void) { return g_hgt_launches; }
extern "C" const char* hgt_last_error(void) { return g_err; }
extern "C" int hgt_abi_version(void) { return 2; }

__global__ void k_ordered_sum(const float* __restrict__ part, const hgt_sum_seg* __restrict__ segs, int64_t n,
                              float* __restrict__ dst) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const hgt_sum_seg s = segs[blockIdx.y];
  dst[s.dst + i] += hgt_chunk_sum(part + s.part + i, s.chunks, n);
}

int hgt_ordered_sum_launch(const float* part, const hgt_sum_seg* segs, int n_segs, int64_t n, float* dst,
                           cudaStream_t st) {
  if (n_segs == 0 || n == 0) return 0;
  HGT_REQUIRE(n_segs <= 65535, "hgt_ordered_sum_launch: %d segments exceed the grid limit", n_segs);
  k_ordered_sum<<<dim3((unsigned)((n + 255) / 256), (unsigned)n_segs), 256, 0, st>>>(part, segs, n, dst);
  HGT_LAUNCH_CHECK();
  return 0;
}
