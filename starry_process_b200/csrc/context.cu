// Context management, error reporting, launch accounting for libspb200.
#include <stdlib.h>

#include <mutex>

#include "common.cuh"
#include "spb_tables.h"

int spb_wigner_init(spb_context *ctx);  // wigner.cu: constant-bank copy of the Rx(pi/2) non-zeros

static thread_local std::string g_last_error;

void spb_set_error(const std::string &msg) { g_last_error = msg; }

extern "C" const char *spb_last_error(void) { return g_last_error.c_str(); }
extern "C" int spb_version(void) { return 100; }

// Everything spb_create allocates; released by spb_destroy AND by every early return of spb_create
// (the guard below), so a failed construction leaks nothing.
static void spb_release(spb_context *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->d_tables) cudaFree(ctx->d_tables);
  if (ctx->d_counters) cudaFree(ctx->d_counters);
  if (ctx->d_scratch) cudaFree(ctx->d_scratch);
  delete ctx;
}

namespace {
struct CtxGuard {
  spb_context *ctx;
  ~CtxGuard() { spb_release(ctx); }
  spb_context *release() {
    spb_context *c = ctx;
    ctx = nullptr;
    return c;
  }
};
}  // namespace

extern "C" int spb_create(int device, const double *tables_host, size_t tables_count,
                          spb_context **out) {
  SPB_REQUIRE(out != nullptr, "spb_create: null output pointer");
  int ndev = 0;
  SPB_CHECK_CUDA(cudaGetDeviceCount(&ndev));
  SPB_REQUIRE(device >= 0 && device < ndev, "spb_create: no such CUDA device");
  SPB_CHECK_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  SPB_CHECK_CUDA(cudaGetDeviceProperties(&prop, device));
  SPB_REQUIRE(prop.major >= 10, "spb_create: libspb200 is built for sm_100a (B200) only");
  CtxGuard guard{new spb_context()};
  spb_context *ctx = guard.ctx;
  ctx->device = device;
  ctx->num_sms = prop.multiProcessorCount;
  ctx->d_tables = nullptr;
  ctx->tables_count = tables_count;
  ctx->launches = 0;
  ctx->d_counters = nullptr;
  ctx->counter_next = 0;
  ctx->d_scratch = nullptr;
  ctx->opt_no_tma = getenv("SPB_NO_TMA") != nullptr;          // defaults of the A/B switches
  ctx->opt_no_cluster = getenv("SPB_NO_CLUSTER") != nullptr;
  ctx->opt_syrk_i8 = getenv("SPB_SYRK_I8") ? atoi(getenv("SPB_SYRK_I8")) : 1;   // default: INT8 tensor cores
  for (int k = 0; k < 3; ++k) ctx->max_active_clusters[k] = -1;
  SPB_CHECK_CUDA(cudaMalloc(&ctx->d_counters, SPB_NUM_COUNTERS * sizeof(unsigned int)));
  SPB_CHECK_CUDA(cudaMemset(ctx->d_counters, 0, SPB_NUM_COUNTERS * sizeof(unsigned int)));
  SPB_CHECK_CUDA(cudaMalloc(&ctx->d_scratch,
                            (size_t)SPB_NUM_COUNTERS * SPB_SCRATCH_PER_SLOT * sizeof(double)));
  if (tables_count > 0) {
    SPB_REQUIRE(tables_host != nullptr, "spb_create: null table blob");
    SPB_CHECK_CUDA(cudaMalloc(&ctx->d_tables, tables_count * sizeof(double)));
    SPB_CHECK_CUDA(cudaMemcpy(ctx->d_tables, tables_host, tables_count * sizeof(double),
                              cudaMemcpyHostToDevice));
    if (tables_count == SPB_TAB_TOTAL) {
      int st = spb_wigner_init(ctx);
      if (st) return st;
    }
  }
  *out = guard.release();
  return 0;
}

extern "C" void spb_destroy(spb_context *ctx) { spb_release(ctx); }

extern "C" int spb_set_option(spb_context *ctx, const char *name, int value) {
  SPB_REQUIRE(ctx != nullptr && name != nullptr, "spb_set_option: null argument");
  const std::string key(name);
  if (key == "moments_syrk_i8") {
    ctx->opt_syrk_i8 = value ? 1 : 0;
    return 0;
  }
  if (key == "cholesky_tma") ctx->opt_no_tma = value ? 0 : 1;
  else if (key == "cholesky_cluster") ctx->opt_no_cluster = value ? 0 : 1;
  else SPB_REQUIRE(false, "spb_set_option: unknown option");
  return 0;
}

extern "C" int spb_device(const spb_context *ctx) { return ctx ? ctx->device : -1; }

extern "C" int spb_launch_count(const spb_context *ctx, long long *count_host) {
  SPB_REQUIRE(ctx != nullptr && count_host != nullptr, "spb_launch_count: null argument");
  *count_host = ctx->launches;
  return 0;
}

// ---------------------------------------------------------------------------------------------
// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time libcuda
// dependency): 3-D fp64 tensor, 128-byte swizzle, used by the TMA store path of the design-matrix
// kernel.  dim0 is the contiguous dimension; strides in bytes for dims 1 and 2.
// ---------------------------------------------------------------------------------------------
typedef CUresult (*spb_encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                  const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// The driver's cuTensorMapEncodeTiled, looked up once (thread-safe).
static int spb_encode_fn_get(spb_encode_fn *out) {
  static spb_encode_fn fn = nullptr;
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  if (!fn) {
    void *ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    SPB_CHECK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres));
    SPB_REQUIRE(ptr != nullptr && qres == cudaDriverEntryPointSuccess,
                "cuTensorMapEncodeTiled is not available in this driver");
    fn = reinterpret_cast<spb_encode_fn>(ptr);
  }
  *out = fn;
  return 0;
}

int spb_encode_tmap_3d_f64(CUtensorMap *out, void *base, unsigned long long d0,
                           unsigned long long d1, unsigned long long d2, unsigned long long s1,
                           unsigned long long s2, unsigned b0, unsigned b1, unsigned b2) {
  spb_encode_fn fn;
  if (const int st = spb_encode_fn_get(&fn)) return st;
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {s1, s2};
  cuuint32_t box[3] = {b0, b1, b2};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, base, dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SPB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (alignment / stride constraints)");
  return 0;
}

// 4-D tensor map of bytes (digit planes of the INT8 Cholesky path), 32-byte swizzle.
int spb_encode_tmap_u8_4d(CUtensorMap *out, void *base, const unsigned long long dims_[4],
                          const unsigned long long strides_[3], const unsigned box_[4]) {
  spb_encode_fn fn;
  if (const int st = spb_encode_fn_get(&fn)) return st;
  cuuint64_t dims[4] = {dims_[0], dims_[1], dims_[2], dims_[3]};
  cuuint64_t strides[3] = {strides_[0], strides_[1], strides_[2]};
  cuuint32_t box[4] = {box_[0], box_[1], box_[2], box_[3]};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, base, dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B,
                  CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SPB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (digit planes)");
  return 0;
}
