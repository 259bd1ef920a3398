// Shared device/host helpers for libspb200 (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <mutex>
#include <string>

#include "../../include/spb200.h"

#define SPB_LMAX 15
// Ring of per-launch work counters / scratch slots.  A slot is reused after SPB_NUM_COUNTERS further
// launches through the same context; a CUDA device cannot hold that many launches in flight (the
// launch queues block the host long before), so two running kernels never share a slot.
#define SPB_NUM_COUNTERS 4096
#define SPB_SCRATCH_PER_SLOT 256  // doubles per launch slot (cluster Cholesky: one per CTA)
#define SPB_NSM_DEFAULT 148

struct spb_context {
  int device;
  int num_sms;
  double *d_tables;       // device copy of the packed constant blob
  size_t tables_count;
  std::atomic<long long> launches;   // number of kernels launched through this context
  // run-time switches (spb_set_option): A/B measurements and the bit-for-bit stress tests
  int opt_no_tma;         // Cholesky operand ring: cp.async instead of TMA
  int opt_no_cluster;     // Cholesky: never use the one-matrix-per-cluster kernel
  int opt_syrk_i8;        // second-moment SYRK of the Ylm moments on the INT8 tensor cores (syrk_i8.cu)
  int max_active_clusters[3];   // cudaOccupancyMaxActiveClusters for cluster sizes 8, 4, 2 (-1: unknown)
  // ring of work counters for kernels that claim their work items dynamically (one per launch,
  // zeroed in-stream before the launch, so that concurrent streams never share one)
  unsigned int *d_counters;
  unsigned int counter_next;
  double *d_scratch;      // SPB_NUM_COUNTERS x SPB_SCRATCH_PER_SLOT doubles, same ring
  // offsets (in doubles) into d_tables, see spb_tables.h
  const double *tab(size_t off) const { return d_tables + off; }
};

void spb_set_error(const std::string &msg);

// One-time per-device initialisation (function attributes, __constant__ uploads) that is safe
// against concurrent callers: the header promises re-entrancy across streams and devices.
struct spb_once_flag {
  std::mutex mu;
  bool done[64] = {};
};
template <class F>
inline int spb_once_per_device(spb_once_flag &f, int device, F &&fn) {
  std::lock_guard<std::mutex> lock(f.mu);
  if (f.done[device & 63]) return 0;
  const int st = fn();
  if (st == 0) f.done[device & 63] = true;
  return st;
}
int spb_encode_tmap_3d_f64(CUtensorMap *out, void *base, unsigned long long d0,
                           unsigned long long d1, unsigned long long d2, unsigned long long s1,
                           unsigned long long s2, unsigned b0, unsigned b1, unsigned b2);
int spb_encode_tmap_u8_4d(CUtensorMap *out, void *base, const unsigned long long dims[4],
                          const unsigned long long strides[3], const unsigned box[4]);

// syrk_i8.cu: cov[b] = scale[b] (ldeg[b] o (X[b] X[b]^T) - vec[b] vec[b]^T) + diag on the INT8 tensor cores
size_t spb_syrk_i8_workspace_bytes(int Bc);
size_t spb_gemm_i8_lower_workspace_bytes(int Bc, int nt);
int spb_gemm_i8_lower(spb_context *ctx, int Bc, int nt, const double *T, const double *A, long long A_stride,
                      double *C, int ldc, void *workspace, cudaStream_t stream);
int spb_syrk_i8(spb_context *ctx, int Bc, const double *X, const int *rkeep, const double *scale,
                const double *vec, const double *diag, const double *ldeg, double *C, void *workspace,
                cudaStream_t stream);

#define SPB_CHECK_CUDA(expr)                                                          \
  do {                                                                                \
    cudaError_t _e = (expr);                                                          \
    if (_e != cudaSuccess) {                                                          \
      spb_set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));              \
      return 1;                                                                       \
    }                                                                                 \
  } while (0)

#define SPB_REQUIRE(cond, msg)                                                        \
  do {                                                                                \
    if (!(cond)) {                                                                    \
      spb_set_error(std::string("spb200: ") + msg);                                   \
      return 2;                                                                       \
    }                                                                                 \
  } while (0)

#define SPB_LAUNCH_CHECK(ctx)                                                         \
  do {                                                                                \
    (ctx)->launches += 1;                                                             \
    cudaError_t _e = cudaGetLastError();                                              \
    if (_e != cudaSuccess) {                                                          \
      spb_set_error(std::string("kernel launch: ") + cudaGetErrorString(_e));         \
      return 1;                                                                       \
    }                                                                                 \
  } while (0)

// ---- FP64 tensor-core MMA (DMMA): D(8x8) += A(8x4, row) * B(4x8, col) ------------------------
// fragment layout (PTX ISA, mma.m8n8k4 .f64): g = lane>>2, tg = lane&3
//   a = A[g][tg]      b = B[tg][g]      d0,d1 = D[g][2*tg + {0,1}]
__device__ __forceinline__ void dmma_m8n8k4(double &d0, double &d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

// ---- cp.async (LDGSTS) 16-byte copy with zero-fill when src_bytes == 0 ------------------------
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc, int src_bytes) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gsrc),
               "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

// ---- mbarrier (shared::cta) helpers: asynchronous producer/consumer hand-off without CTA-wide
// rendezvous.  cp.async completions of the executing thread arrive on the barrier (noinc: the
// expected count is fixed at init time). ------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
  unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(a), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.shared::cta.b64 st, [%0];\n}\n" ::"r"(a) : "memory");
}
__device__ __forceinline__ void mbar_cp_async_arrive(uint64_t *bar) {
  unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];\n" ::"r"(a) : "memory");
}
__device__ __forceinline__ bool mbar_test(uint64_t *bar, unsigned parity) {  // non-blocking
  unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  unsigned ok;
  asm volatile(
      "{\n.reg .pred p;\nmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n}\n"
      : "=r"(ok)
      : "r"(a), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
  unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile(
      "{\n.reg .pred p;\nLAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra LAB_DONE;\nbra LAB_WAIT;\nLAB_DONE:\n}\n" ::"r"(a),
      "r"(parity)
      : "memory");
}

// ---- TMA tensor load global -> shared (3-D tensor map), completion on an mbarrier ---------------
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, unsigned bytes) {
  unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n}\n" ::"r"(a),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_load_3d(void *sdst, const void *tmap, uint64_t *bar, int c0,
                                            int c1, int c2) {
  unsigned s = (unsigned)__cvta_generic_to_shared(sdst);
  unsigned b = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n" ::"r"(s),
      "l"(tmap), "r"(b), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// Orders this thread's earlier generic-proxy writes to GLOBAL memory (st.global) before later
// async-proxy accesses (TMA loads of the same addresses) -- a __threadfence() does not.
__device__ __forceinline__ void fence_proxy_async_global() {
  asm volatile("fence.proxy.async.global;\n" ::: "memory");
}

// ---- TMA tensor store shared::cta -> global (cp.async.bulk.tensor, 3-D tensor map) ------------
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
}
__device__ __forceinline__ void tma_store_3d(const void *tmap, const void *ssrc, int c0, int c1,
                                             int c2) {
  unsigned s = (unsigned)__cvta_generic_to_shared(ssrc);
  asm volatile(
      "cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];\n" ::"l"(tmap),
      "r"(c0), "r"(c1), "r"(c2), "r"(s)
      : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;\n" ::"n"(N) : "memory");
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- phase basis of the light curve: every kernel that evaluates a function of the phase ---------
// theta = 2 pi mod(t / p, 1) (flux.py:261); *wraps, if given, receives floor(t / p).
__device__ __forceinline__ double spb_phase(double t, double period, double *wraps = nullptr) {
  const double x = t / period;
  const double w = floor(x);
  if (wraps) *wraps = w;
  return 2.0 * 3.14159265358979323846 * (x - w);
}

// cs[m] = cos(m theta), sn[m] = sin(m theta) for m <= SPB_LMAX by the Chebyshev recurrences of wigner.h:311-316.
// The design matrix (wigner.cu, -fmad=false) and the rank-31 basis Phi(t) (lowrank.cu, -fmad=true) must round
// identically, since Phi B_inc is exactly the design matrix: the product is rounded on its own (__dmul_rn), so
// no translation unit can fuse it into the subtraction; the doubling is exact.
__device__ __forceinline__ void spb_harmonics(double theta, double *cs, double *sn) {
  cs[0] = 1.0;
  sn[0] = 0.0;
  cs[1] = cos(theta);
  sn[1] = sin(theta);
#pragma unroll
  for (int k = 2; k <= SPB_LMAX; ++k) {
    cs[k] = __dmul_rn(2.0 * cs[k - 1], cs[1]) - cs[k - 2];
    sn[k] = __dmul_rn(2.0 * sn[k - 1], cs[1]) - sn[k - 2];
  }
}

// ---- normalisation series of the flux covariance (norm.py:26-44, sp.py:700-727) -------------------
// From m, the mean of the raw covariance Sig, the normalised covariance is
// s[0] Sig + s[1] (1 - q)(1 - q)^T - s[2] q q^T; *z (if given) receives z.  z depends on t, i, p and u, so
// the SPB_INFO_Z_RANGE bit of *info (if given) is re-evaluated on every call, as the reference does
// (sp.py:1178-1183): it is WRITTEN, not OR-ed into the process' persistent flags.
__device__ __forceinline__ void spb_norm_series(double m, double gp_mean, int order, double zmax, double *s,
                                                double *z_out, int32_t *info) {
  const double mu = 1.0 + gp_mean;  // sp.py:700-701
  const double z = m / (mu * mu);
  double fac = 1.0, alpha = 0.0, beta = 0.0;
  for (int n = 0; n <= order; ++n) {
    alpha += fac;
    beta += 2 * n * fac;
    fac *= z * (2 * n + 3);
  }
  s[0] = alpha / (mu * mu);
  s[1] = z * (alpha + beta);
  s[2] = z * alpha;
  if (z_out) *z_out = z;
  if (info) *info = (*info & ~SPB_INFO_Z_RANGE) | ((z > zmax) ? SPB_INFO_Z_RANGE : 0);
}
