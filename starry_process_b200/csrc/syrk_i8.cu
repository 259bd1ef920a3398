// FP64 GEMMs of the path evaluated exactly on the INT8 tensor cores (tcgen05 + TMEM), on the digit planes of
// i8_planes.cuh: the second-moment SYRK of the Ylm moments and the lower triangle of the conditional flux
// covariance (A Sigma) A^T (end of the file).
//
//     cov_ylm[b] = scale_b ( ldeg_b o (X_b X_b^T) - mom1_b mom1_b^T ) + diag(lambda)      (contrast.py:21-33,
//                                                                  size.py:116-125 for the ldeg factor)
//
// with X_b = sqrtC_lon (256 x 31 rk) -- the same product gemm_nt<EPI_SYRK_COV> evaluates on DMMA:
//   1. slice_rows_kernel: every row of X_b is scaled by a power of two taken from its largest entry, rounded to
//      55 bits and cut into 7 balanced 8-bit digits; the kept eigen-columns (the first rk4 of every 32-wide
//      group) are packed contiguously, zero-padded to a multiple of 32 -> planes (B, 7, 256, 1024) int8;
//   2. syrk_i8_kernel: per 128 x 64 tile of the lower triangle, the 7 TMEM blocks combined in fp64, the
//      covariance epilogue applied and the tile and its mirror image stored.
// Both GEMMs run on one pipeline (i8_gemm): persistent, one CTA per SM; one thread streams the plane chunks
// of a tile by 4-D TMA into a 5-stage ring, one thread issues the MMAs, 8 warps read the blocks back and run
// the GEMM's epilogue.
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "i8_planes.cuh"

namespace {

constexpr int SY_S = 7, SY_RB = 8;   // 7 planes of balanced 8-bit digits
constexpr int SY_LDQ = 1024;         // bytes per plane row (31 x 32 = 992 entries at most)

struct SyrkParams {
  const double *X;        // (B, 256, 992)
  const int *rkeep;       // (B)
  uint8_t *Q;             // (B, 7, 256, 1024)
  double *E;              // (B, 256) row scales
  double *C;              // (B, 256, 256)
  const double *scale;    // (B)
  const double *vec;      // (B, 256)
  const double *diag;     // (256)
  const double *ldeg;     // (B, 16, 16) or NULL
  int B;
};

__device__ __forceinline__ int sy_chunks(int rkeep) {   // k-chunks of 32 packed entries
  const int rk4 = (rkeep + 3) & ~3;
  return (31 * rk4 + I8_KCH - 1) / I8_KCH;
}

// ---- 1. digit planes of X ------------------------------------------------------------------------
__global__ void __launch_bounds__(256) slice_rows_kernel(SyrkParams p) {
  const int b = blockIdx.y, row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int rk4 = (p.rkeep[b] + 3) & ~3;
  const int KQ = 31 * rk4 / 4;                       // quads of packed entries (rk4 % 4 == 0)
  const int KPQ = sy_chunks(p.rkeep[b]) * (I8_KCH / 4);   // quads incl. the zero padding
  const double *xr = p.X + ((size_t)b * 256 + row) * 992;
  // pass 1: the largest entry of the row; the kept entries are parked in shared memory (8 KB per warp) so
  // that pass 2 neither re-reads them from DRAM (ncu: the second read missed L2) nor holds them in 64 registers
  extern __shared__ __align__(16) double sy_stage[];
  double *stg = sy_stage + (size_t)(threadIdx.x >> 5) * 992;
  double mx = 0.0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int q = lane + 32 * j;
    if (q < KQ) {
      const int kk = 4 * q, e2 = kk / rk4, e = kk - e2 * rk4;
      const double4 t = *reinterpret_cast<const double4 *>(xr + e2 * 32 + e);
      *reinterpret_cast<double4 *>(stg + 4 * q) = t;
      mx = fmax(mx, fmax(fmax(fabs(t.x), fabs(t.y)), fmax(fabs(t.z), fabs(t.w))));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  // 2^e > 2.02 max: balanced base-256 digits need |x| <= 1/2
  int ex;
  const double E = i8_scale_exp(mx, ex) ? ldexp(1.0, ex + 1) : 1.0;
  if (lane == 0) p.E[(size_t)b * 256 + row] = E;
  const double sinv = ldexp(1.0 / E, SY_RB * SY_S);
  uint8_t *qrow = p.Q + ((size_t)b * SY_S * 256 + row) * SY_LDQ;
  const size_t pstride = (size_t)256 * SY_LDQ;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int q = lane + 32 * j;
    if (q >= KPQ) continue;
    double v4[4] = {0.0, 0.0, 0.0, 0.0};
    if (q < KQ) {
      const double4 t = *reinterpret_cast<const double4 *>(stg + 4 * q);   // this lane's own copy
      v4[0] = t.x; v4[1] = t.y; v4[2] = t.z; v4[3] = t.w;
    }
    uint32_t W[SY_S];
#pragma unroll
    for (int s = 0; s < SY_S; ++s) W[s] = 0u;
#pragma unroll
    for (int c = 0; c < 4; ++c) (void)i8_cut<SY_S, SY_RB>(v4[c] * sinv, 8 * c, W);
#pragma unroll
    for (int s = 0; s < SY_S; ++s)
      *reinterpret_cast<uint32_t *>(qrow + (size_t)s * pstride + 4 * q) = i8_recentre<SY_RB>(s, W[s]);
  }
}

// ---- the pipeline of both GEMMs ----------------------------------------------------------------------
struct SmemGemm {
  static constexpr int STAGES = 5;
  uint8_t A[STAGES][SY_S][I8_TM][I8_KCH];
  uint8_t B[STAGES][SY_S][I8_TN][I8_KCH];
  uint64_t full[STAGES], empty[STAGES], tmem_full, tmem_empty;
  uint32_t tmem_base;
};

// Persistent loop over the work items of a Job, 128 x 64 output tiles:
//   Job::Item                            integer type of the item index
//   nitems()                             number of items
//   tile(item, b, tm, tn, bB)            A rows tm * 128.. of batch b against B rows tn * 64.. of batch bB
//   chunks(item)                         k-chunks of 32 bytes
//   epilogue(item, wrow, lane, tw, wait) one draining warp (tile rows wrow .. wrow + 15, TMEM address tw):
//                                        loads what it needs, calls wait() and then reads TMEM
template <class Job>
__device__ __forceinline__ void i8_gemm(const Job &job, const CUtensorMap &tmA, const CUtensorMap &tmB) {
  using Item = typename Job::Item;
  constexpr int STAGES = SmemGemm::STAGES;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  SmemGemm &sm = *reinterpret_cast<SmemGemm *>(smem_raw);
  const int tid = threadIdx.x, pw = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    i8_ring_init(sm);
    fence_mbarrier_init();
  }
  if (pw == I8_ISSUER_WARP) i8_tmem_alloc(&sm.tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_base;
  const Item nitems = job.nitems();

  if (pw == I8_PRODUCER_WARP) {
    if (lane == 0) {
      unsigned x = 0;
      for (Item item = blockIdx.x; item < nitems; item += gridDim.x) {
        int b, tm, tn, bB;
        job.tile(item, b, tm, tn, bB);
        const int nch = job.chunks(item);
        for (int ch = 0; ch < nch; ++ch, ++x) {
          const unsigned st = x % STAGES;
          if (x >= (unsigned)STAGES) mbar_wait_sleep(&sm.empty[st], ((x / STAGES) + 1u) & 1u, 60);
          mbar_arrive_expect_tx(&sm.full[st], (unsigned)(SY_S * (I8_TM + I8_TN) * I8_KCH));
          tma_load_4d(&sm.A[st][0][0][0], &tmA, &sm.full[st], ch * I8_KCH, tm * I8_TM, 0, b);
          tma_load_4d(&sm.B[st][0][0][0], &tmB, &sm.full[st], ch * I8_KCH, tn * I8_TN, 0, bB);
        }
      }
    }
  } else if (pw == I8_ISSUER_WARP) {
    if (lane == 0) {
      unsigned x = 0, tq = 0;
      for (Item item = blockIdx.x; item < nitems; item += gridDim.x, ++tq) {
        const int nch = job.chunks(item);
        if (tq > 0) mbar_wait_sleep(&sm.tmem_empty, (tq + 1u) & 1u, 60);
        tc_fence_after();
        for (int ch = 0; ch < nch; ++ch, ++x) {
          const unsigned st = x % STAGES;
          mbar_wait_sleep(&sm.full[st], (x / STAGES) & 1u, 40);
          tc_fence_after();
          i8_issue_chunk<SY_S>(tmem, sm.A[st], sm.B[st], ch > 0);
          i8_commit(&sm.empty[st]);
        }
        i8_commit(&sm.tmem_full);
      }
    }
  } else {
    // TMEM lane rule: warp pw reads lanes 32 (pw % 4) + 16 (pw / 4) .. + 15 = its 16 tile rows
    const int wrow = 32 * (pw & 3) + 16 * ((pw >> 2) & 1);
    const uint32_t tw = tmem + ((uint32_t)wrow << 16);
    unsigned tq = 0;
    for (Item item = blockIdx.x; item < nitems; item += gridDim.x, ++tq) {
      job.epilogue(item, wrow, lane, tw, [&] {
        mbar_wait_sleep(&sm.tmem_full, tq & 1u, 40);
        tc_fence_after();
      });
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&sm.tmem_empty);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (pw == I8_ISSUER_WARP) i8_tmem_dealloc(tmem);
}

// ---- 2. the SYRK ------------------------------------------------------------------------------------
struct SyrkJob {
  using Item = int;
  SyrkParams p;
  __device__ __forceinline__ Item nitems() const { return 6 * p.B; }
  // lower-triangle tiles of the 256 x 256 output: (row block of 128, column block of 64), 6 per sample
  __device__ __forceinline__ void tile(Item item, int &b, int &tm, int &tn, int &bB) const {
    b = item / 6;
    const int t = item - 6 * b;
    tm = (t < 2) ? 0 : 1;
    tn = (t < 2) ? t : t - 2;
    bB = b;
  }
  __device__ __forceinline__ int chunks(Item item) const { return sy_chunks(p.rkeep[item / 6]); }
  template <class Wait>
  __device__ __forceinline__ void epilogue(Item item, int wrow, int lane, uint32_t tw, Wait wait) const {
    const int g = lane >> 2, tg = lane & 3;
    int b, tm, tn, bB;
    tile(item, b, tm, tn, bB);
    const int nch = chunks(item);
    const int m0 = tm * I8_TM + wrow, n0 = tn * I8_TN;
    const double *Eb = p.E + (size_t)b * 256;
    const double *vb = p.vec + (size_t)b * 256;
    const double sc = p.scale[b];
    double *Cb = p.C + (size_t)b * 65536;
    double em[2], vm[2];
    int lm[2];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const int m = m0 + mt * 8 + g;
      em[mt] = ldexp(Eb[m], -2 * SY_RB);
      vm[mt] = vb[m];
      lm[mt] = (int)sqrt((double)m);
    }
    wait();
#pragma unroll
    for (int cq = 0; cq < 4; ++cq) {
      uint32_t v[SY_S][8];
      i8_tmem_ld<SY_S>(tw, 16 * cq, v);
#pragma unroll
      for (int bl = 0; bl < 2; ++bl) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int n = n0 + 16 * cq + 8 * bl + 2 * tg + e;
          const double en = Eb[n], vn = vb[n];
          const int ln = p.ldeg ? (int)sqrt((double)n) : 0;
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) {
            const int m = m0 + mt * 8 + g;
            if (n > m) continue;
            const double t = (nch > 0) ? i8_horner<SY_S, SY_RB>(v, 4 * bl + 2 * mt + e) : 0.0;
            double val = em[mt] * en * t;
            if (p.ldeg) val *= p.ldeg[(size_t)b * 256 + lm[mt] * 16 + ln];
            val = sc * (val - vm[mt] * vn);
            if (m == n) val += p.diag[m];
            Cb[(size_t)m * 256 + n] = val;
            Cb[(size_t)n * 256 + m] = val;
          }
        }
      }
    }
  }
};

__global__ void __launch_bounds__(I8_NTHREADS, 1)
    syrk_i8_kernel(SyrkParams p, const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB) {
  i8_gemm(SyrkJob{p}, tmA, tmB);
}


// =====================================================================================================
// Lower triangle of  C[b] = T[b] A[b]^T  with 256-wide rows (the conditional flux covariance
// K = (A Sigma) A^T of flux.py:335-343 for long light curves): planes of the rows of T (per sample) and of
// A (shared or per sample), K = 256 = 8 chunks per 128 x 64 tile.
// =====================================================================================================
struct GemmLParams {
  const uint8_t *QT, *QA;   // planes (B, 7, nt, 256), (nA, 7, nt, 256)
  const double *ET, *EA;    // row scales (B, nt), (nA, nt)
  double *C;                // (B, nt, ldc)
  long long strideC;
  int ldc, B, nt, nA, tilesM, tilesN, ntile;
};

// digit planes of `rows` rows of 256 doubles: src (nb, rows, 256) -> Q (nb, 7, rows, 256), E (nb, rows)
//   * a row holding an inf or a NaN, or whose maximum is 1e300 or more (2^e would not fit), gets E = NaN:
//     every product touching it comes out NaN, as on the FP64 GEMM, instead of a finite value from
//     digits that cannot represent it;
//   * E >= 2^-1058, so that the epilogue's E 2^-16 does not underflow for rows of subnormals; such rows
//     are scaled by 2^200 before the cut (x 2^56 / E alone would overflow below 2^-967), exactly.
__global__ void __launch_bounds__(256) slice256_kernel(const double *src, long long stride_b, int rows, uint8_t *Q,
                                                       double *E) {
  const int b = blockIdx.y, row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const double *xr = src + (size_t)b * stride_b + (size_t)row * 256;
  double v[2][4];
  double mx = 0.0, nf = 0.0;   // nf: x - x summed over the entries, NaN iff one is inf or NaN
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const double4 t = *reinterpret_cast<const double4 *>(xr + 4 * (lane + 32 * j));
    v[j][0] = t.x; v[j][1] = t.y; v[j][2] = t.z; v[j][3] = t.w;
    mx = fmax(mx, fmax(fmax(fabs(t.x), fabs(t.y)), fmax(fabs(t.z), fabs(t.w))));
    nf += ((t.x - t.x) + (t.y - t.y)) + ((t.z - t.z) + (t.w - t.w));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  const bool bad = __any_sync(0xffffffffu, nf != 0.0) || mx >= 1e300;
  int ex;
  double Ev = i8_scale_exp(mx, ex) ? ldexp(1.0, ex + 1 > -1058 ? ex + 1 : -1058) : 1.0;
  if (bad) Ev = __longlong_as_double(0x7ff8000000000000ll);
  if (lane == 0) E[(size_t)b * rows + row] = Ev;
  const double pre = (Ev < 0x1p-900) ? 0x1p+200 : 1.0;
  const double sinv = ldexp(1.0 / (Ev * pre), SY_RB * SY_S);
  uint8_t *qrow = Q + ((size_t)b * SY_S * rows + row) * 256;
  const size_t pstride = (size_t)rows * 256;
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    uint32_t W[SY_S];
#pragma unroll
    for (int s = 0; s < SY_S; ++s) W[s] = 0u;
#pragma unroll
    for (int c = 0; c < 4; ++c) (void)i8_cut<SY_S, SY_RB>(v[j][c] * pre * sinv, 8 * c, W);
#pragma unroll
    for (int s = 0; s < SY_S; ++s)
      *reinterpret_cast<uint32_t *>(qrow + (size_t)s * pstride + 4 * (lane + 32 * j)) = i8_recentre<SY_RB>(s, W[s]);
  }
}

struct GemmLowerJob {
  using Item = long long;
  GemmLParams p;
  __device__ __forceinline__ Item nitems() const { return (long long)p.ntile * p.B; }
  // tile r of a sample (row-block-major over the lower triangle): row block tm has min(2 tm + 2, tilesN) tiles
  __device__ __forceinline__ void tile(Item item, int &b, int &tm, int &tn, int &bB) const {
    b = (int)(item / p.ntile);
    const int r = (int)(item - (long long)b * p.ntile);
    tm = (int)((sqrt(4.0 * (double)r + 1.0) - 1.0) * 0.5);
    while (tm * (tm + 1) > r) --tm;
    while ((tm + 1) * (tm + 2) <= r) ++tm;
    tn = r - tm * (tm + 1);
    bB = (p.nA == 1) ? 0 : b;
  }
  __device__ __forceinline__ int chunks(Item) const { return 256 / I8_KCH; }
  template <class Wait>
  __device__ __forceinline__ void epilogue(Item item, int wrow, int lane, uint32_t tw, Wait wait) const {
    const int g = lane >> 2, tg = lane & 3;
    int b, tm, tn, ba;
    tile(item, b, tm, tn, ba);
    const int m0 = tm * I8_TM + wrow, n0 = tn * I8_TN;
    const double *Et = p.ET + (size_t)b * p.nt;
    const double *Ea = p.EA + (size_t)ba * p.nt;
    double *Cb = p.C + (size_t)b * p.strideC;
    double em[2];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const int m = m0 + mt * 8 + g;
      em[mt] = (m < p.nt) ? ldexp(Et[m], -2 * SY_RB) : 0.0;
    }
    wait();
#pragma unroll
    for (int cq = 0; cq < 4; ++cq) {
      uint32_t v[SY_S][8];
      i8_tmem_ld<SY_S>(tw, 16 * cq, v);
#pragma unroll
      for (int bl = 0; bl < 2; ++bl) {
        const int n = n0 + 16 * cq + 8 * bl + 2 * tg;
        if (n >= p.nt) continue;
        const double en0 = Ea[n], en1 = (n + 1 < p.nt) ? Ea[n + 1] : 0.0;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          const int m = m0 + mt * 8 + g;
          if (m >= p.nt) continue;
          // both columns in one loop (not two i8_horner calls: that order changes this kernel's schedule)
          double t0 = (double)(int)v[SY_S - 1][4 * bl + 2 * mt], t1 = (double)(int)v[SY_S - 1][4 * bl + 2 * mt + 1];
#pragma unroll
          for (int d = SY_S - 2; d >= 0; --d) {
            t0 = fma(t0, 0.00390625, (double)(int)v[d][4 * bl + 2 * mt]);
            t1 = fma(t1, 0.00390625, (double)(int)v[d][4 * bl + 2 * mt + 1]);
          }
          double *c = Cb + (size_t)m * p.ldc + n;
          if (n + 1 < p.nt) *reinterpret_cast<double2 *>(c) = make_double2(em[mt] * en0 * t0, em[mt] * en1 * t1);
          else *c = em[mt] * en0 * t0;
        }
      }
    }
  }
};

__global__ void __launch_bounds__(I8_NTHREADS, 1)
    gemm_i8_lower_kernel(GemmLParams p, const __grid_constant__ CUtensorMap tmT, const __grid_constant__ CUtensorMap tmA) {
  i8_gemm(GemmLowerJob{p}, tmT, tmA);
}

}  // namespace

size_t spb_syrk_i8_workspace_bytes(int Bc) {
  return (size_t)Bc * SY_S * 256 * SY_LDQ + (size_t)Bc * 256 * sizeof(double) + 512;
}

// cov[b] = scale[b] (ldeg[b] o (X[b] X[b]^T) - vec[b] vec[b]^T) + diag  for b < Bc  (see the file header)
int spb_syrk_i8(spb_context *ctx, int Bc, const double *X, const int *rkeep, const double *scale,
                const double *vec, const double *diag, const double *ldeg, double *C, void *workspace,
                cudaStream_t stream) {
  SyrkParams p;
  p.X = X;
  p.rkeep = rkeep;
  uintptr_t w = ((uintptr_t)workspace + 255) & ~(uintptr_t)255;
  p.Q = reinterpret_cast<uint8_t *>(w);
  p.E = reinterpret_cast<double *>(w + (size_t)Bc * SY_S * 256 * SY_LDQ);
  p.C = C;
  p.scale = scale;
  p.vec = vec;
  p.diag = diag;
  p.ldeg = ldeg;
  p.B = Bc;
  CUtensorMap tmA, tmB;
  memset(&tmA, 0, sizeof(tmA));
  memset(&tmB, 0, sizeof(tmB));
  {
    const unsigned long long dims[4] = {SY_LDQ, 256, SY_S, (unsigned long long)Bc};
    const unsigned long long strides[3] = {SY_LDQ, 256ull * SY_LDQ, (unsigned long long)SY_S * 256 * SY_LDQ};
    const unsigned boxA[4] = {I8_KCH, I8_TM, SY_S, 1};
    const unsigned boxB[4] = {I8_KCH, I8_TN, SY_S, 1};
    int st = spb_encode_tmap_u8_4d(&tmA, p.Q, dims, strides, boxA);
    if (st) return st;
    st = spb_encode_tmap_u8_4d(&tmB, p.Q, dims, strides, boxB);
    if (st) return st;
  }
  static spb_once_flag attr_once;
  {
    const int st = spb_once_per_device(attr_once, ctx->device, [&]() -> int {
      SPB_CHECK_CUDA(cudaFuncSetAttribute(syrk_i8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)sizeof(SmemGemm)));
      SPB_CHECK_CUDA(cudaFuncSetAttribute(slice_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)(8 * 992 * sizeof(double))));
      return 0;
    });
    if (st) return st;
  }
  dim3 gs(32, Bc);
  slice_rows_kernel<<<gs, 256, 8 * 992 * sizeof(double), stream>>>(p);
  SPB_LAUNCH_CHECK(ctx);
  const int grid = 6 * Bc < ctx->num_sms ? 6 * Bc : ctx->num_sms;
  syrk_i8_kernel<<<grid, I8_NTHREADS, sizeof(SmemGemm), stream>>>(p, tmA, tmB);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

// ---- lower triangle of C[b] = T[b] A[b]^T (256-wide rows) on the INT8 tensor cores ------------------------
size_t spb_gemm_i8_lower_workspace_bytes(int Bc, int nt) {
  // digit planes + scales of T (Bc samples) and of A (up to Bc operands)
  return 2 * ((size_t)Bc * SY_S * nt * 256 + (size_t)Bc * nt * sizeof(double)) + 1024;
}

int spb_gemm_i8_lower(spb_context *ctx, int Bc, int nt, const double *T, const double *A, long long A_stride,
                      double *C, int ldc, void *workspace, cudaStream_t stream) {
  const int nA = (A_stride == 0) ? 1 : Bc;
  uintptr_t w = ((uintptr_t)workspace + 255) & ~(uintptr_t)255;
  uint8_t *QT = reinterpret_cast<uint8_t *>(w);
  w += (size_t)Bc * SY_S * nt * 256;
  uint8_t *QA = reinterpret_cast<uint8_t *>(w);
  w += (size_t)nA * SY_S * nt * 256;
  w = (w + 255) & ~(uintptr_t)255;
  double *ET = reinterpret_cast<double *>(w);
  double *EA = ET + (size_t)Bc * nt;
  dim3 gT((nt + 7) / 8, Bc), gA((nt + 7) / 8, nA);
  slice256_kernel<<<gT, 256, 0, stream>>>(T, (long long)nt * 256, nt, QT, ET);
  SPB_LAUNCH_CHECK(ctx);
  slice256_kernel<<<gA, 256, 0, stream>>>(A, A_stride, nt, QA, EA);
  SPB_LAUNCH_CHECK(ctx);
  GemmLParams p;
  p.QT = QT;
  p.QA = QA;
  p.ET = ET;
  p.EA = EA;
  p.C = C;
  p.strideC = (long long)nt * ldc;
  p.ldc = ldc;
  p.B = Bc;
  p.nt = nt;
  p.nA = nA;
  p.tilesM = (nt + I8_TM - 1) / I8_TM;
  p.tilesN = (nt + I8_TN - 1) / I8_TN;
  // every row block keeps its 2 tm + 2 column blocks (the last ones may lie wholly beyond nt: their loads are
  // zero-filled by TMA and their stores masked)
  p.ntile = p.tilesM * (p.tilesM + 1);
  CUtensorMap tmT, tmA;
  memset(&tmT, 0, sizeof(tmT));
  memset(&tmA, 0, sizeof(tmA));
  {
    const unsigned long long dT[4] = {256, (unsigned long long)nt, SY_S, (unsigned long long)Bc};
    const unsigned long long dA[4] = {256, (unsigned long long)nt, SY_S, (unsigned long long)nA};
    const unsigned long long st[3] = {256, 256ull * nt, (unsigned long long)SY_S * 256 * nt};
    const unsigned boxA[4] = {I8_KCH, I8_TM, SY_S, 1};
    const unsigned boxB[4] = {I8_KCH, I8_TN, SY_S, 1};
    int e = spb_encode_tmap_u8_4d(&tmT, QT, dT, st, boxA);
    if (e) return e;
    e = spb_encode_tmap_u8_4d(&tmA, QA, dA, st, boxB);
    if (e) return e;
  }
  static spb_once_flag attr_once;
  {
    const int e = spb_once_per_device(attr_once, ctx->device, [&]() -> int {
      SPB_CHECK_CUDA(cudaFuncSetAttribute(gemm_i8_lower_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)sizeof(SmemGemm)));
      return 0;
    });
    if (e) return e;
  }
  gemm_i8_lower_kernel<<<ctx->num_sms, I8_NTHREADS, sizeof(SmemGemm), stream>>>(p, tmT, tmA);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}
