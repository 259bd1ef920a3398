// Generic batched FP64 tensor-core "NT" GEMM used by several stages of the lnlike path:
//
//     C[b][m][n] = epilogue( sum_k A[b][m][k] * Bm[b][n][k] )
//
// Both operands are read with k contiguous (row-major A (M x K) and row-major Bm (N x K)), which
// is the natural layout of every contraction on this path:
//   * mom2 = sqrtC sqrtC^T                 (contrast.py:21)            A = Bm = sqrtC_lon
//   * T = A_design cov_ylm ; K = T A_design^T   (flux.py:343)          cov_ylm symmetric
//   * a_m = <Omega_m, cov_ylm>             (flux.py:317, wigner.h:410-459 re-associated)
//   * y = u L^T + mean                     (sp.py:505-509)
// CTA tile 128 x 64, 8 warps each owning 16 full rows x 64 columns in DMMA accumulators
// (mma.sync.m8n8k4.f64), operands staged through a 3-stage cp.async shared-memory pipeline with a
// 20-double row stride (conflict-free 8x4 fragment loads).  2 CTAs/SM.
#pragma once
#include "common.cuh"

namespace gnt {

constexpr int TM = 128, TN = 64, KC = 16, KS = KC + 4, STAGES = 3, NTHREADS = 256;

enum Epilogue { EPI_STORE = 0, EPI_SYRK_COV = 1, EPI_MIRROR = 2, EPI_ADD_ROWVEC = 3, EPI_AXPBY = 4 };

struct Desc {
  const double *A;
  long long strideA;
  int lda;
  const double *Bm;
  long long strideB;
  int ldb;
  double *C;
  long long strideC;
  int ldc;
  int M, N, K, batch;
  int ksplit;              // >1: partial sums are written to C + split*strideSplit
  long long strideSplit;
  int lower_only;          // schedule only tiles that touch the lower triangle (M == N)
  // EPI_SYRK_COV: C = scale[b]*(acc - v[b][m] v[b][n]) + (m==n) diag[m], mirrored
  const double *scale;     // (batch)
  const double *vec;       // (batch, M)  (EPI_ADD_ROWVEC: added along n, (batch, N))
  long long strideVec;
  const double *diag;      // (M)
  const int *rkeep;        // optional (batch): sqrtC chunk-skip rule, see k-loop
  const double *ldeg;      // optional (batch, 16, 16): acc is multiplied by ldeg[b][l(m)][l(n)] first
                           // (spot-size second moment of the uniform-dr prior, moments.cu)
  double alpha;
  double beta;             // EPI_AXPBY: C = alpha acc + beta C (C is not read when beta == 0)
};

struct Smem {
  double As[STAGES][TM][KS];
  double Bs[STAGES][TN][KS];
};

template <int EPI>
__global__ void __launch_bounds__(NTHREADS, 2) gemm_nt_kernel(Desc d) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem &sm = *reinterpret_cast<Smem *>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, tg = lane & 3;

  const int tilesM = (d.M + TM - 1) / TM, tilesN = (d.N + TN - 1) / TN;
  int idx = blockIdx.x;
  const int split = idx % d.ksplit;
  idx /= d.ksplit;
  const int tn = idx % tilesN, tm = idx / tilesN;
  const int b = blockIdx.y;
  if (tm >= tilesM) return;
  const int m0 = tm * TM, n0 = tn * TN;
  if (d.lower_only && n0 > m0 + TM - 1) return;

  const double *Ab = d.A + (size_t)b * d.strideA;
  const double *Bb = d.Bm + (size_t)b * d.strideB;

  // k-range of this split, in chunks of KC
  int nch_total = (d.K + KC - 1) / KC;
  int kstep = KC;          // distance between consecutive chunk starts
  int rk4 = 32;            // kept eigen-columns of this batch element, rounded up to 4
  if (d.rkeep) {
    // sqrtC_lon rows are laid out [e2 (31)][e (32)] and only the first rk4 e-columns of every
    // 32-wide group exist: with rk4 <= 16 every second 16-wide chunk is skipped altogether, and
    // otherwise the second chunk of each pair is only (rk4 - 16) wide -- its copies and its
    // DMMA steps are trimmed accordingly (the kernel is L2-bandwidth-bound on these operands).
    rk4 = (d.rkeep[b] + 3) & ~3;
    if (rk4 <= 16) {
      nch_total = d.K / 32;
      kstep = 32;
    }
  }
  const int per = (nch_total + d.ksplit - 1) / d.ksplit;
  const int ch_begin = split * per;
  const int ch_end = min(nch_total, ch_begin + per);

  double acc[2][8][2];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;

  const int seg = tid & 7;
  const double *arow[4];
  bool aok[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = m0 + (tid >> 3) + 32 * i;
    aok[i] = r < d.M;
    arow[i] = Ab + (size_t)(aok[i] ? r : 0) * d.lda;
  }
  const double *brow[2];
  bool bok[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int r = n0 + (tid >> 3) + 32 * i;
    bok[i] = r < d.N;
    brow[i] = Bb + (size_t)(bok[i] ? r : 0) * d.ldb;
  }
  // live width of chunk ch (multiple of 4, <= 16)
  auto chunk_width = [&](int ch) -> int {
    if (!d.rkeep) return KC;
    const int base = (kstep == 32) ? 0 : 16 * (ch & 1);
    const int wdt = rk4 - base;
    return wdt > 16 ? 16 : wdt;
  };
  auto load_chunk = [&](int ch, int st) {
    const int k = ch * kstep + seg * 2;
    const bool kok = (k < d.K) && (seg * 2 < chunk_width(ch));
    const int kk = kok ? k : 0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      cp_async16(&sm.As[st][(tid >> 3) + 32 * i][seg * 2], arow[i] + kk, (aok[i] && kok) ? 16 : 0);
#pragma unroll
    for (int i = 0; i < 2; ++i)
      cp_async16(&sm.Bs[st][(tid >> 3) + 32 * i][seg * 2], brow[i] + kk, (bok[i] && kok) ? 16 : 0);
  };

  // lower_only: this warp's 16 rows only need the 8-column groups that reach the diagonal
  // (columns n0 + 8 nt <= last row); groups strictly above it are neither multiplied nor stored.
  int nt_lim = 8;
  if (d.lower_only) {
    const int last_row = m0 + warp * 16 + 15;
    nt_lim = (last_row - n0) / 8 + 1;       // may be <= 0: the whole warp tile is above the diagonal
    nt_lim = nt_lim < 0 ? 0 : (nt_lim > 8 ? 8 : nt_lim);
  }
  // narrow outputs (N = 31 quadratic forms of the marginal kernel, N = 1 matrix-vector products of
  // predict): 8-column groups beyond N are neither loaded nor multiplied
  {
    const int nt_n = (d.N - n0 + 7) / 8;
    if (nt_n < nt_lim) nt_lim = nt_n;
  }
  const int nch = ch_end - ch_begin;
  // prologue: STAGES-1 chunks in flight (empty commit groups keep the accounting uniform)
#pragma unroll
  for (int s = 0; s < STAGES - 1; ++s) {
    if (s < nch) load_chunk(ch_begin + s, s);
    cp_async_commit();
  }
  for (int c = 0; c < nch; ++c) {
    const int st = c % STAGES;
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    if (c + STAGES - 1 < nch) load_chunk(ch_begin + c + STAGES - 1, (c + STAGES - 1) % STAGES);
    cp_async_commit();
    const int kk_lim = chunk_width(ch_begin + c) >> 2;
    if (nt_lim == 8) {
#pragma unroll
      for (int kk = 0; kk < KC / 4; ++kk) {
        if (kk >= kk_lim) break;
        double a[2], bf[8];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) a[mt] = sm.As[st][warp * 16 + mt * 8 + g][kk * 4 + tg];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) bf[nt] = sm.Bs[st][nt * 8 + g][kk * 4 + tg];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
          for (int nt = 0; nt < 8; ++nt) dmma_m8n8k4(acc[mt][nt][0], acc[mt][nt][1], a[mt], bf[nt]);
      }
    } else if (nt_lim > 0) {
#pragma unroll
      for (int kk = 0; kk < KC / 4; ++kk) {
        if (kk >= kk_lim) break;
        double a[2];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) a[mt] = sm.As[st][warp * 16 + mt * 8 + g][kk * 4 + tg];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          if (nt < nt_lim) {
            const double bfv = sm.Bs[st][nt * 8 + g][kk * 4 + tg];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) dmma_m8n8k4(acc[mt][nt][0], acc[mt][nt][1], a[mt], bfv);
          }
        }
      }
    }
  }

  // ---- epilogue
  double *Cb = d.C + (size_t)b * d.strideC + (size_t)split * d.strideSplit;
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
    const int m = m0 + warp * 16 + mt * 8 + g;
    if (m >= d.M) continue;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int n = n0 + nt * 8 + 2 * tg + e;
        if (n >= d.N) continue;
        double v = acc[mt][nt][e];
        if (EPI == EPI_STORE) {
          // lower_only: the strict upper triangle of a diagonal tile stays untouched
          if (!d.lower_only || n <= m) Cb[(size_t)m * d.ldc + n] = d.alpha * v;
        } else if (EPI == EPI_AXPBY) {
          double *c = Cb + (size_t)m * d.ldc + n;
          *c = (d.beta == 0.0) ? d.alpha * v : fma(d.alpha, v, d.beta * *c);
        } else if (EPI == EPI_ADD_ROWVEC) {
          Cb[(size_t)m * d.ldc + n] = v + d.vec[(size_t)b * d.strideVec + n];
        } else if (EPI == EPI_MIRROR) {
          if (n <= m) {
            Cb[(size_t)m * d.ldc + n] = v;
            Cb[(size_t)n * d.ldc + m] = v;
          }
        } else {  // EPI_SYRK_COV
          if (n <= m) {
            const double *vb = d.vec + (size_t)b * d.strideVec;
            if (d.ldeg) {
              // degree of a Ylm index: l = floor(sqrt(n)), exact for n < 2^52
              const int lm_ = (int)sqrt((double)m), ln_ = (int)sqrt((double)n);
              v *= d.ldeg[(size_t)b * 256 + lm_ * 16 + ln_];
            }
            v = d.scale[b] * (v - vb[m] * vb[n]);
            if (m == n) v += d.diag[m];
            Cb[(size_t)m * d.ldc + n] = v;
            Cb[(size_t)n * d.ldc + m] = v;
          }
        }
      }
    }
  }
}

template <int EPI>
inline int launch(spb_context *ctx, const Desc &d, cudaStream_t stream) {
  SPB_REQUIRE(d.M > 0 && d.N > 0 && d.K > 0 && d.batch > 0, "gemm_nt: empty problem");
  SPB_REQUIRE((d.lda % 2) == 0 && (d.ldb % 2) == 0 && (d.K % 2) == 0,
              "gemm_nt: K and the operand leading dimensions must be even");
  SPB_REQUIRE(d.lda >= d.K && d.ldb >= d.K && d.ldc >= d.N,
              "gemm_nt: leading dimensions must be lda >= K, ldb >= K and ldc >= N");
  SPB_REQUIRE(((uintptr_t)d.A % 16) == 0 && ((uintptr_t)d.Bm % 16) == 0 &&
                  (d.strideA % 2) == 0 && (d.strideB % 2) == 0,
              "gemm_nt: operands must be 16-byte aligned");
  SPB_REQUIRE(d.batch <= 65535, "gemm_nt: batch too large for one launch");
  static spb_once_flag attr_once;   // function attributes are per device (one flag per EPI)
  const size_t smem = sizeof(Smem);
  {
    const int st = spb_once_per_device(attr_once, ctx->device, [&]() -> int {
      SPB_CHECK_CUDA(cudaFuncSetAttribute(gemm_nt_kernel<EPI>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      return 0;
    });
    if (st) return st;
  }
  const int tilesM = (d.M + TM - 1) / TM, tilesN = (d.N + TN - 1) / TN;
  dim3 grid(tilesM * tilesN * d.ksplit, d.batch);
  gemm_nt_kernel<EPI><<<grid, NTHREADS, smem, stream>>>(d);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

}  // namespace gnt
