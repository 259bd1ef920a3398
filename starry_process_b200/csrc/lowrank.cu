// Rank-31 form of the conditional (fixed-inclination) log-likelihood, linear in the number of time
// stamps (DESIGN.md section 4.6).
//
//   K = A Sigma A^T (normalised: sp.py:705-727) + baseline_var + D,   A = Phi(t) B_inc   (flux.py:335-343)
//     = Phi C~ Phi^T + D,   C~ (31 x 31) per element,  D diagonal > 0 (sp.py:1135-1151)
//   D^-1/2 Phi = Q R                (thin Householder QR, once per (t, p, data_cov): spb_lowrank_basis)
//   N = I + R C~ R^T                (K is PD  <=>  N is PD)
//   logdet K = sum log D + logdet N,  r^T K^-1 r = |y - Q w|^2 + w^T N^-1 w,  y = D^-1/2 r, w = Q^T y
//                                   (sp.py:1154-1188: spb_lowrank_lnlike)
//
// The rank is padded to 32 (Phi column 31 and B_inc row 31 are zero).  R is never inverted: light curves
// covering less than one period, or repeating one phase, have a singular R and still work.  Nothing of size
// nt^2 or nt x 256 is formed.  Every reduction runs in a fixed order over fixed row chunks (which depend on nt
// only), so an element's result does not depend on the batch size or on its position in the batch, and
// repeated calls are bitwise equal.
#include <string.h>

#include "common.cuh"
#include "gemm_nt.cuh"

namespace {

constexpr int LR = 32;            // padded rank
constexpr int QR_ROWS = 256;      // rows per TSQR block
constexpr int QR_GROUP = 8;       // R factors stacked into one block above the leaves
constexpr int QR_LD = 33;         // shared-memory row stride (conflict-free row and column walks)
constexpr int SOLVE_CH = 2048;    // time stamps per CTA of the solve (8 warps x 256)
constexpr int SOLVE_EB = 8;       // batch elements per CTA of the solve
constexpr int COV_CHUNK = 512;    // elements per (B_inc Sigma) workspace chunk

// Phi(t) = [1, cos(m theta), sin(m theta), 0] (m = 1 .. 15): the phase basis of design_rows_kernel
__device__ __forceinline__ void phase_row(double t, double period, double *row) {
  double cs[SPB_LMAX + 1], sn[SPB_LMAX + 1];
  spb_harmonics(spb_phase(t, period), cs, sn);
#pragma unroll
  for (int k = 0; k <= SPB_LMAX; ++k) row[k] = cs[k];
#pragma unroll
  for (int k = 1; k <= SPB_LMAX; ++k) row[SPB_LMAX + k] = sn[k];
  row[LR - 1] = 0.0;
}

__device__ __forceinline__ double data_var(int kind, const double *dc, long long i) {
  return kind == 0 ? dc[0] : dc[i];
}

// ---------------------------------------------------------------------------------------------------
// TSQR.  Level 0 factors the whitened Phi in blocks of <= 256 rows (an even split of nt, so every block
// of a multi-block level has >= 128 rows and Householder yields 32 orthonormal columns even when a
// block is rank-deficient); level l > 0 factors the stacked 32 x 32 R factors of level l - 1 in groups
// of 8.  Each block writes its explicit Q (rows x 32) and R; the final Q is assembled top-down
// (qr_combine_kernel): Q_l[block b] <- Q_l[block b] Q_{l+1}[rows 32 b .. 32 b + 31].
// ---------------------------------------------------------------------------------------------------
struct QRLevel {
  long long nrows;
  int nblk;
  int leaf;
  const double *X;        // (nrows, 32) input of an upper level
  double *Q;              // (nrows, 32) out
  double *R;              // (nblk, 32, 32) out
  const double *t;        // leaf: time stamps, period and the data variance
  double period;
  int data_kind;
  const double *data_cov;
  double *part;           // leaf: (nblk, 33) column sums of the unwhitened Phi and sum log D
};

__device__ __forceinline__ void qr_block_range(const QRLevel &p, int b, long long &r0, long long &r1) {
  if (p.leaf) {
    r0 = (long long)b * p.nrows / p.nblk;
    r1 = (long long)(b + 1) * p.nrows / p.nblk;
  } else {
    r0 = (long long)b * QR_GROUP * LR;
    r1 = r0 + QR_GROUP * LR < p.nrows ? r0 + QR_GROUP * LR : p.nrows;
  }
}

// X[k:n, c] <- (I - tau v v^T) X[k:n, c] for the columns c0 <= c < 32, v = (1, V[k+1:n, k]): one warp per
// column, fixed-order dot products
__device__ __forceinline__ void qr_apply(double *X, const double *V, int k, int n, double tau, int c0) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int c = c0 + warp; c < LR; c += 8) {
    const double xk = X[k * QR_LD + c];   // read by every lane before lane 0 updates it
    double d = 0.0;
    for (int i = k + 1 + lane; i < n; i += 32) d += V[i * QR_LD + k] * X[i * QR_LD + c];
    d = warp_sum(d) + xk;
    const double s = tau * d;
    if (lane == 0) X[k * QR_LD + c] -= s;
    for (int i = k + 1 + lane; i < n; i += 32) X[i * QR_LD + c] -= s * V[i * QR_LD + k];
  }
}

__global__ void __launch_bounds__(256) qr_block_kernel(QRLevel p) {
  extern __shared__ double qsm[];
  double *A = qsm;                        // (256, 33): the block, then R above / reflectors below the diagonal
  double *E = A + QR_ROWS * QR_LD;        // (256, 33): explicit Q
  double *tau = E + QR_ROWS * QR_LD;      // (32)
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  long long r0, r1;
  qr_block_range(p, b, r0, r1);
  const int n = (int)(r1 - r0);
  if (p.leaf) {
    if (tid < n) {
      const long long i = r0 + tid;
      double row[LR];
      phase_row(p.t[i], p.period, row);
      const double d = data_var(p.data_kind, p.data_cov, i);
      const double rs = 1.0 / sqrt(d);
#pragma unroll
      for (int c = 0; c < LR; ++c) {
        E[tid * QR_LD + c] = row[c];
        A[tid * QR_LD + c] = row[c] * rs;
      }
      E[tid * QR_LD + LR] = log(d);
    }
    __syncthreads();
    if (tid <= LR) {   // s = Phi^T 1 (unwhitened) and sum log D over this block, fixed order
      double s = 0.0;
      for (int i = 0; i < n; ++i) s += E[i * QR_LD + tid];
      p.part[(size_t)b * (LR + 1) + tid] = s;
    }
  } else {
    for (int idx = tid; idx < n * LR; idx += 256) {
      const int i = idx / LR, c = idx % LR;
      A[i * QR_LD + c] = p.X[(size_t)(r0 + i) * LR + c];
    }
  }
  __syncthreads();
  const int K = n < LR ? n : LR;
  for (int k = 0; k < K; ++k) {
    if (warp == 0) {   // dlarfg: beta = -sign(alpha) |x|, v = x / (alpha - beta), tau = (beta - alpha) / beta
      const double alpha = A[k * QR_LD + k];   // read by every lane before lane 0 overwrites it
      double sg = 0.0;
      for (int i = k + 1 + lane; i < n; i += 32) sg += A[i * QR_LD + k] * A[i * QR_LD + k];
      sg = warp_sum(sg);
      double tk = 0.0, scale = 0.0;
      if (sg > 0.0) {
        const double beta = -copysign(sqrt(alpha * alpha + sg), alpha);
        tk = (beta - alpha) / beta;
        scale = 1.0 / (alpha - beta);
        if (lane == 0) A[k * QR_LD + k] = beta;
      }
      if (lane == 0) tau[k] = tk;
      for (int i = k + 1 + lane; i < n; i += 32) A[i * QR_LD + k] *= scale;
    }
    __syncthreads();
    qr_apply(A, A, k, n, tau[k], k + 1);
    __syncthreads();
  }
  // R (rows >= n are zero), then Q = H_0 ... H_{K-1} [I; 0]
  for (int idx = tid; idx < LR * LR; idx += 256) {
    const int r = idx / LR, c = idx % LR;
    p.R[(size_t)b * LR * LR + idx] = (r < n && c >= r) ? A[r * QR_LD + c] : 0.0;
  }
  for (int idx = tid; idx < n * LR; idx += 256) {
    const int i = idx / LR, c = idx % LR;
    E[i * QR_LD + c] = (i == c) ? 1.0 : 0.0;
  }
  __syncthreads();
  for (int k = K - 1; k >= 0; --k) {
    qr_apply(E, A, k, n, tau[k], k);
    __syncthreads();
  }
  for (int idx = tid; idx < n * LR; idx += 256) {
    const int i = idx / LR, c = idx % LR;
    p.Q[(size_t)(r0 + i) * LR + c] = E[i * QR_LD + c];
  }
}

__global__ void __launch_bounds__(256) qr_combine_kernel(QRLevel p, const double *Qup) {
  __shared__ double G[LR * QR_LD];
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  long long r0, r1;
  qr_block_range(p, b, r0, r1);
  for (int idx = tid; idx < LR * LR; idx += 256)
    G[(idx / LR) * QR_LD + idx % LR] = Qup[(size_t)b * LR * LR + idx];
  __syncthreads();
  for (long long i = r0 + warp; i < r1; i += 8) {
    double *row = p.Q + (size_t)i * LR;
    const double q = row[lane];
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < LR; ++k) acc += __shfl_sync(0xffffffffu, q, k) * G[k * QR_LD + lane];
    row[lane] = acc;
  }
}

// phi_aux = [s = Phi^T 1 (32) | Phi(t_0) (32) | sum log D]
__global__ void basis_aux_kernel(int nblk, const double *part, const double *t, double period,
                                 double *aux) {
  const int tid = threadIdx.x;
  if (tid <= LR) {
    double s = 0.0;
    for (int b = 0; b < nblk; ++b) s += part[(size_t)b * (LR + 1) + tid];
    aux[tid < LR ? tid : 2 * LR] = s;
  }
  if (tid == 64) {
    double row[LR];
    phase_row(t[0], period, row);
    for (int c = 0; c < LR; ++c) aux[LR + c] = row[c];
  }
}

struct QRPlan {
  int levels;
  long long nrows[40];
  int nblk[40];
};

QRPlan qr_plan(int nt) {
  QRPlan pl;
  pl.levels = 0;
  long long rows = nt;
  int nb = (int)((rows + QR_ROWS - 1) / QR_ROWS);
  while (true) {
    pl.nrows[pl.levels] = rows;
    pl.nblk[pl.levels] = nb;
    ++pl.levels;
    if (nb == 1) break;
    rows = (long long)nb * LR;
    nb = (nb + QR_GROUP - 1) / QR_GROUP;
  }
  return pl;
}

// workspace: leaf partials | per upper level: Q (nrows x 32) | R of every level below the top
size_t basis_ws_doubles(int nt) {
  const QRPlan pl = qr_plan(nt);
  size_t n = (size_t)pl.nblk[0] * (LR + 1) + 32;
  for (int l = 0; l < pl.levels; ++l) {
    if (l > 0) n += (size_t)pl.nrows[l] * LR;
    if (l + 1 < pl.levels) n += (size_t)pl.nblk[l] * LR * LR;
  }
  return n;
}

// ---------------------------------------------------------------------------------------------------
// Per element: GP mean, normalisation (spb_norm_series, as norm_scalars_kernel), C~ (written back over C for
// lowrank_post_kernel), T = R C~ R^T, Cholesky of N = I + T, logdet.
// ---------------------------------------------------------------------------------------------------
struct CovParams {
  int nt;
  const double *Binc;
  long long Binc_stride;
  const double *mean_ylm;
  double *C;                // (B, 32, 32) in: B_inc Sigma B_inc^T, out: C~
  const double *R;          // (32, 32)
  const double *aux;        // s | Phi(t0) | sum log D
  spb_noise_model nm;
  const double *bmean;
  long long bm_stride;
  double *L;                // (B, 32, 32) out: Cholesky factor of N (lower)
  double *off;              // (B) out: residual offset (GP mean unless normalised, + baseline mean)
  double *logdet;           // (B) out: logdet K
  double *gp_mean;          // (B) out, optional
  double *z_out;
  int32_t *info;
};

__global__ void __launch_bounds__(256) lowrank_cov_kernel(CovParams p) {
  __shared__ double Cs[LR * QR_LD], Rs[LR * QR_LD], Ps[LR * QR_LD];
  __shared__ double bmv[LR], cs[LR], qh[LR], ph[LR], sc[5];
  __shared__ int bad;
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const double *Bb = p.Binc + (size_t)b * p.Binc_stride;
  const double *s = p.aux;
  // B_inc mean_ylm
  for (int k = warp; k < LR; k += 8) {
    double v = 0.0;
    for (int n = lane; n < 256; n += 32) v += Bb[k * 256 + n] * p.mean_ylm[(size_t)b * 256 + n];
    v = warp_sum(v);
    if (lane == 0) bmv[k] = v;
  }
  // C, lower triangle mirrored (what the Cholesky of the dense path reads)
  for (int idx = tid; idx < LR * LR; idx += 256) {
    const int i = idx / LR, j = idx % LR;
    Cs[i * QR_LD + j] = p.C[(size_t)b * LR * LR + (i >= j ? i * LR + j : j * LR + i)];
    Rs[i * QR_LD + j] = p.R[idx];
  }
  if (tid == 0) bad = 0;
  __syncthreads();
  if (tid == 0) {
    double g = 0.0;
    for (int k = 0; k < LR; ++k) g += s[LR + k] * bmv[k];   // (A mean_ylm)[0], flux.py:340
    sc[0] = g;
    if (p.gp_mean) p.gp_mean[b] = g;
  }
  if (p.nm.normalized && tid < LR) {
    double v = 0.0;
    for (int j = 0; j < LR; ++j) v += Cs[tid * QR_LD + j] * s[j];
    cs[tid] = v;   // Sigma_flux 1 = Phi cs
  }
  __syncthreads();
  const double gp_mean = sc[0];
  double s1 = 1.0, s2 = 0.0, s3 = 0.0;
  if (p.nm.normalized) {
    if (tid == 0) {
      double tot = 0.0;
      for (int k = 0; k < LR; ++k) tot += s[k] * cs[k];
      const double K = (double)p.nt;
      const double m = tot / (K * K);             // tt.mean(Sig)
      spb_norm_series(m, gp_mean, p.nm.normalization_order, p.nm.normalization_zmax, sc + 1,
                      p.z_out ? p.z_out + b : nullptr, p.info ? p.info + b : nullptr);
      sc[4] = K * m;
    }
    __syncthreads();
    if (tid < LR) {
      const double q = cs[tid] / sc[4];           // q = Sigma_flux 1 / (nt m) = Phi qh
      qh[tid] = q;
      ph[tid] = (tid == 0 ? 1.0 : 0.0) - q;       // 1 - q = Phi (e0 - qh)
    }
    __syncthreads();
    s1 = sc[1];
    s2 = sc[2];
    s3 = sc[3];
    for (int idx = tid; idx < LR * LR; idx += 256) {
      const int i = idx / LR, j = idx % LR;
      Cs[i * QR_LD + j] = s1 * Cs[i * QR_LD + j] + (s2 * (ph[i] * ph[j]) - s3 * (qh[i] * qh[j]));
    }
  } else if (tid == 0 && p.z_out) {
    p.z_out[b] = 0.0;
  }
  __syncthreads();
  if (tid == 0 && p.nm.baseline_var) Cs[0] += p.nm.baseline_var[(size_t)b * p.nm.base_stride];
  __syncthreads();
  // P = R C~, then N = I + P R^T (lower triangle, mirrored)
  for (int idx = tid; idx < LR * LR; idx += 256) {
    const int i = idx / LR, j = idx % LR;
    double v = 0.0;
    for (int k = 0; k < LR; ++k) v += Rs[i * QR_LD + k] * Cs[k * QR_LD + j];
    Ps[i * QR_LD + j] = v;
    p.C[(size_t)b * LR * LR + idx] = Cs[i * QR_LD + j];
  }
  __syncthreads();
  for (int idx = tid; idx < LR * LR; idx += 256) {
    const int i = idx / LR, j = idx % LR;
    if (j > i) continue;
    double v = 0.0;
    for (int k = 0; k < LR; ++k) v += Ps[i * QR_LD + k] * Rs[j * QR_LD + k];
    v += (i == j) ? 1.0 : 0.0;
    Cs[i * QR_LD + j] = v;
    Cs[j * QR_LD + i] = v;
  }
  __syncthreads();
  // right-looking Cholesky of N (math.py:75-91: a non-positive pivot flags the element)
  for (int j = 0; j < LR; ++j) {
    const double d = Cs[j * QR_LD + j];
    __syncthreads();
    if (!(d > 0.0)) {
      if (tid == 0) bad = 1;
      break;
    }
    const double ljj = sqrt(d);
    if (tid > j && tid < LR) Cs[tid * QR_LD + j] /= ljj;
    __syncthreads();
    if (tid == 0) Cs[j * QR_LD + j] = ljj;
    for (int idx = tid; idx < LR * LR; idx += 256) {
      const int r = idx / LR, c = idx % LR;
      if (c > j && r >= c) Cs[r * QR_LD + c] -= Cs[r * QR_LD + j] * Cs[c * QR_LD + j];
    }
    __syncthreads();
  }
  __syncthreads();
  for (int idx = tid; idx < LR * LR; idx += 256) {
    const int i = idx / LR, j = idx % LR;
    p.L[(size_t)b * LR * LR + idx] = (j <= i && !bad) ? Cs[i * QR_LD + j] : 0.0;
  }
  if (tid == 0) {
    double ld = 0.0;
    for (int j = 0; j < LR; ++j) ld += log(Cs[j * QR_LD + j]);
    p.logdet[b] = bad ? NAN : s[2 * LR] + 2.0 * ld;
    p.off[b] = (p.nm.normalized ? 0.0 : gp_mean) + (p.bmean ? p.bmean[(size_t)b * p.bm_stride] : 0.0);
    if (p.info) {
      const int prev = p.info[b] & ~SPB_INFO_NOT_PD;
      p.info[b] = prev | (bad ? SPB_INFO_NOT_PD : 0);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Solve.  CTA (chunk of SOLVE_CH time stamps, group of SOLVE_EB elements); each warp owns 256 rows and
// walks them in 32-row tiles of Q staged in its own shared memory.  Residual rows are formed explicitly:
// y = (flux - off) / sqrt(D).  Pass 1: partial w = Q^T y; pass 2: partial |y - Q w|^2.  Per-warp partials
// are combined in warp order, per-chunk partials in chunk order.
// ---------------------------------------------------------------------------------------------------
struct SolveParams {
  int B, nt, M, nch;
  const double *Q;
  const double *flux;
  int ldf;
  long long flux_stride;
  int data_kind;
  const double *data_cov;
  const double *off;
  const double *w;        // (B, M, 32) pass 2 input
  double *wpart;          // (nch, B, M, 32) pass 1 out
  double *sqpart;         // (nch, B, M) pass 2 out
};

template <bool PASS2>
__global__ void __launch_bounds__(256) lowrank_solve_kernel(SolveParams p) {
  extern __shared__ double solve_smem[];
  double (*Qs)[32 * QR_LD] = reinterpret_cast<double (*)[32 * QR_LD]>(solve_smem);             // per warp
  double (*red)[SOLVE_EB][LR] = reinterpret_cast<double (*)[SOLVE_EB][LR]>(solve_smem + 8 * 32 * QR_LD);
  double (*ws)[LR] = reinterpret_cast<double (*)[LR]>(solve_smem + 8 * 32 * QR_LD + 8 * SOLVE_EB * LR);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ch = blockIdx.x, e0 = blockIdx.y * SOLVE_EB;
  const long long row0 = (long long)ch * SOLVE_CH + warp * (SOLVE_CH / 8);
  const long long rowe = min(row0 + SOLVE_CH / 8, (long long)p.nt);
  double *Qw = Qs[warp];
  double offv[SOLVE_EB];
#pragma unroll
  for (int e = 0; e < SOLVE_EB; ++e) offv[e] = (e0 + e < p.B) ? p.off[e0 + e] : 0.0;
  for (int m = 0; m < p.M; ++m) {
    if (PASS2) {
      __syncthreads();
      for (int idx = tid; idx < SOLVE_EB * LR; idx += 256) {
        const int e = idx / LR, k = idx % LR;
        ws[e][k] = (e0 + e < p.B) ? p.w[((size_t)(e0 + e) * p.M + m) * LR + k] : 0.0;
      }
      __syncthreads();
    }
    double acc[SOLVE_EB];
#pragma unroll
    for (int e = 0; e < SOLVE_EB; ++e) acc[e] = 0.0;
    for (long long r = row0; r < rowe; r += 32) {
      const int nr = (int)min(32LL, rowe - r);
      __syncwarp();
      for (int j = 0; j < nr; ++j) Qw[j * QR_LD + lane] = p.Q[(size_t)(r + j) * LR + lane];
      __syncwarp();
      // this lane's row r + lane, whitened residual of every element of the group
      double y[SOLVE_EB];
      const bool have = lane < nr;
      const long long i = r + lane;
      const double rs = have ? 1.0 / sqrt(data_var(p.data_kind, p.data_cov, i)) : 0.0;
#pragma unroll
      for (int e = 0; e < SOLVE_EB; ++e) {
        y[e] = 0.0;
        if (have && e0 + e < p.B)
          y[e] = (p.flux[(size_t)(e0 + e) * p.flux_stride + (size_t)m * p.ldf + i] - offv[e]) * rs;
      }
      if (!PASS2) {
        for (int j = 0; j < nr; ++j) {
          const double q = Qw[j * QR_LD + lane];
#pragma unroll
          for (int e = 0; e < SOLVE_EB; ++e) acc[e] += q * __shfl_sync(0xffffffffu, y[e], j);
        }
      } else if (have) {
#pragma unroll
        for (int e = 0; e < SOLVE_EB; ++e) {
          double v = y[e];
          for (int k = 0; k < LR; ++k) v -= Qw[lane * QR_LD + k] * ws[e][k];
          acc[e] += v * v;
        }
      }
    }
    if (PASS2) {
#pragma unroll
      for (int e = 0; e < SOLVE_EB; ++e) acc[e] = warp_sum(acc[e]);
      if (lane == 0)
        for (int e = 0; e < SOLVE_EB; ++e) red[warp][e][0] = acc[e];
    } else {
#pragma unroll
      for (int e = 0; e < SOLVE_EB; ++e) red[warp][e][lane] = acc[e];
    }
    __syncthreads();
    if (!PASS2) {
      for (int idx = tid; idx < SOLVE_EB * LR; idx += 256) {
        const int e = idx / LR, k = idx % LR;
        if (e0 + e >= p.B) continue;
        double v = 0.0;
        for (int w = 0; w < 8; ++w) v += red[w][e][k];
        p.wpart[(((size_t)ch * p.B + e0 + e) * p.M + m) * LR + k] = v;
      }
    } else if (tid < SOLVE_EB && e0 + tid < p.B) {
      double v = 0.0;
      for (int w = 0; w < 8; ++w) v += red[w][tid][0];
      p.sqpart[((size_t)ch * p.B + e0 + tid) * p.M + m] = v;
    }
    __syncthreads();
  }
}

// w = sum over chunks, then |L^-1 w|^2 (one warp per (element, light curve))
__global__ void __launch_bounds__(256) lowrank_wsum_kernel(int B, int M, int nch, const double *wpart,
                                                           const double *L, double *w, double *qn) {
  const long long pr = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (pr >= (long long)B * M) return;
  const int b = (int)(pr / M);
  double v = 0.0;
  for (int c = 0; c < nch; ++c) v += wpart[((size_t)c * B * M + pr) * LR + lane];
  w[(size_t)pr * LR + lane] = v;
  const double *Lb = L + (size_t)b * LR * LR;
  double x = v, q = 0.0;   // column-oriented forward substitution, lane = row
  for (int i = 0; i < LR; ++i) {
    const double xi = __shfl_sync(0xffffffffu, x, i) / Lb[i * LR + i];
    q += xi * xi;
    if (lane > i) x -= Lb[lane * LR + i] * xi;
  }
  if (lane == 0) qn[pr] = q;
}

__global__ void lowrank_final_kernel(int B, int M, int nt, int nch, const double *sqpart, const double *qn,
                                     const double *logdet, const int32_t *info, double *lnlike, double *quad,
                                     double *logdet_out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double tot = 0.0;
  for (int m = 0; m < M; ++m) {
    double q = qn[(size_t)b * M + m];
    for (int c = 0; c < nch; ++c) q += sqpart[((size_t)c * B + b) * M + m];
    if (quad) quad[(size_t)b * M + m] = q;
    tot += q;
  }
  const double ld = logdet[b];
  if (logdet_out) logdet_out[b] = ld;
  const double ll = -0.5 * tot - 0.5 * M * ld - 0.5 * (double)nt * M * 1.8378770664093454836;  // log(2 pi)
  const bool flagged = (info && info[b] != 0) || isnan(ll);
  lnlike[b] = flagged ? -INFINITY : ll;
}

// ---------------------------------------------------------------------------------------------------
// Predictive distribution of the unnormalised process given one light curve.  K(ts, t) = Phi_s C~ Phi^T and
// K(ts, ts) = Phi_s C~ Phi_s^T, so with (Q T Q^T + I)^-1 = I - Q (I - N^-1) Q^T:
//   mean(ts) = gp_mean + Phi_s a,        a = C~ R^T N^-1 w
//   cov(ts)  = Phi_s P Phi_s^T,          P = C~ - V^T V,  V = L_N^-1 R C~
// and draws use G G^T = P (eigenvectors of P scaled by the square roots of its eigenvalues, negative ones
// clipped to zero): any square root gives the same distribution, and this one exists for a singular P.
// Row and column 31 of C~, and therefore of P, are the zero padding.
// ---------------------------------------------------------------------------------------------------
// An eigenvalue of P below -1e-10 max(lambda_max(P), max_k C~_kk) sets SPB_INFO_NOT_PD: the subtraction
// C~ - V^T V rounds at eps max C~_kk, which can exceed 1e-10 lambda_max(P) where the data pin every mode down.
constexpr double POST_NEG_TOL = 1e-10;
constexpr int JACOBI_SWEEPS = 30;
constexpr int EVAL_EB = 8;               // elements per CTA of the evaluation
constexpr int EVAL_SB = 32;              // draws per CTA of the evaluation

struct PostParams {
  const double *C;          // (B, 32, 32) C~ (lowrank_cov_kernel)
  const double *R;          // (32, 32)
  const double *L;          // (B, 32, 32) Cholesky factor of N (lowrank_cov_kernel)
  const double *w;          // (B, 32) Q^T y (lowrank_wsum_kernel)
  double *a, *P, *G;
  int32_t *info;
};

__global__ void __launch_bounds__(256) lowrank_post_kernel(PostParams p) {
  __shared__ double Cs[LR * QR_LD], Rs[LR * QR_LD], Ls[LR * QR_LD], Vs[LR * QR_LD];
  __shared__ double us[LR];
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  double *ab = p.a + (size_t)b * LR, *Pb = p.P + (size_t)b * LR * LR, *Gb = p.G + (size_t)b * LR * LR;
  for (int idx = tid; idx < LR * LR; idx += 256) {
    const int i = idx / LR, j = idx % LR;
    Cs[i * QR_LD + j] = p.C[(size_t)b * LR * LR + idx];
    Rs[i * QR_LD + j] = p.R[idx];
    Ls[i * QR_LD + j] = p.L[(size_t)b * LR * LR + idx];
  }
  if (p.info[b] & SPB_INFO_NOT_PD) {   // N (hence K(t, t)) is not PD: no posterior
    for (int idx = tid; idx < LR * LR; idx += 256) {
      Pb[idx] = NAN;
      Gb[idx] = NAN;
      if (idx < LR) ab[idx] = NAN;
    }
    return;
  }
  __syncthreads();
  if (warp == 0) {   // a = C~ R^T N^-1 w: forward and back substitution with L_N, lane = row
    double x = p.w[(size_t)b * LR + lane];
    for (int i = 0; i < LR; ++i) {
      const double xi = __shfl_sync(0xffffffffu, x, i) / Ls[i * QR_LD + i];
      if (lane == i) x = xi;
      else if (lane > i) x -= Ls[lane * QR_LD + i] * xi;
    }
    for (int i = LR - 1; i >= 0; --i) {
      const double xi = __shfl_sync(0xffffffffu, x, i) / Ls[i * QR_LD + i];
      if (lane == i) x = xi;
      else if (lane < i) x -= Ls[i * QR_LD + lane] * xi;
    }
    double u = 0.0;
    for (int i = 0; i < LR; ++i) u += Rs[i * QR_LD + lane] * __shfl_sync(0xffffffffu, x, i);
    us[lane] = u;
    __syncwarp();
    double av = 0.0;
    for (int j = 0; j < LR; ++j) av += Cs[lane * QR_LD + j] * us[j];
    ab[lane] = av;
  }
  // R C~, then V = L_N^-1 (R C~) (one column per thread)
  for (int idx = tid; idx < LR * LR; idx += 256) {
    const int i = idx / LR, j = idx % LR;
    double v = 0.0;
    for (int k = 0; k < LR; ++k) v += Rs[i * QR_LD + k] * Cs[k * QR_LD + j];
    Vs[i * QR_LD + j] = v;
  }
  __syncthreads();
  if (tid < LR) {
    for (int i = 0; i < LR; ++i) {
      double v = Vs[i * QR_LD + tid];
      for (int k = 0; k < i; ++k) v -= Ls[i * QR_LD + k] * Vs[k * QR_LD + tid];
      Vs[i * QR_LD + tid] = v / Ls[i * QR_LD + i];
    }
  }
  __syncthreads();
  // P = C~ - V^T V, exactly symmetric (entries (i, j) and (j, i) are the same products in the same order);
  // it replaces R, and the eigenvectors replace L_N
  for (int idx = tid; idx < LR * LR; idx += 256) {
    const int i = idx / LR, j = idx % LR;
    double v = 0.0;
    for (int k = 0; k < LR; ++k) v += Vs[k * QR_LD + i] * Vs[k * QR_LD + j];
    v = Cs[i * QR_LD + j] - v;
    Rs[i * QR_LD + j] = v;
    Pb[idx] = v;
  }
  __syncthreads();
  if (warp == 0) {
    // cyclic Jacobi on the leading 31 x 31 block (the round-robin of moments_k1b: 15 disjoint rotations per
    // round, index 31 the bye), lane = column in the row phase and row in the column phase
    double *A = Rs, *U = Ls;
    for (int r = 0; r < LR; ++r) U[r * QR_LD + lane] = (r == lane) ? 1.0 : 0.0;
    double amax = 0.0;
    for (int k = 0; k < LR - 1; ++k) amax = fmax(amax, fabs(A[k * QR_LD + k]));
    const double floor2 = (1e-20 * amax) * (1e-20 * amax);
    __syncwarp();
    for (int sweep = 0; sweep < JACOBI_SWEEPS; ++sweep) {
      bool rotated = false;
      for (int rnd = 0; rnd < LR - 1; ++rnd) {
        double cl = 1.0, sl = 0.0;
        if (lane >= 1 && lane < 16) {
          int pk = rnd + lane, qk = rnd - lane + 31;
          pk -= (pk >= 31) ? 31 : 0;
          qk -= (qk >= 31) ? 31 : 0;
          const int pi = min(pk, qk), qi = max(pk, qk);
          const double apq = A[pi * QR_LD + qi], app = A[pi * QR_LD + pi], aqq = A[qi * QR_LD + qi];
          if (apq * apq > fmax(floor2, 1.6e-29 * fabs(app * aqq))) {
            const double tau = (aqq - app) / (2.0 * apq);
            const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
            cl = 1.0 / sqrt(1.0 + t * t);
            sl = t * cl;
          }
        }
        rotated |= __any_sync(0xffffffffu, sl != 0.0);
        int P_[15], Q_[15];
        double C_[15], S_[15];
#pragma unroll
        for (int k = 0; k < 15; ++k) {
          int pk = rnd + k + 1, qk = rnd - k - 1 + 31;
          pk -= (pk >= 31) ? 31 : 0;
          qk -= (qk >= 31) ? 31 : 0;
          P_[k] = min(pk, qk);
          Q_[k] = max(pk, qk);
          C_[k] = __shfl_sync(0xffffffffu, cl, k + 1);
          S_[k] = __shfl_sync(0xffffffffu, sl, k + 1);
        }
        __syncwarp();
        // rows: A <- J^T A (lane = column); the 15 rotations touch disjoint pairs
#pragma unroll
        for (int k = 0; k < 15; ++k) {
          const double ap = A[P_[k] * QR_LD + lane], aq = A[Q_[k] * QR_LD + lane];
          A[P_[k] * QR_LD + lane] = C_[k] * ap - S_[k] * aq;
          A[Q_[k] * QR_LD + lane] = S_[k] * ap + C_[k] * aq;
        }
        __syncwarp();
        // columns: A <- A J, U <- U J (lane = row)
#pragma unroll
        for (int k = 0; k < 15; ++k) {
          const double ap = A[lane * QR_LD + P_[k]], aq = A[lane * QR_LD + Q_[k]];
          A[lane * QR_LD + P_[k]] = C_[k] * ap - S_[k] * aq;
          A[lane * QR_LD + Q_[k]] = S_[k] * ap + C_[k] * aq;
          const double up = U[lane * QR_LD + P_[k]], uq = U[lane * QR_LD + Q_[k]];
          U[lane * QR_LD + P_[k]] = C_[k] * up - S_[k] * uq;
          U[lane * QR_LD + Q_[k]] = S_[k] * up + C_[k] * uq;
        }
        __syncwarp();
      }
      if (!rotated) break;
    }
    const double lam = lane < LR - 1 ? A[lane * QR_LD + lane] : 0.0;
    double lmax = lam, lmin = lam, cmax = fabs(Cs[lane * QR_LD + lane]);
    for (int o = 16; o > 0; o >>= 1) {
      lmax = fmax(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
      lmin = fmin(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
      cmax = fmax(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
    }
    // only the draws need the square root: a and P stay valid, G is NaN
    const bool bad = !(lmin >= -POST_NEG_TOL * fmax(lmax, cmax));
    const double sq = sqrt(fmax(lam, 0.0));
    for (int k = 0; k < LR; ++k) {   // G[lane][k] = U[lane][k] sqrt(lambda_k)
      const double g = U[lane * QR_LD + k] * __shfl_sync(0xffffffffu, sq, k);
      Gb[lane * LR + k] = bad ? NAN : g;
    }
    if (lane == 0 && bad) p.info[b] |= SPB_INFO_NOT_PD;
  }
}

// gz[b][s] = G_b z1 (the first 32 unit normals of draw s)
__global__ void __launch_bounds__(256) lowrank_gz_kernel(int B, int S, int nts, const double *G, const double *z,
                                                         long long z_stride, double *gz) {
  const long long pr = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (pr >= (long long)B * S) return;
  const int b = (int)(pr / S), s = (int)(pr % S);
  const double *zr = z + (size_t)b * z_stride + (size_t)s * (LR + nts);
  const double *Gb = G + (size_t)b * LR * LR;
  double v = 0.0;
  for (int j = 0; j < LR; ++j) v += Gb[lane * LR + j] * zr[j];
  gz[(size_t)pr * LR + lane] = v;
}

struct EvalParams {
  int B, nts, S;
  const double *ts;
  double period;
  const double *a, *P, *gp_mean;
  const double *gz;         // (B, S, 32)
  const double *z;          // unit normals (S, 32 + nts) per element, z_stride elements apart
  long long z_stride;
  double sq_eps;
  double *mean, *var, *draws;
};

// CTA (256 output points x EVAL_EB elements x EVAL_SB draws).  Phi(ts) is rebuilt with phase_row (the
// rounding of the basis rows); the mean and variance are written by the CTAs of the first draw group.
__global__ void __launch_bounds__(256) lowrank_eval_kernel(EvalParams p) {
  __shared__ double Ps[LR * LR];
  __shared__ double as[LR];
  const int tid = threadIdx.x;
  const long long i = (long long)blockIdx.x * 256 + tid;
  const bool have = i < p.nts;
  const int e0 = blockIdx.y * EVAL_EB, s0 = blockIdx.z * EVAL_SB;
  const int s1 = min(p.S, s0 + EVAL_SB);
  const bool first = blockIdx.z == 0;
  double row[LR];
  phase_row(have ? p.ts[i] : 0.0, p.period, row);
  for (int e = 0; e < EVAL_EB && e0 + e < p.B; ++e) {
    const int b = e0 + e;
    __syncthreads();
    if (tid < LR) as[tid] = p.a[(size_t)b * LR + tid];
    if (p.var && first)
      for (int idx = tid; idx < LR * LR; idx += 256) Ps[idx] = p.P[(size_t)b * LR * LR + idx];
    __syncthreads();
    if (!have) continue;
    double d = 0.0;
#pragma unroll
    for (int k = 0; k < LR; ++k) d += row[k] * as[k];
    const double m = p.gp_mean[b] + d;
    if (first) {
      p.mean[(size_t)b * p.nts + i] = m;
      if (p.var) {   // sum_k (Phi P)_k Phi_k: the association of the two products that form the full matrix
        double v = 0.0;
#pragma unroll
        for (int k = 0; k < LR; ++k) {
          double tk = 0.0;
#pragma unroll
          for (int j = 0; j < LR; ++j) tk += row[j] * Ps[k * LR + j];
          v += tk * row[k];
        }
        p.var[(size_t)b * p.nts + i] = v;
      }
    }
    for (int s = s0; s < s1; ++s) {
      const double *g = p.gz + ((size_t)b * p.S + s) * LR;
      double d2 = 0.0;
#pragma unroll
      for (int k = 0; k < LR; ++k) d2 += row[k] * g[k];
      const double z2 = p.z[(size_t)b * p.z_stride + (size_t)s * (LR + p.nts) + LR + i];
      p.draws[((size_t)b * p.S + s) * p.nts + i] = m + d2 + p.sq_eps * z2;
    }
  }
}

// Phi(ts) (n, 32), the left factor of the full predictive covariance
__global__ void __launch_bounds__(256) lowrank_phi_kernel(int n, const double *t, double period, double *Phi) {
  const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  double row[LR];
  phase_row(t[i], period, row);
  for (int c = 0; c < LR; ++c) Phi[(size_t)i * LR + c] = row[c];
}

struct LnlikeLayout {
  double *T, *C, *L, *off, *logdet, *wpart, *w, *qn, *sqpart;
  size_t bytes;
};

LnlikeLayout lnlike_layout(void *ws, int B, int M, int nt) {
  const int nch = (nt + SOLVE_CH - 1) / SOLVE_CH;
  const size_t Bc = B < COV_CHUNK ? B : COV_CHUNK;
  size_t sizes[9] = {Bc * LR * 256, (size_t)B * LR * LR, (size_t)B * LR * LR, (size_t)B, (size_t)B,
                     (size_t)nch * B * M * LR, (size_t)B * M * LR, (size_t)B * M, (size_t)nch * B * M};
  double *ptrs[9];
  size_t off = 0;
  for (int k = 0; k < 9; ++k) {
    ptrs[k] = ws ? reinterpret_cast<double *>(reinterpret_cast<unsigned char *>(ws) + off) : nullptr;
    off += ((sizes[k] * sizeof(double) + 255) / 256) * 256;
  }
  LnlikeLayout l = {ptrs[0], ptrs[1], ptrs[2], ptrs[3], ptrs[4], ptrs[5], ptrs[6], ptrs[7], ptrs[8], off};
  return l;
}

// predict_eval workspace: G z1 (B, S, 32) | full covariance only: Phi(ts) (nts, 32) | Phi(ts) P (B, nts, 32)
struct EvalLayout {
  double *gz, *Phi, *T;
  size_t bytes;
};

EvalLayout eval_layout(void *ws, int B, int nts, int S, int full_cov) {
  const size_t sizes[3] = {(size_t)B * S * LR, full_cov ? (size_t)nts * LR : 0,
                           full_cov ? (size_t)B * nts * LR : 0};
  double *ptrs[3];
  size_t off = 0;
  for (int k = 0; k < 3; ++k) {
    ptrs[k] = ws ? reinterpret_cast<double *>(reinterpret_cast<unsigned char *>(ws) + off) : nullptr;
    off += ((sizes[k] * sizeof(double) + 255) / 256) * 256;
  }
  EvalLayout l = {ptrs[0], ptrs[1], ptrs[2], off};
  return l;
}

constexpr size_t QR_SMEM = (2 * QR_ROWS * QR_LD + LR) * sizeof(double);
constexpr size_t SOLVE_SMEM = (8 * 32 * QR_LD + 8 * SOLVE_EB * LR + SOLVE_EB * LR) * sizeof(double);

int set_smem_attributes(spb_context *ctx) {
  static spb_once_flag attr_once;   // function attributes are per device
  return spb_once_per_device(attr_once, ctx->device, [&]() -> int {
    SPB_CHECK_CUDA(cudaFuncSetAttribute(qr_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)QR_SMEM));
    SPB_CHECK_CUDA(cudaFuncSetAttribute(lowrank_solve_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)SOLVE_SMEM));
    SPB_CHECK_CUDA(cudaFuncSetAttribute(lowrank_solve_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)SOLVE_SMEM));
    return 0;
  });
}

// The part of the conditional evaluation shared by the log-likelihood and the predictive posterior:
// C = B_inc Sigma B_inc^T, lowrank_cov_kernel (GP mean, C~, Cholesky of N), pass 1 of the solve and the
// w sums.  `sp` is left filled in for pass 2.
int lowrank_front(spb_context *ctx, int B, int nt, const double *Binc, long long Binc_stride,
                  const double *mean_ylm, const double *cov_ylm, const double *Q, const double *R,
                  const double *phi_aux, const spb_noise_model *noise, int M, const double *flux, int ldf,
                  long long flux_stride, const double *baseline_mean, long long bm_stride, double *gp_mean,
                  double *z_out, int32_t *info, const LnlikeLayout &ly, SolveParams &sp, cudaStream_t stream) {
  const int nch = (nt + SOLVE_CH - 1) / SOLVE_CH;
  int st = set_smem_attributes(ctx);
  if (st) return st;
  // C[b] = B_inc (Sigma B_inc^T): each Sigma is read from HBM once, by the first product
  for (int b0 = 0; b0 < B; b0 += COV_CHUNK) {
    const int Bc = (B - b0 < COV_CHUNK) ? B - b0 : COV_CHUNK;
    gnt::Desc d1 = {};
    d1.A = Binc + (size_t)b0 * Binc_stride;
    d1.strideA = Binc_stride;
    d1.lda = 256;
    d1.Bm = cov_ylm + (size_t)b0 * 65536;
    d1.strideB = 65536;
    d1.ldb = 256;
    d1.C = ly.T;
    d1.strideC = (long long)LR * 256;
    d1.ldc = 256;
    d1.M = LR;
    d1.N = 256;
    d1.K = 256;
    d1.batch = Bc;
    d1.ksplit = 1;
    d1.alpha = 1.0;
    st = gnt::launch<gnt::EPI_STORE>(ctx, d1, stream);
    if (st) return st;
    gnt::Desc d2 = {};
    d2.A = ly.T;
    d2.strideA = (long long)LR * 256;
    d2.lda = 256;
    d2.Bm = Binc + (size_t)b0 * Binc_stride;
    d2.strideB = Binc_stride;
    d2.ldb = 256;
    d2.C = ly.C + (size_t)b0 * LR * LR;
    d2.strideC = (long long)LR * LR;
    d2.ldc = LR;
    d2.M = LR;
    d2.N = LR;
    d2.K = 256;
    d2.batch = Bc;
    d2.ksplit = 1;
    d2.alpha = 1.0;
    st = gnt::launch<gnt::EPI_STORE>(ctx, d2, stream);
    if (st) return st;
  }
  CovParams cp;
  cp.nt = nt;
  cp.Binc = Binc;
  cp.Binc_stride = Binc_stride;
  cp.mean_ylm = mean_ylm;
  cp.C = ly.C;
  cp.R = R;
  cp.aux = phi_aux;
  cp.nm = *noise;
  cp.bmean = baseline_mean;
  cp.bm_stride = bm_stride;
  cp.L = ly.L;
  cp.off = ly.off;
  cp.logdet = ly.logdet;
  cp.gp_mean = gp_mean;
  cp.z_out = z_out;
  cp.info = info;
  lowrank_cov_kernel<<<B, 256, 0, stream>>>(cp);
  SPB_LAUNCH_CHECK(ctx);
  sp.B = B;
  sp.nt = nt;
  sp.M = M;
  sp.nch = nch;
  sp.Q = Q;
  sp.flux = flux;
  sp.ldf = ldf;
  sp.flux_stride = flux_stride;
  sp.data_kind = noise->data_kind;
  sp.data_cov = noise->data_cov;
  sp.off = ly.off;
  sp.w = ly.w;
  sp.wpart = ly.wpart;
  sp.sqpart = ly.sqpart;
  const dim3 grid(nch, (B + SOLVE_EB - 1) / SOLVE_EB);
  lowrank_solve_kernel<false><<<grid, 256, SOLVE_SMEM, stream>>>(sp);
  SPB_LAUNCH_CHECK(ctx);
  const long long pairs = (long long)B * M;
  lowrank_wsum_kernel<<<(unsigned)((pairs + 7) / 8), 256, 0, stream>>>(B, M, nch, ly.wpart, ly.L, ly.w, ly.qn);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

}  // namespace

extern "C" size_t spb_lowrank_basis_workspace_bytes(const spb_context *ctx, int nt) {
  (void)ctx;
  return basis_ws_doubles(nt > 0 ? nt : 1) * sizeof(double) + 256;
}

extern "C" int spb_lowrank_basis(spb_context *ctx, int nt, const double *t, double period, int data_kind,
                                 const double *data_cov, double *Q, double *R, double *phi_aux,
                                 void *workspace, size_t workspace_bytes, void *stream_) {
  SPB_REQUIRE(ctx != nullptr && nt >= SPB_NEIG && t && Q && R && phi_aux && data_cov,
              "lowrank_basis: bad arguments (nt must be >= 31)");
  SPB_REQUIRE(data_kind == 0 || data_kind == 1, "lowrank_basis: data_kind must be 0 (scalar) or 1 (vector)");
  SPB_REQUIRE(period > 0.0, "lowrank_basis: period must be positive");
  SPB_REQUIRE(workspace != nullptr && workspace_bytes >= spb_lowrank_basis_workspace_bytes(ctx, nt),
              "lowrank_basis: workspace too small");
  cudaStream_t stream = (cudaStream_t)stream_;
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  int st = set_smem_attributes(ctx);
  if (st) return st;
  const QRPlan pl = qr_plan(nt);
  double *ws = reinterpret_cast<double *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  double *part = ws;
  double *cur = part + (size_t)pl.nblk[0] * (LR + 1) + 32;
  QRLevel lv[40];
  for (int l = 0; l < pl.levels; ++l) {
    QRLevel &p = lv[l];
    memset(&p, 0, sizeof(p));
    p.nrows = pl.nrows[l];
    p.nblk = pl.nblk[l];
    p.leaf = l == 0;
    p.X = l == 0 ? nullptr : lv[l - 1].R;
    if (l == 0) {
      p.Q = Q;
    } else {
      p.Q = cur;
      cur += (size_t)p.nrows * LR;
    }
    if (l + 1 < pl.levels) {
      p.R = cur;
      cur += (size_t)p.nblk * LR * LR;
    } else {
      p.R = R;
    }
    p.t = t;
    p.period = period;
    p.data_kind = data_kind;
    p.data_cov = data_cov;
    p.part = part;
    qr_block_kernel<<<p.nblk, 256, QR_SMEM, stream>>>(p);
    SPB_LAUNCH_CHECK(ctx);
  }
  for (int l = pl.levels - 2; l >= 0; --l) {
    qr_combine_kernel<<<lv[l].nblk, 256, 0, stream>>>(lv[l], lv[l + 1].Q);
    SPB_LAUNCH_CHECK(ctx);
  }
  basis_aux_kernel<<<1, 96, 0, stream>>>(pl.nblk[0], part, t, period, phi_aux);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" size_t spb_lowrank_lnlike_workspace_bytes(const spb_context *ctx, int B, int M, int nt) {
  (void)ctx;
  if (B < 1) B = 1;
  if (M < 1) M = 1;
  if (nt < 1) nt = 1;
  return lnlike_layout(nullptr, B, M, nt).bytes + 256;
}

extern "C" int spb_lowrank_lnlike(spb_context *ctx, int B, int nt, const double *Binc, long long Binc_stride,
                                  const double *mean_ylm, const double *cov_ylm, const double *Q,
                                  const double *R, const double *phi_aux, const spb_noise_model *noise, int M,
                                  const double *flux, int ldf, long long flux_stride,
                                  const double *baseline_mean, long long bm_stride, double *lnlike,
                                  double *quad, double *logdet, double *z_out, int32_t *info, void *workspace,
                                  size_t workspace_bytes, void *stream_) {
  SPB_REQUIRE(ctx != nullptr && B > 0 && nt >= SPB_NEIG && M > 0 && noise != nullptr,
              "lowrank_lnlike: bad arguments");
  SPB_REQUIRE(Binc && mean_ylm && cov_ylm && Q && R && phi_aux && flux && lnlike,
              "lowrank_lnlike: missing operand");
  SPB_REQUIRE(Binc_stride == 0 || Binc_stride == (long long)LR * 256,
              "lowrank_lnlike: Binc_stride must be 0 (shared) or 32 * 256");
  SPB_REQUIRE(ldf >= nt, "lowrank_lnlike: ldf must be >= nt");
  SPB_REQUIRE(noise->data_cov != nullptr && (noise->data_kind == 0 || noise->data_kind == 1) &&
                  noise->data_stride == 0,
              "lowrank_lnlike: data_cov must be one scalar or one (nt) vector shared by the batch");
  SPB_REQUIRE(noise->baseline_var == nullptr || noise->base_kind == 0,
              "lowrank_lnlike: baseline_var must be a scalar (or one per element)");
  SPB_REQUIRE(noise->temporal_kind == 0, "lowrank_lnlike: temporal kernels are not low-rank");
  SPB_REQUIRE(workspace != nullptr && workspace_bytes >= spb_lowrank_lnlike_workspace_bytes(ctx, B, M, nt),
              "lowrank_lnlike: workspace too small");
  SPB_REQUIRE(((uintptr_t)Binc % 16) == 0 && ((uintptr_t)cov_ylm % 16) == 0,
              "lowrank_lnlike: Binc and cov_ylm must be 16-byte aligned");
  SPB_REQUIRE((long long)B <= 65535LL * SOLVE_EB, "lowrank_lnlike: batch too large for one launch");
  cudaStream_t stream = (cudaStream_t)stream_;
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  void *ws = reinterpret_cast<void *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  const LnlikeLayout ly = lnlike_layout(ws, B, M, nt);
  const int nch = (nt + SOLVE_CH - 1) / SOLVE_CH;
  SolveParams sp;
  int st = lowrank_front(ctx, B, nt, Binc, Binc_stride, mean_ylm, cov_ylm, Q, R, phi_aux, noise, M, flux, ldf,
                         flux_stride, baseline_mean, bm_stride, nullptr, z_out, info, ly, sp, stream);
  if (st) return st;
  const dim3 grid(nch, (B + SOLVE_EB - 1) / SOLVE_EB);
  lowrank_solve_kernel<true><<<grid, 256, SOLVE_SMEM, stream>>>(sp);
  SPB_LAUNCH_CHECK(ctx);
  lowrank_final_kernel<<<(B + 127) / 128, 128, 0, stream>>>(B, M, nt, nch, ly.sqpart, ly.qn, ly.logdet, info,
                                                            lnlike, quad, logdet);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" size_t spb_lowrank_posterior_workspace_bytes(const spb_context *ctx, int B, int nt) {
  return spb_lowrank_lnlike_workspace_bytes(ctx, B, 1, nt);
}

extern "C" int spb_lowrank_posterior(spb_context *ctx, int B, int nt, const double *Binc, long long Binc_stride,
                                     const double *mean_ylm, const double *cov_ylm, const double *Q,
                                     const double *R, const double *phi_aux, const spb_noise_model *noise,
                                     const double *flux, const double *baseline_mean, long long bm_stride,
                                     double *a, double *P, double *G, double *gp_mean, int32_t *info,
                                     void *workspace, size_t workspace_bytes, void *stream_) {
  SPB_REQUIRE(ctx != nullptr && B > 0 && nt >= SPB_NEIG && noise != nullptr, "lowrank_posterior: bad arguments");
  SPB_REQUIRE(Binc && mean_ylm && cov_ylm && Q && R && phi_aux && flux && a && P && G && gp_mean && info,
              "lowrank_posterior: missing operand");
  SPB_REQUIRE(Binc_stride == 0 || Binc_stride == (long long)LR * 256,
              "lowrank_posterior: Binc_stride must be 0 (shared) or 32 * 256");
  SPB_REQUIRE(!noise->normalized, "lowrank_posterior: the predictive distribution of a normalised process is "
                                  "not defined");
  SPB_REQUIRE(noise->data_cov != nullptr && (noise->data_kind == 0 || noise->data_kind == 1) &&
                  noise->data_stride == 0,
              "lowrank_posterior: data_cov must be one scalar or one (nt) vector shared by the batch");
  SPB_REQUIRE(noise->baseline_var == nullptr || noise->base_kind == 0,
              "lowrank_posterior: baseline_var must be a scalar (or one per element)");
  SPB_REQUIRE(noise->temporal_kind == 0, "lowrank_posterior: temporal kernels are not low-rank");
  SPB_REQUIRE(workspace != nullptr && workspace_bytes >= spb_lowrank_posterior_workspace_bytes(ctx, B, nt),
              "lowrank_posterior: workspace too small");
  SPB_REQUIRE(((uintptr_t)Binc % 16) == 0 && ((uintptr_t)cov_ylm % 16) == 0,
              "lowrank_posterior: Binc and cov_ylm must be 16-byte aligned");
  SPB_REQUIRE((long long)B <= 65535LL * SOLVE_EB, "lowrank_posterior: batch too large for one launch");
  cudaStream_t stream = (cudaStream_t)stream_;
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  void *ws = reinterpret_cast<void *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  const LnlikeLayout ly = lnlike_layout(ws, B, 1, nt);
  SolveParams sp;
  int st = lowrank_front(ctx, B, nt, Binc, Binc_stride, mean_ylm, cov_ylm, Q, R, phi_aux, noise, 1, flux, nt, 0,
                         baseline_mean, bm_stride, gp_mean, nullptr, info, ly, sp, stream);
  if (st) return st;
  PostParams pp;
  pp.C = ly.C;
  pp.R = R;
  pp.L = ly.L;
  pp.w = ly.w;
  pp.a = a;
  pp.P = P;
  pp.G = G;
  pp.info = info;
  lowrank_post_kernel<<<B, 256, 0, stream>>>(pp);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" size_t spb_lowrank_predict_eval_workspace_bytes(const spb_context *ctx, int B, int nts, int nsamples,
                                                           int full_cov) {
  (void)ctx;
  if (B < 1) B = 1;
  if (nts < 1) nts = 1;
  if (nsamples < 0) nsamples = 0;
  return eval_layout(nullptr, B, nts, nsamples, full_cov).bytes + 256;
}

extern "C" int spb_lowrank_predict_eval(spb_context *ctx, int B, int nts, const double *t_sample, double period,
                                        const double *a, const double *P, const double *G,
                                        const double *gp_mean, int nsamples, const double *unit_normals,
                                        long long un_stride, double eps, double *mean, double *var,
                                        double *cov, int ldc, double *draws, void *workspace,
                                        size_t workspace_bytes, void *stream_) {
  SPB_REQUIRE(ctx != nullptr && B > 0 && nts > 0 && nsamples >= 0, "lowrank_predict_eval: bad arguments");
  SPB_REQUIRE(t_sample && a && P && gp_mean && mean, "lowrank_predict_eval: missing operand");
  SPB_REQUIRE(period > 0.0, "lowrank_predict_eval: period must be positive");
  SPB_REQUIRE(nsamples == 0 || (G && unit_normals && draws && eps >= 0.0 &&
                                (un_stride == 0 || un_stride == (long long)nsamples * (LR + nts))),
              "lowrank_predict_eval: draws need G, unit normals (nsamples, 32 + nts) shared (un_stride 0) or "
              "per element (un_stride nsamples * (32 + nts)) and eps >= 0");
  SPB_REQUIRE(cov == nullptr || (ldc >= nts && ((uintptr_t)P % 16) == 0),
              "lowrank_predict_eval: cov needs ldc >= nts and a 16-byte aligned P");
  SPB_REQUIRE((long long)B <= 65535LL * EVAL_EB && (long long)nsamples <= 65535LL * EVAL_SB,
              "lowrank_predict_eval: batch or draw count too large for one launch");
  SPB_REQUIRE(workspace != nullptr &&
                  workspace_bytes >= spb_lowrank_predict_eval_workspace_bytes(ctx, B, nts, nsamples, cov != nullptr),
              "lowrank_predict_eval: workspace too small");
  cudaStream_t stream = (cudaStream_t)stream_;
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  void *ws = reinterpret_cast<void *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  const EvalLayout ly = eval_layout(ws, B, nts, nsamples, cov != nullptr);
  if (nsamples > 0) {
    const long long pairs = (long long)B * nsamples;
    lowrank_gz_kernel<<<(unsigned)((pairs + 7) / 8), 256, 0, stream>>>(B, nsamples, nts, G, unit_normals, un_stride,
                                                                       ly.gz);
    SPB_LAUNCH_CHECK(ctx);
  }
  EvalParams ep;
  ep.B = B;
  ep.nts = nts;
  ep.S = nsamples;
  ep.ts = t_sample;
  ep.period = period;
  ep.a = a;
  ep.P = P;
  ep.gp_mean = gp_mean;
  ep.gz = ly.gz;
  ep.z = unit_normals;
  ep.z_stride = un_stride;
  ep.sq_eps = sqrt(eps);
  ep.mean = mean;
  ep.var = var;
  ep.draws = draws;
  dim3 grid((nts + 255) / 256, (B + EVAL_EB - 1) / EVAL_EB, nsamples > 0 ? (nsamples + EVAL_SB - 1) / EVAL_SB : 1);
  lowrank_eval_kernel<<<grid, 256, 0, stream>>>(ep);
  SPB_LAUNCH_CHECK(ctx);
  if (cov) {   // Phi_s P Phi_s^T: T = Phi_s P (P symmetric), cov = T Phi_s^T
    lowrank_phi_kernel<<<(nts + 255) / 256, 256, 0, stream>>>(nts, t_sample, period, ly.Phi);
    SPB_LAUNCH_CHECK(ctx);
    for (int b0 = 0; b0 < B; b0 += 65535) {
      const int Bc = (B - b0 < 65535) ? B - b0 : 65535;
      gnt::Desc d1 = {};
      d1.A = ly.Phi;
      d1.strideA = 0;
      d1.lda = LR;
      d1.Bm = P + (size_t)b0 * LR * LR;
      d1.strideB = (long long)LR * LR;
      d1.ldb = LR;
      d1.C = ly.T;
      d1.strideC = (long long)nts * LR;
      d1.ldc = LR;
      d1.M = nts;
      d1.N = LR;
      d1.K = LR;
      d1.batch = Bc;
      d1.ksplit = 1;
      d1.alpha = 1.0;
      int st = gnt::launch<gnt::EPI_STORE>(ctx, d1, stream);
      if (st) return st;
      gnt::Desc d2 = {};
      d2.A = ly.T;
      d2.strideA = (long long)nts * LR;
      d2.lda = LR;
      d2.Bm = ly.Phi;
      d2.strideB = 0;
      d2.ldb = LR;
      d2.C = cov + (size_t)b0 * nts * ldc;
      d2.strideC = (long long)nts * ldc;
      d2.ldc = ldc;
      d2.M = nts;
      d2.N = nts;
      d2.K = LR;
      d2.batch = Bc;
      d2.ksplit = 1;
      d2.alpha = 1.0;
      st = gnt::launch<gnt::EPI_STORE>(ctx, d2, stream);
      if (st) return st;
    }
  }
  return 0;
}
