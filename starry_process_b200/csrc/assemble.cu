// Assembly of the GP covariance that is factorised by the Cholesky kernel.
//
//   marginal kernel interpolation    flux.py:256-276  (cubic in the phase lag on the covpts grid)
//   normalisation series             sp.py:705-727, ops/norm/norm.py:26-44
//   data covariance + baseline       sp.py:1135-1151
//
// The dense (nt x nt) matrix is written exactly ONCE: for the normalised process the row sums that
// the series needs are obtained by re-evaluating the (cheap) interpolant in a compute-only pass
// instead of writing K, reading it back and rewriting it.
#include "common.cuh"

namespace {

struct AsmParams {
  int B, nt, ldk, covpts;
  const double *t;
  double period;
  const double *coef;     // (B,4,covpts+1)   marginal only
  const double *var;      // (B)
  const double *gp_mean;  // (B)
  spb_noise_model nm;
  double *K;              // (B,nt,ldk)
  double *rowq;           // (B,nt)  workspace: row sums, then q_i
  double *colpart;        // (B,RS_G,nt) workspace: column-sum partials of the symmetric pass
  double *scal;           // (B,4)   workspace: s1, s2, s3
  double *z_out;
  int32_t *info;
  int marginal;
};

__device__ __forceinline__ double interp_cov(const double *cf, int nc, double inv_dx, double thi,
                                             double thj) {
  // flux.py:262-271: x = |theta_i - theta_j|, inds = floor(x / dx), x0 = (x - xp[inds + 1]) / dx
  // with xp[k] = (k - 1) dx, i.e. x0 = x / dx - inds.  Evaluated with one multiplication by 1/dx
  // instead of two FP64 divisions: x / dx <= covpts, so x0 moves by <= covpts * 2^-53 and the
  // (continuous) interpolant by a relative ~1e-14, far inside the 1e-8 lnlike tolerance.
  const double s = fabs(thi - thj) * inv_dx;
  const int ind = (int)s;
  const double x0 = s - (double)ind;
  const double x2 = x0 * x0;
  return cf[ind] + cf[nc + ind] * x0 + cf[2 * nc + ind] * x2 + cf[3 * nc + ind] * (x2 * x0);
}

// Temporal kernels of time-variable surfaces (temporal.py:8-16), Hadamard-multiplied into the flux
// covariance BEFORE the normalisation (sp.py:697-698).  kind 1 = Matern-3/2, 2 = squared exponential.
__device__ __forceinline__ double temporal_k(int kind, double ti, double tj, double tau) {
  const double dt = fabs(ti - tj);
  if (kind == 1) {
    const double x = sqrt(3.0) * dt / tau;
    return (1.0 + x) * exp(-x);
  }
  return exp(-(dt * dt) / (2.0 * tau));
}

// ---- pass A (normalised conditional): row sums of K -----------------------------------------
__global__ void __launch_bounds__(256) rowsum_kernel(AsmParams p) {
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = blockIdx.x * 8 + warp; i < p.nt; i += gridDim.x * 8) {
    const double *row = p.K + ((size_t)b * p.nt + i) * p.ldk;
    double s = 0.0;
    for (int j = lane; j < p.nt; j += 32) s += row[j];
    s = warp_sum(s);
    if (lane == 0) p.rowq[(size_t)b * p.nt + i] = s;
  }
}

// ---- pass A', marginal kernel: the covariance is symmetric, so only the strict lower triangle is
// interpolated (half the evaluations); every value is added to its row sum AND to the sum of its
// column, which is the row sum of the mirrored element.  Deterministic (no atomics): a warp owns
// whole rows (interleaved by 64 for balance), lanes own columns j = lane mod 32 and keep their
// column sums in registers; the 8 warps are combined through shared memory in a fixed order and
// each of the RS_G CTAs of a sample leaves one partial vector that pass S adds up.
constexpr int RS_G = 8;      // CTAs per sample
constexpr int RS_CB = 512;   // columns per register block (16 per lane: 3 CTAs per SM)

// How an entry v(i, j) of the raw covariance is obtained: one policy per kind of light curve, each a
// compile-time parameter of rowsum_sym_kernel so that no policy costs another registers or predicated
// instructions in the inner loop.  A policy stages its shared-memory tables (stage: per time stamp, beside
// the phase table; tables: once that is complete, together with its per-CTA constants, whose FP64 divisions
// then overlap the latency of the staging loads), fixes the row (row) and returns v(i, j) for j < i
// (operator()) and v(i, i) for nt > 1 (diag).
//
// General time stamps: the cubic interpolant of flux.py:256-276 at |theta_i - theta_j|.
struct GeneralEntry {
  const double *cf, *th;
  int nc;
  double inv_dx, thi;
  __device__ GeneralEntry(const AsmParams &p, int b, const double *cf_, const double *th_, double *tail)
      : cf(cf_), th(th_), nc(p.covpts + 1) {}
  __device__ void stage(int k, double wraps) {}
  __device__ void tables(const AsmParams &p) { inv_dx = (double)p.covpts / (2.0 * 3.14159265358979323846); }
  __device__ void row(int i) { thi = th[i]; }
  __device__ double operator()(int i, int j) const { return interp_cov(cf, nc, inv_dx, thi, th[j]); }
  __device__ double diag() const { return interp_cov(cf, nc, inv_dx, thi, thi); }
};

// Time-variable surfaces: the interpolant times the temporal kernel (which is 1 on the diagonal).
struct TemporalEntry : GeneralEntry {
  const double *t;
  double *tm;   // tail: t (nt)
  int tkind;
  double tau, ti;
  __device__ TemporalEntry(const AsmParams &p, int b, const double *cf_, const double *th_, double *tail)
      : GeneralEntry(p, b, cf_, th_, tail), t(p.t), tm(tail), tkind(p.nm.temporal_kind),
        tau(p.nm.tau[(size_t)b * p.nm.tau_stride]) {}
  __device__ void stage(int k, double wraps) { tm[k] = t[k]; }
  __device__ void row(int i) {
    GeneralEntry::row(i);
    ti = tm[i];
  }
  __device__ double operator()(int i, int j) const {
    return GeneralEntry::operator()(i, j) * temporal_k(tkind, ti, tm[j], tau);
  }
};

// EQUALLY SPACED time stamps (spb_noise_model.uniform_dt).
// theta_i - theta_j = 2 pi ((t_i - t_j) / p - (floor(t_i / p) - floor(t_j / p))) = 2 pi (d dt / p - m) with
// d = i - j and m one of floor(d dt / p), floor(d dt / p) + 1: the interpolant is tabulated once per CTA
// for the 2 nt possible arguments (G[0][d], G[1][d]) and an entry costs two conflict-free shared-memory
// loads (the wrap count of column j and the table value) instead of the phase load and four coefficient
// gathers of the general policy, which is bound by exactly those (shared-memory LSU 77 %).  Entries whose
// wrap count is neither of the two candidates (cannot happen in exact arithmetic) take the general formula.
struct UniformEntry : GeneralEntry {
  double *G;      // tail: G (2 nt) | wraps (nt ints) | m0 (nt ints)
  int *fl, *m0t;  // floor(t_k / p) per stamp, floor(d dt / p) per lag
  int nt, fli;
  __device__ UniformEntry(const AsmParams &p, int b, const double *cf_, const double *th_, double *tail)
      : GeneralEntry(p, b, cf_, th_, tail), G(tail), fl(reinterpret_cast<int *>(tail + 2 * p.nt)), m0t(fl + p.nt),
        nt(p.nt) {}
  __device__ void stage(int k, double wraps) { fl[k] = (int)wraps; }
  __device__ void tables(const AsmParams &p) {
    GeneralEntry::tables(p);
    const double dtp = p.nm.uniform_dt / p.period;
    for (int d = threadIdx.x; d < nt; d += 256) {
      const double x = (double)d * dtp, m0 = floor(x);
      G[d] = interp_cov(cf, nc, inv_dx, 2.0 * 3.14159265358979323846 * (x - m0), 0.0);
      G[nt + d] = interp_cov(cf, nc, inv_dx, 2.0 * 3.14159265358979323846 * (m0 + 1.0 - x), 0.0);
      m0t[d] = (int)m0;
    }
    __syncthreads();
  }
  __device__ void row(int i) {
    GeneralEntry::row(i);
    fli = fl[i];
  }
  __device__ double operator()(int i, int j) const {
    const int d = i - j;
    const int w = (fli - fl[j]) - m0t[d];   // 0 or 1
    return ((unsigned)w <= 1u) ? G[w * nt + d] : GeneralEntry::operator()(i, j);
  }
  __device__ double diag() const { return G[0]; }
};

template <class Entry>
__global__ void __launch_bounds__(256, 3) rowsum_sym_kernel(AsmParams p) {
  extern __shared__ double sh[];  // coef (4*nc) | theta (nt) | part (8 x RS_CB) | the entry's own tables
  const int b = blockIdx.y, c = blockIdx.x;
  const int nc = p.covpts + 1;
  double *cf = sh, *th = sh + 4 * nc, *part = th + p.nt;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  Entry e(p, b, cf, th, part + 8 * RS_CB);
  for (int k = tid; k < 4 * nc; k += 256) cf[k] = p.coef[(size_t)b * 4 * nc + k];
  for (int k = tid; k < p.nt; k += 256) {
    double wraps;
    th[k] = spb_phase(p.t[k], p.period, &wraps);
    e.stage(k, wraps);
  }
  __syncthreads();
  e.tables(p);
  double *rowq = p.rowq + (size_t)b * p.nt;
  double *colp = p.colpart + ((size_t)b * RS_G + c) * p.nt;
  for (int cb0 = 0; cb0 < p.nt; cb0 += RS_CB) {
    double cs[RS_CB / 32];
#pragma unroll
    for (int k = 0; k < RS_CB / 32; ++k) cs[k] = 0.0;
    for (int i = c * 8 + warp; i < p.nt; i += RS_G * 8) {
      if (i < cb0) continue;
      e.row(i);
      double *Krow = p.K + ((size_t)b * p.nt + i) * p.ldk;
      double rs = 0.0;
#pragma unroll
      for (int k = 0; k < RS_CB / 32; ++k) {
        const int j = cb0 + 32 * k + lane;
        if (cb0 + 32 * k <= i) {        // warp-uniform
          if (j < i) {
            const double v = e(i, j);
            rs += v;
            cs[k] += v;
            if (p.nm.defer) Krow[j] = v;   // raw covariance, written once (coalesced along j)
          } else if (j == i) {
            const double v = (p.nt == 1) ? p.var[b] : e.diag();
            rs += v;
            if (p.nm.defer) Krow[j] = v;
          }
        }
      }
      rs = warp_sum(rs);
      if (lane == 0) rowq[i] = (cb0 == 0) ? rs : rowq[i] + rs;
    }
#pragma unroll
    for (int k = 0; k < RS_CB / 32; ++k) part[warp * RS_CB + 32 * k + lane] = cs[k];
    __syncthreads();
    for (int j = tid; j < RS_CB && cb0 + j < p.nt; j += 256) {
      double t = 0.0;
#pragma unroll
      for (int w = 0; w < 8; ++w) t += part[w * RS_CB + j];
      colp[cb0 + j] = t;
    }
    __syncthreads();
  }
}

// ---- pass S: per-sample scalars of the normalisation series ---------------------------------
__global__ void __launch_bounds__(256) norm_scalars_kernel(AsmParams p) {
  __shared__ double red[8];
  __shared__ double mshare;
  const int b = blockIdx.x, tid = threadIdx.x;
  double s = 0.0;
  for (int i = tid; i < p.nt; i += 256) {
    double r = p.rowq[(size_t)b * p.nt + i];
    if (p.marginal) {  // add the mirrored (column) contributions of the symmetric pass
      for (int c = 0; c < RS_G; ++c) r += p.colpart[((size_t)b * RS_G + c) * p.nt + i];
      p.rowq[(size_t)b * p.nt + i] = r;
    }
    s += r;
  }
  s = warp_sum(s);
  if ((tid & 31) == 0) red[tid >> 5] = s;
  __syncthreads();
  if (tid == 0) {
    double tot = 0.0;
    for (int k = 0; k < 8; ++k) tot += red[k];
    const double K = (double)p.nt;
    const double m = tot / (K * K);             // tt.mean(Sig)
    mshare = m;
    p.scal[4 * b + 3] = m;
    spb_norm_series(m, p.gp_mean[b], p.nm.normalization_order, p.nm.normalization_zmax, p.scal + 4 * b,
                    p.z_out ? p.z_out + b : nullptr, p.info ? p.info + b : nullptr);
  }
  __syncthreads();
  const double km = (double)p.nt * mshare;
  for (int i = tid; i < p.nt; i += 256) p.rowq[(size_t)b * p.nt + i] /= km;  // q = Sig 1 / (K m)
}

__device__ __forceinline__ double noise_term(const spb_noise_model &nm, int b, int i, int j, int nt) {
  double v = 0.0;
  if (nm.data_cov) {
    if (nm.data_kind == 0) {
      if (i == j) v += nm.data_cov[(size_t)b * nm.data_stride];
    } else if (nm.data_kind == 1) {
      if (i == j) v += nm.data_cov[(size_t)b * nm.data_stride + i];
    } else {
      v += nm.data_cov[(size_t)b * nm.data_stride + (size_t)i * nt + j];
    }
  }
  if (nm.baseline_var) {
    if (nm.base_kind == 0) v += nm.baseline_var[(size_t)b * nm.base_stride];
    else v += nm.baseline_var[(size_t)b * nm.base_stride + (size_t)i * nt + j];
  }
  return v;
}

// ---- pass W: write K (marginal) or update it in place (conditional) ---------------------------
template <bool TEMPORAL>
__global__ void __launch_bounds__(256) write_kernel(AsmParams p) {
  extern __shared__ double sh[];
  const int b = blockIdx.y;
  const int nc = p.covpts + 1;
  double *cf = sh, *th = sh + (p.marginal ? 4 * nc : 0), *q = th + (p.marginal ? p.nt : 0);
  double *tm = q + (p.nm.normalized ? p.nt : 0);
  const int tid = threadIdx.x;
  const int tkind = (TEMPORAL && p.marginal) ? p.nm.temporal_kind : 0;
  const double tau = tkind ? p.nm.tau[(size_t)b * p.nm.tau_stride] : 1.0;
  if (p.marginal) {
    for (int k = tid; k < 4 * nc; k += 256) cf[k] = p.coef[(size_t)b * 4 * nc + k];
    for (int k = tid; k < p.nt; k += 256) th[k] = spb_phase(p.t[k], p.period);
    if (TEMPORAL && tkind)
      for (int k = tid; k < p.nt; k += 256) tm[k] = p.t[k];
  }
  double s1 = 1.0, s2 = 0.0, s3 = 0.0;
  if (p.nm.normalized) {
    for (int k = tid; k < p.nt; k += 256) q[k] = p.rowq[(size_t)b * p.nt + k];
    s1 = p.scal[4 * b + 0];
    s2 = p.scal[4 * b + 1];
    s3 = p.scal[4 * b + 2];
  }
  __syncthreads();
  const double dx = (double)p.covpts / (2.0 * 3.14159265358979323846);  // 1 / dx
  // each CTA owns a band of rows; threads run along columns (coalesced 8-byte stores).  With
  // lower_only (the log-likelihood path: the Cholesky kernel never reads above the diagonal) only
  // columns j <= i are produced, halving both the interpolation work and the HBM writes.
  for (int i = blockIdx.x; i < p.nt; i += gridDim.x) {
    double *row = p.K + ((size_t)b * p.nt + i) * p.ldk;
    const double thi = p.marginal ? th[i] : 0.0;
    const double qi = p.nm.normalized ? q[i] : 0.0;
    const int jend = (p.marginal && p.nm.lower_only) ? i + 1 : p.nt;
    for (int j = tid; j < jend; j += 256) {
      double v;
      if (p.marginal) {
        v = (p.nt == 1) ? p.var[b] : interp_cov(cf, nc, dx, thi, th[j]);
        if (TEMPORAL && tkind) v *= temporal_k(tkind, tm[i], tm[j], tau);
      } else {
        v = row[j];
      }
      if (p.nm.normalized) {
        const double qj = q[j];
        v = s1 * v + (s2 * ((1.0 - qi) * (1.0 - qj)) - s3 * (qi * qj));  // sp.py:721-726
      }
      v += noise_term(p.nm, b, i, j, p.nt);
      row[j] = v;
    }
  }
}

int run_assemble(spb_context *ctx, AsmParams &p, void *workspace, size_t workspace_bytes,
                 cudaStream_t stream) {
  SPB_REQUIRE(p.B > 0 && p.nt > 0 && p.ldk >= p.nt, "assemble: bad arguments");
  SPB_REQUIRE(p.B <= 65535, "assemble: batch too large for one launch");
  const size_t need = ((size_t)p.B * p.nt * (1 + RS_G) + (size_t)p.B * 4) * sizeof(double);
  SPB_REQUIRE(workspace != nullptr && workspace_bytes >= need, "assemble: workspace too small");
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  p.rowq = reinterpret_cast<double *>(workspace);
  p.scal = p.rowq + (size_t)p.B * p.nt;
  p.colpart = p.scal + (size_t)p.B * 4;
  const int nc = p.covpts + 1;
  const size_t smT = (p.marginal && p.nm.temporal_kind) ? (size_t)p.nt * sizeof(double) : 0;
  const size_t smA = (p.marginal ? (4 * nc + p.nt) : 0) * sizeof(double) + smT;
  const size_t smW = smA + (p.nm.normalized ? p.nt : 0) * sizeof(double);
  SPB_REQUIRE(p.nm.temporal_kind >= 0 && p.nm.temporal_kind <= 2, "assemble: unknown temporal kernel");
  SPB_REQUIRE(!p.nm.temporal_kind || p.nm.tau != nullptr, "assemble: temporal kernel without tau");
  SPB_REQUIRE(smW <= 200 * 1024, "assemble: nt too large for the shared-memory staging");
  static spb_once_flag attr_once;   // function attributes are per device
  {
    const int st = spb_once_per_device(attr_once, ctx->device, [&]() -> int {
      SPB_CHECK_CUDA(cudaFuncSetAttribute(write_kernel<false>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      SPB_CHECK_CUDA(cudaFuncSetAttribute(write_kernel<true>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      SPB_CHECK_CUDA(cudaFuncSetAttribute(rowsum_sym_kernel<GeneralEntry>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      SPB_CHECK_CUDA(cudaFuncSetAttribute(rowsum_sym_kernel<TemporalEntry>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      SPB_CHECK_CUDA(cudaFuncSetAttribute(rowsum_sym_kernel<UniformEntry>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      return 0;
    });
    if (st) return st;
  }
  if (p.nm.normalized) {
    if (p.marginal) {
      const size_t smS = smA + (size_t)8 * RS_CB * sizeof(double);
      SPB_REQUIRE(smS <= 200 * 1024, "assemble: nt too large for the shared-memory staging");
      dim3 gridS(RS_G, p.B);
      const size_t smU = smS + (size_t)p.nt * (2 * sizeof(double) + 2 * sizeof(int)) + 16;
      if (p.nm.temporal_kind) rowsum_sym_kernel<TemporalEntry><<<gridS, 256, smS, stream>>>(p);
      else if (p.nm.uniform_dt > 0.0 && p.nt > 1 && smU <= 200 * 1024)
        rowsum_sym_kernel<UniformEntry><<<gridS, 256, smU, stream>>>(p);
      else rowsum_sym_kernel<GeneralEntry><<<gridS, 256, smS, stream>>>(p);
    } else {
      dim3 gridA(min((p.nt + 7) / 8, 16), p.B);
      rowsum_kernel<<<gridA, 256, 0, stream>>>(p);
    }
    SPB_LAUNCH_CHECK(ctx);
    norm_scalars_kernel<<<p.B, 256, 0, stream>>>(p);
    SPB_LAUNCH_CHECK(ctx);
  } else if (p.z_out) {
    SPB_CHECK_CUDA(cudaMemsetAsync(p.z_out, 0, (size_t)p.B * sizeof(double), stream));
  }
  if (p.nm.defer) {
    SPB_REQUIRE(p.marginal && p.nm.lower_only && p.nm.data_kind != 2 && p.nm.base_kind != 2,
                "assemble: defer needs the marginal lower-only path without full-matrix noise terms");
    if (p.nm.normalized) return 0;   // rowsum_sym_kernel already wrote the raw lower triangle
    AsmParams raw = p;               // raw interpolant only; the Cholesky kernel adds the noise
    raw.nm.data_cov = nullptr;
    raw.nm.baseline_var = nullptr;
    dim3 gridR(min(p.nt, 32), p.B);
    if (p.marginal && p.nm.temporal_kind) write_kernel<true><<<gridR, 256, smW, stream>>>(raw);
    else write_kernel<false><<<gridR, 256, smW, stream>>>(raw);
    SPB_LAUNCH_CHECK(ctx);
    return 0;
  }
  dim3 gridW(min(p.nt, 32), p.B);
  if (p.marginal && p.nm.temporal_kind) write_kernel<true><<<gridW, 256, smW, stream>>>(p);
  else write_kernel<false><<<gridW, 256, smW, stream>>>(p);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

}  // namespace

namespace {
// Rectangular marginal kernel K(ts, t) of predict (sp.py:887-902): the same cubic interpolant as
// flux.py:256-276 evaluated at |theta_ts,i - theta_t,j|, one output row per warp pass.
__global__ void __launch_bounds__(256) cross_marginal_kernel(int nts, int nt, int covpts,
                                                             const double *ts, const double *t,
                                                             double period, const double *coef,
                                                             const double *offset,
                                                             long long offset_stride, double *out,
                                                             int ld, long long out_stride) {
  extern __shared__ double sh[];  // coef (4*nc) | theta_t (nt)
  const int b = blockIdx.y;
  const int nc = covpts + 1;
  double *cf = sh, *th = sh + 4 * nc;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int k = tid; k < 4 * nc; k += 256) cf[k] = coef[(size_t)b * 4 * nc + k];
  for (int k = tid; k < nt; k += 256) th[k] = spb_phase(t[k], period);
  __syncthreads();
  const double inv_dx = (double)covpts / (2.0 * 3.14159265358979323846);
  const double off = offset ? offset[(size_t)b * offset_stride] : 0.0;
  for (int i = blockIdx.x * 8 + warp; i < nts; i += gridDim.x * 8) {
    const double thi = spb_phase(ts[i], period);
    double *row = out + (size_t)b * out_stride + (size_t)i * ld;
    for (int j = lane; j < ld; j += 32)
      row[j] = (j < nt) ? interp_cov(cf, nc, inv_dx, thi, th[j]) + off : 0.0;
  }
}
}  // namespace

namespace {
__global__ void __launch_bounds__(256) temporal_scale_kernel(int n1, int n2, const double *t1,
                                                             const double *t2, int kind,
                                                             const double *tau, long long tau_stride,
                                                             const double *offset,
                                                             long long offset_stride, double *K,
                                                             int ld, long long stride) {
  const int b = blockIdx.y;
  const double tb = tau[(size_t)b * tau_stride];
  const double off = offset ? offset[(size_t)b * offset_stride] : 0.0;
  for (int i = blockIdx.x; i < n1; i += gridDim.x) {
    const double ti = t1[i];
    double *row = K + (size_t)b * stride + (size_t)i * ld;
    for (int j = threadIdx.x; j < n2; j += 256)
      row[j] = fma(row[j], temporal_k(kind, ti, t2[j], tb), off);
  }
}
}  // namespace

extern "C" int spb_temporal_scale(spb_context *ctx, int B, int n1, int n2, const double *t1,
                                  const double *t2, int kind, const double *tau,
                                  long long tau_stride, const double *offset,
                                  long long offset_stride, double *K, int ld, long long K_stride,
                                  void *stream) {
  SPB_REQUIRE(ctx != nullptr && B > 0 && n1 > 0 && n2 > 0 && ld >= n2 && K != nullptr && tau != nullptr,
              "temporal_scale: bad arguments");
  SPB_REQUIRE(kind == 1 || kind == 2, "temporal_scale: unknown kernel");
  SPB_REQUIRE(B <= 65535, "temporal_scale: batch too large for one launch");
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  int gx = n1 < 8 * ctx->num_sms ? n1 : 8 * ctx->num_sms;
  temporal_scale_kernel<<<dim3(gx, B), 256, 0, (cudaStream_t)stream>>>(
      n1, n2, t1, t2, kind, tau, tau_stride, offset, offset_stride, K, ld, K_stride);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int spb_cross_marginal(spb_context *ctx, int B, int nts, int nt, const double *ts,
                                  const double *t, double period, int covpts, const double *coef,
                                  const double *offset, long long offset_stride, double *K_ts_t,
                                  int ld, long long K_stride, void *stream) {
  SPB_REQUIRE(ctx != nullptr && ts != nullptr && t != nullptr && coef != nullptr && K_ts_t != nullptr,
              "cross_marginal: null argument");
  SPB_REQUIRE(B > 0 && nts > 0 && nt > 0 && ld >= nt, "cross_marginal: bad arguments");
  SPB_REQUIRE(covpts >= 4, "cross_marginal: covpts must be >= 4");
  SPB_REQUIRE(period > 0.0, "cross_marginal: period must be positive");
  SPB_REQUIRE(B <= 65535, "cross_marginal: batch too large for one launch");
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  const size_t smem = (size_t)(4 * (covpts + 1) + nt) * sizeof(double);
  SPB_REQUIRE(smem <= 200 * 1024, "cross_marginal: nt too large for the shared-memory phase table");
  SPB_CHECK_CUDA(cudaFuncSetAttribute(cross_marginal_kernel,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int gx = (nts + 7) / 8;
  if (gx > 4 * ctx->num_sms) gx = 4 * ctx->num_sms;
  cross_marginal_kernel<<<dim3(gx, B), 256, smem, (cudaStream_t)stream>>>(
      nts, nt, covpts, ts, t, period, coef, offset, offset_stride, K_ts_t, ld, K_stride);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" size_t spb_assemble_workspace_bytes(const spb_context *ctx, int B, int nt) {
  (void)ctx;
  return ((size_t)B * nt * (1 + RS_G) + (size_t)B * 4) * sizeof(double) + 256;
}

extern "C" void spb_assemble_workspace_layout(int B, int nt, void *workspace, double **q,
                                              double **scal) {
  double *rowq = reinterpret_cast<double *>(workspace);
  if (q) *q = rowq;
  if (scal) *scal = rowq + (size_t)B * nt;
}

extern "C" int spb_assemble_marginal(spb_context *ctx, int B, int nt, const double *t, double period,
                                     int covpts, const double *coef, const double *var,
                                     const double *gp_mean, const spb_noise_model *noise, double *K,
                                     int ldk, double *z_out, int32_t *info, void *workspace,
                                     size_t workspace_bytes, void *stream) {
  SPB_REQUIRE(ctx != nullptr && noise != nullptr && t != nullptr && coef != nullptr,
              "assemble_marginal: null argument");
  SPB_REQUIRE(period > 0.0, "assemble_marginal: period must be positive");
  AsmParams p = {};
  p.B = B;
  p.nt = nt;
  p.ldk = ldk;
  p.covpts = covpts;
  p.t = t;
  p.period = period;
  p.coef = coef;
  p.var = var;
  p.gp_mean = gp_mean;
  p.nm = *noise;
  p.K = K;
  p.z_out = z_out;
  p.info = info;
  p.marginal = 1;
  return run_assemble(ctx, p, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int spb_assemble_conditional(spb_context *ctx, int B, int nt, const double *gp_mean,
                                        const spb_noise_model *noise, double *K, int ldk,
                                        double *z_out, int32_t *info, void *workspace,
                                        size_t workspace_bytes, void *stream) {
  SPB_REQUIRE(ctx != nullptr && noise != nullptr, "assemble_conditional: null argument");
  AsmParams p = {};
  p.B = B;
  p.nt = nt;
  p.ldk = ldk;
  p.covpts = 1;
  p.period = 1.0;
  p.gp_mean = gp_mean;
  p.nm = *noise;
  p.K = K;
  p.z_out = z_out;
  p.info = info;
  p.marginal = 0;
  return run_assemble(ctx, p, workspace, workspace_bytes, (cudaStream_t)stream);
}
