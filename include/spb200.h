/*
 * spb200.h -- C ABI of libspb200.so: the B200-native (sm_100a) batched log-likelihood hot path of
 * rodluger/starry_process, for ydeg = 15 (N = 256 spherical-harmonic coefficients), fp64.
 *
 * This is the drop-in boundary.  Every entry point replaces one (or a fused group) of the
 * reference's Theano ops / Python glue on the lnlike path; the reference interface each one
 * replaces is cited as file:line under starry_process/.  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host; all arrays are C-contiguous
 *     row-major float64 (as the reference enforces, ops/include/theano_helpers.h:55-63);
 *   - the caller owns all memory (outputs and workspaces); workspace sizes come from the
 *     *_workspace_bytes functions;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default
 *     stream), re-entrant across streams/devices, and performs no host synchronisation;
 *   - return value: 0 on success, non-zero on a usage / CUDA error (message: spb_last_error());
 *   - per-batch-element numerical failures (non positive-definite K, normalised process outside
 *     its validity range, hyperparameters out of bounds, a latitude eigen-solve that did not
 *     converge) never fail the call: they set info[b] != 0 and lnlike[b] = -inf (the bits of
 *     SPB_INFO_NEG_INF), the batched analogue of the reference's NaN -> -inf convention
 *     (math.py:82-91, sp.py:1178-1188);
 *   - Ylm index n = l^2 + l + m; angles in radians at this level (the Python surface takes degrees).
 */
#ifndef SPB200_H
#define SPB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPB_YDEG 15
#define SPB_N 256      /* (ydeg+1)^2,                         ops/include/constants.h:27 */
#define SPB_NWIG 5456  /* packed Wigner matrix size,          ops/include/constants.h:33-34 */
#define SPB_NEIG 31    /* 2*ydeg+1, rank of the Wigner integrals, integrals.py:112-114 */

typedef struct spb_context spb_context;

/* info[] bits */
#define SPB_INFO_NOT_PD 1       /* Cholesky met a non-positive pivot (math.py:82-91) */
#define SPB_INFO_Z_RANGE 2      /* normalised process: z > normalization_zmax (sp.py:1178-1183) */
#define SPB_INFO_BOUNDS 4       /* hyperparameter outside CheckBoundsOp range (ops/exceptions.py:30-48) */
#define SPB_INFO_EIG_NOCONV 8   /* latitude eigen-solve did not converge (eigh.py:12-16 -> NaN) */
#define SPB_INFO_I8_RANGE 16    /* transient: spb_cholesky_lnlike_i8 re-ran this matrix on the DMMA kernel */
/* The bits that force lnlike[b] = -inf on every log-likelihood route (dense Cholesky kernels, the INT8
 * Cholesky, the rank-31 route): each marks an element whose reference value is NaN (-> -inf).  A NaN
 * lnlike maps to -inf as well.  SPB_INFO_I8_RANGE is not among them: it only records a re-run.          */
#define SPB_INFO_NEG_INF (SPB_INFO_NOT_PD | SPB_INFO_Z_RANGE | SPB_INFO_BOUNDS | SPB_INFO_EIG_NOCONV)

const char *spb_last_error(void);
int spb_version(void);

/* ---------------------------------------------------------------------------------------------
 * Context: holds the hyperparameter-independent constant tables in device memory.
 *
 * `tables_host` is a packed host blob produced by starry_process_b200/_tables.py (the host-side
 * mirror of the reference's graph-build-time NumPy precomputations: size.py:10-43 Spot operator,
 * wigner.py:295-372 polynomial Wigner tensors, longitude.py:9-49 + integrals.py:116-124 longitude
 * tensors, flux.py:107-179 inclination-marginalisation integrals).  Layout: spb_tables.h.
 * ------------------------------------------------------------------------------------------- */
int spb_create(int device, const double *tables_host, size_t tables_count, spb_context **out);
void spb_destroy(spb_context *ctx);
int spb_device(const spb_context *ctx);

/* ---------------------------------------------------------------------------------------------
 * (a1) gauss2beta -- latitude.py:14-77.  mu, sigma in DEGREES (as the reference takes them).
 * ------------------------------------------------------------------------------------------- */
int spb_gauss2beta(spb_context *ctx, int B, const double *mu_deg, const double *sigma_deg,
                   double *a, double *b, void *stream);

/* log-Jacobian of the (a, b) -> (mu, sigma) transform of the latitude prior, one value per element:
 * LatitudeIntegral._log_jac, latitude.py:221-241, 281-316 (used by calibrate/log_prob.py:87-90);
 * -inf where sigma > sigma_max (degrees, defaults.py: 45).                                      */
int spb_log_jac(spb_context *ctx, int B, const double *a, const double *b, double sigma_max_deg,
                double *log_jac, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (a2-a9) Ylm moment integrals: size -> latitude -> longitude -> contrast.
 * Replaces SizeIntegral/LatitudeIntegral/LongitudeIntegral/ContrastIntegral
 * (size.py:93-115, latitude.py:171-212 + ops/latitude/latitude.cc:19-81 + ops/include/latitude.h:22-173
 *  + special.h:173-232, integrals.py:116-151, math.py:121-139 + ops/eigh/eigh.py:11-20,
 *  longitude.py:9-49, contrast.py:9-33).
 *   r_deg, a, b, c, n : (B) hyperparameters (r in degrees; a, b the Beta shape parameters)
 *   mean_ylm          : (B, 256)       out
 *   cov_ylm           : (B, 256, 256)  out
 *   info              : (B)            out (bit mask above)
 * ------------------------------------------------------------------------------------------- */
/* Keyword options of the moment integrals that the reference threads through its constructor
 * (sp.py:241-262, defaults.py:4-35).  A NULL pointer / zero field selects the reference default.
 *   Bp            (16, 1000) spot profile operator S A (size.py:10-43) for a lower spherical-harmonic
 *                 degree: rows l > ydeg zero.  The degree-15 machinery then evaluates the ydeg < 15
 *                 process exactly (the latitude / longitude rotations are block-diagonal in l), the
 *                 caller reads the leading (ydeg+1)^2 block of mean_ylm / cov_ylm
 *   lambda        (256) diagonal jitter: epsy for l < 15, epsy15 for l = 15 (contrast.py:26-32); zero
 *                 for l > ydeg when a lower degree is embedded
 *   abmin, log_alpha_max, log_beta_max      latitude.py:171-200                                  */
typedef struct {
  const double *Bp;
  const double *lambda;
  double abmin;
  double log_alpha_max;
  double log_beta_max;
} spb_moments_options;

size_t spb_ylm_moments_workspace_bytes(const spb_context *ctx, int B);
int spb_ylm_moments(spb_context *ctx, int B, const double *r_deg, const double *a, const double *b,
                    const double *c, const double *n, double *mean_ylm, double *cov_ylm,
                    int32_t *info, void *workspace, size_t workspace_bytes, void *stream);
/* Same with a UNIFORM prior on the spot radius over [r - dr, r + dr] (size.py:55-89, 116-125:
 * Spot.get_e, Spot.get_eigE): dr_deg (B) in degrees, or NULL for the delta prior above.          */
int spb_ylm_moments_dr(spb_context *ctx, int B, const double *r_deg, const double *dr_deg,
                       const double *a, const double *b, const double *c, const double *n,
                       const spb_moments_options *opt, double *mean_ylm, double *cov_ylm,
                       int32_t *info, void *workspace, size_t workspace_bytes, void *stream);
int spb_gauss2beta_opt(spb_context *ctx, int B, const double *mu_deg, const double *sigma_deg,
                       const spb_moments_options *opt, double *a, double *b, void *stream);
int spb_log_jac_opt(spb_context *ctx, int B, const double *a, const double *b, double sigma_max_deg,
                    const spb_moments_options *opt, double *log_jac, void *stream);

/* (f-4) Ylm moments AND their derivatives with respect to (r [deg], a, b, c, n), for the gradient of
 * the log-likelihood (the reference: Theano reverse mode through ops/include/latitude.h:22-173
 * derivative lanes, eigh.h:19-65, integrals.py:116-151).  Delta prior on the spot radius.
 * Returns 11 VARIANTS of the moments per sample, variant-major (slot v * B + b):
 *   v = 0 base;  1,2: r + eps, r - eps;  3,4: a +-;  5,6: b +-;  7,8: c +-;  9,10: n +-
 * where variants 1..6 move (S = Z^T Q Z, q_l, mom1) along their ANALYTIC tangents (Beta-moment
 * derivative lanes, profile derivative) and then run the unchanged eigen-solve / longitude / SYRK
 * pipeline, which is linear in S and quadratic in (q_l, mom1): the central difference
 * (out[v+] - out[v-]) / (2 eps) of any linear / quadratic functional of (mean_ylm, cov_ylm) is its
 * exact directional derivative.  eps: (5, B) absolute steps (rel_step times base / tangent scale).
 *   mean_ylm: (11 B, 256) out;  cov_ylm: (11 B, 256, 256) out;  info: (B) out                      */
size_t spb_ylm_moments_grad_workspace_bytes(const spb_context *ctx, int B);
int spb_ylm_moments_grad(spb_context *ctx, int B, const double *r_deg, const double *a,
                         const double *b, const double *c, const double *n,
                         const spb_moments_options *opt, double rel_step, double *mean_ylm,
                         double *cov_ylm, double *eps, int32_t *info, void *workspace,
                         size_t workspace_bytes, void *stream);

/* Cholesky factor of cov_ylm and prior draws -- sp.py:265-271, 489-509.
 *   L_ylm : (B,256,256) out, lower triangle (upper zeroed);  unit_normals: (B, nsamples, 256)
 *   y     : (B, nsamples, 256) out = mean + L u                                              */
int spb_cho_cov_ylm(spb_context *ctx, int B, const double *cov_ylm, double *L_ylm, int32_t *info,
                    void *stream);
int spb_sample_ylm(spb_context *ctx, int B, int nsamples, const double *mean_ylm,
                   const double *L_ylm, const double *unit_normals, double *y, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (a13) flux operator rTA1 / rTA1L(u) -- ops/flux/rTA1.cc:7-30, rTA1L.cc:22-60,
 * ops/include/flux.h:302-309, 501-523.  u: (nu, 2) quadratic limb darkening; out: (nu, 256).
 * ------------------------------------------------------------------------------------------- */
int spb_flux_operator(spb_context *ctx, int nu, const double *u, double *rTA1, void *stream);

/* (a10) real Wigner x-rotation matrices, packed -- ops/wigner/Rx.cc:10-49, wigner.h:37-284.
 *   theta: (nang) radians; Rx: (nang, 5456)                                                   */
int spb_Rx(spb_context *ctx, int nang, const double *theta, double *Rx, void *stream);

/* (a11) tensordotRz -- ops/wigner/tensordotRz.cc:10-56, wigner.h:290-339.
 *   M: (K,256), theta: (K) -> f: (K,256)                                                      */
int spb_tensordotRz(spb_context *ctx, int K, const double *M, const double *theta, double *f,
                    void *stream);

/* (a12) design matrix A(t; i, p, u) -- flux.py:88-105, 278-281, 345-350.
 *   t: (nt); inc_rad: (I); period: (I) or NULL (=> 1.0); rTA1: (I,256) or (1,256) broadcast
 *   (rTA1_stride = 256 or 0);  A: (I, nt, 256)                                                */
size_t spb_design_matrix_workspace_bytes(const spb_context *ctx, int I, int nt);
int spb_design_matrix(spb_context *ctx, int I, int nt, const double *t, const double *inc_rad,
                      const double *period, const double *rTA1, int rTA1_stride, double *A,
                      void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (a14-a18) flux-space GP mean and covariance.
 *
 * Marginalised over inclination -- flux.py:55-62, 181-231, 256-276, 295-333 and
 * ops/wigner/special_tensordotRz.cc:10-65 (wigner.h:410-459):
 *   mean_ylm (B,256), cov_ylm (B,256,256), rTA1 (256) [shared], t (nt), period p, covpts
 *   -> gp_mean (B) (the scalar flux mean), kernel coefficient table coef (B, 4, covpts+1),
 *      var (B) (the nt == 1 variance).  The dense (nt,nt) covariance is then materialised from the
 *      table by spb_assemble_marginal (and the rectangular K(ts, t) of predict by
 *      spb_cross_marginal).
 *
 * Conditional on inclination -- flux.py:335-343:
 *   K[b] = A cov_ylm[b] A^T, gp_mean[b] = (A mean_ylm[b])[0];  A: (nt,256) shared by the batch
 *   (A_stride = 0) or one design matrix per element (A_stride = nt*256, e.g. one inclination each).
 * ------------------------------------------------------------------------------------------- */
size_t spb_flux_marginal_workspace_bytes(const spb_context *ctx, int B);
int spb_flux_marginal(spb_context *ctx, int B, const double *mean_ylm, const double *cov_ylm,
                      const double *rTA1, int covpts, double *gp_mean, double *var, double *coef,
                      void *workspace, size_t workspace_bytes, void *stream);

size_t spb_flux_conditional_workspace_bytes(const spb_context *ctx, int B, int nt);
int spb_flux_conditional(spb_context *ctx, int B, int nt, const double *A, long long A_stride,
                         const double *mean_ylm, const double *cov_ylm, double *gp_mean, double *K,
                         int ldk, void *workspace, size_t workspace_bytes, void *stream);
/* Same, but only the lower triangle (and the diagonal) of K is written: for callers that factorise K
 * next (flux.py:335-343 feeding sp.py:1135-1176); the strict upper triangle is left untouched. */
int spb_flux_conditional_lower(spb_context *ctx, int B, int nt, const double *A, long long A_stride,
                         const double *mean_ylm, const double *cov_ylm, double *gp_mean, double *K,
                         int ldk, void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (a17, a19, a21) assemble the GP covariance that is factorised:
 *   marginal:  K_ij = cubic(|theta_i - theta_j|) from coef            (flux.py:256-276)
 *   normalised (normalized != 0): K <- (alpha/mu^2) K + z((alpha+beta) p p^T - alpha q q^T),
 *              mu = 1 + gp_mean, z = mean(K)/mu^2                      (sp.py:705-727, norm.py:26-44)
 *   K += data_cov (scalar | per-point vector | full matrix) + baseline_var (scalar | matrix)
 *                                                                      (sp.py:1135-1151)
 * data_kind / base_kind: 0 = scalar (pointer to 1 or B values, stride given), 1 = (nt) vector,
 * 2 = (nt,nt) matrix; strides are in elements between batch entries (0 = shared).
 *   z_out: (B) the normalisation series parameter (0 when not normalised).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int normalized;            /* sp.py:699-701 */
  int normalization_order;   /* defaults.py:19 (20) */
  double normalization_zmax; /* defaults.py:20 (0.023) */
  int data_kind;
  const double *data_cov;
  long long data_stride;
  int base_kind;
  const double *baseline_var;
  long long base_stride;
  int lower_only;            /* marginal assembly: write only K[i][j], j <= i (what the Cholesky
                                kernel reads); the strict upper triangle is left untouched */
  int defer;                 /* leave K RAW (lower triangle) and only produce the normalisation
                                scalars / row-sum vector in the workspace: the affine map and the
                                noise terms are applied by spb_cholesky_lnlike_affine.  Requires
                                lower_only and no full-matrix data_cov / baseline_var.            */
  /* (f-3) time-variable surfaces: the raw covariance is multiplied elementwise by the temporal
   * kernel k(|t_i - t_j|; tau) before the normalisation (temporal.py:8-16, sp.py:697-698).
   * Applied inside spb_assemble_marginal; the conditional branch scales K with
   * spb_temporal_scale before spb_assemble_conditional.                                       */
  int temporal_kind;         /* 0 none, 1 Matern-3/2, 2 squared exponential */
  const double *tau;         /* one value, or one per batch element (tau_stride 0 | 1) */
  long long tau_stride;
  /* Hint for the marginal assembly: the time stamps are equally spaced, t_k = t_0 + k uniform_dt (to
   * rounding).  The covariance then only depends on (i - j, number of period wraps between t_j and
   * t_i), so the cubic interpolant is tabulated once per sample for the 2 nt possible arguments and the
   * per-entry coefficient gathers disappear.  0 = general time stamps (the interpolant is evaluated per
   * entry).  The caller vouches for the spacing (sp.py checks it); values agree with the general path to
   * the rounding of |theta_i - theta_j| (1e-15 relative).                                          */
  double uniform_dt;
} spb_noise_model;

size_t spb_assemble_workspace_bytes(const spb_context *ctx, int B, int nt);
/* Where spb_assemble_* leaves q (B,nt) and scal (B,4) inside `workspace` (for spb_affine). */
void spb_assemble_workspace_layout(int B, int nt, void *workspace, double **q, double **scal);
int spb_assemble_marginal(spb_context *ctx, int B, int nt, const double *t, double period, int covpts,
                          const double *coef, const double *var, const double *gp_mean,
                          const spb_noise_model *noise, double *K, int ldk, double *z_out,
                          int32_t *info, void *workspace, size_t workspace_bytes, void *stream);
int spb_assemble_conditional(spb_context *ctx, int B, int nt, const double *gp_mean,
                             const spb_noise_model *noise, double *K, int ldk, double *z_out,
                             int32_t *info, void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (a20, a21) batched Cholesky + triangular solve + log-determinant -> log-likelihood.
 * Replaces cho_factor / cho_solve (math.py:75-100 -> LAPACK dpotrf/dtrtrs) and the lnlike
 * reduction of sp.py:1154-1188.
 *   K      : (B, nt, ldk) in: symmetric (lower triangle read); out: L in the lower triangle
 *   resid  : (B, M, ldr)  in: residual light curves r = flux - mean, one per ROW;
 *                         out: y = L^{-1} r   (resid_stride elements between batch entries)
 *   lnlike : (B) out = -1/2 sum y^2 - M sum log L_ii - 1/2 nt M log(2 pi); -inf when info[b] != 0
 *   quad   : (B, M) out or NULL: per-light-curve r^T K^{-1} r;  logdet: (B) or NULL: sum log L_ii
 * ldk and ldr must be even and the base pointers 16-byte aligned.
 * ------------------------------------------------------------------------------------------- */
int spb_cholesky_lnlike(spb_context *ctx, int B, int nt, double *K, int ldk, long long K_stride,
                        int M, double *resid, int ldr, long long resid_stride, double *lnlike,
                        double *quad, double *logdet, int32_t *info, void *stream);

/* Same factorisation with the LAST ASSEMBLY STEP FUSED INTO ITS LOADS: the kernel reads every entry
 * of the raw covariance exactly once (to initialise its accumulators) and applies there
 *     K'_ij = s1 K_ij + s2 (1 - q_i)(1 - q_j) - s3 q_i q_j + offset + [i == j] diag_i
 * i.e. the normalisation of sp.py:705-727 (s1 = alpha/mu^2, s2 = z (alpha+beta), s3 = z alpha, q the
 * scaled row sums; all produced by spb_assemble_* with noise->defer = 1), the scalar / per-point
 * data covariance and the scalar baseline variance of sp.py:1135-1151.  The dense matrix is then
 * written once (raw) and never re-read or re-written by an assembly pass.
 *   scal: (B,4) [s1, s2, s3, -] or NULL (identity);  q: (B,nt) or NULL
 *   diag: NULL | one value per batch element (diag_kind 0, diag_stride 0 or 1) | (nt) values
 *         (diag_kind 1, diag_stride 0 or nt);  offset: NULL | one value (offset_stride 0 or 1)   */
typedef struct {
  const double *scal;
  const double *q;
  const double *diag;
  int diag_kind;
  long long diag_stride;
  const double *offset;
  long long offset_stride;
} spb_affine;

int spb_cholesky_lnlike_affine(spb_context *ctx, int B, int nt, double *K, int ldk,
                               long long K_stride, const spb_affine *affine, int M, double *resid,
                               int ldr, long long resid_stride, double *lnlike, double *quad,
                               double *logdet, int32_t *info, void *stream);

/* The same log-likelihood with the panel updates of the factorisation evaluated on the INT8 tensor
 * cores (tcgen05.mma.kind::i8, accumulators in TMEM) from 7-bit digit planes of L -- an error-free
 * (Ozaki-style) emulation of the FP64 products.  `planes`: 78 = seven planes of balanced 8-bit digits
 * (55 bits relative to each row's maximum: results at the rounding-noise level of the FP64 kernel, 28
 * plane products -- the fastest), 8 or 87 = eight planes of 7-bit digits (56 bits, 36 products), 7 or 77 =
 * seven planes of 7-bit digits (49 bits).  Replaces the same
 * reference lines as spb_cholesky_lnlike_affine (math.py:75-100, sp.py:1154-1188).  Differences:
 *   K is only READ (the factor is not returned);  a diagonal lower bound diag(d) <= K' is needed to
 *   scale the right-hand-side rows (|y_k|^2 <= sum_k r_k^2 / d_k): d = `lambda_min` > 0 (e.g. the
 *   white-noise variance already added to K), or, when lambda_min <= 0, the affine diagonal
 *   affine->diag (`affine` may be NULL otherwise);  workspace of
 *   spb_cholesky_i8_workspace_bytes(B, nt, M, planes) bytes (digit planes + row scales);
 *   matrices whose digits overflow (SPB_INFO_I8_RANGE, never observed) are re-run through the FP64
 *   kernel, which overwrites THEIR K with L.
 * resid / lnlike / quad / logdet / info as spb_cholesky_lnlike.                                    */
size_t spb_cholesky_i8_workspace_bytes(int B, int nt, int M, int planes);
int spb_cholesky_lnlike_i8(spb_context *ctx, int B, int nt, double *K, int ldk, long long K_stride,
                           const spb_affine *affine, int M, double *resid, int ldr,
                           long long resid_stride, double *lnlike, double *quad, double *logdet,
                           int32_t *info, int planes, double lambda_min, void *workspace,
                           size_t workspace_bytes, void *stream);

/* Forward solve y = L^{-1} r for many right-hand sides against ONE factor, the RHS rows split
 * across the whole GPU (config "1 factorisation + 1024 RHS").  quad: (M) out.               */
int spb_cholesky_solve_rows(spb_context *ctx, int nt, const double *L, int ldk, int M, double *resid,
                            int ldr, double *quad, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Rank-31 conditional log-likelihood, linear in nt (DESIGN.md section 4.6).  Replaces, for a static
 * process conditional on inclination with scalar / per-point data_cov and a scalar / per-element
 * baseline_var, the dense chain flux.py:335-343 (K = A cov_ylm A^T), sp.py:705-727 (normalisation)
 * and sp.py:1052-1188 (noise terms, Cholesky, lnlike).  Every design-matrix row is
 * Phi(t) B_inc with Phi = [1, cos(m theta), sin(m theta)] (m = 1..15, theta = 2 pi frac(t / p)),
 * padded to 32 columns, so K = Phi C~ Phi^T + D with C~ of size 32.  Nothing of size nt^2 or
 * nt x 256 is formed; an element's result does not depend on the batch it is evaluated in.
 *
 * spb_lowrank_inclination : B_inc (I, 32, 256) for inclinations inc_rad (I) and the flux operator
 *                           rTA1 (rTA1_stride 0 | 256, as spb_design_matrix); workspace of
 *                           spb_lowrank_inclination_workspace_bytes(I) bytes, 16-byte aligned.
 * spb_lowrank_basis       : once per (t, period, data_cov), for any batch: the thin QR
 *                           D^-1/2 Phi = Q R (Householder TSQR; Q (nt, 32) with orthonormal
 *                           columns, R (32, 32), possibly singular) and
 *                           phi_aux (65) = [Phi^T 1 (32) | Phi(t_0) (32) | sum log D].
 *                           data_kind 0: data_cov is one value; 1: (nt) values.  nt >= 31.
 * spb_lowrank_lnlike      : per element, C = B_inc cov_ylm B_inc^T (Binc_stride 0 = shared, or
 *                           32 * 256), the GP mean (A mean_ylm)[0], the normalisation of
 *                           spb_assemble_* (noise->normalized, same z, SPB_INFO_Z_RANGE), the
 *                           baseline variance (noise->baseline_var, base_kind 0, base_stride 0 | 1),
 *                           N = I + R C~ R^T, its Cholesky factor (SPB_INFO_NOT_PD), and
 *                             lnlike = -1/2 sum_m (|y - Q w|^2 + w^T N^-1 w) - M/2 logdet K - nt M/2 log 2 pi
 *                           with y = D^-1/2 (flux - mean - baseline_mean), w = Q^T y; -inf where info != 0.
 *                           noise->data_kind / data_cov must be the ones given to spb_lowrank_basis
 *                           (data_stride 0).  flux: (M, ldf) shared (flux_stride 0) or per element
 *                           (flux_stride elements between elements); baseline_mean: NULL | one value
 *                           (bm_stride 0) | one per element (bm_stride 1).  quad (B, M), logdet (B)
 *                           (= logdet K), z_out (B) may be NULL.
 *
 * Predictive distribution (predict / sample_conditional) of an unnormalised process given one light curve:
 *   mean(ts) = gp_mean + Phi(ts) a,   cov(ts, ts) = Phi(ts) P Phi(ts)^T,   draws = mean + Phi(ts) G z1 + sqrt(eps) z2
 * spb_lowrank_posterior   : per element, from the operands of spb_lowrank_lnlike with M = 1 and a flux (nt)
 *                           shared by the batch (noise->normalized must be 0): a (B, 32) = C~ R^T N^-1 w,
 *                           P (B, 32, 32) = C~ - V^T V with V = L_N^-1 R C~, G (B, 32, 32) with G G^T = P
 *                           (eigenvectors scaled by sqrt(max(lambda, 0))), gp_mean (B).  info (B) in/out:
 *                           SPB_INFO_NOT_PD is set where N is not PD (a, P and G are then NaN) or where
 *                           P has an eigenvalue below -1e-10 max(lambda_max(P), max_k C~_kk) (G is then
 *                           NaN: no draws; a and P stay valid).  Other bits are kept.
 *                           Workspace of spb_lowrank_posterior_workspace_bytes(B, nt) bytes.
 * spb_lowrank_predict_eval: for nts time stamps t_sample and the posterior above: mean (B, nts); var (B, nts)
 *                           = diag(Phi P Phi^T) or NULL; cov (B, nts, ldc) = Phi P Phi^T or NULL (two DMMA
 *                           products; P 16-byte aligned); with nsamples > 0, draws (B, nsamples, nts) from
 *                           unit_normals (nsamples, 32 + nts) per draw [z1 (32) | z2 (nts)], shared by the
 *                           batch (un_stride 0) or per element (un_stride nsamples * (32 + nts)).  Workspace of
 *                           spb_lowrank_predict_eval_workspace_bytes(B, nts, nsamples, cov != NULL) bytes.
 *                           Nothing of size nts^2 is formed unless cov is requested.
 * ------------------------------------------------------------------------------------------- */
size_t spb_lowrank_inclination_workspace_bytes(const spb_context *ctx, int I);
int spb_lowrank_inclination(spb_context *ctx, int I, const double *inc_rad, const double *rTA1,
                            int rTA1_stride, double *Binc, void *workspace, size_t workspace_bytes,
                            void *stream);
size_t spb_lowrank_basis_workspace_bytes(const spb_context *ctx, int nt);
int spb_lowrank_basis(spb_context *ctx, int nt, const double *t, double period, int data_kind,
                      const double *data_cov, double *Q, double *R, double *phi_aux, void *workspace,
                      size_t workspace_bytes, void *stream);
size_t spb_lowrank_lnlike_workspace_bytes(const spb_context *ctx, int B, int M, int nt);
int spb_lowrank_lnlike(spb_context *ctx, int B, int nt, const double *Binc, long long Binc_stride,
                       const double *mean_ylm, const double *cov_ylm, const double *Q, const double *R,
                       const double *phi_aux, const spb_noise_model *noise, int M, const double *flux,
                       int ldf, long long flux_stride, const double *baseline_mean, long long bm_stride,
                       double *lnlike, double *quad, double *logdet, double *z_out, int32_t *info,
                       void *workspace, size_t workspace_bytes, void *stream);
size_t spb_lowrank_posterior_workspace_bytes(const spb_context *ctx, int B, int nt);
int spb_lowrank_posterior(spb_context *ctx, int B, int nt, const double *Binc, long long Binc_stride,
                          const double *mean_ylm, const double *cov_ylm, const double *Q, const double *R,
                          const double *phi_aux, const spb_noise_model *noise, const double *flux,
                          const double *baseline_mean, long long bm_stride, double *a, double *P, double *G,
                          double *gp_mean, int32_t *info, void *workspace, size_t workspace_bytes,
                          void *stream);
size_t spb_lowrank_predict_eval_workspace_bytes(const spb_context *ctx, int B, int nts, int nsamples,
                                                int full_cov);
int spb_lowrank_predict_eval(spb_context *ctx, int B, int nts, const double *t_sample, double period,
                             const double *a, const double *P, const double *G, const double *gp_mean,
                             int nsamples, const double *unit_normals, long long un_stride, double eps,
                             double *mean, double *var, double *cov, int ldc, double *draws, void *workspace,
                             size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------
 * (f-2) building blocks of predict / sample / sample_conditional / sample_ylm_conditional
 * (sp.py:518-641, 729-765, 767-1002).  Together with spb_cholesky_lnlike (whose "residual" rows are
 * any set of right-hand sides: out = L^{-1} rhs, one per row) they cover
 *   K_ts_t        spb_cross_marginal (marginalised, sp.py:887-902) | two spb_gemm_nt (sp.py:903-906)
 *   mu, K         mu = mean + V w,  K = K_ts_ts - V V^T  with V = (L^{-1} K_t_ts)^T, w = L^{-1}(y - mean)
 *   draws         spb_tril + spb_gemm_nt:  x = mu + L u
 *
 * spb_gemm_nt : C[b] = alpha A[b] Bm[b]^T + beta C[b];  A: (M, K) row-major (lda), Bm: (N, K)
 *               row-major (ldb), C: (M, N) (ldc); K, lda, ldb even, operands 16-byte aligned;
 *               batch strides in elements (0 = shared operand).
 * spb_tril    : zero the strict upper triangle of B (n x n) matrices (the Cholesky kernel leaves the
 *               upper triangle of its in-place factor untouched).
 * spb_cross_marginal : K_ts_t[b][i][j] = k_b(|theta(ts_i) - theta(t_j)|) + offset[b], the cubic
 *               interpolant of flux.py:256-276 on the coef table of spb_flux_marginal; columns
 *               nt..ld-1 are zeroed (ld even: the rows are right-hand sides of the solve); K_stride
 *               elements between batch entries.
 * ------------------------------------------------------------------------------------------- */
/* (f-3) K[b][i][j] = K[b][i][j] * k(|t1_i - t2_j|; tau_b) + offset_b  -- temporal.py:8-16 applied to
 * a (n1 x n2) block (sp.py:697-698 square, sp.py:893-895 rectangular K(ts, t) followed by the
 * baseline variance).  kind: 1 Matern-3/2, 2 squared exponential; offset may be NULL.          */
int spb_temporal_scale(spb_context *ctx, int B, int n1, int n2, const double *t1, const double *t2,
                       int kind, const double *tau, long long tau_stride, const double *offset,
                       long long offset_stride, double *K, int ld, long long K_stride, void *stream);

int spb_gemm_nt(spb_context *ctx, int batch, int M, int N, int K, double alpha, const double *A,
                int lda, long long strideA, const double *Bm, int ldb, long long strideB,
                double beta, double *C, int ldc, long long strideC, void *stream);
int spb_tril(spb_context *ctx, int B, int n, double *L, int ld, long long stride, void *stream);
int spb_cross_marginal(spb_context *ctx, int B, int nts, int nt, const double *ts, const double *t,
                       double period, int covpts, const double *coef, const double *offset,
                       long long offset_stride, double *K_ts_t, int ld, long long K_stride,
                       void *stream);

/* ---------------------------------------------------------------------------------------------
 * Measurement helpers (not part of the reference interface): FP64 tensor-pipe (DMMA) peak
 * micro-benchmark used as the roofline denominator; returns achieved TFLOP/s via *tflops_host.
 * ------------------------------------------------------------------------------------------- */
int spb_dmma_peak(spb_context *ctx, int iters, double *tflops_host, double *ms_host);
/* Run-time switches for A/B measurements and the bit-for-bit stress tests (defaults: everything on;
 * the environment variables SPB_NO_TMA / SPB_NO_CLUSTER set the defaults at spb_create):
 *   "cholesky_tma"     1 | 0   operand ring of the batched Cholesky fed by TMA | by cp.async
 *   "cholesky_cluster" 1 | 0   few matrices: one matrix per thread-block cluster | per CTA
 *   "moments_syrk_i8"  1 | 0   the FP64 GEMMs with an INT8-tensor-core form -- the second-moment SYRK of
 *                              spb_ylm_moments* (contrast.py:21-33) and, for nt >= 1024, the product
 *                              (A Sigma) A^T of spb_flux_conditional_lower (flux.py:335-343) -- on the INT8
 *                              tensor cores (exact 7 x 8-bit digit planes, tcgen05 + TMEM; cov_ylm within
 *                              1e-15 of its maximum of the FP64 result) | on the FP64 (DMMA) tensor cores;
 *                              on the INT8 form, entries of K that involve a row of A Sigma or A holding an
 *                              inf / NaN, or an entry of magnitude >= 1e300, are NaN (DESIGN.md 4.4);
 *                              environment default SPB_SYRK_I8                                     */
int spb_set_option(spb_context *ctx, const char *name, int value);
int spb_launch_count(const spb_context *ctx, long long *count_host);

#ifdef __cplusplus
}
#endif
#endif /* SPB200_H */
