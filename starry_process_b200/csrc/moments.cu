// Ylm moment integrals: (r, a, b, c, n) -> mean_ylm (256), cov_ylm (256 x 256), batched.
//
// Replaces the reference chain  SizeIntegral -> LatitudeIntegral -> LongitudeIntegral ->
// ContrastIntegral  (size.py:93-115; latitude.py:171-212 + ops/include/latitude.h:22-173;
// integrals.py:116-151; math.py:121-139 + ops/eigh/eigh.py:11-20; longitude.py:9-49;
// contrast.py:9-33).  Built with -fmad=false: the Beta-moment recurrences and the binomial double
// sums of latitude.h are reproduced with the reference's unfused operation order; bulk
// contractions use explicit fma().
//
// B200-first re-organisation (DESIGN.md "moments"):
//   K1  one CTA per hyperparameter sample:
//         spot profile -> q_size (16 values)                         size.py:45-53
//         Beta moments B(k), even/even binomial table term(2a,2b)    latitude.h:48-60,112-143
//           (the odd-index "F"/2F1 lane of latitude.h:63-109 only ever feeds entries that the
//            scatter of latitude.h:146-172 never reads -- l+m and l-m have equal parity -- so it
//            is not evaluated)
//         the 256x256 eigenproblem of math.py:121-139 is solved in the 31-dimensional range of
//         Q (constant orthonormal basis Z): S = Z^T Q Z, parallel cyclic Jacobi in shared
//         memory, eigenvalues <= 1e-15 clipped exactly as matrix_sqrt does
//         -> sqrtC_lat (256 x r), first moments through the folded tensors R0, t_lon
//   K2  sqrtC_lon = T_lon . sqrtC_lat  (integrals.py:133-138) as small DMMA GEMMs, the T_lon
//       fragments register-resident and re-used across 32 samples
//   K3  cov = (pi c)^2 n (sqrtC_lon sqrtC_lon^T - mom1 mom1^T) + diag(lambda) on the FP64 tensor
//       pipe (gemm_nt.cuh, lower tiles mirrored); the longitude re-factorisation of
//       integrals.py:144-150 only clips <=1e-15 modes of an explicitly PSD product and is skipped.
#include "gemm_nt.cuh"
#include "spb_tables.h"

namespace {

constexpr int NT1 = 256;
constexpr int JS = 33;  // Jacobi smem stride

struct K1Params {
  const double *r_deg, *a, *b, *c, *n;
  const double *Bp;      // (16,1000) spot profile operator (context table, or a per-process one for ydeg < 15)
  double abmin, lam, lbm;   // latitude.py:178-200: clamp of a, b; log_alpha_max; log_beta_max
  const double *dr_deg;  // (B) half-width of the uniform spot-radius prior, or nullptr (delta prior)
  double *E2;            // (B,16,16) spot-size second moment Etilde (dr prior only)
  int B;
  const double *tab;
  double *mom1;      // (B,256)   first moment before the contrast scaling
  double *mean_ylm;  // (B,256)
  double *S_lat;     // (B,256,32) sqrtC_lat, first rkeep columns non-zero
  double *scale;     // (B)       (pi c)^2 n
  int *rkeep;        // (B)
  int32_t *info;     // (B)
  double *Sred;      // (B,32,32) workspace: S = Z^T Q Z (K1a) -> V diag(sqrt w), compacted (K1b)
  double *qs;        // (B,16)    workspace: spot-size coefficients q_l
};

// K1 is split in three so that the latency-bound eigen-solve (a chain of FP64 divisions and square
// roots per Jacobi round, ~280 rounds) runs with ONE WARP per sample and a dozen samples in flight
// per SM, instead of one 256-thread CTA per sample with 15 of its 16 warps idle:
//   K1a (256 threads / sample)  profile, Beta moments, term table, S = Z^T Q Z, first moments
//   K1b (1 warp / sample)       cyclic Jacobi on S, clip, X = V diag(sqrt w)
//   K1c (256 threads / sample)  sqrtC_lat = q_l H X
struct K1Smem {
  double Zs[32][36];      // 32 (permuted) rows of the range basis Z at a time; first member:
                          // 16-byte aligned; pitch 36 = 4 (mod 16): conflict-free B fragments
  unsigned char kj[256], ki[256], kl[256];   // (m + l, l - m, l) of the permuted Ylm index
  double bprof[1000];
  double qs[16];
  double Bk[64];
  double tt[31][31];      // term(2a, 2b)
  double Y[256][33];      // Q Z
  double A[32][JS];       // S, symmetrised
  double V[32][JS];       // staging
  double m1lat[256];
};

constexpr int K1B_WARPS = 4;   // samples per CTA of the eigen-solve kernel
struct K1bWarp {
  double A[32][JS];       // Jacobi iterate
  double V[32][JS];       // eigenvectors
  int order[32];
  int rotated;
  int rk;
};

__device__ __forceinline__ void lm_of(int n, int &l, int &m) {
  l = (int)floor(sqrt((double)n));
  while (l * l > n) --l;
  while ((l + 1) * (l + 1) <= n) ++l;
  m = n - l * l - l;
}

// Ylm rows sorted by the parity of l - m (even first); see the Y = Q Z stage of K1a
__constant__ int k1_perm[256];
// term-table work list: k1_tt_sched[slot * 256 + tid] = a * 31 + b, or -1
__constant__ int k1_tt_sched[3 * 256];

int k1_upload_perm(int device) {
  static std::mutex mu;                 // concurrent first calls from several host threads
  std::lock_guard<std::mutex> lock(mu);
  static bool done_dev[64] = {false};   // __constant__ banks are per device
  bool &done = done_dev[device & 63];
  if (!done) {
    int perm[256], n = 0;
    for (int par = 0; par < 2; ++par)
      for (int l = 0; l <= SPB_LMAX; ++l)
        for (int m = -l; m <= l; ++m)
          if (((l - m) & 1) == par) perm[n++] = l * l + l + m;
    if (cudaMemcpyToSymbol(k1_perm, perm, sizeof(perm)) != cudaSuccess) return 1;
    // longest-processing-time-first assignment of the (a, b) pairs with a + b <= 30
    int sched[3 * 256], cnt[256] = {0};
    long load[256] = {0};
    for (int i = 0; i < 3 * 256; ++i) sched[i] = -1;
    bool used[961] = {false};
    for (;;) {
      int best = -1, bt = 0;
      for (int idx = 0; idx < 961; ++idx) {
        const int a2 = idx / 31, b2 = idx % 31;
        if (used[idx] || a2 + b2 > 30) continue;
        const int t = (a2 + 1) * (b2 + 1);
        if (t > bt) {
          bt = t;
          best = idx;
        }
      }
      if (best < 0) break;
      used[best] = true;
      int k = -1;
      for (int t = 0; t < 256; ++t)
        if (cnt[t] < 3 && (k < 0 || load[t] < load[k])) k = t;
      if (k < 0) return 1;
      sched[cnt[k] * 256 + k] = best;
      ++cnt[k];
      load[k] += bt;
    }
    if (cudaMemcpyToSymbol(k1_tt_sched, sched, sizeof(sched)) != cudaSuccess) return 1;
    done = true;
  }
  return 0;
}

// ---- sm.Bk (61 raw moments, or one of their derivative lanes) -> sm.tt (term table) -> sm.Y = Q Z
// -> sm.A = S = Z^T Q Z symmetrised (31 x 31 padded to 32).  Shared by the value kernel (K1a) and the
// tangent kernel (K1a_tan: the same linear chain applied to dB/dalpha, dB/dbeta).
__device__ __forceinline__ void k1a_S_from_moments(K1Smem &sm, const double *tab, int tid, int warp,
                                                    int lane) {
  // ---- term(2a, 2b) = sum_k1 sum_k2 C(a,k1) (-1)^k2 C(b,k2) B(k1+k2), latitude.h:112-143
  // The signed binomial products come from the LAT_FAC table (built on the host with the
  // reference's ratio recurrences, bit-identical to evaluating them here); the accumulation order
  // is the reference's.  The heavy (a, b) pairs are dealt out first so the tail is short.
  {
    // Work list: the 496 non-zero (a, b) pairs are dealt to the 256 threads longest-first (LPT,
    // k1_tt_sched): the longest chain is then the single heaviest pair (256 terms) instead of 374
    // terms.  The factors live in L2 (371 KB table) and are streamed ahead of the (serial,
    // reference-ordered) accumulation.
    const double *fac = tab + SPB_TAB_LAT_FAC;
    const double *facoff = tab + SPB_TAB_LAT_FACOFF;
    for (int idx = tid; idx < 31 * 31; idx += NT1) {
      const int a2 = idx / 31, b2 = idx % 31;
      if (a2 + b2 > 30) sm.tt[a2][b2] = 0.0;
    }
#pragma unroll 1
    for (int slot = 0; slot < 3; ++slot) {
      const int idx = k1_tt_sched[slot * 256 + tid];
      if (idx < 0) continue;
      const int a2 = idx / 31, b2 = idx % 31;
      double acc = 0.0;
      const double *f = fac + (int)facoff[idx];
      // the rows of the double sum are contiguous in the table: one flat, software-pipelined stream
      // (16 factors in flight while the previous 16 are accumulated in the reference's order)
      const int T = (a2 + 1) * (b2 + 1), w = b2 + 1;
      double nxt[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) nxt[u] = (u < T) ? __ldg(f + u) : 0.0;
      int k1 = 0, k2 = 0;
      for (int n0 = 0; n0 < T; n0 += 16) {
        double cur[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) cur[u] = nxt[u];
        if (n0 + 16 < T) {
#pragma unroll
          for (int u = 0; u < 16; ++u) nxt[u] = (n0 + 16 + u < T) ? __ldg(f + n0 + 16 + u) : 0.0;
        }
        // branch-free: slots past the end carry a zero factor (adding 0 is exact), and k1 + k2
        // stays inside Bk[64]
#pragma unroll
        for (int u = 0; u < 16; ++u) {
          acc += cur[u] * sm.Bk[k1 + k2];
          ++k2;
          const bool wrap = (k2 == w);
          k2 = wrap ? 0 : k2;
          k1 += wrap ? 1 : 0;
        }
      }
      sm.tt[a2][b2] = acc;
    }
  }
  __syncthreads();

  // ---- Y = Q Z with Q(n1,n2) = term(j1+j2, i1+i2) 2^-(l1+l2)   (latitude.h:146-172)
  // A (256 x 256) x (256 x 31) product on the FP64 tensor pipe.  Q(n1, n2) vanishes unless l - m
  // has the same parity for both indices, so rows AND the contraction index run in parity-sorted
  // order (k1_perm: 136 even, then 120 odd; 8-row tiles and 4-wide k-steps never straddle the
  // boundary) and every (m-tile, k-step) pair of opposite parity is skipped as a whole: half the
  // DMMAs.  The Q entries are generated in the A-fragment layout from the term table (the 2^-(l1+l2)
  // scaling is an exact exponent adjustment); Z is staged 32 permuted rows at a time, 36-double
  // pitch (conflict-free B fragments).
  int l1, m1;
  lm_of(tid, l1, m1);
  {
    // (j, i, l) of the permuted index tid, for the k side
    {
      int lp, mp;
      lm_of(k1_perm[tid], lp, mp);
      sm.kj[tid] = (unsigned char)(mp + lp);
      sm.ki[tid] = (unsigned char)(lp - mp);
      sm.kl[tid] = (unsigned char)lp;
    }
    const int g = lane >> 2, tg = lane & 3;
    int rj[4], ri[4], rl[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      int lp, mp;
      lm_of(k1_perm[32 * warp + 8 * q + g], lp, mp);
      rj[q] = mp + lp;
      ri[q] = lp - mp;
      rl[q] = lp;
    }
    double acc[4][4][2];
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) acc[q][nt][0] = acc[q][nt][1] = 0.0;
    const double *Z = tab + SPB_TAB_LAT_Z;
    for (int c0 = 0; c0 < 256; c0 += 32) {
      __syncthreads();
      for (int k = tid; k < 32 * 16; k += NT1) {
        const int r = k >> 4, c = k & 15;
        const double2 z2 = __ldg(reinterpret_cast<const double2 *>(Z + k1_perm[c0 + r] * 32) + c);
        *reinterpret_cast<double2 *>(&sm.Zs[r][2 * c]) = z2;
      }
      __syncthreads();
#pragma unroll
      for (int ks = 0; ks < 8; ++ks) {
        const int kp = c0 + 4 * ks;              // permuted contraction index of this k-step
        const bool k_even = kp < 136;
        const int kj = sm.kj[kp + tg], ki = sm.ki[kp + tg], kl = sm.kl[kp + tg];
        double bf[4];
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) bf[nt] = sm.Zs[4 * ks + tg][8 * nt + g];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const bool m_even = 32 * warp + 8 * q < 136;   // warp-uniform
          if (m_even == k_even) {
            const double t = sm.tt[(rj[q] + kj) >> 1][(ri[q] + ki) >> 1];
            // t * 2^-(l1 + l2): exact (ldexp in the scalar form)
            const double av = t * __hiloint2double((1023 - (rl[q] + kl)) << 20, 0);
#pragma unroll
            for (int nt = 0; nt < 4; ++nt) dmma_m8n8k4(acc[q][nt][0], acc[q][nt][1], av, bf[nt]);
          }
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int n1 = k1_perm[32 * warp + 8 * q + g];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const int col = 8 * nt + 2 * tg;
        sm.Y[n1][col] = acc[q][nt][0];
        if (col + 1 < 31) sm.Y[n1][col + 1] = acc[q][nt][1];
      }
    }
  }
  __syncthreads();
  // ---- S = Z^T Y (31 x 31), symmetrised, padded to 32: a (32 x 256) x (256 x 32) product on DMMA,
  // warp w owns the 8 x 16 block  rows 8 (w / 2),  columns 16 (w % 2)
  {
    const double *Z = tab + SPB_TAB_LAT_Z;
    const int g = lane >> 2, tg = lane & 3;
    const int a0 = 8 * (warp >> 1), c0 = 16 * (warp & 1);
    double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
#pragma unroll 1
    for (int k0 = 0; k0 < 256; k0 += 32) {
      double av[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) av[u] = __ldg(Z + (k0 + 4 * u + tg) * 32 + a0 + g);
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int k = k0 + 4 * u + tg;
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
          dmma_m8n8k4(acc[nt][0], acc[nt][1], av[u], sm.Y[k][c0 + 8 * nt + g]);
      }
    }
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int a = a0 + g, c = c0 + 8 * nt + 2 * tg + e;
        sm.V[a][c] = (a < 31 && c < 31) ? acc[nt][e] : 0.0;   // staging
      }
  }
  __syncthreads();
  for (int idx = tid; idx < 32 * 32; idx += NT1) {
    const int a = idx >> 5, c2 = idx & 31;
    sm.A[a][c2] = 0.5 * (sm.V[a][c2] + sm.V[c2][a]);
  }
  __syncthreads();
}

__global__ void __launch_bounds__(NT1, 2) moments_k1a(K1Params p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  K1Smem &sm = *reinterpret_cast<K1Smem *>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.x;
  const double *tab = p.tab;

  const double ang = 3.14159265358979323846 / 180.0;
  const double r = p.r_deg[b] * ang;
  double aa = p.a[b], bb = p.b[b];
  const double cc = p.c[b], nn = p.n[b];
  // CheckBoundsOp semantics (ops/exceptions.py:30-48; size.py:103, latitude.py:179-181,
  // contrast.py:15): the batched path flags the element instead of raising.
  const double tol = 1e-6;
  bool bad = !(r >= -tol && r <= 0.5 * 3.14159265358979323846 + tol) || !(aa >= -tol && aa <= 1 + tol) ||
             !(bb >= -tol && bb <= 1 + tol) || !(nn >= -tol);
  const bool has_dr = p.dr_deg != nullptr;
  const double dr = has_dr ? p.dr_deg[b] * ang : 0.0;
  if (has_dr) bad = bad || !(dr >= -tol && dr <= 0.5 * 3.14159265358979323846 + tol);   // size.py:120
  if (aa < p.abmin) aa = p.abmin;  // latitude.py:180-182 (abmin)
  if (bb < p.abmin) bb = p.abmin;

  // ---- spot profile, size.py:45-53 (sfac = 300); uniform radius prior: its mean over
  // [r - dr, r + dr], size.py:55-62 (Spot.get_e)
  for (int s = tid; s < 1000; s += NT1) {
    const double th = tab[SPB_TAB_THETA + s];
    if (has_dr) {
      const double chim = exp(300.0 * (r - dr - th));
      const double chip = exp(300.0 * (r + dr - th));
      sm.bprof[s] = 1.0 / (2 * dr * 300.0) * log((1 + chim) / (1 + chip));
    } else {
      const double z = 300.0 * (th - r);
      sm.bprof[s] = 1.0 / (1.0 + exp(-z)) - 1.0;
    }
  }
  __syncthreads();
  if (has_dr) {
    // ---- spot-size SECOND moment Etilde = Bp C Bp^T (16 x 16), size.py:64-86 (Spot.get_eigE before
    // its matrix square root): C_ij = E[b(theta_i) b(theta_j)] under the uniform radius prior, only
    // for theta < cutoff (r + dr), cutoff = 1.5.  The reference then carries sqrt(Etilde) through
    // the latitude / longitude integrals and re-compresses twice; all of it is linear in the second
    // moment, so the Ylm covariance is  Etilde[l1][l2] * (delta-prior second moment with q_l = 1)
    // -- applied as a Hadamard factor in the SYRK epilogue (measured against the unmodified
    // reference: 5e-14 relative on cov_ylm; its 1e-15 eigenvalue clips are below that).
    //   W = C Bp^T in 256-row chunks (one row per thread, staged in sm.Y), then Etilde += Bp W.
    int kmax = 0;   // numpy argmax of a boolean array: first True, 0 when none
    for (int s = 0; s < 1000; ++s)
      if (tab[SPB_TAB_THETA + s] / (r + dr) > 1.5) {
        kmax = s;
        break;
      }
    double *Wst = &sm.Y[0][0];          // [256][16] staging (Y is not live yet)
    double *Bst = Wst + 256 * 16;       // [16][64]  Bp tile
    double eacc = 0.0;                  // thread (l1, l2) = (tid / 16, tid % 16)
    const double inv2 = 1.0 / (2 * dr * 300.0);
    for (int i0 = 0; i0 < kmax; i0 += NT1) {
      const int i = i0 + tid;
      const bool live = i < kmax;
      const double ti = live ? tab[SPB_TAB_THETA + i] : 0.0;
      double term_i = 0.0, diag_i = 0.0;
      if (live) {
        const double chim = exp(300.0 * (r - dr - ti)), chip = exp(300.0 * (r + dr - ti));
        term_i = log(1 + chim) - log(1 + chip);
        diag_i = 1 / (1 + chip) + chim / (1 + chim) - term_i - 1;
      }
      double wrow[16];
#pragma unroll
      for (int l = 0; l < 16; ++l) wrow[l] = 0.0;
      for (int j0 = 0; j0 < kmax; j0 += 64) {
        __syncthreads();
        for (int k = tid; k < 16 * 64; k += NT1) {
          const int l = k >> 6, jj = k & 63;
          Bst[k] = (j0 + jj < kmax) ? p.Bp[(size_t)l * 1000 + j0 + jj] : 0.0;
        }
        __syncthreads();
        if (live) {
          const int jn = min(64, kmax - j0);
          for (int jj = 0; jj < jn; ++jj) {
            const int j = j0 + jj;
            const double tj = tab[SPB_TAB_THETA + j];
            double cij;
            if (j == i) {
              cij = diag_i;
            } else {
              const double chim = exp(300.0 * (r - dr - tj)), chip = exp(300.0 * (r + dr - tj));
              const double term_j = log(1 + chim) - log(1 + chip);
              const double ex = exp(300.0 * (tj - ti));
              cij = (ex * term_j - term_i) / (1 - ex + 1.0e-15);
            }
            cij *= inv2;
#pragma unroll
            for (int l = 0; l < 16; ++l) wrow[l] = fma(cij, Bst[l * 64 + jj], wrow[l]);
          }
        }
      }
      __syncthreads();
#pragma unroll
      for (int l = 0; l < 16; ++l) Wst[tid * 16 + l] = live ? wrow[l] : 0.0;
      __syncthreads();
      {
        const int l1 = tid >> 4, l2 = tid & 15;
        const int in = min(NT1, kmax - i0);
        const double *bp = p.Bp + (size_t)l1 * 1000 + i0;
        for (int ii = 0; ii < in; ++ii) eacc = fma(bp[ii], Wst[ii * 16 + l2], eacc);
      }
    }
    p.E2[(size_t)b * 256 + tid] = bad ? NAN : eacc;
    __syncthreads();
  }
  for (int row = warp; row < 16; row += NT1 / 32) {
    const double *bp = p.Bp + (size_t)row * 1000;
    double acc = 0.0;
    for (int s = lane; s < 1000; s += 32) acc = fma(bp[s], sm.bprof[s], acc);
    acc = warp_sum(acc);
    if (lane == 0) sm.qs[row] = acc;
  }

  // ---- Beta moments, latitude.py:197-200 and latitude.h:48-60
  if (tid == 0) {
    const double alpha0 = exp(aa * p.lam);
    const double beta0 = exp(log(0.5) + bb * (p.lbm - log(0.5)));
    const double alpha = alpha0 > 0.0 ? alpha0 : 0.0;  // ops/latitude/latitude.cc:47-48
    const double beta = beta0 > 0.0 ? beta0 : 0.0;
    sm.Bk[0] = 1.0;
    for (int k = 1; k < 61; ++k) {
      const double c1 = 1.0 / (alpha + beta + k - 1.0);
      const double c2 = (alpha + k - 1.0) * c1;
      sm.Bk[k] = c2 * sm.Bk[k - 1];
    }
  }
  __syncthreads();

  k1a_S_from_moments(sm, tab, tid, warp, lane);
  int l1, m1;
  lm_of(tid, l1, m1);
  // S goes to the eigen-solve kernel
  for (int idx = tid; idx < 32 * 32; idx += NT1) p.Sred[(size_t)b * 1024 + idx] = sm.A[idx >> 5][idx & 31];
  if (tid < 16) p.qs[(size_t)b * 16 + tid] = sm.qs[tid];
  const double qsl = sm.qs[l1];

  // ---- first moments (integrals.py:126-131): latitude then longitude
  {
    const int w = 2 * l1 + 1;
    const double *R0 = tab + SPB_TAB_LAT_R0 + (size_t)(l1 * (2 * l1 - 1) * (2 * l1 + 1)) / 3 +
                       (size_t)(m1 + l1) * w;
    double acc = 0.0;
    for (int k = 0; k < w; ++k) {
      const int I = 2 * l1 - k;
      double ql = 0.0;
      if (!(k & 1)) ql = ldexp(sm.tt[k >> 1][I >> 1], -l1);
      acc = fma(R0[k], ql, acc);
    }
    sm.m1lat[tid] = qsl * acc;
  }
  __syncthreads();
  {
    const int w = 2 * l1 + 1;
    const double *T1 = tab + SPB_TAB_LON_T1 + (size_t)(l1 * (2 * l1 - 1) * (2 * l1 + 1)) / 3 +
                       (size_t)(m1 + l1) * w;
    double acc = 0.0;
    for (int m = 0; m < w; ++m) acc = fma(T1[m], sm.m1lat[l1 * l1 + m], acc);
    const double pi = 3.14159265358979323846;
    p.mom1[(size_t)b * 256 + tid] = bad ? NAN : acc;
    p.mean_ylm[(size_t)b * 256 + tid] = bad ? NAN : (pi * cc * nn) * acc;  // contrast.py:22
  }
  if (tid == 0) {
    const double pi = 3.14159265358979323846;
    p.scale[b] = (pi * cc) * (pi * cc) * nn;  // contrast.py:23-25
    p.info[b] = bad ? SPB_INFO_BOUNDS : 0;
  }
}



// ------------------------------------------------------------------------------------------
// Tangent lanes for the gradient of the log-likelihood (SURVEY.md 8(f) rank 4).  The only
// non-linear, hyperparameter-dependent inputs of the Ylm moments are the Beta moments B(k) of the
// latitude distribution and the spot profile; everything downstream of (S = Z^T Q Z, q_l, mom1) is
// linear / quadratic.  K1a_tan evaluates, per sample,
//   dS/da, dS/db   : the K1a chain applied to the derivative lanes dB/dalpha, dB/dbeta of
//                    ops/include/latitude.h:48-60 (chain factors d alpha / d a = 10 alpha,
//                    d beta / d b = (10 - ln 1/2) beta; zero below the abmin clamp)
//   dq_l / dr      : Bp . d b(theta; r) / d r   (size.py:45-53), per DEGREE of r
//   d mom1 / d(r, a, b)
// and moments_expand_kernel turns them into +-eps perturbed copies of (S, q, mom1) that run through
// the unchanged K1b / K1c / K2 / SYRK pipeline.  Because that pipeline is linear in S and quadratic
// in (q, mom1), the central difference of its outputs along a tangent is the exact directional
// derivative (no truncation error); the reference instead back-propagates through eigh
// (ops/include/eigh.h:19-65, integrals.py:133-151).
// ------------------------------------------------------------------------------------------
struct K1TanParams {
  const double *r_deg, *a, *b;
  const double *Bp;
  double abmin, lam, lbm;
  int B;
  const double *tab;
  double *dS;     // (B,2,32,32)
  double *dqs;    // (B,16)
  double *dmom1;  // (B,3,256): r, a, b
};

__global__ void __launch_bounds__(NT1, 2) moments_k1a_tan(K1TanParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  K1Smem &sm = *reinterpret_cast<K1Smem *>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.x;
  const double *tab = p.tab;
  const double ang = 3.14159265358979323846 / 180.0;
  const double r = p.r_deg[b] * ang;
  double aa = p.a[b], bb = p.b[b];
  const bool a_free = aa > p.abmin, b_free = bb > p.abmin;   // latitude.py:180-182 (abmin clamp)
  if (!a_free) aa = p.abmin;
  if (!b_free) bb = p.abmin;
  __shared__ double dqs_s[16];
  __shared__ double lanes[3][64];   // B, dB/dalpha, dB/dbeta
  __shared__ double chain[2];

  // ---- spot profile and its r-derivative: b = sigma(z) - 1, z = 300 (theta - r),
  // d b / d r = -300 sigma (1 - sigma)
  for (int pass = 0; pass < 2; ++pass) {
    for (int s = tid; s < 1000; s += NT1) {
      const double z = 300.0 * (tab[SPB_TAB_THETA + s] - r);
      const double sg = 1.0 / (1.0 + exp(-z));
      sm.bprof[s] = pass == 0 ? sg - 1.0 : -300.0 * sg * (1.0 - sg) * ang;
    }
    __syncthreads();
    for (int row = warp; row < 16; row += NT1 / 32) {
      const double *bp = p.Bp + (size_t)row * 1000;
      double acc = 0.0;
      for (int s = lane; s < 1000; s += 32) acc = fma(bp[s], sm.bprof[s], acc);
      acc = warp_sum(acc);
      if (lane == 0) (pass == 0 ? sm.qs[row] : dqs_s[row]) = acc;
    }
    __syncthreads();
  }
  if (tid < 16) p.dqs[(size_t)b * 16 + tid] = dqs_s[tid];

  // ---- Beta moments and their derivative lanes, latitude.h:48-60
  if (tid == 0) {
    const double alpha0 = exp(aa * p.lam);
    const double beta0 = exp(log(0.5) + bb * (p.lbm - log(0.5)));
    const double alpha = alpha0 > 0.0 ? alpha0 : 0.0;
    const double beta = beta0 > 0.0 ? beta0 : 0.0;
    chain[0] = a_free ? p.lam * alpha : 0.0;
    chain[1] = b_free ? (p.lbm - log(0.5)) * beta : 0.0;
    lanes[0][0] = 1.0;
    lanes[1][0] = 0.0;
    lanes[2][0] = 0.0;
    for (int k = 1; k < 61; ++k) {
      const double c1 = 1.0 / (alpha + beta + k - 1.0);
      const double c2 = (alpha + k - 1.0) * c1;
      const double c3 = beta * c1 * c1;
      const double c4 = (1 - k - alpha) * c1 * c1;
      lanes[0][k] = c2 * lanes[0][k - 1];
      lanes[1][k] = c3 * lanes[0][k - 1] + c2 * lanes[1][k - 1];
      lanes[2][k] = c4 * lanes[0][k - 1] + c2 * lanes[2][k - 1];
    }
  }
  __syncthreads();

  int l1, m1;
  lm_of(tid, l1, m1);
  const int w = 2 * l1 + 1;
  const double *R0 = tab + SPB_TAB_LAT_R0 + (size_t)(l1 * (2 * l1 - 1) * (2 * l1 + 1)) / 3 +
                     (size_t)(m1 + l1) * w;
  const double *T1 = tab + SPB_TAB_LON_T1 + (size_t)(l1 * (2 * l1 - 1) * (2 * l1 + 1)) / 3 +
                     (size_t)(m1 + l1) * w;
  double glat[3];   // (R0 . q_lat) of this Ylm index for the three lanes
  for (int v = 0; v < 3; ++v) {
    if (tid < 64) sm.Bk[tid] = lanes[v][tid];
    __syncthreads();
    k1a_S_from_moments(sm, tab, tid, warp, lane);   // -> sm.tt, sm.A (ends with a barrier)
    if (v > 0) {
      const double f = chain[v - 1];
      for (int idx = tid; idx < 32 * 32; idx += NT1)
        p.dS[((size_t)b * 2 + (v - 1)) * 1024 + idx] = f * sm.A[idx >> 5][idx & 31];
    }
    double acc = 0.0;
    for (int k = 0; k < w; ++k) {
      const int I = 2 * l1 - k;
      double ql = 0.0;
      if (!(k & 1)) ql = ldexp(sm.tt[k >> 1][I >> 1], -l1);
      acc = fma(R0[k], ql, acc);
    }
    glat[v] = acc;
    __syncthreads();
  }
  // ---- d mom1: longitude first-moment map applied to the three latitude tangents
  for (int d = 0; d < 3; ++d) {
    double val;
    if (d == 0) val = dqs_s[l1] * glat[0];
    else val = chain[d - 1] * sm.qs[l1] * glat[d];
    sm.m1lat[tid] = val;
    __syncthreads();
    double acc = 0.0;
    for (int m = 0; m < w; ++m) acc = fma(T1[m], sm.m1lat[l1 * l1 + m], acc);
    p.dmom1[((size_t)b * 3 + d) * 256 + tid] = acc;
    __syncthreads();
  }
}

// Variants of the moment inputs, variant-major: slot v * B + b, v = 0 base (already written by K1a),
// 1,2: r +-; 3,4: a +-; 5,6: b +-.  eps[d * B + b] is the absolute step of direction d (r in
// degrees): rel_step times the ratio of the largest base entry to the largest tangent entry.
struct ExpandParams {
  int B;
  double rel_step;
  const double *c, *n;
  const double *dS, *dqs, *dmom1;
  double *Sred, *qs, *mom1, *mean_ylm, *scale;
  int32_t *info;
  double *eps;   // (5, B): r, a, b, c, n
};

__global__ void __launch_bounds__(256) moments_expand_kernel(ExpandParams p) {
  __shared__ double red[8];
  __shared__ double mx[5];
  const int b = blockIdx.x, tid = threadIdx.x, B = p.B;
  auto block_max = [&](double v) {
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    if ((tid & 31) == 0) red[tid >> 5] = v;
    __syncthreads();
    double t = 0.0;
    for (int k = 0; k < 8; ++k) t = fmax(t, red[k]);
    return t;
  };
  const double *S0 = p.Sred + (size_t)b * 1024;
  const double *Sa = p.dS + ((size_t)b * 2 + 0) * 1024, *Sb = p.dS + ((size_t)b * 2 + 1) * 1024;
  double m0 = 0.0, ma = 0.0, mb = 0.0;
  for (int i = tid; i < 1024; i += 256) {
    m0 = fmax(m0, fabs(S0[i]));
    ma = fmax(ma, fabs(Sa[i]));
    mb = fmax(mb, fabs(Sb[i]));
  }
  m0 = block_max(m0);
  ma = block_max(ma);
  mb = block_max(mb);
  double q0 = tid < 16 ? fabs(p.qs[(size_t)b * 16 + tid]) : 0.0;
  double q1 = tid < 16 ? fabs(p.dqs[(size_t)b * 16 + tid]) : 0.0;
  q0 = block_max(q0);
  q1 = block_max(q1);
  if (tid == 0) {
    mx[0] = (q1 > 0.0) ? p.rel_step * q0 / q1 : 1.0;
    mx[1] = (ma > 0.0) ? p.rel_step * m0 / ma : 1.0;
    mx[2] = (mb > 0.0) ? p.rel_step * m0 / mb : 1.0;
    mx[3] = p.rel_step * fabs(p.c[b]);
    mx[4] = p.rel_step * fabs(p.n[b]);
    if (!(mx[3] > 0.0)) mx[3] = p.rel_step;
    if (!(mx[4] > 0.0)) mx[4] = p.rel_step;
    for (int d = 0; d < 5; ++d) p.eps[(size_t)d * B + b] = mx[d];
  }
  __syncthreads();
  const double pi = 3.14159265358979323846;
  const double fac = pi * p.c[b] * p.n[b];
  for (int v = 1; v < 7; ++v) {
    const int d = (v - 1) >> 1;
    const double e = ((v - 1) & 1) ? -mx[d] : mx[d];
    const size_t slot = (size_t)v * B + b;
    for (int i = tid; i < 1024; i += 256) {
      double val = S0[i];
      if (d == 1) val = fma(e, Sa[i], val);
      if (d == 2) val = fma(e, Sb[i], val);
      p.Sred[slot * 1024 + i] = val;
    }
    if (tid < 16) {
      double val = p.qs[(size_t)b * 16 + tid];
      if (d == 0) val = fma(e, p.dqs[(size_t)b * 16 + tid], val);
      p.qs[slot * 16 + tid] = val;
    }
    {
      const double m1v = fma(e, p.dmom1[((size_t)b * 3 + d) * 256 + tid], p.mom1[(size_t)b * 256 + tid]);
      p.mom1[slot * 256 + tid] = m1v;
      p.mean_ylm[slot * 256 + tid] = fac * m1v;
    }
    if (tid == 0) {
      p.scale[slot] = p.scale[b];
      p.info[slot] = p.info[b];
    }
  }
}

// Variants 7..10 (c +-, n +-): Sigma = (pi c)^2 n C + lambda and mean = pi c n mom1 are monomials in
// (c, n), so these are rescalings of the base moments (contrast.py:20-33).
__global__ void __launch_bounds__(256) moments_scale_variants_kernel(int B, const double *c,
                                                                     const double *n, const double *eps,
                                                                     const double *lambda,
                                                                     double *mean_ylm, double *cov_ylm) {
  const int b = blockIdx.x, v = 7 + blockIdx.y, tid = threadIdx.x;
  const int d = 3 + ((v - 7) >> 1);
  const double e = ((v - 7) & 1) ? -eps[(size_t)d * B + b] : eps[(size_t)d * B + b];
  const double cb = c[b], nb = n[b];
  const double c2 = (d == 3) ? cb + e : cb, n2 = (d == 4) ? nb + e : nb;
  const double fm = (c2 * n2) / (cb * nb);
  const double fc = (c2 * c2 * n2) / (cb * cb * nb);
  const size_t slot = (size_t)v * B + b;
  mean_ylm[slot * 256 + tid] = fm * mean_ylm[(size_t)b * 256 + tid];
  const double *src = cov_ylm + (size_t)b * 65536;
  double *dst = cov_ylm + slot * 65536;
  for (int i = tid; i < 65536; i += 256) {
    const int row = i >> 8, col = i & 255;
    const double lam = (row == col) ? lambda[row] : 0.0;
    dst[i] = fma(fc, src[i] - lam, lam);
  }
}

__device__ __forceinline__ double jrcp(double x) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  double e = fma(-x, y, 1.0);
  y = fma(y, e, y);
  e = fma(-x, y, 1.0);
  return fma(y, e, y);
}
__device__ __forceinline__ double jrsqrt(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  double e = fma(-x * y, y, 1.0);
  y = fma(0.5 * y, e, y);
  e = fma(-x * y, y, 1.0);
  return fma(0.5 * y, e, y);
}

// ---- K1b: one warp per sample.  Same round-robin ordering, thresholds and clipping as the
// CTA-wide version it replaces; the 16 disjoint rotations of
// a round are computed by lanes 0-15, the row phase runs one column per lane and the column phase
// one row per lane (both conflict-free with the 33-double stride), with __syncwarp in between.
__global__ void __launch_bounds__(32 * K1B_WARPS) moments_k1b(K1Params p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * K1B_WARPS + warp;
  if (b >= p.B) return;
  K1bWarp &sm = reinterpret_cast<K1bWarp *>(smem_raw)[warp];
  double *Sg = p.Sred + (size_t)b * 1024;
  for (int a = 0; a < 32; ++a) {
    sm.A[a][lane] = Sg[a * 32 + lane];
    sm.V[a][lane] = (a == lane) ? 1.0 : 0.0;
  }
  __syncwarp();
  double amax = 0.0;
  for (int a = 0; a < 31; ++a) amax = fmax(amax, fabs(sm.A[a][a]));
  const double rot_tol = 1e-20 * amax;
  bool converged = false;
  for (int sweep = 0; sweep < 16 && !converged; ++sweep) {
    if (lane == 0) sm.rotated = 0;
    __syncwarp();
    for (int rnd = 0; rnd < 31; ++rnd) {
      double cth_l = 1.0, sth_l = 0.0;
      if (lane < 16) {
        int pi, qi;
        if (lane == 0) {
          pi = rnd;
          qi = 31;
        } else {
          pi = (rnd + lane) % 31;
          qi = (rnd - lane + 31) % 31;
        }
        if (pi > qi) {
          const int t = pi;
          pi = qi;
          qi = t;
        }
        const double apq = sm.A[pi][qi];
        const double app = sm.A[pi][pi], aqq = sm.A[qi][qi];
        // rotate unless a_pq is negligible against sqrt(a_pp a_qq) (relative criterion for PSD
        // matrices) or against the absolute floor 1e-20 max|a_ii| -- compared squared, no sqrt
        const double thr2 = fmax(rot_tol * rot_tol, 1.6e-29 * fabs(app * aqq));
        if (apq * apq > thr2 && qi < 31) {
          // Jacobi rotation  t = sgn(tau) / (|tau| + sqrt(1 + tau^2)),  tau = (a_qq - a_pp) / (2 a_pq),
          // written as t = sgn |o| / (|d| + sqrt(d^2 + o^2)) with d = a_qq - a_pp, o = 2 a_pq, and
          // evaluated with MUFU-seeded reciprocal / reciprocal square root (two Newton steps each):
          // the round's critical path is this chain, and IEEE division and square root cost ~15
          // dependent FP64 instructions apiece where these cost five.
          const double d = aqq - app, o = 2.0 * apq;
          const double r2 = fma(d, d, o * o);
          const double h = r2 * jrsqrt(r2);
          const double sg = (((d >= 0.0) == (o >= 0.0)) || d == 0.0) ? 1.0 : -1.0;   // sgn(tau), tau = d / o
          const double t = sg * fabs(o) * jrcp(fabs(d) + h);
          cth_l = jrsqrt(fma(t, t, 1.0));
          sth_l = t * cth_l;
          sm.rotated = 1;
        }
      }
      // pair indices are lane-invariant functions of (rnd, k); (c, s) come from lane k by shuffle:
      // no shared-memory broadcast loads in the update phases (they were half of the LSU traffic
      // that bounds this kernel)
      int P[16], Q[16];
      double C[16], S[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        int pk, qk;
        if (k == 0) {
          pk = rnd;
          qk = 31;
        } else {
          pk = rnd + k;
          pk -= (pk >= 31) ? 31 : 0;
          qk = rnd - k + 31;
          qk -= (qk >= 31) ? 31 : 0;
        }
        P[k] = min(pk, qk);
        Q[k] = max(pk, qk);
        C[k] = __shfl_sync(0xffffffffu, cth_l, k);
        S[k] = __shfl_sync(0xffffffffu, sth_l, k);
      }
      // The 16 rotations of a round touch disjoint row (column) pairs, so all operands are loaded
      // first and all results stored last: the compiler cannot prove the shared-memory accesses of
      // different rotations independent, and would otherwise serialise load -> FP64 -> store 16x.
      // rows: A <- J^T A   (lane = column)
      {
        double ap[16], aq[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          ap[k] = sm.A[P[k]][lane];
          aq[k] = sm.A[Q[k]][lane];
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const double cth = C[k], sth = S[k];
          const double np_ = cth * ap[k] - sth * aq[k];
          const double nq_ = sth * ap[k] + cth * aq[k];
          ap[k] = np_;
          aq[k] = nq_;
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          sm.A[P[k]][lane] = ap[k];
          sm.A[Q[k]][lane] = aq[k];
        }
      }
      __syncwarp();
      // columns: A <- A J, V <- V J   (lane = row)
      {
        double ap[16], aq[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          ap[k] = sm.A[lane][P[k]];
          aq[k] = sm.A[lane][Q[k]];
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const double cth = C[k], sth = S[k];
          const double np_ = cth * ap[k] - sth * aq[k];
          const double nq_ = sth * ap[k] + cth * aq[k];
          ap[k] = np_;
          aq[k] = nq_;
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          sm.A[lane][P[k]] = ap[k];
          sm.A[lane][Q[k]] = aq[k];
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          ap[k] = sm.V[lane][P[k]];
          aq[k] = sm.V[lane][Q[k]];
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const double cth = C[k], sth = S[k];
          const double np_ = cth * ap[k] - sth * aq[k];
          const double nq_ = sth * ap[k] + cth * aq[k];
          ap[k] = np_;
          aq[k] = nq_;
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          sm.V[lane][P[k]] = ap[k];
          sm.V[lane][Q[k]] = aq[k];
        }
      }
      __syncwarp();
    }
    converged = (sm.rotated == 0);
    __syncwarp();
  }
  if (!converged) {
    // rotations at the rounding floor can keep a sweep "busy"; the solve has failed only if a
    // significant off-diagonal element survives
    double offmax = 0.0;
    for (int a = 0; a < 31; ++a)
      for (int c2 = a + 1; c2 < 31; ++c2) offmax = fmax(offmax, fabs(sm.A[a][c2]));
    converged = offmax <= 1e-13 * amax;
  }
  // ---- matrix_sqrt clip (math.py:133-136): keep w > 1e-15, compact kept modes to the front
  if (lane == 0) {
    int rk = 0;
    for (int e = 0; e < 31; ++e)
      if (sm.A[e][e] > 1e-15) sm.order[rk++] = e;
    sm.rk = rk;
  }
  __syncwarp();
  const int rk = sm.rk;
  for (int a = 0; a < 32; ++a) {   // lane = kept mode e
    double v = 0.0;
    if (lane < rk && a < 31) {
      const int src = sm.order[lane];
      v = sm.V[a][src] * sqrt(sm.A[src][src]);
    }
    Sg[a * 32 + lane] = v;
  }
  if (lane == 0) {
    p.rkeep[b] = rk;
    if (!converged) atomicOr(&p.info[b], SPB_INFO_EIG_NOCONV);
  }
}

// ---- K1c: sqrtC_lat row (integrals.py:133-138 with eigE = q_size column, T = R_lat U)
__global__ void __launch_bounds__(NT1) moments_k1c(K1Params p) {
  __shared__ double Xs[32][JS];
  const int tid = threadIdx.x, b = blockIdx.x;
  for (int idx = tid; idx < 1024; idx += NT1) Xs[idx >> 5][idx & 31] = p.Sred[(size_t)b * 1024 + idx];
  __syncthreads();
  int l1, m1;
  lm_of(tid, l1, m1);
  // dr prior: the spot-size factor enters as Etilde[l1][l2] in the SYRK epilogue instead
  const double qsl = p.dr_deg ? 1.0 : p.qs[(size_t)b * 16 + l1];
  const bool bad = (p.info[b] & SPB_INFO_BOUNDS) != 0;
  const double *H = p.tab + SPB_TAB_LAT_H + (size_t)tid * 32;
  double out[32];
#pragma unroll
  for (int e = 0; e < 32; ++e) out[e] = 0.0;
  for (int a = 0; a < 31; ++a) {
    const double h = H[a];
#pragma unroll
    for (int e = 0; e < 32; ++e) out[e] = fma(h, Xs[a][e], out[e]);
  }
  double *dst = p.S_lat + ((size_t)b * 256 + tid) * 32;
#pragma unroll
  for (int e = 0; e < 32; ++e) dst[e] = bad ? NAN : qsl * out[e];
}

// ------------------------------------------------------------------------------------------
// K2: X[b][(l,m')][e2][e] = sum_m T_lon[l][m'][e2][m] * S_lat[b][(l,m)][e]
// grid.x = (l, 256-row chunk) work list, grid.y = groups of 32 samples
// ------------------------------------------------------------------------------------------
struct K2Item {
  int l, row0, nrows, toff;
};
__constant__ K2Item k2_items[64];

struct K2Params {
  const double *tab;
  const double *S_lat;  // (B,256,32)
  const int *rkeep;
  double *X;  // (B,256,31*32)
  int B;
};

constexpr int K2_GROUP = 32;
constexpr int K2_SP = 36;   // shared-memory pitch of the S_lat slice: 36 = 4 (mod 16) makes the
                            // (k = tg, n = g) fragment loads of m8n8k4 conflict-free

// For each l this is a small GEMM  X_l (31 w x rk) = T_l (31 w x w) . S_l (w x rk),  w = 2l + 1, and it
// runs on the FP64 tensor pipe: a warp owns 32 rows (4 m-tiles) of the constant tensor and keeps
// their A fragments IN REGISTERS for all 32 samples of its group (the tensor never goes through
// shared memory); per sample only the S_lat slice is staged (double-buffered, one barrier) and
// read as B fragments.  k is padded to a multiple of 4 and the kept eigen-columns to n-tiles of 8;
// only the first rk4 = 4 ceil(rkeep / 4) columns are written (the SYRK never reads the rest).
// The scalar-FMA form of this kernel was shared-memory-LSU-bound (one wavefront per ~4 FMAs).
__global__ void __launch_bounds__(256, 2) moments_k2(K2Params p) {
  __shared__ __align__(16) double Ssh[2][32][K2_SP];
  const K2Item it = k2_items[blockIdx.x];
  const int w = 2 * it.l + 1;
  const int nkk = (w + 3) >> 2;   // k-steps of 4
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, tg = lane & 3;
  const double *Tl = p.tab + SPB_TAB_LON_T + it.toff + (size_t)it.row0 * w;
  // A fragments: a[mt][kk] = T[row = 32 warp + 8 mt + g][k = 4 kk + tg]
  double a[4][8];
#pragma unroll
  for (int mt = 0; mt < 4; ++mt) {
    const int r = 32 * warp + 8 * mt + g;
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
      const int k = 4 * kk + tg;
      a[mt][kk] = (r < it.nrows && k < w) ? __ldg(Tl + (size_t)r * w + k) : 0.0;
    }
  }
  const bool warp_live = 32 * warp < it.nrows;
  const int b0 = blockIdx.y * K2_GROUP;
  const int b1 = min(p.B, b0 + K2_GROUP);
  for (int b = b0; b < b1; ++b) {
    double(*Sb)[K2_SP] = Ssh[(b - b0) & 1];
    const double *src = p.S_lat + ((size_t)b * 256 + it.l * it.l) * 32;
    // rows k >= w of the padded slice are zero (4 nkk <= 32 rows)
    for (int idx = tid; idx < 4 * nkk * 32; idx += 256) {
      const int k = idx >> 5, e = idx & 31;
      Sb[k][e] = (k < w) ? src[idx] : 0.0;
    }
    __syncthreads();
    const int rk4 = (p.rkeep[b] + 3) & ~3;
    const int nnt = (rk4 + 7) >> 3;
    double *Xb = p.X + (size_t)b * (256 * 992) + ((size_t)it.l * it.l * 31 + it.row0) * 32;
    if (warp_live) {
      for (int nt = 0; nt < nnt; ++nt) {
        double acc[4][2];
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) acc[mt][0] = acc[mt][1] = 0.0;
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
          if (kk < nkk) {
            const double bf = Sb[4 * kk + tg][8 * nt + g];
#pragma unroll
            for (int mt = 0; mt < 4; ++mt) dmma_m8n8k4(acc[mt][0], acc[mt][1], a[mt][kk], bf);
          }
        }
        const int col = 8 * nt + 2 * tg;
        if (col < rk4) {
#pragma unroll
          for (int mt = 0; mt < 4; ++mt) {
            const int r = 32 * warp + 8 * mt + g;
            if (r < it.nrows)
              *reinterpret_cast<double2 *>(Xb + (size_t)r * 32 + col) = make_double2(acc[mt][0], acc[mt][1]);
          }
        }
      }
    }
    // the double-buffered Ssh makes one barrier per sample sufficient
  }
}

int k2_upload_items(int device, int *nitems_out) {
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  static bool done_dev[64] = {false};
  static int nitems_dev[64] = {0};
  bool &done = done_dev[device & 63];
  int &nitems = nitems_dev[device & 63];
  if (!done) {
    K2Item items[64];
    int toff = 0;
    for (int l = 0; l <= SPB_LMAX; ++l) {
      const int w = 2 * l + 1, rows = w * 31;
      for (int r0 = 0; r0 < rows; r0 += 256) {
        items[nitems].l = l;
        items[nitems].row0 = r0;
        items[nitems].nrows = (rows - r0 < 256) ? rows - r0 : 256;
        items[nitems].toff = toff;
        ++nitems;
      }
      toff += w * 31 * w;
    }
    if (cudaMemcpyToSymbol(k2_items, items, sizeof(K2Item) * nitems) != cudaSuccess) return 1;
    done = true;
  }
  *nitems_out = nitems;
  return 0;
}

constexpr int MOM_CHUNK = 1024;  // samples per pass (bounds the sqrtC_lon workspace to 2 GB)

struct MomWs {
  double *mom1, *S_lat, *scale, *X, *Sred, *qs, *E2;
  int *rkeep;
  void *i8ws;   // digit planes + row scales of the INT8 SYRK (one chunk)
};

size_t mom_ws_layout(int B, unsigned char *base, MomWs *ws) {
  const int Bc = B < MOM_CHUNK ? B : MOM_CHUNK;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off += (bytes + 255) & ~(size_t)255;
    return o;
  };
  size_t o_mom1 = take((size_t)B * 256 * 8);
  size_t o_S = take((size_t)B * 256 * 32 * 8);
  size_t o_scale = take((size_t)B * 8);
  size_t o_rk = take((size_t)B * 4);
  size_t o_X = take((size_t)Bc * 256 * 992 * 8);
  size_t o_Sred = take((size_t)B * 1024 * 8);
  size_t o_qs = take((size_t)B * 16 * 8);
  size_t o_E2 = take((size_t)B * 256 * 8);
  size_t o_i8 = take(spb_syrk_i8_workspace_bytes(Bc));
  if (ws) {
    ws->E2 = reinterpret_cast<double *>(base + o_E2);
    ws->i8ws = base + o_i8;
    ws->Sred = reinterpret_cast<double *>(base + o_Sred);
    ws->qs = reinterpret_cast<double *>(base + o_qs);
    ws->mom1 = reinterpret_cast<double *>(base + o_mom1);
    ws->S_lat = reinterpret_cast<double *>(base + o_S);
    ws->scale = reinterpret_cast<double *>(base + o_scale);
    ws->rkeep = reinterpret_cast<int *>(base + o_rk);
    ws->X = reinterpret_cast<double *>(base + o_X);
  }
  return off;
}

// gauss2beta, latitude.py:62-77
__global__ void gauss2beta_kernel(int B, const double *mu, const double *sigma, double *a,
                                  double *b, double lam, double lbm) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const double ang = 3.14159265358979323846 / 180.0;
  const double m = mu[i] * ang;
  const double v = (sigma[i] * ang) * (sigma[i] * ang);
  const double c1 = cos(m), c2 = cos(2 * m), c3 = cos(3 * m);
  const double ch = cos(0.5 * m);
  const double term = 1.0 / (16 * v * (ch * ch * ch * ch));
  const double alpha = (2 + 4 * v + (3 + 8 * v) * c1 + 2 * c2 + c3) * term;
  const double beta = (c1 + 2 * v * (3 + c2) - c3) * term;
  a[i] = log(alpha) / lam;
  b[i] = fmax(0.0, (log(beta) - log(0.5)) / (lbm - log(0.5)));
}

// log |d(a, b) / d(mu, sigma)|, latitude.py:221-241 (mode and width of the latitude pdf from the
// Beta shape parameters) and 281-316; -inf when sigma > sigma_max.
__global__ void log_jac_kernel(int B, const double *a, const double *b, double sigma_max_rad,
                               double *out, double abmin, double lam, double lbm) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  double aa = a[i], bb = b[i];
  if (aa < abmin) aa = abmin;  // latitude.py:178-182 (abmin)
  if (bb < abmin) bb = abmin;
  const double al = exp(aa * lam);
  const double be = exp(log(0.5) + bb * (lbm - log(0.5)));
  double term = 4 * al * al - 8 * al - 6 * be + 4 * al * be + be * be + 5;
  const double mu = 2 * atan(sqrt(2 * al + be - 2 - sqrt(term)));
  const double cm = cos(mu), sn = sin(mu);
  term = 1 - al + be + (be - 1) * cm + (al - 1) / (cm * cm);
  const double sigma = sqrt(sn * sn / term);
  const double c1 = 1 + cm, s2 = sin(2 * mu);
  const double num = al * be * (c1 * c1 * c1) * (s2 * s2 * s2);
  const double f1 = -3 + 2 * al + be + (-1 + 2 * al + be) * cm;
  const double f2 = 2 * (-1 + al + be) + 3 * (-1 + be) * cm - 2 * (-1 + al - be) * cos(2 * mu) +
                    (-1 + be) * cos(3 * mu);
  const double lj = log(fabs(num / (sigma * f1 * (f2 * f2))));
  out[i] = (sigma > sigma_max_rad) ? -INFINITY : lj;
}

}  // namespace

// Options of the moment integrals that the reference threads through as keywords (sp.py:241-262):
// NULL or zero-initialised fields mean the reference defaults (defaults.py:4-35).
static void resolve_options(const spb_context *ctx, const spb_moments_options *opt, const double **Bp,
                            const double **lambda, double *abmin, double *lam, double *lbm) {
  *Bp = (opt && opt->Bp) ? opt->Bp : ctx->d_tables + SPB_TAB_BP;
  *lambda = (opt && opt->lambda) ? opt->lambda : ctx->d_tables + SPB_TAB_LAMBDA;
  *abmin = (opt && opt->abmin > 0.0) ? opt->abmin : 1e-12;
  *lam = (opt && opt->log_alpha_max > 0.0) ? opt->log_alpha_max : 10.0;
  *lbm = (opt && opt->log_beta_max > 0.0) ? opt->log_beta_max : 10.0;
}

extern "C" int spb_log_jac(spb_context *ctx, int B, const double *a, const double *b,
                           double sigma_max_deg, double *log_jac, void *stream) {
  return spb_log_jac_opt(ctx, B, a, b, sigma_max_deg, nullptr, log_jac, stream);
}

extern "C" int spb_log_jac_opt(spb_context *ctx, int B, const double *a, const double *b,
                               double sigma_max_deg, const spb_moments_options *opt, double *log_jac,
                               void *stream) {
  SPB_REQUIRE(ctx != nullptr && B > 0, "log_jac: bad arguments");
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  const double *Bp, *lambda;
  double abmin, lam, lbm;
  resolve_options(ctx, opt, &Bp, &lambda, &abmin, &lam, &lbm);
  log_jac_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      B, a, b, sigma_max_deg * 3.14159265358979323846 / 180.0, log_jac, abmin, lam, lbm);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int spb_gauss2beta(spb_context *ctx, int B, const double *mu_deg,
                              const double *sigma_deg, double *a, double *b, void *stream) {
  return spb_gauss2beta_opt(ctx, B, mu_deg, sigma_deg, nullptr, a, b, stream);
}

extern "C" int spb_gauss2beta_opt(spb_context *ctx, int B, const double *mu_deg,
                                  const double *sigma_deg, const spb_moments_options *opt, double *a,
                                  double *b, void *stream) {
  SPB_REQUIRE(ctx != nullptr && B > 0, "gauss2beta: bad arguments");
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  const double *Bp, *lambda;
  double abmin, lam, lbm;
  resolve_options(ctx, opt, &Bp, &lambda, &abmin, &lam, &lbm);
  gauss2beta_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(B, mu_deg, sigma_deg, a, b, lam,
                                                                     lbm);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

// K1b -> K1c -> K2 -> SYRK for B samples whose (Sred, qs, mom1, scale, info) are in place.
static int moments_tail(spb_context *ctx, int B, K1Params &p1, MomWs &ws, double *cov_ylm, bool has_dr,
                        const double *lambda, cudaStream_t stream) {
  moments_k1b<<<(B + K1B_WARPS - 1) / K1B_WARPS, 32 * K1B_WARPS, K1B_WARPS * sizeof(K1bWarp), stream>>>(p1);
  SPB_LAUNCH_CHECK(ctx);
  moments_k1c<<<B, NT1, 0, stream>>>(p1);
  SPB_LAUNCH_CHECK(ctx);

  int nitems = 0;
  SPB_REQUIRE(k2_upload_items(ctx->device, &nitems) == 0, "ylm_moments: constant upload failed");
  for (int b0 = 0; b0 < B; b0 += MOM_CHUNK) {
    const int Bc = (B - b0 < MOM_CHUNK) ? B - b0 : MOM_CHUNK;
    K2Params p2;
    p2.tab = ctx->d_tables;
    p2.S_lat = ws.S_lat + (size_t)b0 * 256 * 32;
    p2.rkeep = ws.rkeep + b0;
    p2.X = ws.X;
    p2.B = Bc;
    dim3 grid2(nitems, (Bc + K2_GROUP - 1) / K2_GROUP);
    moments_k2<<<grid2, 256, 0, stream>>>(p2);
    SPB_LAUNCH_CHECK(ctx);

    gnt::Desc d = {};
    d.A = ws.X;
    d.strideA = 256 * 992;
    d.lda = 992;
    d.Bm = ws.X;
    d.strideB = 256 * 992;
    d.ldb = 992;
    d.C = cov_ylm + (size_t)b0 * 65536;
    d.strideC = 65536;
    d.ldc = 256;
    d.M = 256;
    d.N = 256;
    d.K = 992;
    d.batch = Bc;
    d.ksplit = 1;
    d.strideSplit = 0;
    d.lower_only = 1;
    d.scale = ws.scale + b0;
    d.vec = ws.mom1 + (size_t)b0 * 256;
    d.strideVec = 256;
    d.diag = lambda;
    d.rkeep = ws.rkeep + b0;
    d.ldeg = has_dr ? ws.E2 + (size_t)b0 * 256 : nullptr;
    d.alpha = 1.0;
    int st;
    if (ctx->opt_syrk_i8)
      st = spb_syrk_i8(ctx, Bc, ws.X, d.rkeep, d.scale, d.vec, d.diag, d.ldeg, d.C, ws.i8ws, stream);
    else
      st = gnt::launch<gnt::EPI_SYRK_COV>(ctx, d, stream);
    if (st) return st;
  }
  return 0;
}

extern "C" size_t spb_ylm_moments_workspace_bytes(const spb_context *ctx, int B) {
  (void)ctx;
  return mom_ws_layout(B, nullptr, nullptr);
}

extern "C" int spb_ylm_moments(spb_context *ctx, int B, const double *r_deg, const double *a,
                               const double *b, const double *c, const double *n, double *mean_ylm,
                               double *cov_ylm, int32_t *info, void *workspace,
                               size_t workspace_bytes, void *stream_) {
  return spb_ylm_moments_dr(ctx, B, r_deg, nullptr, a, b, c, n, nullptr, mean_ylm, cov_ylm, info,
                            workspace, workspace_bytes, stream_);
}

extern "C" int spb_ylm_moments_dr(spb_context *ctx, int B, const double *r_deg, const double *dr_deg,
                                  const double *a, const double *b, const double *c, const double *n,
                                  const spb_moments_options *opt, double *mean_ylm, double *cov_ylm,
                                  int32_t *info, void *workspace, size_t workspace_bytes,
                                  void *stream_) {
  SPB_REQUIRE(ctx != nullptr && B > 0, "ylm_moments: bad arguments");
  SPB_REQUIRE(ctx->tables_count == SPB_TAB_TOTAL, "ylm_moments: context has no constant tables");
  SPB_REQUIRE(workspace_bytes >= mom_ws_layout(B, nullptr, nullptr) && workspace != nullptr,
              "ylm_moments: workspace too small");
  SPB_REQUIRE(((uintptr_t)workspace % 256) == 0, "ylm_moments: workspace must be 256-byte aligned");
  cudaStream_t stream = (cudaStream_t)stream_;
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  MomWs ws;
  mom_ws_layout(B, reinterpret_cast<unsigned char *>(workspace), &ws);

  static spb_once_flag attr1_once;
  {
    const int st = spb_once_per_device(attr1_once, ctx->device, [&]() -> int {
      SPB_CHECK_CUDA(cudaFuncSetAttribute(moments_k1a, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)sizeof(K1Smem)));
      SPB_CHECK_CUDA(cudaFuncSetAttribute(moments_k1b, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)(K1B_WARPS * sizeof(K1bWarp))));
      return 0;
    });
    if (st) return st;
  }
  SPB_REQUIRE(k1_upload_perm(ctx->device) == 0, "ylm_moments: constant upload failed");
  const double *Bp, *lambda;
  double abmin, lam, lbm;
  resolve_options(ctx, opt, &Bp, &lambda, &abmin, &lam, &lbm);
  K1Params p1;
  p1.Bp = Bp;
  p1.abmin = abmin;
  p1.lam = lam;
  p1.lbm = lbm;
  p1.r_deg = r_deg;
  p1.dr_deg = dr_deg;
  p1.E2 = ws.E2;
  p1.a = a;
  p1.b = b;
  p1.c = c;
  p1.n = n;
  p1.B = B;
  p1.tab = ctx->d_tables;
  p1.mom1 = ws.mom1;
  p1.mean_ylm = mean_ylm;
  p1.S_lat = ws.S_lat;
  p1.scale = ws.scale;
  p1.rkeep = ws.rkeep;
  p1.info = info;
  p1.Sred = ws.Sred;
  p1.qs = ws.qs;
  moments_k1a<<<B, NT1, sizeof(K1Smem), stream>>>(p1);
  SPB_LAUNCH_CHECK(ctx);
  return moments_tail(ctx, B, p1, ws, cov_ylm, dr_deg != nullptr, lambda, stream);
}

// Workspace of the gradient call: the moments workspace of 7 B samples plus the tangent arrays.
static size_t grad_ws_layout(int B, unsigned char *base, MomWs *ws, double **dS, double **dqs,
                             double **dmom1, int32_t **info7) {
  size_t off = mom_ws_layout(7 * B, base, ws);
  auto take = [&](size_t bytes) {
    size_t o = off;
    off += (bytes + 255) & ~(size_t)255;
    return o;
  };
  const size_t o1 = take((size_t)B * 2 * 1024 * 8), o2 = take((size_t)B * 16 * 8),
               o3 = take((size_t)B * 3 * 256 * 8), o4 = take((size_t)7 * B * 4);
  if (base) {
    *dS = reinterpret_cast<double *>(base + o1);
    *dqs = reinterpret_cast<double *>(base + o2);
    *dmom1 = reinterpret_cast<double *>(base + o3);
    *info7 = reinterpret_cast<int32_t *>(base + o4);
  }
  return off;
}

extern "C" size_t spb_ylm_moments_grad_workspace_bytes(const spb_context *ctx, int B) {
  (void)ctx;
  return grad_ws_layout(B, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
}

extern "C" int spb_ylm_moments_grad(spb_context *ctx, int B, const double *r_deg, const double *a,
                                    const double *b, const double *c, const double *n,
                                    const spb_moments_options *opt, double rel_step, double *mean_ylm,
                                    double *cov_ylm, double *eps, int32_t *info, void *workspace,
                                    size_t workspace_bytes, void *stream_) {
  SPB_REQUIRE(ctx != nullptr && B > 0 && rel_step > 0.0, "ylm_moments_grad: bad arguments");
  SPB_REQUIRE(ctx->tables_count == SPB_TAB_TOTAL, "ylm_moments_grad: context has no constant tables");
  SPB_REQUIRE(workspace != nullptr && workspace_bytes >= spb_ylm_moments_grad_workspace_bytes(ctx, B),
              "ylm_moments_grad: workspace too small");
  SPB_REQUIRE(((uintptr_t)workspace % 256) == 0, "ylm_moments_grad: workspace must be 256-byte aligned");
  cudaStream_t stream = (cudaStream_t)stream_;
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  MomWs ws;
  double *dS, *dqs, *dmom1;
  int32_t *info7;
  grad_ws_layout(B, reinterpret_cast<unsigned char *>(workspace), &ws, &dS, &dqs, &dmom1, &info7);
  static spb_once_flag attr_once;
  {
    const int st = spb_once_per_device(attr_once, ctx->device, [&]() -> int {
      SPB_CHECK_CUDA(cudaFuncSetAttribute(moments_k1a, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)sizeof(K1Smem)));
      SPB_CHECK_CUDA(cudaFuncSetAttribute(moments_k1a_tan, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)sizeof(K1Smem)));
      SPB_CHECK_CUDA(cudaFuncSetAttribute(moments_k1b, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)(K1B_WARPS * sizeof(K1bWarp))));
      return 0;
    });
    if (st) return st;
  }
  SPB_REQUIRE(k1_upload_perm(ctx->device) == 0, "ylm_moments_grad: constant upload failed");
  // base sample: K1a into the first B slots of the 7 B arrays
  const double *Bp, *lambda;
  double abmin, lam, lbm;
  resolve_options(ctx, opt, &Bp, &lambda, &abmin, &lam, &lbm);
  K1Params p1;
  p1.Bp = Bp;
  p1.abmin = abmin;
  p1.lam = lam;
  p1.lbm = lbm;
  p1.r_deg = r_deg;
  p1.dr_deg = nullptr;
  p1.E2 = ws.E2;
  p1.a = a;
  p1.b = b;
  p1.c = c;
  p1.n = n;
  p1.B = B;
  p1.tab = ctx->d_tables;
  p1.mom1 = ws.mom1;
  p1.mean_ylm = mean_ylm;
  p1.S_lat = ws.S_lat;
  p1.scale = ws.scale;
  p1.rkeep = ws.rkeep;
  p1.info = info7;
  p1.Sred = ws.Sred;
  p1.qs = ws.qs;
  moments_k1a<<<B, NT1, sizeof(K1Smem), stream>>>(p1);
  SPB_LAUNCH_CHECK(ctx);
  K1TanParams pt;
  pt.Bp = Bp;
  pt.abmin = abmin;
  pt.lam = lam;
  pt.lbm = lbm;
  pt.r_deg = r_deg;
  pt.a = a;
  pt.b = b;
  pt.B = B;
  pt.tab = ctx->d_tables;
  pt.dS = dS;
  pt.dqs = dqs;
  pt.dmom1 = dmom1;
  moments_k1a_tan<<<B, NT1, sizeof(K1Smem), stream>>>(pt);
  SPB_LAUNCH_CHECK(ctx);
  ExpandParams pe;
  pe.B = B;
  pe.rel_step = rel_step;
  pe.c = c;
  pe.n = n;
  pe.dS = dS;
  pe.dqs = dqs;
  pe.dmom1 = dmom1;
  pe.Sred = ws.Sred;
  pe.qs = ws.qs;
  pe.mom1 = ws.mom1;
  pe.mean_ylm = mean_ylm;
  pe.scale = ws.scale;
  pe.info = info7;
  pe.eps = eps;
  moments_expand_kernel<<<B, 256, 0, stream>>>(pe);
  SPB_LAUNCH_CHECK(ctx);
  // the unchanged pipeline on the 7 B variants
  p1.B = 7 * B;
  int st = moments_tail(ctx, 7 * B, p1, ws, cov_ylm, false, lambda, stream);
  if (st) return st;
  moments_scale_variants_kernel<<<dim3(B, 4), 256, 0, stream>>>(B, c, n, eps, lambda, mean_ylm,
                                                               cov_ylm);
  SPB_LAUNCH_CHECK(ctx);
  // flags of the base sample (bounds, eigen-solve) are what the caller sees
  SPB_CHECK_CUDA(cudaMemcpyAsync(info, info7, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToDevice,
                                 stream));
  return 0;
}
