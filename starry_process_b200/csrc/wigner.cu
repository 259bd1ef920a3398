// Real Wigner rotations and the flux design matrix.
//
//   spb_Rx            Rx(theta), all l <= 15, packed (5456)      ops/wigner/Rx.cc:10-49 ->
//                     rotar / dlmn                               ops/include/wigner.h:37-284
//   spb_tensordotRz   f = M . Rz(theta_k) row by row             ops/wigner/tensordotRz.cc:10-56,
//                                                                wigner.h:290-339
//   spb_design_matrix A(t; i, p, u) = rTA1 . Rx(-i) . Rz(theta) . Rx(pi/2)
//                                                                flux.py:88-105, 278-281
//
// Built with -fmad=false: the Alvarez-Collado recurrences are evaluated with the same unfused
// multiply/add sequence as the reference's `g++ -O2` build, but PARALLEL over the (m', m) entries
// of each degree (the reference walks them serially): one CTA per angle, the complex matrices
// D[l] for all l kept in shared memory (43.6 KB).
#include <string.h>

#include "common.cuh"
#include "spb_tables.h"

namespace {

__host__ __device__ __forceinline__ int nwig(int l) { return ((l + 1) * (2 * l + 1) * (2 * l + 3)) / 3; }

// integer cos/sin of k*pi/2 style phase tables used by rotar (wigner.h:232-270)
__device__ __forceinline__ void phase_al(int mp, int &c, int &s) {
  // (cosmal, sinmal) starts (0,-1) at mp = 1 and maps (c, s) -> (s, -c)
  const int k = (mp - 1) & 3;
  c = (k == 0) ? 0 : (k == 1) ? -1 : (k == 2) ? 0 : 1;
  s = (k == 0) ? -1 : (k == 1) ? 0 : (k == 2) ? 1 : 0;
}
__device__ __forceinline__ void phase_ga(int m, int &c, int &s) {
  // (cosmga, sinmga) starts (0, 1) at m = 1 and maps (c, s) -> (-s, c)
  const int k = (m - 1) & 3;
  c = (k == 0) ? 0 : (k == 1) ? -1 : (k == 2) ? 0 : 1;
  s = (k == 0) ? 1 : (k == 1) ? 0 : (k == 2) ? -1 : 0;
}

__global__ void __launch_bounds__(256) rx_kernel(int nang, const double *theta, double sign_in,
                                                 double *Rout) {
  __shared__ double D[SPB_NWIG];
  const int tid = threadIdx.x;
  const int ia = blockIdx.x;
  if (ia >= nang) return;
  double *R = Rout + (size_t)ia * SPB_NWIG;
  const double th = sign_in * theta[ia];
  const double root_two = sqrt(2.0);
  const double c2 = cos(th), s2 = sin(th);

  if (tid == 0) {
    // wigner.h:164-206
    D[0] = 1.0;
    D[9] = 0.5 * (1.0 + c2);
    D[8] = -s2 / root_two;
    D[7] = 0.5 * (1.0 - c2);
    D[6] = -D[8];
    D[5] = D[9] - D[7];
    D[4] = D[8];
    D[3] = D[7];
    D[2] = D[6];
    D[1] = D[9];
    R[0] = 1.0;
    R[1] = D[9] - D[7];
    R[2] = -root_two * D[6];
    R[3] = 0;
    R[4] = -root_two * D[8];
    R[5] = D[5];
    R[6] = 0;
    R[7] = 0;
    R[8] = 0;
    R[9] = D[9] + D[7];
  }
  __syncthreads();
  double tgbet2;
  if (fabs(s2) < 1.0e-14) tgbet2 = s2;  // SP_WIGNER_TOL, constants.h:71-73
  else tgbet2 = (1.0 - c2) / s2;

  for (int l = 2; l <= SPB_LMAX; ++l) {
    const int w = 2 * l + 1, w1 = w - 2, w2 = w - 4;
    double *Dl = D + nwig(l - 1);
    const double *Dm1 = D + nwig(l - 2);
    const double *Dm2 = D + nwig(l - 3);
    double *Rl = R + nwig(l - 1);
#define DL(r, c) Dl[(r)*w + (c)]
#define DM1(r, c) Dm1[(r)*w1 + (c)]
#define DM2(r, c) Dm2[(r)*w2 + (c)]
    // (a) top row by recurrence, wigner.h:57-73 (serial in m)
    if (tid == 0) {
      const int isup = l - 1, iinf = 1 - l;
      DL(2 * l, 2 * l) = 0.5 * DM1(isup + l - 1, isup + l - 1) * (1.0 + c2);
      DL(2 * l, 0) = 0.5 * DM1(isup + l - 1, -isup + l - 1) * (1.0 - c2);
      for (int m = isup; m > iinf - 1; --m)
        DL(2 * l, m + l) = -tgbet2 * sqrt((double)(l + m + 1) / (l - m)) * DL(2 * l, m + 1 + l);
    }
    // (b) upper quarter triangle, wigner.h:77-110: rows mp in [0, l-1], columns m in [-mp, mp]
    {
      const int al = l, al1 = l - 1, tal1 = al + al1;
      const double ali = 1.0 / al1;
      const double cosaux = c2 * al * al1;
      for (int idx = tid; idx < l * w; idx += 256) {
        const int mp = idx / w, m = idx % w - l;
        if (m < -mp || m > mp) continue;
        const int laux = l + mp, lbux = l - mp;
        const double aux = ali / sqrt((double)(laux * lbux));
        const double cux = sqrt((double)((laux - 1) * (lbux - 1))) * al;
        const int lauz = l + m, lbuz = l - m;
        const double auz = 1.0 / sqrt((double)(lauz * lbuz));
        const double fact = aux * auz;
        double term = tal1 * (cosaux - (double)(m * mp)) * DM1(mp + l - 1, m + l - 1);
        if ((lbuz != 1) && (lbux != 1)) {
          const double cuz = sqrt((double)((lauz - 1) * (lbuz - 1)));
          term = term - DM2(mp + l - 2, m + l - 2) * cux * cuz;
        }
        DL(mp + l, m + l) = fact * term;
      }
    }
    __syncthreads();
    // (c) reflection, wigner.h:117-129: D(mp, m) = (-1)^(mp+m) D(m, mp), m in [1, l], mp in [-m, m-1]
    for (int idx = tid; idx < l * w; idx += 256) {
      const int m = idx / w + 1, mp = idx % w - l;
      if (mp < -m || mp > m - 1) continue;
      const double sg = ((mp + m) & 1) ? -1.0 : 1.0;
      DL(mp + l, m + l) = sg * DL(m + l, mp + l);
    }
    __syncthreads();
    // (d) inversion, wigner.h:131-142: D(mp, m) = (-1)^(mp+m) D(-mp, -m), m in [-l, l-1], mp in [-l, -m-1]
    for (int idx = tid; idx < w * w; idx += 256) {
      const int m = idx / w - l, mp = idx % w - l;
      if (m > l - 1 || mp > -m - 1) continue;
      const double sg = ((mp + m) & 1) ? -1.0 : 1.0;
      DL(mp + l, m + l) = sg * DL(-mp + l, -m + l);
    }
    __syncthreads();
    // (e) real matrices from the complex ones, wigner.h:226-270
    if (tid == 0) Rl[l * w + l] = DL(l, l);
    for (int idx = tid; idx < l; idx += 256) {
      const int mp = idx + 1;
      int cal, sal;
      phase_al(mp, cal, sal);
      Rl[(mp + l) * w + l] = root_two * DL(l, mp + l) * cal;
      Rl[(-mp + l) * w + l] = root_two * DL(l, mp + l) * sal;
      // the axis entries R(l, +-m) are rewritten identically for every mp in the reference
      const int m = mp;
      int cga, sga;
      phase_ga(m, cga, sga);
      Rl[l * w + (m + l)] = root_two * DL(m + l, l) * cga;
      Rl[l * w + (-m + l)] = -root_two * DL(m + l, l) * sga;
    }
    for (int idx = tid; idx < l * l; idx += 256) {
      const int mp = idx / l + 1, m = idx % l + 1;
      int cal, sal, cga, sga;
      phase_al(mp, cal, sal);
      phase_ga(m, cga, sga);
      const int sgn = (mp & 1) ? -1 : 1;
      const double d1 = DL(-mp + l, -m + l);
      const double d2 = sgn * DL(mp + l, -m + l);
      const int cosag = cal * cga - sal * sga;
      const int cosagm = cal * cga + sal * sga;
      const int sinag = sal * cga + cal * sga;
      const int sinagm = sal * cga - cal * sga;
      Rl[(mp + l) * w + (m + l)] = d1 * cosag + d2 * cosagm;
      Rl[(mp + l) * w + (-m + l)] = -d1 * sinag + d2 * sinagm;
      Rl[(-mp + l) * w + (m + l)] = d1 * sinag + d2 * sinagm;
      Rl[(-mp + l) * w + (-m + l)] = d1 * cosag - d2 * cosagm;
    }
    __syncthreads();
#undef DL
#undef DM1
#undef DM2
  }
}

// cos(n theta), sin(n theta) by the recurrences of wigner.h:307-316
__device__ __forceinline__ void cheb_cs(double theta, double *cs, double *sn) {
  cs[0] = 1.0;
  sn[0] = 0.0;
  cs[1] = cos(theta);
  sn[1] = sin(theta);
  for (int n = 2; n <= SPB_LMAX; ++n) {
    cs[n] = 2.0 * cs[n - 1] * cs[1] - cs[n - 2];
    sn[n] = 2.0 * sn[n - 1] * cs[1] - sn[n - 2];
  }
}

__global__ void __launch_bounds__(256) tensordotRz_kernel(int K, const double *M, const double *theta,
                                                          double *f) {
  __shared__ double cs[16], sn[16];
  const int k = blockIdx.x, n = threadIdx.x;
  if (k >= K) return;
  if (n == 0) cheb_cs(theta[k], cs, sn);
  __syncthreads();
  const int l = (int)floor(sqrt((double)n) + 1e-9);
  const int j = n - l * l, m = j - l;
  const double *Mk = M + (size_t)k * 256;
  const double cm = cs[m < 0 ? -m : m];
  const double sm = m < 0 ? -sn[-m] : sn[m];
  f[(size_t)k * 256 + n] = Mk[n] * cm + Mk[l * l + 2 * l - j] * sm;
}

// ------------------------------------------------------------------------------------------
// Design matrix  A(t; i, p, u) = rTA1 . Rx(-i) . Rz(theta_t) . Rx(pi/2)      flux.py:88-105
//
//   design_v_kernel   v = rTA1 . Rx(-i) once per inclination (identical for every timestamp:
//                     hoisted out of the reference's tile(rTA1, (nt, 1)) product), stored as the
//                     pairs (v[n], +-v[mirror(n)]) that the z-rotation consumes
//   design_rows_kernel  one THREAD per timestamp.  cos/sin(m theta) by the reference's Chebyshev
//                     recurrences in registers; the row is produced degree by degree by the
//                     fully unrolled body of design_gen.inc, which visits only the 1372
//                     structurally non-zero entries of Rx(pi/2) (of 5456) and fetches their values
//                     as warp-uniform 16-byte shared-memory broadcasts; finished columns leave
//                     through TMA tensor stores.  2048 B written + 8 B read per row: the kernel
//                     is bound by HBM writes (DESIGN.md "design matrix").
// ------------------------------------------------------------------------------------------
constexpr int DM_THREADS = 128;
constexpr int RX90_NZ = (int)SPB_TAB_RX90_NZ_COUNT;  // 1372

struct DesignParams {
  int I, nt;
  const double *t, *period;
  const double *VV;     // (I, 256, 2)
  const double *RxNZ;   // (1372) non-zeros of Rx(pi/2), consumption order
  double *A;
};

__global__ void __launch_bounds__(256) design_v_kernel(int I, const double *rTA1, int rTA1_stride,
                                                       const double *RxInc, double *VV) {
  __shared__ double v[256];
  const int n = threadIdx.x, ii = blockIdx.x;
  if (ii >= I) return;
  const int l = (int)floor(sqrt((double)n) + 1e-9);
  const int j = n - l * l, m = j - l, w = 2 * l + 1;
  // v[(l, m)] = sum_m' rTA1[(l, m')] Rx(-i)_l[m'][m]   (flux.py:95-96, 74-86)
  const double *rt = rTA1 + (size_t)ii * rTA1_stride + l * l;
  const double *rx = RxInc + (size_t)ii * SPB_NWIG + nwig(l - 1);
  double acc = 0.0;
  for (int mp = 0; mp < w; ++mp) acc += rt[mp] * rx[mp * w + j];
  v[n] = acc;
  __syncthreads();
  // f[l^2 + j] = v[l^2 + j] cos(m theta) + v[l^2 + 2l - j] sin(m theta), sin(-|m| theta) folded
  // into the sign of the partner (wigner.h:319-337)
  const double vb = v[l * l + 2 * l - j];
  double2 *out = reinterpret_cast<double2 *>(VV) + (size_t)ii * 256 + n;
  *out = make_double2(acc, m < 0 ? -vb : vb);
}

// Inclination basis of the rank-31 conditional path (DESIGN.md section 4.6): a design-matrix row is
// f(theta) . Rx(pi/2) with f[n] = VV.x[n] cos(|m_n| theta) + VV.y[n] sin(|m_n| theta), so
//   A = Phi(t) B_inc,  Phi = [1, cos(m theta) (m = 1..15), sin(m theta) (m = 1..15)]
//   B_inc[m]      = sum over |m_n| = m of VV.x[n] Rx90[n, :]      (rows 0..15)
//   B_inc[15 + m] = sum over |m_n| = m of VV.y[n] Rx90[n, :]      (rows 16..30);  row 31 = 0.
// One thread per output column n' = l^2 + j' (Rx(pi/2) is block-diagonal in l).
__global__ void __launch_bounds__(256) lowrank_binc_kernel(int I, const double *VV, const double *Rx90,
                                                           double *Binc) {
  __shared__ double2 v[256];
  const int c = threadIdx.x, ii = blockIdx.x;
  if (ii >= I) return;
  v[c] = reinterpret_cast<const double2 *>(VV)[(size_t)ii * 256 + c];
  __syncthreads();
  const int l = (int)floor(sqrt((double)c) + 1e-9);
  const int jp = c - l * l, w = 2 * l + 1;
  const double *rx = Rx90 + nwig(l - 1);
  double *out = Binc + (size_t)ii * 32 * 256 + c;
  for (int k = 0; k <= SPB_LMAX; ++k) {
    double a = 0.0, b = 0.0;
    if (k <= l) {
      const int j1 = l + k;
      a = v[l * l + j1].x * rx[j1 * w + jp];
      b = v[l * l + j1].y * rx[j1 * w + jp];
      if (k > 0) {
        const int j2 = l - k;
        a += v[l * l + j2].x * rx[j2 * w + jp];
        b += v[l * l + j2].y * rx[j2 * w + jp];
      }
    }
    out[k * 256] = a;
    if (k > 0) out[(SPB_LMAX + k) * 256] = b;
  }
  out[31 * 256] = 0.0;
}

// Store path: the warp collects a (32 timestamps x 16 columns) tile in shared memory -- 128-byte rows
// in the TMA 128B-swizzle layout, so the lanes' 16-byte stores are conflict-free -- and one elected
// lane hands it to the TMA engine (cp.async.bulk.tensor.3d shared -> global through a tensor map of A,
// which also clips the rows past nt); double-buffered per warp, the LSU only sees the STS.128.
// (DESIGN.md section 4.2 records it against direct 32-byte global stores.)
// The 1372 coefficients come from shared memory as warp-uniform broadcasts.  (A constant-bank
// variant -- LDCU into uniform registers -- measured 13 % slower: profiles/r01_time_design_variants.log.)
constexpr int DM_CW = 16;                        // columns per TMA box (128 bytes)
constexpr int DM_BOX_BYTES = 32 * DM_CW * 8;     // 32 rows x 128 B = 4096
constexpr int DM_STAGE_BYTES = (DM_THREADS / 32) * 2 * DM_BOX_BYTES;

__global__ void __launch_bounds__(DM_THREADS, 3)
    design_rows_kernel(DesignParams p, const __grid_constant__ CUtensorMap tmapA) {
  extern __shared__ __align__(1024) unsigned char dm_smem[];
  // the swizzle pattern is a function of the shared-memory ADDRESS: align the tiles to its 1 KB atom
  unsigned char *stage = dm_smem;                                          // [warp][2][4096]
  {
    const unsigned a = (unsigned)__cvta_generic_to_shared(dm_smem);
    stage += (1024u - (a & 1023u)) & 1023u;
  }
  double2 *Rs2 = reinterpret_cast<double2 *>(stage + DM_STAGE_BYTES);
  double2 *Vs2 = Rs2 + RX90_NZ / 2;                                        // 256
  const int tid = threadIdx.x, ii = blockIdx.y, warp = tid >> 5, lane = tid & 31;
  for (int k = tid; k < RX90_NZ / 2; k += DM_THREADS)
    Rs2[k] = reinterpret_cast<const double2 *>(p.RxNZ)[k];
  for (int k = tid; k < 256; k += DM_THREADS)
    Vs2[k] = reinterpret_cast<const double2 *>(p.VV)[(size_t)ii * 256 + k];
  __syncthreads();
  unsigned char *wstage = stage + warp * 2 * DM_BOX_BYTES;
  const double per = p.period ? p.period[ii] : 1.0;
  const int ntiles = (p.nt + DM_THREADS - 1) / DM_THREADS;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int t = tile * DM_THREADS + tid;
    // rows past nt are computed on a clamped timestamp and clipped by the tensor map
    double cs[SPB_LMAX + 1], sn[SPB_LMAX + 1];
    spb_harmonics(spb_phase(p.t[t < p.nt ? t : p.nt - 1], per), cs, sn);
    const int trow0 = tile * DM_THREADS + warp * 32;   // first timestamp of this warp's tile
    double o0, o1, o2, o3;
#define RS2(q) Rs2[q]
    // chunk q uses buffer q & 1; before refilling it, the store issued two chunks ago must have
    // finished reading shared memory (at most the most recent store may still be in flight)
#define DM_BEGIN(q)                                                                 \
  do {                                                                              \
    if (lane == 0) bulk_wait_read<1>();                                             \
    __syncwarp();                                                                   \
  } while (0)
#define DM_STORE4(c, a, b, cc, d)                                                   \
  do {                                                                              \
    unsigned char *b_ = wstage + (((c) >> 4) & 1) * DM_BOX_BYTES + lane * 128;      \
    const int j_ = ((c) & 15) >> 1;                                                 \
    *reinterpret_cast<double2 *>(b_ + ((j_ ^ (lane & 7)) << 4)) = make_double2(a, b);        \
    *reinterpret_cast<double2 *>(b_ + (((j_ + 1) ^ (lane & 7)) << 4)) = make_double2(cc, d); \
  } while (0)
#define DM_FLUSH(q)                                                                 \
  do {                                                                              \
    fence_proxy_async_smem();                                                       \
    __syncwarp();                                                                   \
    if (lane == 0) {                                                                \
      tma_store_3d(&tmapA, wstage + ((q) & 1) * DM_BOX_BYTES, (q) * DM_CW, trow0, ii); \
      bulk_commit();                                                                \
    }                                                                               \
  } while (0)
#include "design_gen.inc"
#undef DM_BEGIN
#undef DM_STORE4
#undef DM_FLUSH
#undef RS2
  }
  if (lane == 0) bulk_wait_read<0>();  // TMA must be done reading this CTA's shared memory
}

}  // namespace

int spb_wigner_init(spb_context *ctx) {
  (void)ctx;
  return 0;
}

extern "C" int spb_Rx(spb_context *ctx, int nang, const double *theta, double *Rx, void *stream) {
  SPB_REQUIRE(ctx != nullptr && nang > 0, "Rx: bad arguments");
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  rx_kernel<<<nang, 256, 0, (cudaStream_t)stream>>>(nang, theta, 1.0, Rx);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int spb_tensordotRz(spb_context *ctx, int K, const double *M, const double *theta,
                               double *f, void *stream) {
  SPB_REQUIRE(ctx != nullptr && K > 0, "tensordotRz: bad arguments");
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  tensordotRz_kernel<<<K, 256, 0, (cudaStream_t)stream>>>(K, M, theta, f);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" size_t spb_design_matrix_workspace_bytes(const spb_context *ctx, int I, int nt) {
  (void)ctx;
  (void)nt;
  return (size_t)I * (SPB_NWIG + 512) * sizeof(double);
}

extern "C" int spb_design_matrix(spb_context *ctx, int I, int nt, const double *t,
                                 const double *inc_rad, const double *period, const double *rTA1,
                                 int rTA1_stride, double *A, void *workspace,
                                 size_t workspace_bytes, void *stream_) {
  SPB_REQUIRE(ctx != nullptr && I > 0 && nt > 0, "design_matrix: bad arguments");
  SPB_REQUIRE(ctx->tables_count == SPB_TAB_TOTAL, "design_matrix: context has no constant tables");
  SPB_REQUIRE(workspace != nullptr &&
                  workspace_bytes >= (size_t)I * (SPB_NWIG + 512) * sizeof(double),
              "design_matrix: workspace too small");
  SPB_REQUIRE(((uintptr_t)A % 32) == 0 && ((uintptr_t)workspace % 16) == 0,
              "design_matrix: A must be 32-byte aligned (workspace 16-byte)");
  SPB_REQUIRE(I <= 65535, "design_matrix: too many inclinations for one launch");
  cudaStream_t stream = (cudaStream_t)stream_;
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  double *VV = reinterpret_cast<double *>(workspace);          // (I, 512), 16-byte aligned
  double *RxInc = VV + (size_t)I * 512;                        // (I, 5456)
  rx_kernel<<<I, 256, 0, stream>>>(I, inc_rad, -1.0, RxInc);  // Rx(-i), flux.py:96
  SPB_LAUNCH_CHECK(ctx);
  design_v_kernel<<<I, 256, 0, stream>>>(I, rTA1, rTA1_stride, RxInc, VV);
  SPB_LAUNCH_CHECK(ctx);
  DesignParams p;
  p.I = I;
  p.nt = nt;
  p.t = t;
  p.period = period;
  p.VV = VV;
  p.RxNZ = ctx->d_tables + SPB_TAB_RX90_NZ;
  p.A = A;
  // row tiles per inclination; CTAs loop over tiles so that the 15 KB table prologue is amortised
  // once there is more than enough work to fill the GPU (3 CTAs per SM resident)
  const int ntiles = (nt + DM_THREADS - 1) / DM_THREADS;
  const long long want = 3LL * ctx->num_sms * 4;
  int gx = ntiles;
  if ((long long)ntiles * I > want) {
    gx = (int)((want + I - 1) / I);
    if (gx < 1) gx = 1;
    if (gx > ntiles) gx = ntiles;
  }
  dim3 grid(gx, I);
  const size_t smem = (RX90_NZ / 2 + 256) * sizeof(double2) + DM_STAGE_BYTES + 1024;
  CUtensorMap tmap;
  memset(&tmap, 0, sizeof(tmap));
  // 3-D view of A: (256 columns, nt timestamps, I inclinations), box = 16 columns x 32 timestamps,
  // 128-byte swizzle (matches the kernel's shared-memory tile layout)
  int st = spb_encode_tmap_3d_f64(&tmap, A, 256, (unsigned long long)nt, (unsigned long long)I,
                                  256ull * 8, (unsigned long long)nt * 256 * 8, DM_CW, 32, 1);
  if (st) return st;
  static spb_once_flag attr_once;
  st = spb_once_per_device(attr_once, ctx->device, [&]() -> int {
    SPB_CHECK_CUDA(cudaFuncSetAttribute(design_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)smem));
    return 0;
  });
  if (st) return st;
  design_rows_kernel<<<grid, DM_THREADS, smem, stream>>>(p, tmap);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" size_t spb_lowrank_inclination_workspace_bytes(const spb_context *ctx, int I) {
  return spb_design_matrix_workspace_bytes(ctx, I, 0);
}

extern "C" int spb_lowrank_inclination(spb_context *ctx, int I, const double *inc_rad, const double *rTA1,
                                       int rTA1_stride, double *Binc, void *workspace,
                                       size_t workspace_bytes, void *stream_) {
  SPB_REQUIRE(ctx != nullptr && I > 0, "lowrank_inclination: bad arguments");
  SPB_REQUIRE(ctx->tables_count == SPB_TAB_TOTAL, "lowrank_inclination: context has no constant tables");
  SPB_REQUIRE(workspace != nullptr && workspace_bytes >= spb_lowrank_inclination_workspace_bytes(ctx, I) &&
                  ((uintptr_t)workspace % 16) == 0,
              "lowrank_inclination: workspace too small or not 16-byte aligned");
  cudaStream_t stream = (cudaStream_t)stream_;
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  double *VV = reinterpret_cast<double *>(workspace);          // (I, 512)
  double *RxInc = VV + (size_t)I * 512;                        // (I, 5456)
  rx_kernel<<<I, 256, 0, stream>>>(I, inc_rad, -1.0, RxInc);  // Rx(-i), flux.py:96
  SPB_LAUNCH_CHECK(ctx);
  design_v_kernel<<<I, 256, 0, stream>>>(I, rTA1, rTA1_stride, RxInc, VV);
  SPB_LAUNCH_CHECK(ctx);
  lowrank_binc_kernel<<<I, 256, 0, stream>>>(I, VV, ctx->d_tables + SPB_TAB_RX90, Binc);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}
