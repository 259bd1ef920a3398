// Batched dense Cholesky + forward solve + log-determinant -> log-likelihood, FP64 tensor cores.
//
// Replaces, for a batch of B independent GP covariances, the reference's
//   cho_factor  -> scipy.linalg.cholesky  (LAPACK dpotrf)        math.py:75-94
//   cho_solve   -> 2 x solve_triangular   (LAPACK dtrtrs)        math.py:20-38, 97-100
//   lnlike = -1/2 r^T K^-1 r - M sum(log diag L) - 1/2 K M log 2pi   sp.py:1154-1188
//
// Design (B200-first, not a LAPACK transliteration)
//   * one CTA (256 threads, 8 warps) owns one matrix at a time; grid = min(B, 2 x #SM) persistent
//     CTAs, 2 CTAs resident per SM so one CTA's latency-bound diagonal-block work overlaps the
//     other's tensor-pipe work;
//   * LEFT-looking blocked factorisation, panel width NB = 64: every block column is read once
//     as the C operand and the already-factored part of L is streamed as A/B operands, so HBM/L2
//     traffic is ~n^3/(6 NB) reads + one write of L (a right-looking update would re-write the
//     trailing matrix once per panel);
//   * the panel update  P = K[:, j] - L[:, :j] L[j, :j]^T  runs on mma.sync.m8n8k4.f64 (DMMA) from
//     a 3-slot shared-memory ring handed off through mbarriers (no CTA-wide rendezvous in the
//     k-loop); tiles that lie wholly inside K are fetched by TMA (cp.async.bulk.tensor through a
//     tensor map of the batch, hardware 128-byte swizzle), tiles that mix matrix rows with appended
//     right-hand-side rows by per-thread cp.async writing the same swizzle; each warp owns 16 full
//     rows x 64 columns of the panel in registers;
//   * the triangular solve  X = P L_jj^-T  is done IN REGISTERS on the tensor pipe as an 8x8-blocked
//     forward substitution (accumulator fragments are re-shaped into A fragments with warp
//     shuffles), so the panel never round-trips through shared memory;
//   * the residual light curves r are appended as extra ROWS of the matrix ("augmented" Cholesky):
//     the same panel loop then produces y = L^-1 r, so lnlike needs no back substitution:
//         r^T K^-1 r = |y|^2;
//   * the 64x64 diagonal block is factorised IN THE ACCUMULATOR REGISTERS of warps 0-3
//     (potf2_regs): 8x8 diagonal tiles by their owner warp with shuffles only (potf2_tile8), the
//     tiles below solved and the trailing tiles updated with DMMA, two 128-thread named barriers per
//     8-column sub-panel.
//   * memory-model note: the factor is written with ordinary st.global (generic proxy) and re-read
//     by TMA (async proxy) in later panels, so every thread executes fence.proxy.async.global after
//     its stores of a panel and before the barrier that ends the panel.
//
// Algorithmic flops per matrix: nt^3/3 (factor) + nt^2 M (forward solve); see DESIGN.md.
#include <cooperative_groups.h>
#include <stddef.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "i8_planes.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int NB = 64;         // panel width
constexpr int KC = 16;         // k-chunk per pipeline stage (one 128-byte row segment)
constexpr int LS = NB + 4;     // smem stride of the diagonal block: 68
constexpr int DS = 12;         // smem stride of the 8x8 diagonal-inverse blocks

// Tile geometry of the FP64 kernels: a CTA of 8 warps owns TM = 128 rows of a panel at a time (16 rows
// x 64 columns per warp) and streams its operands through a ring of STAGES chunks.  The alternatives
// measured against it (4-warp tiles, deeper rings, a producer warp) lost inside the bench step:
// DESIGN.md section 4.1 (ii).
constexpr int TM = 128;
constexpr int NTHREADS = 2 * TM;
constexpr int STAGES = 3;      // operand ring depth (look-ahead = STAGES - 1 chunks)

enum { KIND_NONE = 0, KIND_DIAG = 1, KIND_PAD = 2, KIND_BELOW = 3, KIND_RHS = 4 };
enum { MODE_FACTOR = 1, MODE_SOLVE = 0 };

struct PotrfParams {
  double *K;
  int n, ld;
  long long strideK;
  double *R;
  int M, ldr;
  long long strideR;
  double *lnlike, *quad, *logdet;
  int32_t *info;
  int B;
  int mode;
  int rows_per_cta;  // MODE_SOLVE: RHS rows per work item
  unsigned int *counter;  // zeroed before the launch: work items beyond the first wave are claimed here
  double *scratch;        // cluster kernel: (B, CLUSTER) per-CTA partial sums of |y|^2
  int use_tma;            // operand tiles that lie wholly inside K come through TMA (tensor map of K)
  int only_flag;          // != 0: only matrices whose info has this bit are processed (the bit is cleared)
  spb_affine aff;    // fused last assembly step (scal == q == diag == offset == NULL: none)
  int aff_on;
};

struct RowMap {
  double *Kb, *Rb;
  int n, M, ld, ldr, c0, nbelow, mode, rb, nrhs;
  __device__ __forceinline__ double *row(int v, int &kind) const {
    if (mode == MODE_FACTOR) {
      if (v < NB) {
        int r = c0 + v;
        if (r < n) {
          kind = KIND_DIAG;
          return Kb + (size_t)r * ld;
        }
        kind = KIND_PAD;
        return nullptr;
      }
      int w = v - NB;
      if (w < nbelow) {
        kind = KIND_BELOW;
        return Kb + (size_t)(c0 + NB + w) * ld;
      }
      w -= nbelow;
      if (w < M) {
        kind = KIND_RHS;
        return Rb + (size_t)w * ldr;
      }
      kind = KIND_NONE;
      return nullptr;
    }
    if (v < nrhs) {
      kind = KIND_RHS;
      return Rb + (size_t)(rb + v) * ldr;
    }
    kind = KIND_NONE;
    return nullptr;
  }
};

// Stage buffers are unpadded 16-double (128-byte) rows with an XOR swizzle of the 16-byte chunk
// index: chunk' = chunk ^ (2 * (row & 3)).  For the m8n8k4 fragment pattern (lane -> row g,
// k = 4 kk + tg) every half-warp then touches 16 distinct 8-byte banks: conflict-free LDS.64
// without the 25 % padding, which is what lets three stages fit beside the diagonal block at
// two CTAs per SM.
// L_jj storage: row stride 68 (conflict-free for the m8n8k4 fragment pattern).
struct LdStore {
  double v[NB * LS];
  __device__ __forceinline__ double &at(int i, int j) { return v[i * LS + j]; }
  __device__ __forceinline__ const double &at(int i, int j) const { return v[i * LS + j]; }
};

struct Smem {
  double As[STAGES][TM][KC];
  double Bs[STAGES][NB][KC];
  LdStore Ld;   // diagonal block L_jj (lower), valid after potf2
  double Dv[NB][DS];   // the 8 inverses of the 8x8 diagonal blocks of L_jj: Dv[8*nb + r][c]
  double red[NTHREADS / 32];
  double dpiv[NB];         // pivots L_ii^2 of the current diagonal block
  double af[4];            // fused affine map of this matrix: s1, s2, s3, offset
  uint64_t full[STAGES];   // chunk landed: 256 cp.async arrivals (one per thread)
  uint64_t empty[STAGES];  // chunk consumed: 8 arrivals (one per warp)
  int bad;
  int next_item;
};

static_assert(offsetof(Smem, Dv) == offsetof(Smem, Ld) + sizeof(double) * NB * LS,
              "Ld and Dv must be adjacent (copied as one block by the cluster kernel)");

// element index inside a stage row: the TMA 128-byte swizzle (16-byte chunk index XOR row mod 8),
// used by the cp.async path as well so that both fill the ring in the same layout
__device__ __forceinline__ int swz(int row, int k) {
  return (((k >> 1) ^ (row & 7)) << 1) | (k & 1);
}

__device__ __forceinline__ double negate(double x) {  // sign flip on the integer pipe
  return __hiloint2double(__double2hiint(x) ^ (int)0x80000000, __double2loint(x));
}

// ------------------------------------------------------------------------------------------
// Initialise the accumulators with the K (or residual) values of the two rows this thread owns in
// each m-tile; the k-loop then accumulates (-L) L^T, leaving the Schur complement
// P = K - L L^T.  `full` (block-uniform: the whole 64-column panel lies inside the matrix, so no
// padding rows/columns exist) selects the fast path: plain 16-byte loads straight into the
// accumulator registers with NO dependent instruction, so that their HBM latency overlaps the
// cp.async prologue of the k-loop instead of stalling the warp before it starts.  Rows past the
// last virtual row load a dummy row (never stored); the strictly upper part of the diagonal block
// may be uninitialised memory (lower-only assembly) and is never consumed.
// ------------------------------------------------------------------------------------------
// The fused affine map (spb_affine): applied to covariance rows only, never to residual rows.
struct AffRow {
  const double *q;   // (nt) scaled row sums of this matrix, or nullptr
  const double *dg;  // diagonal add: pointer to this matrix' value(s), or nullptr
  int dg_vec;        // dg is an (nt) vector
  bool norm;         // s1, s2, s3 present
};

// AffRow of matrix `item`; thread 0 stores its scalars s1, s2, s3, offset in sm.af (the identity map
// when p.aff_on == 0).
template <class SM>
__device__ __forceinline__ AffRow aff_setup(const PotrfParams &p, int item, SM &sm, int tid) {
  AffRow af;
  af.q = nullptr;
  af.dg = nullptr;
  af.dg_vec = 0;
  af.norm = false;
  if (p.aff_on) {
    af.norm = (p.aff.scal != nullptr) && (p.aff.q != nullptr);
    if (af.norm) af.q = p.aff.q + (size_t)item * p.n;
    if (p.aff.diag) {
      af.dg = p.aff.diag + (size_t)item * p.aff.diag_stride;
      af.dg_vec = (p.aff.diag_kind == 1);
    }
  }
  if (tid == 0) {
    const double *sc = af.norm ? p.aff.scal + 4 * (size_t)item : nullptr;
    sm.af[0] = sc ? sc[0] : 1.0;
    sm.af[1] = sc ? sc[1] : 0.0;
    sm.af[2] = sc ? sc[2] : 0.0;
    sm.af[3] = (p.aff_on && p.aff.offset) ? p.aff.offset[(size_t)item * p.aff.offset_stride] : 0.0;
  }
  return af;
}

// K' = s1 K + s2 (1 - q_i)(1 - q_j) - s3 q_i q_j + offset  ==  s1 K + C_i - D_i q_j  with the per-row
// constants C_i = s2 (1 - q_i) + offset and D_i = s2 (1 - q_i) + s3 q_i: two FMAs per entry on the
// accumulator-load path (the re-association moves K' by a few 1e-16 of the rank-one terms, which are
// themselves ~1e-3 of K: far below the 1e-8 lnlike tolerance).
template <class SM>
__device__ __forceinline__ void aff_row_consts(const SM &sm, const AffRow &af, int gi, double &Ci, double &Di) {
  Ci = sm.af[3];
  Di = 0.0;
  if (af.norm) {
    const double qi = af.q[gi];
    const double a = sm.af[1] * (1.0 - qi);
    Ci += a;
    Di = a + sm.af[2] * qi;
  }
}

template <class SM>
__device__ __forceinline__ double aff_apply(const SM &sm, const AffRow &af, double k, double Ci,
                                            double Di, bool diag_row, int gi, int gc) {
  if (af.norm) k = fma(sm.af[0], k, fma(-Di, af.q[gc], Ci));
  else k += Ci;
  if (diag_row && gc == gi && af.dg) k += af.dg_vec ? af.dg[gi] : af.dg[0];  // sp.py:1135-1144
  return k;
}

// The affine arithmetic of a full-panel covariance row (rows of the diagonal block and below it), applied
// to accumulators that hold the raw K values: see aff_apply.
template <class SM>
__device__ __forceinline__ void aff_full_row(const SM &sm, const AffRow &af, bool diag_row, int gi, int v,
                                             int c0, int tg, double Ci, double Di, double (&accrow)[8][2]) {
  {
      if (af.norm) {
        const double s1 = sm.af[0];
        const double *qp = af.q + c0 + 2 * tg;
#pragma unroll
        for (int h = 0; h < 2; ++h) {   // two batches of 8 loads: bounded register footprint
          double q0[4], q1[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            q0[k] = __ldg(qp + (4 * h + k) * 8);
            q1[k] = __ldg(qp + (4 * h + k) * 8 + 1);
          }
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int nt = 4 * h + k;
            accrow[nt][0] = fma(s1, accrow[nt][0], fma(-Di, q0[k], Ci));
            accrow[nt][1] = fma(s1, accrow[nt][1], fma(-Di, q1[k], Ci));
          }
        }
      } else {
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          accrow[nt][0] += Ci;
          accrow[nt][1] += Ci;
        }
      }
      if (diag_row && af.dg) {   // data_cov on the diagonal (sp.py:1135-1144): column v of row v
        const double dgv = af.dg_vec ? af.dg[gi] : af.dg[0];
        const bool mine = ((v & 7) >> 1) == tg;
        // unconditional adds of a selected operand: a guarded `accrow[nt] += dgv` is turned into a
        // dynamically indexed access by the compiler, which sends the accumulators to local memory
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const bool hit = mine && nt == (v >> 3);
          accrow[nt][0] += (hit && !(v & 1)) ? dgv : 0.0;
          accrow[nt][1] += (hit && (v & 1)) ? dgv : 0.0;
        }
      }
    }
}

template <class SM, class RM>
__device__ __forceinline__ void init_acc(const SM &sm, const RM &rm, const AffRow &af, bool aff_on,
                                         int v, int c0, int tg, bool full, double (&accrow)[8][2]) {
  int kind;
  const double *p = rm.row(v, kind);
  const bool cov_row = aff_on && (kind == KIND_DIAG || kind == KIND_BELOW);
  const int gi = c0 + v;  // global row of a covariance row (diagonal-block and below rows alike)
  double Ci = 0.0, Di = 0.0;
  if (cov_row) aff_row_consts(sm, af, gi, Ci, Di);
  const bool diag_row = (kind == KIND_DIAG);
  if (full) {
    if (p == nullptr) p = rm.Kb;
    // all global loads first (no dependent instruction or branch in between: one batch of
    // outstanding requests per tile), then the branch-free affine arithmetic
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const double2 kv = *reinterpret_cast<const double2 *>(p + c0 + nt * 8 + 2 * tg);
      accrow[nt][0] = kv.x;
      accrow[nt][1] = kv.y;
    }
    if (cov_row) aff_full_row(sm, af, diag_row, gi, v, c0, tg, Ci, Di, accrow);
    return;
  }
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int col = nt * 8 + 2 * tg;
    const int gc = c0 + col;
    double k0 = 0.0, k1 = 0.0;
    if (kind == KIND_PAD) {
      k0 = (col == v) ? 1.0 : 0.0;
      k1 = (col + 1 == v) ? 1.0 : 0.0;
    } else if (kind != KIND_NONE && gc < rm.n) {
      // ld is even and the base 16-byte aligned: (gc, gc+1) is one aligned 16-byte load that stays
      // inside the row
      const double2 kv = *reinterpret_cast<const double2 *>(p + gc);
      k0 = kv.x;
      k1 = (gc + 1 < rm.n) ? kv.y : 0.0;
      if (cov_row) {
        k0 = aff_apply(sm, af, k0, Ci, Di, diag_row, gi, gc);
        if (gc + 1 < rm.n) k1 = aff_apply(sm, af, k1, Ci, Di, diag_row, gi, gc + 1);
      }
      if (kind == KIND_DIAG) {
        if (col > v) k0 = 0.0;
        if (col + 1 > v) k1 = 0.0;
      }
    }
    accrow[nt][0] = k0;
    accrow[nt][1] = k1;
  }
}

// ------------------------------------------------------------------------------------------
// acc(16 rows x 64 cols per warp) -= sum_k A[v0 + rows][k] * L[c0 + cols][k],  k in [0, c0)
//
// 3-slot cp.async ring handed off through mbarriers instead of __syncthreads: every thread's
// copies of a chunk arrive on full[slot] when they land (cp.async.mbarrier.arrive.noinc), a warp
// starts on a chunk as soon as that barrier flips and releases the slot on empty[slot] when its
// fragments are read, and the copies of chunk c+1 are issued (behind empty[slot], i.e. once every
// warp is past chunk c-2) before chunk c is consumed.  Warps therefore never rendezvous inside
// the k-loop: one may run a full chunk ahead of the slowest.  `it` is the CTA-uniform running chunk
// count (slot = it % 3, barrier phase = it / 3) and persists across tiles, panels and matrices.
// Warps whose 16 rows are all beyond the last virtual row keep feeding the ring but issue no
// tensor work.
// ------------------------------------------------------------------------------------------
// lim0 < 8 (warp w of the diagonal block): only the first lim0 = 2 w + 2 8-column groups reach the
// diagonal, the rest of the warp tile is never consumed and is not multiplied.
// `init` loads (and, on the fused path, transforms) the accumulators; it runs AFTER the first two
// chunks have been requested so that its global-load latency -- and the dependent affine FMAs --
// overlap the cp.async prologue instead of preceding it.
template <class Init>
__device__ __forceinline__ void gemm_tile(Smem &sm, const RowMap &rm, int v0, int c0, int nvirt,
                                          bool diag_tile, unsigned &it, double (&acc)[2][8][2],
                                          Init init, const CUtensorMap *tmK = nullptr,
                                          int item = 0) {
  constexpr int LA = STAGES - 1;
  constexpr int RPP = NTHREADS / 8;      // rows covered by one pass of the per-thread copies
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, tg = lane & 3;
  const int nchunks = c0 / KC;
  const bool diag_warp = diag_tile && warp < 4;
  const int lim0 = diag_warp ? 2 * warp + 2 : 8;
  if (nchunks == 0) {
    init();
    return;
  }
  const bool warp_live = diag_warp || (v0 + warp * 16) < nvirt;

  // this thread's cp.async assignments: A: TM / RPP x 16B, B: NB / RPP x 16B per chunk
  const int seg = tid & 7;                 // 16-byte chunk of the 128-byte row segment
  const int r8 = tid >> 3;                 // 0 .. RPP - 1
  const int sseg = (seg ^ (r8 & 7)) << 1;  // swizzled element offset (row & 7 == r8 & 7: RPP % 8 == 0)
  const double *arow[TM / RPP];
  int abytes[TM / RPP];
#pragma unroll
  for (int i = 0; i < TM / RPP; ++i) {
    int kind;
    double *p = rm.row(v0 + r8 + RPP * i, kind);
    arow[i] = p ? p : rm.Kb;
    abytes[i] = p ? 16 : 0;
  }
  const double *brow[NB / RPP];
  int bbytes[NB / RPP];
#pragma unroll
  for (int i = 0; i < NB / RPP; ++i) {
    int r = c0 + r8 + RPP * i;
    brow[i] = (r < rm.n) ? rm.Kb + (size_t)r * rm.ld : rm.Kb;
    bbytes[i] = (r < rm.n) ? 16 : 0;
  }
  // Tiles whose 128 rows are all rows of K (no appended right-hand-side or padding rows) are
  // fetched by TMA: one thread requests the 128 x 16 and 64 x 16 operand boxes (three
  // cp.async.bulk.tensor of 64 rows each; rows of the B box past the matrix are zero-filled by the
  // tensor map), every other thread only arrives on the barrier.
  const bool tma_tile = tmK != nullptr && rm.mode == MODE_FACTOR && (c0 + v0 + TM <= rm.n);
  // slot / phase of running chunk number x
  auto issue = [&](int ch, unsigned x, bool blocking) -> bool {
    const unsigned st = x % STAGES;
    // previous user of the slot fully read by every warp?
    if (blocking) mbar_wait(&sm.empty[st], ((x / STAGES) + 1u) & 1u);
    else if (!mbar_test(&sm.empty[st], ((x / STAGES) + 1u) & 1u)) return false;
    if (tma_tile) {
      if (tid == 0) {
        mbar_arrive_expect_tx(&sm.full[st], (TM + NB) * KC * (unsigned)sizeof(double));
#pragma unroll
        for (int bx = 0; bx < TM / 64; ++bx)   // boxes of 64 rows x 16 columns
          tma_load_3d(&sm.As[st][64 * bx][0], tmK, &sm.full[st], ch * KC, c0 + v0 + 64 * bx, item);
        tma_load_3d(&sm.Bs[st][0][0], tmK, &sm.full[st], ch * KC, c0, item);
      } else {
        mbar_arrive(&sm.full[st]);
      }
      return true;
    }
    const int k0 = ch * KC + seg * 2;
#pragma unroll
    for (int i = 0; i < TM / RPP; ++i) cp_async16(&sm.As[st][r8 + RPP * i][sseg], arow[i] + k0, abytes[i]);
#pragma unroll
    for (int i = 0; i < NB / RPP; ++i) cp_async16(&sm.Bs[st][r8 + RPP * i][sseg], brow[i] + k0, bbytes[i]);
    mbar_cp_async_arrive(&sm.full[st]);
    return true;
  };

  // per-lane fragment offsets inside a stage row: element (row g, k = 4 kk + tg)
  int koff[KC / 4];
#pragma unroll
  for (int kk = 0; kk < KC / 4; ++kk) koff[kk] = swz(g, kk * 4 + tg);

#pragma unroll
  for (int j = 0; j < LA; ++j)
    if (j < nchunks) issue(j, it + j, true);
  init();
  for (int ch = 0; ch < nchunks; ++ch) {
    const unsigned x = it + ch;
    const unsigned st = x % STAGES;
    // chunk ch + LA goes to the slot of chunk ch - 1.  If every warp is already past that chunk the
    // copies are issued NOW (LA chunks of latency cover); otherwise after this chunk's math (one
    // chunk less, but a warp never waits for a sibling that is at most one chunk behind).
    bool early = false;
    if (ch + LA < nchunks) early = issue(ch + LA, x + LA, false);
    mbar_wait(&sm.full[st], (x / STAGES) & 1u);  // chunk ch landed, for every thread's copies
    if (warp_live) {
      const double *Bw = &sm.Bs[st][g][0];
      const double *Aw = &sm.As[st][warp * 16 + g][0];
      if (lim0 >= 8) {
#pragma unroll
        for (int kk = 0; kk < KC / 4; ++kk) {
          double a[2], b[8];
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) a[mt] = negate(Aw[mt * 8 * KC + koff[kk]]);
#pragma unroll
          for (int nt = 0; nt < 8; ++nt) b[nt] = Bw[nt * 8 * KC + koff[kk]];
#pragma unroll
          for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) dmma_m8n8k4(acc[mt][nt][0], acc[mt][nt][1], a[mt], b[nt]);
        }
      } else {
#pragma unroll
        for (int kk = 0; kk < KC / 4; ++kk) {
          double a[2];
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) a[mt] = negate(Aw[mt * 8 * KC + koff[kk]]);
#pragma unroll
          for (int nt = 0; nt < 8; ++nt) {
            if (nt < lim0) {
              const double b = Bw[nt * 8 * KC + koff[kk]];
#pragma unroll
              for (int mt = 0; mt < 2; ++mt) dmma_m8n8k4(acc[mt][nt][0], acc[mt][nt][1], a[mt], b);
            }
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&sm.empty[st]);
    if (!early && ch + LA < nchunks) issue(ch + LA, x + LA, true);
  }
  it += nchunks;
}

// Accumulator fragment (8x8, C layout) -> A fragment of its k-block q (columns 4q..4q+3).
__device__ __forceinline__ double c_to_a(double d0, double d1, int q, int lane) {
  const int tg = lane & 3;
  const int src = (lane & ~3) | (2 * q + (tg >> 1));
  const double v0 = __shfl_sync(0xffffffffu, d0, src);
  const double v1 = __shfl_sync(0xffffffffu, d1, src);
  return (tg & 1) ? v1 : v0;
}

// In-register TRSM on the tensor pipe for the two 8-row m-tiles of a warp.  On entry acc holds
// P; on exit acc holds X = P L_jj^-T.  RIGHT-looking 8x8-blocked substitution: as soon as the
// block column X_kb = P_kb Dinv_kb^T is known it is pushed into every later block,
// P_nb -= X_kb L[nb,kb]^T, so each step issues 4 (7 - kb) independent DMMAs and only two A
// fragments per m-tile are live (the left-looking form kept all 16 and serialised 2 nb DMMAs).
template <class SM>
__device__ __forceinline__ void trsm_warp(const SM &sm, double (&acc)[2][8][2], int lane) {
  const int g = lane >> 2, tg = lane & 3;
#pragma unroll
  for (int kb = 0; kb < 8; ++kb) {
    double xa[2][2];
    const double d0 = sm.Dv[kb * 8 + g][tg], d1 = sm.Dv[kb * 8 + g][4 + tg];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const double a0 = c_to_a(acc[mt][kb][0], acc[mt][kb][1], 0, lane);
      const double a1 = c_to_a(acc[mt][kb][0], acc[mt][kb][1], 1, lane);
      double x0 = 0.0, x1 = 0.0;
      dmma_m8n8k4(x0, x1, a0, d0);
      dmma_m8n8k4(x0, x1, a1, d1);
      acc[mt][kb][0] = x0;
      acc[mt][kb][1] = x1;
      xa[mt][0] = negate(c_to_a(x0, x1, 0, lane));
      xa[mt][1] = negate(c_to_a(x0, x1, 1, lane));
    }
#pragma unroll
    for (int nb = kb + 1; nb < 8; ++nb) {
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const double b = sm.Ld.at(nb * 8 + g, kb * 8 + q * 4 + tg);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) dmma_m8n8k4(acc[mt][nb][0], acc[mt][nb][1], xa[mt][q], b);
      }
    }
  }
}

// Store X rows (below-diagonal rows of L, or y rows of the RHS) and accumulate |y|^2.
// Called by all 32 lanes of a warp (the shuffles are unconditional).
__device__ __forceinline__ void store_rows(const RowMap &rm, int v, int c0, int tg,
                                           const double (&accrow)[8][2], double &quad_part,
                                           double *quad_out) {
  int kind;
  double *p = rm.row(v, kind);
  const bool live = (kind == KIND_BELOW || kind == KIND_RHS);
  double q = 0.0;
  if (live) {
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int gc = c0 + nt * 8 + 2 * tg;
      if (gc + 1 < rm.n) {
        *reinterpret_cast<double2 *>(p + gc) = make_double2(accrow[nt][0], accrow[nt][1]);
        q += accrow[nt][0] * accrow[nt][0] + accrow[nt][1] * accrow[nt][1];
      } else if (gc < rm.n) {
        p[gc] = accrow[nt][0];
        q += accrow[nt][0] * accrow[nt][0];
      }
    }
  }
  if (kind != KIND_RHS) q = 0.0;
  quad_part += q;
  if (quad_out) {  // uniform across the grid
    // the 4 lanes of a quad share the row: reduce before the atomic
    q += __shfl_xor_sync(0xffffffffu, q, 1);
    q += __shfl_xor_sync(0xffffffffu, q, 2);
    if (kind == KIND_RHS && tg == 0) {
      const int m = (rm.mode == MODE_FACTOR) ? (v - NB - rm.nbelow) : (rm.rb + v);
      atomicAdd(quad_out + m, q);
    }
  }
}

// The inverses of the eight 8x8 diagonal blocks of sm.Ld: thread (blk, c) with c < 8 -> column c of
// block blk (MODE_SOLVE only).
template <class SM>
__device__ __forceinline__ void diag_inverses(SM &sm) {
  const int tid = threadIdx.x;
  if (tid < 64) {
    const int blk = tid >> 3, c = tid & 7;
    const int o = blk * 8;
    double x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      double sacc = (i == c) ? 1.0 : 0.0;
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (k < i && k >= c) sacc -= sm.Ld.at(o + i, o + k) * x[k];
      x[i] = (i >= c) ? sacc / sm.Ld.at(o + i, o + i) : 0.0;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) sm.Dv[o + i][c] = x[i];
  }
  __syncthreads();
}

// ---- reciprocal / reciprocal square root for the pivot chain ---------------------------------
// MUFU seed (~2^-20) + two Newton steps on the FMA pipe: 1 + 4 dependent instructions instead of the
// ~12 of an IEEE division, ~1 ulp.  The pivot recurrence d_{k+1} = a - v^2 / d_k is the serial
// spine of the whole factorisation, and its FP64 instructions queue behind the sibling CTA's DMMAs.
__device__ __forceinline__ double fast_rcp(double d) {
  double x;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
  double e = fma(-d, x, 1.0);
  x = fma(x, e, x);
  e = fma(-d, x, 1.0);
  return fma(x, e, x);
}
__device__ __forceinline__ double fast_rsqrt(double d) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
  double e = fma(-d * y, y, 1.0);
  y = fma(0.5 * y, e, y);
  e = fma(-d * y, y, 1.0);
  return fma(0.5 * y, e, y);
}

__device__ __forceinline__ void bar_diag() {  // warps 0-3 only (named barrier 1)
  asm volatile("bar.sync 1, 128;\n" ::: "memory");
}

// Cholesky of ONE 8x8 tile held in the accumulator layout of a warp (lane (g, tg): row g, columns
// 2 tg, 2 tg + 1), entirely with shuffles: no shared memory, no barrier, no branch.  Gaussian
// elimination without scaling (v_ik = L_ik sqrt(d_k)), the same row operations applied to an
// identity tile, so that L = V diag(d^-1/2) and L^-1 = diag(d^-1/2) W come out together.
// The serial spine is the pivot recurrence d_{k+1} = a_{k+1,k+1} - v_{k+1,k}^2 / d_k; every lane
// carries it redundantly from two values broadcast BEFORE 1/d_k is known, so one pivot costs
// rcp -> mul -> fma and no shuffle or select sits on the chain.  The square roots are taken once,
// lane-parallel, at the end.  The strictly upper part of the tile may be garbage (lower-only
// assembly): it is never used (selects, not multiplications by zero, mask it).
//   on exit: (v0, v1) = L tile, (w0, w1) = L^-1 tile (upper triangle exactly 0), returns d_g
__device__ __forceinline__ double potf2_tile8(double &v0, double &v1, double &w0, double &w1, int lane,
                                              bool &bad) {
  const int g = lane >> 2, tg = lane & 3;
  w0 = (2 * tg == g) ? 1.0 : 0.0;
  w1 = (2 * tg + 1 == g) ? 1.0 : 0.0;
  double d = __shfl_sync(0xffffffffu, v0, 0);  // d_0
  double dmine = 1.0;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    bad = bad || !(d > 0.0);  // also NaN; the matrix is flagged, its numbers are left to rot
    dmine = (g == k) ? d : dmine;
    if (k < 7) {
      const double vk = (k & 1) ? v1 : v0;             // register holding column k
      const double vn = ((k + 1) & 1) ? v1 : v0;       // register holding column k + 1
      const double vik = __shfl_sync(0xffffffffu, vk, (lane & ~3) | (k >> 1));  // v_{g,k}
      const double vj0 = __shfl_sync(0xffffffffu, vk, 8 * tg + (k >> 1));       // v_{2tg,k}
      const double vj1 = __shfl_sync(0xffffffffu, vk, 8 * tg + 4 + (k >> 1));   // v_{2tg+1,k}
      const double wk0 = __shfl_sync(0xffffffffu, w0, 4 * k + tg);
      const double wk1 = __shfl_sync(0xffffffffu, w1, 4 * k + tg);
      const double pk = __shfl_sync(0xffffffffu, vk, 4 * (k + 1) + (k >> 1));        // v_{k+1,k}
      const double qk = __shfl_sync(0xffffffffu, vn, 4 * (k + 1) + ((k + 1) >> 1));  // a_{k+1,k+1}
      const double r = fast_rcp(d);
      d = fma(-(pk * r), pk, qk);
      const double m = (g > k) ? vik * r : 0.0;
      v0 = fma(-m, (2 * tg > k) ? vj0 : 0.0, v0);
      v1 = fma(-m, (2 * tg + 1 > k) ? vj1 : 0.0, v1);
      w0 = fma(-m, wk0, w0);
      w1 = fma(-m, wk1, w1);
    }
  }
  const double rs_row = fast_rsqrt(dmine);
  const double rs_c0 = __shfl_sync(0xffffffffu, rs_row, 8 * tg);
  const double rs_c1 = __shfl_sync(0xffffffffu, rs_row, 8 * tg + 4);
  v0 *= rs_c0;
  v1 *= rs_c1;
  w0 *= rs_row;
  w1 *= rs_row;
  return dmine;
}

// 64x64 Cholesky of the diagonal block, IN THE ACCUMULATOR REGISTERS of warps 0-3 (warp w holds
// rows 16 w .. 16 w + 15 of P = K_jj - L L^T as 2 x 8 accumulator tiles).  Two-level: for each of the
// 8 sub-panels s the owner warp factors the 8x8 diagonal tile with shuffles (potf2_tile8) and
// publishes L_ss and L_ss^-1; every warp solves its tiles below on the tensor pipe
// (X = P L_ss^-T, two DMMAs per tile) and publishes X; the trailing update P_ij -= X_i X_j^T is DMMA
// again.  Only column s + 1 is updated on the critical path; the update of the later columns is
// deferred until after the next diagonal tile has been factored, so the serial spine per sub-panel
// is  8 pivots -> barrier -> 2 DMMAs -> barrier -> 2 DMMAs.  Warps 4-7 (rows below the block) keep
// their accumulators in registers and wait at the CTA barrier that follows.
// Produces sm.Ld (lower; strictly-upper 8x8 tiles untouched), sm.Dv and the pivots sm.dpiv = L_ii^2.
template <class SM>
__device__ __forceinline__ void potf2_regs(SM &sm, double (&acc)[2][8][2], int warp, int lane) {
  const int g = lane >> 2, tg = lane & 3;
  // 8-row blocks of the diagonal tile held by this warp: m-tile mt -> block 2 warp + mt; block b lives
  // in columns 0 .. 8 b + 7
  const int rb[2] = {2 * warp, 2 * warp + 1};
  bool bad = false;
#pragma unroll
  for (int s = 0; s < 8; ++s) {
    // owner of diagonal tile s: warp s / 2, m-tile s % 2
    if (warp == (s >> 1)) {
      double w0, w1;
      double &t0 = acc[s & 1][s][0], &t1 = acc[s & 1][s][1];
      const double dg = potf2_tile8(t0, t1, w0, w1, lane, bad);
      *reinterpret_cast<double2 *>(&sm.Ld.at(8 * s + g, 8 * s + 2 * tg)) = make_double2(t0, t1);
      *reinterpret_cast<double2 *>(&sm.Dv[8 * s + g][2 * tg]) = make_double2(w0, w1);
      if (tg == 0) sm.dpiv[8 * s + g] = dg;
    }
    // deferred part of the previous sub-panel's update: columns beyond s.  The A fragments are
    // re-read from the published X (no registers held across the barriers).
    if (s > 0) {
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        double xq[2];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
          xq[mt] = negate(sm.Ld.at(8 * max(rb[mt], s) + g, 8 * (s - 1) + 4 * q + tg));
#pragma unroll
        for (int nt = s + 1; nt < 8; ++nt) {
          const double b = sm.Ld.at(8 * nt + g, 8 * (s - 1) + 4 * q + tg);
#pragma unroll
          for (int mt = 0; mt < 2; ++mt)
            if (nt <= rb[mt]) dmma_m8n8k4(acc[mt][nt][0], acc[mt][nt][1], xq[mt], b);
        }
      }
    }
    bar_diag();  // L_ss^-1 published
    double xa[2][2] = {{0.0, 0.0}, {0.0, 0.0}};  // -X fragments of this sub-panel
    {
      const double d0 = sm.Dv[8 * s + g][tg], d1 = sm.Dv[8 * s + g][4 + tg];
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        if (rb[mt] > s) {
          const double a0 = c_to_a(acc[mt][s][0], acc[mt][s][1], 0, lane);
          const double a1 = c_to_a(acc[mt][s][0], acc[mt][s][1], 1, lane);
          double x0 = 0.0, x1 = 0.0;
          dmma_m8n8k4(x0, x1, a0, d0);
          dmma_m8n8k4(x0, x1, a1, d1);
          acc[mt][s][0] = x0;
          acc[mt][s][1] = x1;
          *reinterpret_cast<double2 *>(&sm.Ld.at(8 * rb[mt] + g, 8 * s + 2 * tg)) =
              make_double2(x0, x1);
          xa[mt][0] = negate(c_to_a(x0, x1, 0, lane));
          xa[mt][1] = negate(c_to_a(x0, x1, 1, lane));
        }
      }
    }
    bar_diag();  // column block s of L_jj published
    if (s < 7) {  // critical path: column s + 1 only
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const double b = sm.Ld.at(8 * (s + 1) + g, 8 * s + 4 * q + tg);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
          if (s + 1 <= rb[mt])
            dmma_m8n8k4(acc[mt][s + 1][0], acc[mt][s + 1][1], xa[mt][q], b);
      }
    }
  }
  if (bad) sm.bad = 1;
}

// the 8 compute warps of the INT8 kernel (named barrier 2: its producer and issuer warps stay out)
__device__ __forceinline__ void cbar256() { asm volatile("bar.sync 2, 256;\n" ::: "memory"); }

// Sum of v over the 8 warps (256 threads) of a kernel: the whole CTA of the FP64 kernels, the compute
// warps of the INT8 kernel (I8: they meet at cbar256 instead of __syncthreads).
template <bool I8, class SM>
__device__ __forceinline__ double block_sum(SM &sm, double v) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  v = warp_sum(v);
  if (I8) cbar256(); else __syncthreads();
  if (lane == 0) sm.red[warp] = v;
  if (I8) cbar256(); else __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int w = 0; w < NTHREADS / 32; ++w) t += sm.red[w];
  if (I8) cbar256(); else __syncthreads();
  return t;
}

// lnlike, logdet and info of matrix `item` (MODE_FACTOR; called by one thread).  Flags raised by earlier
// stages (bounds, normalisation range, eigen-solve) also map to -inf; the `clear` bits belong to this
// launch and are recomputed: SPB_INFO_NOT_PD from `bad`, plus the bits in `set`.
__device__ __forceinline__ void lnlike_epilogue(const PotrfParams &p, int item, double quad, double logdet,
                                                bool bad, int clear, int set) {
  const int M = p.R ? p.M : 0;
  double ll = -0.5 * quad - (double)M * logdet - 0.5 * (double)p.n * (double)M * 1.8378770664093453;  // log(2 pi)
  const int prev = p.info ? (p.info[item] & ~clear) : 0;
  if (bad || (prev & SPB_INFO_NEG_INF) || ll != ll) ll = -INFINITY;
  if (p.lnlike) p.lnlike[item] = ll;
  if (p.logdet) p.logdet[item] = bad ? NAN : logdet;
  if (p.info) p.info[item] = prev | (bad ? SPB_INFO_NOT_PD : 0) | set;
}

// dynamic shared memory of the three Cholesky kernels (TMA 128-byte swizzle: 1 KB aligned)
extern __shared__ __align__(1024) unsigned char smem_raw[];

__global__ void __launch_bounds__(NTHREADS, 2)
    potrf_lnlike_kernel(PotrfParams p, const __grid_constant__ CUtensorMap tmK) {
  Smem &sm = *reinterpret_cast<Smem *>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, tg = lane & 3;

  int nitems;
  if (p.mode == MODE_FACTOR) nitems = p.B;
  else nitems = (p.M + p.rows_per_cta - 1) / p.rows_per_cta;

  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&sm.full[s], NTHREADS);
      mbar_init(&sm.empty[s], NTHREADS / 32);
    }
  }
  __syncthreads();
  unsigned it = 0;  // running k-chunk count of this CTA (ring slot / barrier phase)

  // Work items (matrices) beyond the first wave are claimed from a global counter: the two CTAs of
  // an SM drift in and out of phase (tensor-pipe phases overlapping or not), so CTA run times for
  // the same number of matrices differ by +-15 %; a static split would wait for the slowest.
  for (int item = blockIdx.x; item < nitems;) {
    if (p.only_flag && !(p.info[item] & p.only_flag)) {   // block-uniform: skip, claim the next matrix
      if (tid == 0) sm.next_item = (int)gridDim.x + (int)atomicAdd(p.counter, 1u);
      __syncthreads();
      item = sm.next_item;
      __syncthreads();
      continue;
    }
    RowMap rm;
    rm.n = p.n;
    rm.ld = p.ld;
    rm.ldr = p.ldr;
    rm.mode = p.mode;
    double *quad_out;
    if (p.mode == MODE_FACTOR) {
      rm.Kb = p.K + (size_t)item * p.strideK;
      rm.Rb = p.R ? p.R + (size_t)item * p.strideR : nullptr;
      rm.M = p.R ? p.M : 0;
      rm.rb = 0;
      rm.nrhs = rm.M;
      quad_out = p.quad ? p.quad + (size_t)item * p.M : nullptr;
    } else {
      rm.Kb = p.K;
      rm.Rb = p.R;
      rm.M = p.M;
      rm.rb = item * p.rows_per_cta;
      rm.nrhs = min(p.rows_per_cta, p.M - rm.rb);
      quad_out = p.quad;
    }
    const AffRow af = aff_setup(p, item, sm, tid);   // aff_on == 0 in MODE_SOLVE
    if (tid == 0) sm.bad = 0;
    if (quad_out) {
      if (p.mode == MODE_FACTOR) {
        for (int m = tid; m < rm.M; m += NTHREADS) quad_out[m] = 0.0;
      } else {
        for (int m = tid; m < rm.nrhs; m += NTHREADS) quad_out[rm.rb + m] = 0.0;
      }
    }
    __syncthreads();

    double logdet_part = 0.0, quad_part = 0.0;
    double acc[2][8][2];

    for (int c0 = 0; c0 < p.n; c0 += NB) {
      rm.c0 = c0;
      rm.nbelow = max(0, p.n - c0 - NB);
      const int nvirt = (p.mode == MODE_FACTOR) ? NB + rm.nbelow + rm.M : rm.nrhs;
      const bool full_panel = (c0 + NB <= p.n);
      if (p.mode == MODE_SOLVE) {
        // fetch L_jj (identity-padded) and invert its 8x8 diagonal blocks
        for (int idx = tid; idx < NB * NB; idx += NTHREADS) {
          const int i = idx >> 6, j = idx & 63;
          double v = 0.0;
          if (j <= i) {
            if (c0 + i < p.n) v = rm.Kb[(size_t)(c0 + i) * p.ld + c0 + j];
            else v = (i == j) ? 1.0 : 0.0;
          }
          sm.Ld.at(i, j) = v;
        }
        __syncthreads();
        diag_inverses(sm);
      }
      for (int v0 = 0; v0 < nvirt; v0 += TM) {
        // MODE_FACTOR, first tile: rows 0..63 are the diagonal block (warps 0-3), rows 64..127 the
        // first rows below it (warps 4-7)
        const bool diag_tile = (p.mode == MODE_FACTOR) && (v0 == 0);
        gemm_tile(sm, rm, v0, c0, nvirt, diag_tile, it, acc, [&]() {
#pragma unroll
          for (int mt = 0; mt < 2; ++mt)
            init_acc(sm, rm, af, p.aff_on != 0, v0 + warp * 16 + mt * 8 + g, c0, tg, full_panel, acc[mt]);
        }, p.use_tma ? &tmK : nullptr, item);   // acc = K - L L^T = P
        if (diag_tile) {
          if (warp < 4) potf2_regs(sm, acc, warp, lane);
          __syncthreads();  // L_jj and the inverses of its diagonal tiles are in shared memory
          if (tid < min(NB, p.n - c0)) logdet_part += 0.5 * log(sm.dpiv[tid]);
          // write L_jj back (lower triangle, valid rows/cols only)
          for (int idx = tid; idx < NB * NB; idx += NTHREADS) {
            const int i = idx >> 6, j = idx & 63;
            if (j <= i && c0 + i < p.n) rm.Kb[(size_t)(c0 + i) * p.ld + c0 + j] = sm.Ld.at(i, j);
          }
        }
        if (!(diag_tile && warp < 4) && (v0 + warp * 16) < nvirt) {
          trsm_warp(sm, acc, lane);
#pragma unroll
          for (int mt = 0; mt < 2; ++mt)
            store_rows(rm, v0 + warp * 16 + mt * 8 + g, c0, tg, acc[mt], quad_part, quad_out);
        }
      }
      // this thread's st.global of the panel (store_rows, the L_jj write-back) must be visible to the
      // async proxy before any thread requests them through TMA in a later panel
      fence_proxy_async_global();
      __syncthreads();  // Ld/Dv are rewritten by the next panel; global writes of this panel done
      __threadfence_block();
    }

    // ---- reductions -> lnlike
    const double quad = block_sum<false>(sm, quad_part);
    const double logdet = block_sum<false>(sm, logdet_part);
    if (p.mode == MODE_FACTOR && tid == 0)
      lnlike_epilogue(p, item, quad, logdet, sm.bad != 0, SPB_INFO_NOT_PD | p.only_flag, 0);
    if (tid == 0) sm.next_item = (int)gridDim.x + (int)atomicAdd(p.counter, 1u);
    __syncthreads();
    item = sm.next_item;
  }
}

#include "potrf_i8.cuh"

// ------------------------------------------------------------------------------------------
// Small batches (B <= #SM / 2): ONE MATRIX PER THREAD-BLOCK CLUSTER of 8, 4 or 2 CTAs (SMs).
//
// A lone CTA needs 2.3 ms for a 1000 x 1000 matrix (one SM's tensor pipe, every serial phase
// exposed), which is the whole latency of a single log-likelihood evaluation -- the regime of a
// single MCMC chain, of predict() and of the conditional samplers.  Here the 128-row tiles of a
// panel are dealt round-robin to the CTAs of a cluster: all k-loops of a panel run concurrently on
// different SMs, CTA 0 owns the diagonal tile (k-loop, in-register factorisation, L_jj written to
// global memory), and two cluster barriers per panel (release / acquire: they order the global
// writes) separate  "L_jj published"  and  "panel complete".  The other CTAs copy L_jj and the
// inverses of its diagonal tiles out of CTA 0's shared memory (DSMEM) and run the same in-register
// TRSM.  Same device functions, same operands per tile as the batch kernel: the factor and the
// solved rows are bit-identical to it (lnlike to rounding: |y|^2 is summed per CTA).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned cluster_rank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_barrier() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n"
               "barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}

template <int CLUSTER>
__global__ void __launch_bounds__(NTHREADS, 1) potrf_cluster_kernel(PotrfParams p) {
  Smem &sm = *reinterpret_cast<Smem *>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, tg = lane & 3;
  const int rank = (int)cluster_rank();
  const int item = blockIdx.x / CLUSTER;

  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&sm.full[s], NTHREADS);
      mbar_init(&sm.empty[s], NTHREADS / 32);
    }
    sm.bad = 0;
  }
  unsigned it = 0;

  RowMap rm;
  rm.n = p.n;
  rm.ld = p.ld;
  rm.ldr = p.ldr;
  rm.mode = MODE_FACTOR;
  rm.Kb = p.K + (size_t)item * p.strideK;
  rm.Rb = p.R ? p.R + (size_t)item * p.strideR : nullptr;
  rm.M = p.R ? p.M : 0;
  rm.rb = 0;
  rm.nrhs = rm.M;
  double *quad_out = p.quad ? p.quad + (size_t)item * p.M : nullptr;
  const AffRow af = aff_setup(p, item, sm, tid);
  // per-RHS accumulators are zeroed by CTA 0 before the first "L_jj published" barrier; every
  // contribution is added after it
  if (quad_out && rank == 0)
    for (int m = tid; m < rm.M; m += NTHREADS) quad_out[m] = 0.0;
  __syncthreads();

  double logdet_part = 0.0, quad_part = 0.0;
  double acc[2][8][2];

  for (int c0 = 0; c0 < p.n; c0 += NB) {
    rm.c0 = c0;
    rm.nbelow = max(0, p.n - c0 - NB);
    const int nvirt = NB + rm.nbelow + rm.M;
    const int ntiles = (nvirt + TM - 1) / TM;
    const bool full_panel = (c0 + NB <= p.n);
    const bool have_tile = rank < ntiles;
    // ---- first tile of this CTA: k-loop (needs nothing from this panel)
    if (have_tile) {
      const int v0 = rank * TM;
      gemm_tile(sm, rm, v0, c0, nvirt, rank == 0, it, acc, [&]() {
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
          init_acc(sm, rm, af, p.aff_on != 0, v0 + warp * 16 + mt * 8 + g, c0, tg, full_panel, acc[mt]);
      });
    }
    if (rank == 0) {
      if (warp < 4) potf2_regs(sm, acc, warp, lane);
      __syncthreads();
      if (tid < min(NB, p.n - c0)) logdet_part += 0.5 * log(sm.dpiv[tid]);
      for (int idx = tid; idx < NB * NB; idx += NTHREADS) {
        const int i = idx >> 6, j = idx & 63;
        if (j <= i && c0 + i < p.n) rm.Kb[(size_t)(c0 + i) * p.ld + c0 + j] = sm.Ld.at(i, j);
      }
      __threadfence();
    }
    cluster_barrier();   // L_jj published
    if (rank != 0 && have_tile) {
      // L_jj and the inverses of its 8x8 diagonal tiles straight from CTA 0's shared memory
      // (distributed shared memory; Ld and Dv are adjacent in Smem): the same operands as CTA 0
      // and the batch kernel use, hence bit-identical rows, and no second trip through L2
      const double2 *src = reinterpret_cast<const double2 *>(
          cg::this_cluster().map_shared_rank(&sm.Ld.v[0], 0));
      double2 *dst = reinterpret_cast<double2 *>(&sm.Ld.v[0]);
      for (int idx = tid; idx < (int)((sizeof(sm.Ld) + sizeof(sm.Dv)) / sizeof(double2)); idx += NTHREADS)
        dst[idx] = src[idx];
      __syncthreads();
    }
    // ---- finish the first tile, then any further tiles of this CTA
    for (int ti = rank; ti < ntiles; ti += CLUSTER) {
      const int v0 = ti * TM;
      if (ti != rank) {
        gemm_tile(sm, rm, v0, c0, nvirt, false, it, acc, [&]() {
#pragma unroll
          for (int mt = 0; mt < 2; ++mt)
            init_acc(sm, rm, af, p.aff_on != 0, v0 + warp * 16 + mt * 8 + g, c0, tg, full_panel, acc[mt]);
        });
      }
      if (!(ti == 0 && warp < 4) && (v0 + warp * 16) < nvirt) {
        trsm_warp(sm, acc, lane);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
          store_rows(rm, v0 + warp * 16 + mt * 8 + g, c0, tg, acc[mt], quad_part, quad_out);
      }
    }
    __threadfence();
    cluster_barrier();   // panel complete: its columns are visible to every CTA of the cluster
  }

  const double quad = block_sum<false>(sm, quad_part);
  const double logdet = block_sum<false>(sm, logdet_part);   // non-zero in CTA 0 only
  // deterministic reduction: one partial per CTA, summed by CTA 0 in rank order
  if (tid == 0) p.scratch[(size_t)item * CLUSTER + rank] = quad;
  __threadfence();
  cluster_barrier();
  if (rank == 0 && tid == 0) {
    double qtot = 0.0;
#pragma unroll
    for (int r = 0; r < CLUSTER; ++r) qtot += __ldcg(p.scratch + (size_t)item * CLUSTER + r);
    lnlike_epilogue(p, item, qtot, logdet, sm.bad != 0, SPB_INFO_NOT_PD | p.only_flag, 0);
  }
}

// cluster sizes of potrf_cluster_kernel, largest first (the order of spb_context::max_active_clusters)
struct ClusterKernel {
  int size;
  void (*kernel)(PotrfParams);
};
constexpr ClusterKernel CLUSTER_KERNELS[3] = {
    {8, potrf_cluster_kernel<8>}, {4, potrf_cluster_kernel<4>}, {2, potrf_cluster_kernel<2>}};

// ------------------------------------------------------------------------------------------
// DMMA peak micro-benchmark: 8 warps x 16 independent accumulator tiles, operands in registers.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256, 2) dmma_peak_kernel(int iters, double *sink) {
  double acc[16][2];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i][0] = acc[i][1] = 0.0;
  double a = 1.0 + threadIdx.x * 1e-9, b = 1.0 - threadIdx.x * 1e-9;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) dmma_m8n8k4(acc[i][0], acc[i][1], a, b);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += acc[i][0] + acc[i][1];
  if (s == 123.456) sink[0] = s;
}

}  // namespace

// PotrfParams of a MODE_FACTOR launch; affine == nullptr: no fused affine map
static PotrfParams factor_params(int B, int nt, double *K, int ldk, long long K_stride,
                                 const spb_affine *affine, int M, double *resid, int ldr,
                                 long long resid_stride, double *lnlike, double *quad, double *logdet,
                                 int32_t *info) {
  PotrfParams p = {};
  p.K = K;
  p.n = nt;
  p.ld = ldk;
  p.strideK = K_stride;
  p.R = (M > 0) ? resid : nullptr;
  p.M = M;
  p.ldr = ldr;
  p.strideR = resid_stride;
  p.lnlike = lnlike;
  p.quad = quad;
  p.logdet = logdet;
  p.info = info;
  p.B = B;
  p.mode = MODE_FACTOR;
  p.aff = affine ? *affine : spb_affine{};
  p.aff_on = affine ? 1 : 0;
  return p;
}

// the layout every kernel of this file assumes: 16-byte loads of (column, column + 1) pairs
static int check_layout(const PotrfParams &p) {
  SPB_REQUIRE(p.n > 0 && p.B > 0, "cholesky: empty problem");
  SPB_REQUIRE(p.ld >= p.n && (p.ld % 2) == 0, "cholesky: ldk must be even and >= nt");
  SPB_REQUIRE(((uintptr_t)p.K % 16) == 0 && (p.strideK % 2) == 0,
              "cholesky: K must be 16-byte aligned with an even batch stride");
  if (p.R) {
    SPB_REQUIRE(p.ldr >= p.n && (p.ldr % 2) == 0, "cholesky: ldr must be even and >= nt");
    SPB_REQUIRE(((uintptr_t)p.R % 16) == 0 && (p.strideR % 2) == 0,
                "cholesky: resid must be 16-byte aligned with an even batch stride");
  }
  return 0;
}

// the next work counter of the context's ring, zeroed in-stream
static int claim_counter(spb_context *ctx, void *stream, unsigned int **counter) {
  *counter = ctx->d_counters + (__atomic_fetch_add(&ctx->counter_next, 1u, __ATOMIC_RELAXED) % SPB_NUM_COUNTERS);
  SPB_CHECK_CUDA(cudaMemsetAsync(*counter, 0, sizeof(unsigned int), (cudaStream_t)stream));
  return 0;
}

static int potrf_launch(spb_context *ctx, PotrfParams &p, void *stream) {
  if (const int st = check_layout(p)) return st;
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  p.scratch = nullptr;
  const size_t smem = sizeof(Smem);   // batch and cluster kernel
  static spb_once_flag attr_once;
  {
    const int st = spb_once_per_device(attr_once, ctx->device, [&]() -> int {
      SPB_CHECK_CUDA(cudaFuncSetAttribute(potrf_lnlike_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)smem));
      SPB_CHECK_CUDA(cudaFuncSetAttribute(potrf_lnlike_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                          cudaSharedmemCarveoutMaxShared));
      for (const ClusterKernel &ck : CLUSTER_KERNELS)
        SPB_CHECK_CUDA(cudaFuncSetAttribute(ck.kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      return 0;
    });
    if (st) return st;
  }
  int nitems = (p.mode == MODE_FACTOR) ? p.B : (p.M + p.rows_per_cta - 1) / p.rows_per_cta;
  // few matrices: one 8-CTA cluster per matrix instead of one CTA (see potrf_cluster_kernel).  The
  // cluster kernel factors every matrix of the batch: never for a pass restricted by only_flag.
  int k_cs = -1;
  if (!ctx->opt_no_cluster && p.mode == MODE_FACTOR && p.only_flag == 0 && p.n > 2 * 128 && ctx->d_scratch &&
      p.B * 2 <= ctx->num_sms) {
    // largest cluster size whose clusters are all co-resident (a second wave of clusters would
    // cost more than a smaller cluster: GPCs host a whole number of clusters), asked of the driver
    static std::mutex occ_mu;
    {
      std::lock_guard<std::mutex> lock(occ_mu);
      if (ctx->max_active_clusters[0] < 0) {
        for (int k = 0; k < 3; ++k) {
          const int c = CLUSTER_KERNELS[k].size;
          cudaLaunchConfig_t q = {};
          q.gridDim = dim3((unsigned)(c * ctx->num_sms));
          q.blockDim = dim3(NTHREADS);
          q.dynamicSmemBytes = smem;
          cudaLaunchAttribute a[1];
          a[0].id = cudaLaunchAttributeClusterDimension;
          a[0].val.clusterDim.x = (unsigned)c;
          a[0].val.clusterDim.y = 1;
          a[0].val.clusterDim.z = 1;
          q.attrs = a;
          q.numAttrs = 1;
          int n = 0;
          const cudaError_t e = cudaOccupancyMaxActiveClusters(&n, CLUSTER_KERNELS[k].kernel, &q);
          ctx->max_active_clusters[k] = (e == cudaSuccess) ? n : 0;
        }
        (void)cudaGetLastError();
      }
    }
    // a cluster size is eligible only if its per-CTA partial sums fit the launch's scratch slot;
    // otherwise fall through to the next size and finally to the one-CTA-per-matrix kernel
    for (int k = 0; k < 3 && k_cs < 0; ++k)
      if (p.B <= ctx->max_active_clusters[k] && CLUSTER_KERNELS[k].size * p.B <= SPB_SCRATCH_PER_SLOT) k_cs = k;
  }
  if (k_cs >= 0) {
    const int cs = CLUSTER_KERNELS[k_cs].size;
    const unsigned slot = __atomic_fetch_add(&ctx->counter_next, 1u, __ATOMIC_RELAXED) % SPB_NUM_COUNTERS;
    p.scratch = ctx->d_scratch + (size_t)slot * SPB_SCRATCH_PER_SLOT;
    p.counter = nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(p.B * cs));
    cfg.blockDim = dim3(NTHREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cs;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SPB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, CLUSTER_KERNELS[k_cs].kernel, p));
    SPB_LAUNCH_CHECK(ctx);
    return 0;
  }
  int grid = nitems < 2 * ctx->num_sms ? nitems : 2 * ctx->num_sms;   // 2 CTAs per SM
  // tensor map of the batch of matrices for the TMA-fed operand ring: (columns, rows, matrix),
  // boxes of 16 columns x 64 rows, 128-byte swizzle
  CUtensorMap tmK;
  memset(&tmK, 0, sizeof(tmK));
  p.use_tma = 0;
  if (!ctx->opt_no_tma && p.mode == MODE_FACTOR && p.n >= TM + NB) {
    const unsigned long long sk = p.strideK > 0 ? (unsigned long long)p.strideK : (unsigned long long)p.n * p.ld;
    int st = spb_encode_tmap_3d_f64(&tmK, p.K, (unsigned long long)p.ld, (unsigned long long)p.n,
                                    (unsigned long long)p.B, (unsigned long long)p.ld * 8, sk * 8, KC,
                                    NB, 1);
    p.use_tma = (st == 0) ? 1 : 0;   // an unencodable layout simply keeps the cp.async path
  }
  if (const int st = claim_counter(ctx, stream, &p.counter)) return st;
  potrf_lnlike_kernel<<<grid, NTHREADS, smem, (cudaStream_t)stream>>>(p, tmK);
  SPB_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int spb_cholesky_lnlike(spb_context *ctx, int B, int nt, double *K, int ldk,
                                   long long K_stride, int M, double *resid, int ldr,
                                   long long resid_stride, double *lnlike, double *quad,
                                   double *logdet, int32_t *info, void *stream) {
  SPB_REQUIRE(ctx != nullptr, "null context");
  PotrfParams p = factor_params(B, nt, K, ldk, K_stride, nullptr, M, resid, ldr, resid_stride, lnlike, quad,
                                logdet, info);
  return potrf_launch(ctx, p, stream);
}

extern "C" int spb_cholesky_lnlike_affine(spb_context *ctx, int B, int nt, double *K, int ldk,
                                          long long K_stride, const spb_affine *affine, int M,
                                          double *resid, int ldr, long long resid_stride,
                                          double *lnlike, double *quad, double *logdet,
                                          int32_t *info, void *stream) {
  SPB_REQUIRE(ctx != nullptr && affine != nullptr, "cholesky_lnlike_affine: null argument");
  SPB_REQUIRE((affine->scal == nullptr) == (affine->q == nullptr),
              "cholesky_lnlike_affine: scal and q must be given together");
  PotrfParams p = factor_params(B, nt, K, ldk, K_stride, affine, M, resid, ldr, resid_stride, lnlike, quad,
                                logdet, info);
  return potrf_launch(ctx, p, stream);
}

// ---- INT8-tensor-core path (potrf_i8.cuh) ----------------------------------------------------------
static inline int i8_n64(int nt) { return (nt + NB - 1) & ~(NB - 1); }

// `planes` of the C ABI: 8 (= 87) eight planes of 7-bit digits, 7 (= 77) seven planes of 7-bit digits,
// 78 seven planes of 8-bit digits
static inline int i8_decode(int planes, int *rb) {
  if (planes == 8 || planes == 87) { *rb = 7; return 8; }
  if (planes == 7 || planes == 77) { *rb = 7; return 7; }
  if (planes == 78) { *rb = 8; return 7; }
  *rb = 0;
  return 0;
}

extern "C" size_t spb_cholesky_i8_workspace_bytes(int B, int nt, int M, int planes) {
  int rb0;
  planes = i8_decode(planes, &rb0);
  if (B <= 0 || nt <= 0 || M < 0 || planes == 0) return 0;
  const size_t NR = (size_t)i8_n64(nt) + (size_t)M, LDQ = (size_t)i8_n64(nt);
  return (size_t)B * ((size_t)planes * NR * LDQ + NR * sizeof(double)) + 1024;
}

extern "C" int spb_cholesky_lnlike_i8(spb_context *ctx, int B, int nt, double *K, int ldk,
                                      long long K_stride, const spb_affine *affine, int M,
                                      double *resid, int ldr, long long resid_stride, double *lnlike,
                                      double *quad, double *logdet, int32_t *info, int planes,
                                      double lambda_min, void *workspace, size_t workspace_bytes,
                                      void *stream) {
  SPB_REQUIRE(ctx != nullptr, "cholesky_lnlike_i8: null context");
  SPB_REQUIRE(lambda_min > 0.0 || (affine != nullptr && affine->diag != nullptr),
              "cholesky_lnlike_i8: lambda_min > 0 or affine->diag (data covariance) is required");
  SPB_REQUIRE(affine == nullptr || (affine->scal == nullptr) == (affine->q == nullptr),
              "cholesky_lnlike_i8: scal and q must be given together");
  int rb = 0;
  planes = i8_decode(planes, &rb);
  SPB_REQUIRE(planes != 0, "cholesky_lnlike_i8: planes must be 7, 8, 77, 78 or 87");
  SPB_REQUIRE(info != nullptr, "cholesky_lnlike_i8: info is required");
  SPB_REQUIRE(nt > NB && nt <= NB * I8_MAXP, "cholesky_lnlike_i8: nt out of range (64 < nt <= 16384)");
  SPB_REQUIRE(workspace != nullptr && workspace_bytes >= spb_cholesky_i8_workspace_bytes(B, nt, M, planes),
              "cholesky_lnlike_i8: workspace too small");
  PotrfParams p = factor_params(B, nt, K, ldk, K_stride, affine, M, resid, ldr, resid_stride, lnlike, quad,
                                logdet, info);
  if (const int st = check_layout(p)) return st;
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  I8Params ip;
  const int n64 = i8_n64(nt);
  ip.NR = n64 + M;
  ip.LDQ = n64;
  ip.lambda_min = lambda_min;
  uintptr_t w = ((uintptr_t)workspace + 255) & ~(uintptr_t)255;
  ip.Q = reinterpret_cast<uint8_t *>(w);
  ip.strideQ = (long long)planes * ip.NR * ip.LDQ;
  ip.E = reinterpret_cast<double *>((w + (size_t)B * ip.strideQ + 255) & ~(uintptr_t)255);
  SPB_REQUIRE((uintptr_t)(ip.E + (size_t)B * ip.NR) <= (uintptr_t)workspace + workspace_bytes,
              "cholesky_lnlike_i8: workspace too small");
  CUtensorMap tmA, tmB;
  memset(&tmA, 0, sizeof(tmA));
  memset(&tmB, 0, sizeof(tmB));
  {
    const unsigned long long dims[4] = {(unsigned long long)ip.LDQ, (unsigned long long)ip.NR,
                                        (unsigned long long)planes, (unsigned long long)B};
    const unsigned long long strides[3] = {(unsigned long long)ip.LDQ,
                                           (unsigned long long)ip.LDQ * ip.NR,
                                           (unsigned long long)ip.strideQ};
    const unsigned boxA[4] = {I8_KCH, I8_TM, (unsigned)planes, 1};
    const unsigned boxB[4] = {I8_KCH, NB, (unsigned)planes, 1};
    int st = spb_encode_tmap_u8_4d(&tmA, ip.Q, dims, strides, boxA);
    if (st) return st;
    st = spb_encode_tmap_u8_4d(&tmB, ip.Q, dims, strides, boxB);
    if (st) return st;
  }
  static spb_once_flag attr_once;
  {
    const int st = spb_once_per_device(attr_once, ctx->device, [&]() -> int {
#define SPB_I8_ATTR(S_, ST_, RB_, KP_)                                                                  \
  SPB_CHECK_CUDA(cudaFuncSetAttribute(potrf_i8_kernel<S_, ST_, RB_, KP_>,                               \
                                      cudaFuncAttributeMaxDynamicSharedMemorySize,                      \
                                      (int)sizeof(SmemI8<S_, ST_, KP_>)))
      SPB_I8_ATTR(8, 3, 7, false);
      SPB_I8_ATTR(7, 3, 7, false);
      SPB_I8_ATTR(7, 3, 8, false);
      SPB_I8_ATTR(7, 2, 7, true);
      SPB_I8_ATTR(7, 2, 8, true);
#undef SPB_I8_ATTR
      return 0;
    });
    if (st) return st;
  }
  const int grid = B < ctx->num_sms ? B : ctx->num_sms;
  if (const int st = claim_counter(ctx, stream, &p.counter)) return st;
  // 7-plane kernels, nt <= 1536: two ring stages + the cp.async prefetch of the next K tile (the per-tile
  // chain dominates there); larger nt: three ring stages (the MMA stream dominates, -8 % with two)
  const bool kpre = (planes == 7) && nt <= 1536;
#define SPB_I8_GO(S_, ST_, RB_, KP_)                                                                    \
  potrf_i8_kernel<S_, ST_, RB_, KP_><<<grid, I8_NTHREADS, sizeof(SmemI8<S_, ST_, KP_>), (cudaStream_t)stream>>>(p, ip, tmA, tmB)
  if (planes == 8) SPB_I8_GO(8, 3, 7, false);
  else if (rb == 7 && kpre) SPB_I8_GO(7, 2, 7, true);
  else if (rb == 7) SPB_I8_GO(7, 3, 7, false);
  else if (kpre) SPB_I8_GO(7, 2, 8, true);
  else SPB_I8_GO(7, 3, 8, false);
#undef SPB_I8_GO
  SPB_LAUNCH_CHECK(ctx);
  // safety net: matrices flagged SPB_INFO_I8_RANGE go through the FP64 kernel (their K is intact)
  p.only_flag = SPB_INFO_I8_RANGE;
  return potrf_launch(ctx, p, stream);
}

extern "C" int spb_cholesky_solve_rows(spb_context *ctx, int nt, const double *L, int ldk, int M,
                                       double *resid, int ldr, double *quad, void *stream) {
  SPB_REQUIRE(ctx != nullptr, "null context");
  SPB_REQUIRE(M > 0 && resid != nullptr, "solve_rows: no right-hand sides");
  PotrfParams p = {};   // no lnlike / logdet / info, no affine map
  p.K = const_cast<double *>(L);
  p.n = nt;
  p.ld = ldk;
  p.R = resid;
  p.M = M;
  p.ldr = ldr;
  p.quad = quad;
  p.B = 1;
  p.mode = MODE_SOLVE;
  // one full 128-row tile per work item (a tile costs the same DMMA time however many of its
  // rows are live, so smaller items would only replicate the streaming of L)
  p.rows_per_cta = TM;
  return potrf_launch(ctx, p, stream);
}

extern "C" int spb_dmma_peak(spb_context *ctx, int iters, double *tflops_host, double *ms_host) {
  SPB_REQUIRE(ctx != nullptr, "null context");
  SPB_CHECK_CUDA(cudaSetDevice(ctx->device));
  double *sink = nullptr;
  SPB_CHECK_CUDA(cudaMalloc(&sink, 8));
  cudaEvent_t e0, e1;
  SPB_CHECK_CUDA(cudaEventCreate(&e0));
  SPB_CHECK_CUDA(cudaEventCreate(&e1));
  const int grid = 2 * ctx->num_sms;
  dmma_peak_kernel<<<grid, 256>>>(iters / 10 + 1, sink);  // warm-up
  SPB_CHECK_CUDA(cudaEventRecord(e0));
  dmma_peak_kernel<<<grid, 256>>>(iters, sink);
  SPB_CHECK_CUDA(cudaEventRecord(e1));
  SPB_CHECK_CUDA(cudaEventSynchronize(e1));
  ctx->launches += 2;
  float ms = 0.f;
  SPB_CHECK_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  const double flops = (double)grid * 8.0 * 16.0 * (double)iters * 512.0;
  if (tflops_host) *tflops_host = flops / (ms * 1e-3) / 1e12;
  if (ms_host) *ms_host = ms;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(sink);
  return 0;
}
