// Batched Cholesky -> lnlike with the trailing updates on the INT8 tensor cores (tcgen05 + TMEM).
// Included by potrf.cu inside its anonymous namespace (shares RowMap, init_acc, potf2_regs, trsm_warp).
//
// FP64 has no tcgen05 form, but the panel update  P = K - L L^T  is a sum of products of numbers whose
// magnitude is known in advance (|L_ik| <= sqrt(K_ii)), so it is evaluated exactly on INT8 digit planes
// (i8_planes.cuh: digit format, MMA stream, TMEM read-back):
//
//   * every stored row of L (and of the appended right-hand sides y = L^-1 r) gets its scale 2^e_i before
//     the factorisation starts; its digits are stored as S int8 planes next to K.  Default: S = 7 planes of
//     balanced RB = 8-bit digits (55 bits per row); S = 8 x RB = 7 (56 bits) and S = 7 x RB = 7 (49 bits)
//     are kept;
//   * for a 128 x 64 tile of the panel the MMA stream accumulates the plane products of the already factored
//     columns in TMEM; the 8 compute warps combine the S blocks in fp64, apply the row scales and subtract
//     from the K values of the tile (copied to shared memory by cp.async during the previous tile when
//     nt <= 1536, loaded directly otherwise); from there on the tile is the round-1 kernel's: in-register
//     potf2 of the diagonal block, in-register TRSM on DMMA, |y|^2 and log-determinant reductions;
//   * the new rows of L are cut into digit planes straight from the accumulator registers and stored;
//     the producer thread waits for exactly the tiles a k-chunk needs (a monotone counter of stored
//     tiles), so the MMA stream of the next tile -- and of the next PANEL, up to its last two k-chunks --
//     runs while the warps are still in the TRSM / stores of the current one (look-ahead for free).
//
// With 55 / 56 bits relative to the row maximum the lnlike differences to the DMMA kernel are at the level of
// fp64 rounding noise (<= 3.8e-12 / 1.2e-12 relative on the bench covariances, cond 1e3 .. 2e7).  K itself is
// only READ.
//
// Safety net: a digit that does not fit (a row bound violated: cannot happen for rows of L, and for
// the right-hand-side rows only if K' - diag were indefinite by more than 15/16 of diag) sets
// SPB_INFO_I8_RANGE for the matrix; the launcher then re-runs exactly those matrices through the DMMA
// kernel (K is untouched, so nothing is lost).

constexpr int I8_MAXP = 256;         // panels per matrix (nt <= 16384)
static_assert(NB == I8_TN, "a panel is one TMEM block wide");

struct I8Params {
  uint8_t *Q;            // (B, S, NR, LDQ) digit planes
  double *E;             // (B, NR) row scales 2^e
  long long strideQ;     // bytes per matrix
  int NR, LDQ;
  double lambda_min;     // > 0: K' >= lambda_min I (else K' >= diag(aff.diag)): bounds the right-hand-side rows
};

// Virtual rows of a panel for this kernel.  A tile's A operand must be ONE box of 128 consecutive plane
// rows, i.e. virtual row v of the panel at column c0 has to be plane row c0 + v; the last panel of a
// matrix whose size is not a multiple of 64 (identity-padded diagonal block, right-hand sides at virtual
// row 64 + m) fixes the plane rows of the right-hand sides at n64 + m, n64 = round_up(nt, 64).  Two layouts:
//   * "gap" (M <= n64 - nt, the bench case): the right-hand-side planes are kept TWICE, at rows nt + m
//     (inside the unused gap nt .. n64 - 1, read by the full panels, where they follow the last matrix row
//     exactly as in the FP64 kernel: no extra tile) and at rows n64 + m (read by the last panel);
//   * otherwise: once, at n64 + m, and every panel carries the n64 - nt unused rows as KIND_NONE rows
//     between the matrix rows and the right-hand sides (nbel counts them).
struct RowMapI8 {
  double *Kb, *Rb;
  int n, M, ld, ldr, c0, nbel;   // nbel: virtual rows between the diagonal block and the right-hand sides
  __device__ __forceinline__ double *row(int v, int &kind) const {
    if (v < NB) {
      const int r = c0 + v;
      if (r < n) {
        kind = KIND_DIAG;
        return Kb + (size_t)r * ld;
      }
      kind = KIND_PAD;
      return nullptr;
    }
    int w = v - NB;
    if (w < nbel) {
      const int r = c0 + NB + w;
      if (r < n) {
        kind = KIND_BELOW;
        return Kb + (size_t)r * ld;
      }
      kind = KIND_NONE;
      return nullptr;
    }
    w -= nbel;
    if (w < M) {
      kind = KIND_RHS;
      return Rb + (size_t)w * ldr;
    }
    kind = KIND_NONE;
    return nullptr;
  }
};

template <int S_, int STAGES_, bool KPRE_ = false>
struct SmemI8 {
  static constexpr int S = S_;
  static constexpr int STAGES = STAGES_;
  uint8_t A[STAGES_][S_][I8_TM][I8_KCH];   // 4 KB per plane
  uint8_t B[STAGES_][S_][NB][I8_KCH];      // 2 KB per plane; planes t0..t1 form one N = 64 (t1 - t0 + 1) operand
  // KPRE: the 128 x 64 K tile of the NEXT tile, copied by cp.async while the current one is processed; chunk c
  // (of 16) of thread t at [(c * 256 + t)]: every thread reads back what it copied, conflict-free both ways
  double2 Kpre[KPRE_ ? 16 * I8_NCT : 1];
  LdStore Ld;
  double Dv[NB][DS];
  double red[I8_NCT / 32];
  double dpiv[NB];
  double af[4];
  uint64_t full[STAGES_], empty[STAGES_], tmem_full, tmem_empty;
  unsigned first[I8_MAXP + 1];   // sequence number of the first tile of every panel of this matrix
  uint32_t tmem_base;
  volatile unsigned stored;      // tiles whose planes are in global memory (monotone over the launch)
  int bad;
  int bad_range;
  int next_item;
};

// The fused affine map (spb_affine) of one accumulator row that holds RAW values of a full panel (the
// arithmetic half of init_acc; used when the values come from the cp.async prefetch buffer).
template <class SM>
__device__ __forceinline__ void i8_apply_aff(const SM &sm, const RowMapI8 &rm, const AffRow &af, int v, int c0,
                                             int tg, double (&accrow)[8][2]) {
  int kind;
  (void)rm.row(v, kind);
  if (kind != KIND_DIAG && kind != KIND_BELOW) return;
  const int gi = c0 + v;
  double Ci, Di;
  aff_row_consts(sm, af, gi, Ci, Di);
  aff_full_row(sm, af, kind == KIND_DIAG, gi, v, c0, tg, Ci, Di, accrow);
}

// number of 128-row tiles of the panel starting at column c0 (NR = nt + M virtual rows in total)
__device__ __forceinline__ int i8_nbel(int n, int n64, bool gap, int c0) {
  return gap ? ((c0 + NB <= n) ? n - c0 - NB : 0) : n64 - c0 - NB;
}
__device__ __forceinline__ int i8_nvirt(int n, int n64, int M, bool gap, int c0) {
  return NB + i8_nbel(n, n64, gap, c0) + M;
}
__device__ __forceinline__ int i8_ntiles(int nvirt) { return (nvirt + I8_TM - 1) / I8_TM; }

template <int S, int STAGES, int RB, bool KPRE>
__global__ void __launch_bounds__(I8_NTHREADS, 1)
    potrf_i8_kernel(PotrfParams p, I8Params ip, const __grid_constant__ CUtensorMap tmA,
                    const __grid_constant__ CUtensorMap tmB) {
  using SM = SmemI8<S, STAGES, KPRE>;
  SM &sm = *reinterpret_cast<SM *>(smem_raw);
  const int tid = threadIdx.x, pw = tid >> 5, lane = tid & 31, g = lane >> 2, tg = lane & 3;
  // TMEM lanes a warp may read: 32 (pw % 4) .. + 31; the fragment-shaped loads take 16 of them, so compute
  // warp pw owns tile rows 32 (pw % 4) + 16 (pw / 4) .. + 15, i.e. it plays LOGICAL warp 2 (pw % 4) + pw / 4
  // of the 8-warp geometry (rows 16 warp .. 16 warp + 15)
  const int warp = 2 * (pw & 3) + ((pw >> 2) & 1);
  const int NR = ip.NR;

  if (tid == 0) {
    i8_ring_init(sm);
    sm.stored = 0;
    fence_mbarrier_init();
  }
  if (pw == I8_ISSUER_WARP) i8_tmem_alloc(&sm.tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_base;

  unsigned xchunk = 0;     // producer / issuer: running k-chunk count (ring slot, barrier phase)
  unsigned tq = 0;         // issuer / compute: running count of tiles that went through TMEM
  unsigned seq_base = 0;   // sequence number of the first tile of the current matrix

  for (int item = blockIdx.x; item < p.B;) {
    // ---------------------------------------------------------------- per-matrix set-up
    RowMapI8 rm;
    rm.n = p.n;
    rm.ld = p.ld;
    rm.ldr = p.ldr;
    rm.Kb = p.K + (size_t)item * p.strideK;
    rm.Rb = p.R ? p.R + (size_t)item * p.strideR : nullptr;
    rm.M = p.R ? p.M : 0;
    const int n64 = (p.n + NB - 1) & ~(NB - 1);
    const int M_ = p.R ? p.M : 0;
    const bool gap = (M_ <= n64 - p.n);   // also true when M = 0; false when nt is a multiple of 64 and M > 0
    double *quad_out = p.quad ? p.quad + (size_t)item * p.M : nullptr;
    const AffRow af = aff_setup(p, item, sm, tid);
    double *Eb = ip.E + (size_t)item * NR;
    uint8_t *Qb = ip.Q + (size_t)item * ip.strideQ;
    if (tid == 0) {
      sm.bad = 0;
      sm.bad_range = 0;
      unsigned f = seq_base;
      int j = 0;
      for (int c0 = 0; c0 < p.n; c0 += NB, ++j) {
        sm.first[j] = f;
        f += (unsigned)i8_ntiles(i8_nvirt(p.n, n64, M_, gap, c0));
      }
      sm.first[j] = f;
    }
    __syncthreads();
    const int npanels = (p.n + NB - 1) / NB;
    const unsigned seq_end = sm.first[npanels];

    if (pw < 8) {
      // ============================================================== COMPUTE WARPS
      if (quad_out)
        for (int m = tid; m < rm.M; m += I8_NCT) quad_out[m] = 0.0;
      // row scales: 2^e_i > 1.0101 sqrt(K'_ii) for the rows of L;  for the right-hand-side rows a bound of
      // |y_k| (below)
      // 2^e (x 2 for balanced 8-bit digits); 1 (2) for a row without a finite positive bound
      const auto row_scale = [](double x) {
        int e;
        return (i8_scale_exp(x, e) ? ldexp(1.0, e) : 1.0) * (RB == 8 ? 2.0 : 1.0);
      };
      for (int r = tid; r < p.n; r += I8_NCT) {
        double kd = rm.Kb[(size_t)r * p.ld + r];
        if (p.aff_on) {
          double Ci, Di;
          aff_row_consts(sm, af, r, Ci, Di);
          kd = aff_apply(sm, af, kd, Ci, Di, true, r, r);
        }
        Eb[r] = row_scale(sqrt(kd));
      }
      for (int m = pw; m < rm.M; m += I8_NCT / 32) {
        const double *rr = rm.Rb + (size_t)m * p.ldr;
        double mx = 0.0;
        for (int k = lane; k < p.n; k += 32) mx = fmax(mx, fabs(rr[k]));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        // |y_k| <= |y| = sqrt(r^T K'^-1 r) <= sqrt(sum_k r_k^2 / d_k) with d = lambda_min or the affine diagonal
        // (K' >= diag(d)): unlike sqrt(nt) max|r| / sqrt(min d) it does not grow with a diagonal scaling of K'
        // or with noise that varies along the light curve (x 4 of margin; summed relative to max|r|)
        const double inv = (mx > 0.0) ? 1.0 / mx : 0.0;
        double s = 0.0;
        for (int k = lane; k < p.n; k += 32) {
          const double x = rr[k] * inv;
          s += x * x / ((ip.lambda_min > 0.0) ? ip.lambda_min : (af.dg_vec ? af.dg[k] : af.dg[0]));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0)
          Eb[n64 + m] = row_scale(4.0 * mx * sqrt(s));
      }
      for (int r = p.n + tid; r < n64; r += I8_NCT) Eb[r] = 1.0;
      __threadfence_block();
      cbar256();

      double logdet_part = 0.0, quad_part = 0.0;
      double acc[2][8][2];
      bool bad_range = false;
      bool have_pre = false;   // KPRE: the prefetch buffer holds this tile's raw values (block-uniform)
      unsigned seq = seq_base;
      for (int c0 = 0; c0 < p.n; c0 += NB) {
        rm.c0 = c0;
        rm.nbel = i8_nbel(p.n, n64, gap, c0);
        const int nvirt = NB + rm.nbel + rm.M;
        const bool full_panel = (c0 + NB <= p.n);
        const bool need_planes = (c0 + NB < p.n);   // a later panel will read these columns
        const int nchunks = c0 / I8_KCH;
        for (int v0 = 0; v0 < nvirt; v0 += I8_TM, ++seq) {
          const bool diag_tile = (v0 == 0);
          const int vr = v0 + warp * 16;            // first tile row of this warp
          if (KPRE && have_pre) {
            // the raw K (or right-hand-side) values of this tile were copied to shared memory during the
            // previous tile: pick them up and apply the affine map
            cp_async_wait<0>();
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
              for (int nt = 0; nt < 8; ++nt) {
                const double2 kv = sm.Kpre[(mt * 8 + nt) * I8_NCT + tid];
                acc[mt][nt][0] = kv.x;
                acc[mt][nt][1] = kv.y;
              }
              if (p.aff_on) i8_apply_aff(sm, rm, af, vr + mt * 8 + g, c0, tg, acc[mt]);
            }
          } else {
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
              init_acc(sm, rm, af, p.aff_on != 0, vr + mt * 8 + g, c0, tg, full_panel, acc[mt]);
          }
          {
            // the K rows of the NEXT tile are read exactly once, from HBM, and their latency (3 us per tile
            // when loaded at the top of the tile) is the largest single item of the per-tile chain: with
            // KPRE they are copied now by cp.async (per thread: its own 16 x 16 bytes) and waited for at the
            // top of the next tile; without, at least requested into L2
            RowMapI8 rn = rm;
            int v0n = v0 + I8_TM;
            if (v0n >= nvirt) {
              v0n = 0;
              rn.c0 = c0 + NB;
              rn.nbel = i8_nbel(p.n, n64, gap, rn.c0);
            }
            have_pre = false;
            if (rn.c0 < p.n) {
              if (KPRE) {
                if (rn.c0 + NB <= p.n) {      // full panels only (block-uniform)
#pragma unroll
                  for (int mt = 0; mt < 2; ++mt) {
                    int kind;
                    const double *pn = rn.row(v0n + warp * 16 + mt * 8 + g, kind);
                    const int bytes = pn ? 16 : 0;
                    const double *src = (pn ? pn : rn.Kb) + rn.c0 + 2 * tg;
#pragma unroll
                    for (int nt = 0; nt < 8; ++nt)
                      cp_async16(&sm.Kpre[(mt * 8 + nt) * I8_NCT + tid], src + nt * 8, bytes);
                  }
                  cp_async_commit();
                  have_pre = true;
                }
              } else {
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
                  int kind;
                  const double *pn = rn.row(v0n + warp * 16 + mt * 8 + g, kind);
                  if (pn != nullptr && rn.c0 + 16 * tg < p.n)
                    asm volatile("prefetch.global.L2 [%0];\n" ::"l"(pn + rn.c0 + 16 * tg));
                }
              }
            }
          }
          if (nchunks > 0) {
            // scales of this thread's rows (plane row = c0 + virtual row for matrix and RHS rows alike)
            double si[2];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
              const int v = vr + mt * 8 + g;
              int kind;
              (void)rm.row(v, kind);
              const int er = (kind == KIND_RHS) ? n64 + (v - NB - rm.nbel) : c0 + v;   // row of the scale table
              const bool valid = (kind == KIND_DIAG || kind == KIND_BELOW || kind == KIND_RHS);
              si[mt] = valid ? -ldexp(Eb[er], -2 * RB) : 0.0;
            }
            mbar_wait_sleep(&sm.tmem_full, tq & 1u, 50);
            tc_fence_after();
            const uint32_t tw = tmem + ((uint32_t)(32 * (pw & 3) + 16 * ((pw >> 2) & 1)) << 16);
#pragma unroll
            for (int cq = 0; cq < 4; ++cq) {
              uint32_t v[S][8];
              i8_tmem_ld<S>(tw, 16 * cq, v);
#pragma unroll
              for (int b = 0; b < 2; ++b) {
                const int nt = 2 * cq + b;
                const int gc = c0 + nt * 8 + 2 * tg;
                const double sj0 = (gc < p.n) ? Eb[gc] : 0.0;
                const double sj1 = (gc + 1 < p.n) ? Eb[gc + 1] : 0.0;
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
                  for (int e = 0; e < 2; ++e) {
                    const double t = i8_horner<S, RB>(v, 4 * b + 2 * mt + e);
                    acc[mt][nt][e] = fma(si[mt] * (e ? sj1 : sj0), t, acc[mt][nt][e]);
                  }
                }
              }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.tmem_empty);
            ++tq;
          }
          const int lw = warp;
          if (diag_tile) {
            if (lw < 4) potf2_regs(sm, acc, lw, lane);
            cbar256();   // L_jj and the inverses of its diagonal tiles are in shared memory
            if (tid < min(NB, p.n - c0)) logdet_part += 0.5 * log(sm.dpiv[tid]);
          }
          // a matrix already found not positive definite turns into NaNs from here on: its digits
          // overflow, but there is nothing to rescue by re-running it on the FP64 kernel
          const bool already_bad = (*(volatile int *)&sm.bad) != 0;
          const int vr2 = v0 + lw * 16;             // first tile row of this warp from here on
          if (!(diag_tile && lw < 4) && vr2 < nvirt) {
            trsm_warp(sm, acc, lane);
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
              const int v = vr2 + mt * 8 + g;
              int kind;
              double *prow = rm.row(v, kind);
              const bool live = (kind == KIND_BELOW || kind == KIND_RHS);
              // ---- fp64: the y rows (output); the rows of L are kept only as digit planes
              double q = 0.0;
              if (kind == KIND_RHS) {
#pragma unroll
                for (int nt = 0; nt < 8; ++nt) {
                  const int gc = c0 + nt * 8 + 2 * tg;
                  if (gc + 1 < rm.n) {
                    *reinterpret_cast<double2 *>(prow + gc) = make_double2(acc[mt][nt][0], acc[mt][nt][1]);
                  } else if (gc < rm.n) {
                    prow[gc] = acc[mt][nt][0];
                  }
                }
              }
              if (kind == KIND_RHS) {
#pragma unroll
                for (int nt = 0; nt < 8; ++nt) {
                  const int gc = c0 + nt * 8 + 2 * tg;
                  if (gc < rm.n) q += acc[mt][nt][0] * acc[mt][nt][0];
                  if (gc + 1 < rm.n) q += acc[mt][nt][1] * acc[mt][nt][1];
                }
              }
              quad_part += q;
              if (quad_out) {
                q += __shfl_xor_sync(0xffffffffu, q, 1);
                q += __shfl_xor_sync(0xffffffffu, q, 2);
                if (kind == KIND_RHS && tg == 0) atomicAdd(quad_out + (v - NB - rm.nbel), q);
              }
              // ---- digit planes of the new rows (read by the MMA stream of later panels).
              // Inside a 64-column panel block the bytes are stored in the order 16 tg + 2 nt + e
              // (column 8 nt + 2 tg + e): a dot product over k does not care about the order as long
              // as both operands use the same one, and this one makes the 16 entries a thread holds of
              // a row contiguous -- one 16-byte store per (row, plane), no shuffles.
              if (need_planes && live) {
                const int mrhs = v - NB - rm.nbel;                      // right-hand-side index (KIND_RHS)
                const int pr = (kind == KIND_RHS) ? n64 + mrhs : c0 + v;   // plane row == row of the scale table
                const double sinv = ldexp(1.0 / Eb[pr], RB * S);   // 2^(RB S - e): exact
                uint8_t *qrow = Qb + (size_t)pr * ip.LDQ + c0 + 16 * tg;
                const size_t pstride = (size_t)NR * ip.LDQ;
                // The cut of i8_cut, written out: 16 entries per thread in 4 words per plane, the range check
                // between the lower digits and the top digit (i8_cut's order changes this kernel's schedule).
                constexpr long long BIAS = i8_bias(S, RB);
                constexpr unsigned FMASK = (1u << RB) - 1u;
                uint32_t W[S][4];
#pragma unroll
                for (int s = 0; s < S; ++s)
#pragma unroll
                  for (int w = 0; w < 4; ++w) W[s][w] = 0u;
#pragma unroll
                for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
                  for (int e = 0; e < 2; ++e) {
                    const long long Xb = __double2ll_rn(acc[mt][nt][e] * sinv) + BIAS;
                    const unsigned mul = 1u << (8 * ((nt & 1) * 2 + e));   // byte position in the word
#pragma unroll
                    for (int jd = 0; jd < S - 1; ++jd)
                      W[S - 1 - jd][nt >> 1] += ((uint32_t)(Xb >> (RB * jd)) & FMASK) * mul;
                    const int top = (int)(Xb >> (RB * (S - 1))) - (1 << (RB - 1));
                    bad_range = bad_range || ((top < -128 || top > 127) && !already_bad);
                    W[0][nt >> 1] += ((uint32_t)top & 255u) * mul;
                  }
                }
#pragma unroll
                for (int s = 0; s < S; ++s) {
                  uint4 o;
                  o.x = i8_recentre<RB>(s, W[s][0]);
                  o.y = i8_recentre<RB>(s, W[s][1]);
                  o.z = i8_recentre<RB>(s, W[s][2]);
                  o.w = i8_recentre<RB>(s, W[s][3]);
                  *reinterpret_cast<uint4 *>(qrow + (size_t)s * pstride) = o;
                  // "gap" layout: second copy of a right-hand-side row, read by the full panels
                  if (gap && kind == KIND_RHS && n64 != p.n)
                    *reinterpret_cast<uint4 *>(qrow + (size_t)s * pstride -
                                               (size_t)(n64 - p.n) * ip.LDQ) = o;
                }
              }
            }
          }
          // the planes (generic-proxy stores) must be visible to the TMA engine before the producer is
          // told about them; the barrier also protects Ld / Dv against the next panel's potf2
          fence_proxy_async_global();
          __threadfence_block();
          cbar256();
          if (tid == 0) {
            __threadfence_block();   // the barrier's view of the other warps' stores before the counter moves
            sm.stored = seq + 1;
          }
        }
      }
      if (bad_range) sm.bad_range = 1;
      // ---- reductions -> lnlike
      const double quad = block_sum<true>(sm, quad_part);
      const double logdet = block_sum<true>(sm, logdet_part);
      if (tid == 0) {
        lnlike_epilogue(p, item, quad, logdet, sm.bad != 0, SPB_INFO_NOT_PD | SPB_INFO_I8_RANGE,
                        sm.bad_range ? SPB_INFO_I8_RANGE : 0);
        sm.next_item = (int)gridDim.x + (int)atomicAdd(p.counter, 1u);
      }
    } else if (pw == I8_PRODUCER_WARP) {
      // ============================================================== TMA PRODUCER (one thread)
      if (lane == 0) {
        unsigned known = sm.stored;
        for (int c0 = NB; c0 < p.n; c0 += NB) {
          const int nvirt = i8_nvirt(p.n, n64, M_, gap, c0);
          const int nchunks = c0 / I8_KCH;
          const bool last_partial = (c0 + NB > p.n);
          for (int v0 = 0; v0 < nvirt; v0 += I8_TM) {
            const int vlast = min(v0 + I8_TM, nvirt) - 1;   // last live virtual row of the tile
            for (int ch = 0; ch < nchunks; ++ch, ++xchunk) {
              // the k-columns of this chunk were written during panel P (a full panel), by the tile that
              // held the tile's last live row there.  Virtual row of that row in panel P: matrix rows and,
              // in full panels, right-hand sides simply shift by c0 - P; in the last (partial) panel the
              // right-hand side m = vlast - 64 sat at NB + nbel(P) + m.
              const int P = (ch * I8_KCH) & ~(NB - 1);
              int vP;
              if (last_partial) {
                const int m = vlast - NB;
                vP = (m >= 0) ? NB + i8_nbel(p.n, n64, gap, P) + m : (p.n - 1 - P);
              } else {
                vP = vlast + (c0 - P);
              }
              const unsigned need = sm.first[P / NB] + (unsigned)(vP / I8_TM) + 1u;
              if ((int)(known - need) < 0) {
                while ((int)((known = sm.stored) - need) < 0) __nanosleep(100);
                __threadfence_block();
                fence_proxy_async_global();
              }
              const unsigned st = xchunk % STAGES;
              if (xchunk >= (unsigned)STAGES) mbar_wait_sleep(&sm.empty[st], ((xchunk / STAGES) + 1u) & 1u, 100);
              mbar_arrive_expect_tx(&sm.full[st], (unsigned)(S * (I8_TM + NB) * I8_KCH));
              tma_load_4d(&sm.A[st][0][0][0], &tmA, &sm.full[st], ch * I8_KCH, c0 + v0, 0, item);
              tma_load_4d(&sm.B[st][0][0][0], &tmB, &sm.full[st], ch * I8_KCH, c0, 0, item);
            }
          }
        }
      }
    } else if (pw == I8_ISSUER_WARP) {
      // ============================================================== MMA ISSUER (one thread)
      if (lane == 0) {
        for (int c0 = NB; c0 < p.n; c0 += NB) {
          const int nvirt = i8_nvirt(p.n, n64, M_, gap, c0);
          const int nchunks = c0 / I8_KCH;
          for (int v0 = 0; v0 < nvirt; v0 += I8_TM, ++tq) {
            if (tq > 0) mbar_wait_sleep(&sm.tmem_empty, (tq + 1u) & 1u, 100);   // the warps have drained TMEM
            tc_fence_after();
            for (int ch = 0; ch < nchunks; ++ch, ++xchunk) {
              const unsigned st = xchunk % STAGES;
              mbar_wait_sleep(&sm.full[st], (xchunk / STAGES) & 1u, 50);
              tc_fence_after();
              i8_issue_chunk<S>(tmem, sm.A[st], sm.B[st], ch > 0);
              i8_commit(&sm.empty[st]);
            }
            i8_commit(&sm.tmem_full);
          }
        }
      }
    }
    __syncthreads();
    item = sm.next_item;
    seq_base = seq_end;
  }
  tc_fence_before();
  __syncthreads();
  if (pw == I8_ISSUER_WARP) i8_tmem_dealloc(tmem);
}
