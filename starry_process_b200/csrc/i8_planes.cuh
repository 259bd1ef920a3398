// INT8 digit planes: error-free emulation of FP64 products on the INT8 tensor cores (tcgen05 + TMEM).
// The digit format and the tcgen05 pipeline pieces shared by the Cholesky panel updates (potrf_i8.cuh) and by
// the second-moment SYRK and the lower-triangle GEMM (syrk_i8.cu).
//
// FP64 has no tcgen05 form, but a product  sum_k x_ik y_jk  whose rows have magnitudes known in advance can
// be evaluated EXACTLY in integer arithmetic (Ozaki-style error-free slicing; accuracy study:
// oracle/study/ozaki_cholesky.py, micro-benchmark: scripts/micro/i8_emul_micro.cu):
//
//   * every row i is scaled by a power of two 2^-e_i (i8_scale_exp), rounded to S x RB bits and cut into S
//     signed RB-bit digits  x_ik 2^-e_i = sum_s d_s(i,k) 2^{-RB (s+1)};  the digits are stored as S int8
//     PLANES (plane s holds digit s of every entry).  Digit widths:
//       RB = 8: balanced base-256 digits in [-128, 127]; all planes use the whole int8 range and the rows are
//               scaled to |x| <= 1/2.  7 planes carry 55 bits -- one bit less than 8 planes of 7 bits, with 28
//               instead of 36 plane products and 7/8 of the operand traffic;
//       RB = 7: digits in [-64, 63] except the leading one, which uses the whole int8 range (|x| <= 0.99);
//   * the cut (i8_cut) needs no carry chain: X = rint(x 2^(RB S - e)), Xb = X + sum_j 2^(RB-1) 2^(RB j)
//     (i8_bias) has plain RB-bit fields u_j in [0, 2^RB); the lower digits are d_j = u_j - 2^(RB-1)
//     (i8_recentre, four bytes at a time), the top field re-centred the same way keeps the sign;
//   * for a 128 x 64 output tile, one thread issues, per 32-byte k-chunk, tcgen05.mma.kind::i8 products of
//     digit plane A_s (128 rows x 32 bytes) with the concatenated planes B_0 .. B_{S-1-s} (N up to 256)
//     into TMEM (i8_issue_chunk): pairs with s + t = d accumulate EXACTLY (int32) in the 64-column block d,
//     and the S blocks of a tile fit the 512 TMEM columns of an SM.  Operands arrive by 4-D TMA (one box of
//     all planes, 32-byte swizzle) in a shared-memory ring; the tensor core runs from shared-memory
//     descriptors, so no warp touches the operands;
//   * the warps draining TMEM read the S blocks back with fragment-shaped tcgen05.ld (16x256b: the same
//     (row g, columns 2 tg) layout as the DMMA accumulators; i8_tmem_ld) and combine them in fp64 (Horner
//     in 2^-RB, i8_horner); the result times 2^(e_i + e_j - 2 RB) is the FP64 product to the rounding of
//     the final fp64 operations.
//
// Roles of a CTA: warps 0-7 drain TMEM (the TMEM lane rule: warp w reads lanes 32 (w % 4) .. + 31), warp 8
// is the TMA producer, warp 9 the MMA issuer and owner of the TMEM allocation; one CTA per SM.
#pragma once
#include "common.cuh"

constexpr int I8_KCH = 32;           // bytes of k per ring stage = K of one tcgen05.mma.kind::i8
constexpr int I8_TM = 128;           // rows of a tile = M of one instruction
constexpr int I8_TN = 64;            // columns of a tile = columns of one TMEM block
constexpr int I8_NCT = 256;          // threads of the warps that drain TMEM (warps 0-7)
constexpr int I8_PRODUCER_WARP = 8;  // TMA producer (one thread)
constexpr int I8_ISSUER_WARP = 9;    // MMA issuer (one thread)
constexpr int I8_NTHREADS = 320;

// ---- digit format -----------------------------------------------------------------------------------------
// sum_{j < S} 2^(RB-1) 2^(RB j): makes every RB-bit field of a signed S-digit number non-negative
__host__ __device__ constexpr long long i8_bias(int S, int RB) {
  long long b = 0;
  for (int j = 0; j < S; ++j) b = (b << RB) + (1ll << (RB - 1));
  return b;
}

// Exponent e of a row scale 2^e: the smallest with 1.0101 x < 2^e (x / 2^e <= 0.99: the leading digit fits
// int8; balanced 8-bit digits take one power of two more).  False for x = 0, inf or NaN, where the caller
// picks the scale.
__device__ __forceinline__ bool i8_scale_exp(double x, int &e) {
  if (!(x > 0.0) || !(x < 1e300)) return false;
  (void)frexp(x * 1.0101, &e);
  return true;
}

// Cuts xs = x 2^(RB S - e) into S digits and ORs them, shifted by `shift` bits, into the plane words W: W[0]
// gets the signed top digit, W[1..S-1] the biased lower digits (to be re-centred by i8_recentre before the
// store).  Returns the top digit: it fits int8 only if the row scale bounded |x|.
template <int S, int RB>
__device__ __forceinline__ int i8_cut(double xs, int shift, uint32_t (&W)[S]) {
  const long long Xb = __double2ll_rn(xs) + i8_bias(S, RB);
#pragma unroll
  for (int j = 0; j < S - 1; ++j) W[S - 1 - j] |= ((uint32_t)(Xb >> (RB * j)) & ((1u << RB) - 1u)) << shift;
  const int top = (int)(Xb >> (RB * (S - 1))) - (1 << (RB - 1));
  W[0] |= ((uint32_t)top & 255u) << shift;
  return top;
}
// the word of plane s as stored: the lower planes' fields minus 2^(RB-1), bytewise
template <int RB>
__device__ __forceinline__ uint32_t i8_recentre(int s, uint32_t w) {
  return (s == 0) ? w : __vsub4(w, RB == 8 ? 0x80808080u : 0x40404040u);
}

// ---- tcgen05 / TMA ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_4d(void *sdst, const void *tmap, uint64_t *bar, int c0, int c1,
                                            int c2, int c3) {
  unsigned s = (unsigned)__cvta_generic_to_shared(sdst);
  unsigned b = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n" ::"r"(s),
      "l"(tmap), "r"(b), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ uint64_t i8_smem_desc(const void *p) {
  // K-major operand, 32-byte swizzle: rows of 32 B, 8-row groups 256 B apart, descriptor version 1
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  uint64_t d = (uint64_t)((a >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(256 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)6 << 61;
  return d;
}
__device__ __forceinline__ uint32_t i8_idesc(int n) {
  // D = s32, A = B = signed 8 bit, both K-major, M = 128
  return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(I8_TM >> 4) << 24);
}
__device__ __forceinline__ void i8_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc,
                                       uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void i8_commit(uint64_t *bar) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(a)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
}
// 16 lanes x 256 bit, x2 = 16 columns: for each 8-column block b, v[4 b], v[4 b + 1] = (row T/4,
// columns 2 (T%4), +1) and v[4 b + 2], v[4 b + 3] = (row T/4 + 8, same columns): the DMMA C layout
__device__ __forceinline__ void tmem_ld_frag16(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }
// Waits of the two single-thread roles: poll with a sleep in between.  A tight try_wait loop keeps the
// warp permanently eligible and its barrier probes share the LSU path with the SHFL / LDS of the compute
// warp on the same scheduler (measured: the shuffle-bound 8x8 pivot chain ran 3.5x slower next to one).
__device__ __forceinline__ void mbar_wait_sleep(uint64_t *bar, unsigned parity, unsigned ns) {
  while (!mbar_test(bar, parity)) __nanosleep(ns);
}

// All 512 TMEM columns of the SM (one CTA per SM); one whole warp executes these.
__device__ __forceinline__ void i8_tmem_alloc(uint32_t *dst_smem) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(dst_smem);
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(a), "r"(512u)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void i8_tmem_dealloc(uint32_t tmem) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "r"(512u) : "memory");
}

// The barriers of the operand ring (full / empty per stage: one TMA transaction, one tcgen05.commit) and of the
// TMEM hand-off (tmem_full: one commit; tmem_empty: one arrival per draining warp); one thread executes this,
// then fence_mbarrier_init.
template <class SM>
__device__ __forceinline__ void i8_ring_init(SM &sm) {
#pragma unroll
  for (int s = 0; s < SM::STAGES; ++s) {
    mbar_init(&sm.full[s], 1);
    mbar_init(&sm.empty[s], 1);
  }
  mbar_init(&sm.tmem_full, 1);
  mbar_init(&sm.tmem_empty, I8_NCT / 32);
}
__device__ __forceinline__ void fence_mbarrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}

// The MMAs of one k-chunk: A_s against B_0 .. B_{S-1-s} (at most 4 planes = N 256 per instruction), pair
// s + t into TMEM block s + t.  The first chunk of a tile (accumulate = false) writes blocks 0 .. S-1 from s = 0.
template <int S>
__device__ __forceinline__ void i8_issue_chunk(uint32_t tmem, const uint8_t (&A)[S][I8_TM][I8_KCH],
                                               const uint8_t (&B)[S][I8_TN][I8_KCH], bool accumulate) {
#pragma unroll
  for (int s = 0; s < S; ++s) {
    const uint64_t da = i8_smem_desc(&A[s][0][0]);
    const int nt = S - s;                       // planes B_0 .. B_{nt-1}
#pragma unroll
    for (int t0 = 0; t0 < nt; t0 += 4) {
      const int np = nt - t0 < 4 ? nt - t0 : 4;
      i8_mma(tmem + (uint32_t)(I8_TN * (s + t0)), da, i8_smem_desc(&B[t0][0][0]), i8_idesc(I8_TN * np),
             (accumulate || s > 0) ? 1u : 0u);
    }
  }
}

// Columns col .. col + 15 of the S TMEM blocks (tw: the warp's TMEM lanes, column 0).
template <int S>
__device__ __forceinline__ void i8_tmem_ld(uint32_t tw, int col, uint32_t (&v)[S][8]) {
#pragma unroll
  for (int d = 0; d < S; ++d) tmem_ld_frag16(tw + (uint32_t)(I8_TN * d + col), v[d]);
  tmem_ld_wait();
}
// Entry i of the fragment: sum_d v[d][i] 2^(-RB d)
template <int S, int RB>
__device__ __forceinline__ double i8_horner(const uint32_t (&v)[S][8], int i) {
  double t = (double)(int)v[S - 1][i];
#pragma unroll
  for (int d = S - 2; d >= 0; --d) t = fma(t, RB == 8 ? 0.00390625 : 0.0078125, (double)(int)v[d][i]);
  return t;
}
