// softmax_math.cuh — the exp2 inner loop shared by the attention kernels.
//
// Per score element: x = s*c - m*c (FFMA), MUFU.EX2, row-sum FADD, half a cvt.  The scale and
// the row sum use the packed fp32 pipe (fma.rn.f32x2 / add.rn.f32x2 -> FFMA2 / FADD2), which
// halves their instruction count.  tools/softmax_rate.cu (profiles/r02_session2l.log): a warp alone
// on its scheduler needs 1150 clk for the 128 scores of a row, 1030 of them the MUFU pipe (8 clk per
// warp instruction = 16 exp/clk/SM) — the loop is MUFU-bound with ~580 issue slots to spare.
// exp_chunk32_mix moves a fixed subset of the pairs onto those slots (polynomial on the FMA pipe).
// Alternatives that were built, verified and measured on B200 at B4 H32 N4096 D128 and dropped:
//   * round 1 (profiles/r01_fmha_variants.txt): 3/16 or 7/16 of the exps through a degree-3 polynomial with a
//     Cody-Waite split: 1256 / 1218 TFLOPS against 1257 without; a polynomial whose range reduction uses
//     floorf / float->int conversions is slower than the MUFU it replaces (softmax_rate: 1597 vs 1193 clk per
//     row at 25 %) — those conversions run on the MUFU pipe themselves;
//   * ex2.approx.f16x2: sm_100a lowers it to two MUFU.EX2.F16, no saving.
#pragma once
#include "sm100_ptx.cuh"

namespace b200 {

B200_DEVICE uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
B200_DEVICE uint64_t f2_pack_u(uint32_t lo, uint32_t hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
  return r;
}
B200_DEVICE void f2_unpack(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
B200_DEVICE uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
B200_DEVICE uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// P = exp2(s*c - m*c) for 32 consecutive scores of one row: 16 packed half2 for the TMEM
// store; row-sum contributions (the un-rounded fp32 values, as the reference accumulates them,
// flash_attn_mma_split_q.cu:459-471) go into 4 independent packed accumulators.
B200_DEVICE void exp_chunk32(const uint32_t (&s)[32], uint64_t c2, uint64_t nmc2, uint32_t (&pk)[16],
                             uint64_t (&acc)[4]) {
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const uint64_t x = f2_fma(f2_pack_u(s[2 * i], s[2 * i + 1]), c2, nmc2);
    float x0, x1;
    f2_unpack(x, x0, x1);
    const float e0 = fast_exp2(x0), e1 = fast_exp2(x1);
    acc[i & 3] = f2_add(acc[i & 3], f2_pack(e0, e1));
    pk[i] = pack_half2(e0, e1);
  }
}

// exp_chunk32 with the pairs selected by kPolyMask (bit i = pair i of the chunk) evaluated WITHOUT the MUFU pipe:
//   x' = max(x, -126);  t = x' + 1.5*2^23 (round-to-nearest integer n = round(x') lands in the low mantissa bits);
//   f = x' - (t - 1.5*2^23) in [-0.5, 0.5];  2^f ~ c0 + f (c1 + f (c2 + f c3))  (minimax, max rel. error 7.6e-5 —
//   a third of the fp16 rounding P gets afterwards);  2^x = bits(2^f) + (bits(t) << 23): the shift drops everything of t
//   but n, negative n wraps to the right exponent decrement.  Per pair: 2 FMNMX, 2 FADD2, 4 FFMA2, 2 LEA — no MUFU, no
//   conversion instruction (FRND / F2I run on the MUFU pipe as well).
template <uint32_t kPolyMask>
B200_DEVICE void exp_chunk32_mix(const uint32_t (&s)[32], uint64_t c2, uint64_t nmc2, uint32_t (&pk)[16],
                                 uint64_t (&acc)[4]) {
  const uint64_t magic2 = f2_pack(12582912.f, 12582912.f), nmagic2 = f2_pack(-12582912.f, -12582912.f);
  const uint64_t neg1_2 = f2_pack(-1.f, -1.f);
  const uint64_t k0 = f2_pack(0.9999276399612427f, 0.9999276399612427f), k1 = f2_pack(0.693252682685852f, 0.693252682685852f);
  const uint64_t k2 = f2_pack(0.24261489510536194f, 0.24261489510536194f), k3 = f2_pack(0.05521666631102562f, 0.05521666631102562f);
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const uint64_t x = f2_fma(f2_pack_u(s[2 * i], s[2 * i + 1]), c2, nmc2);
    float x0, x1, e0, e1;
    f2_unpack(x, x0, x1);
    if ((kPolyMask >> i) & 1u) {
      const uint64_t xc = f2_pack(fmaxf(x0, -126.f), fmaxf(x1, -126.f));
      const uint64_t t = f2_add(xc, magic2);
      const uint64_t f = f2_fma(f2_add(t, nmagic2), neg1_2, xc);
      uint64_t q = f2_fma(k3, f, k2);
      q = f2_fma(q, f, k1);
      q = f2_fma(q, f, k0);
      float q0, q1, t0, t1;
      f2_unpack(q, q0, q1);
      f2_unpack(t, t0, t1);
      e0 = __uint_as_float(__float_as_uint(q0) + (__float_as_uint(t0) << 23));
      e1 = __uint_as_float(__float_as_uint(q1) + (__float_as_uint(t1) << 23));
    } else {
      e0 = fast_exp2(x0);
      e1 = fast_exp2(x1);
    }
    acc[i & 3] = f2_add(acc[i & 3], f2_pack(e0, e1));
    pk[i] = pack_half2(e0, e1);
  }
}

B200_DEVICE float f2_hsum4(const uint64_t (&acc)[4]) {
  float a, b, s = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f2_unpack(acc[i], a, b);
    s += a + b;
  }
  return s;
}

// ---- key extents of causal attention (query row i sees the keys j <= i + Nk - Nq; the host guarantees Nk >= Nq)
// KV tiles of bc keys a work item with query rows [.., q_end) needs: all num_kv of them, or (causal) those up to the
// tile holding the last key its last real row sees.  Every role of a kernel derives the item's loop count from this.
B200_DEVICE int attn_kv_tiles(int causal, int num_kv, int Nq, int Nk, int q_end, int bc) {
  if (!causal) return num_kv;
  const int last_key = min(q_end, Nq) - 1 + (Nk - Nq);
  return min(num_kv, last_key / bc + 1);
}

// one past the last key query row `qrow` sees: the ragged-tail mask of a tile at key k0 becomes "scores at or beyond
// key_end - k0 are -inf" (a padding row past Nq keeps a non-empty range; its output is never stored)
B200_DEVICE int attn_key_end(int causal, int Nq, int Nk, int qrow) {
  return causal ? min(Nk, qrow + (Nk - Nq) + 1) : Nk;
}

}  // namespace b200
