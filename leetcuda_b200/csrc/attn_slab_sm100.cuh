// attn_slab_sm100.cuh — fused attention forward for LARGE head dims (128 < D <= 1024; the output
// columns are split into slabs of <= 256 over sibling CTAs).
//
// Replaces the reference's "QKV-tiling" / FFPA-L1 kernels
// (kernels/flash-attn/mma/basic/flash_attn_mma_tiling_qkv.cu:77-797,
//  ffpa-attn/csrc/cuffpa/ffpa_attn_templates_L1.cuh:7-590; SURVEY.md §8a rows a10, a13),
// which stream 16-wide d-slices of Q, K and V through a tiny smem buffer and keep O in
// fp16 registers.  The constraint that shapes the sm_100a design is TMEM: 512 fp32
// columns per SM.  O[128 x D] alone would take D columns, so the OUTPUT columns are
// split: a CTA owns 128 query rows and a slab of DV <= 256 output columns,
//
//   TMEM: S0 [0,128)  S1 [128,256)  O [256, 256+DV)          (P_b aliases S_b, fp16)
//
// and computes the full S = Q K^T (all D) itself.  For D <= 256 there is one slab (no
// redundancy); D = 512 uses two sibling CTAs per query tile that both compute S (QK is
// done twice, PV once: 3/4 of the tensor work is useful... 2/3 at the margin), which needs
// no cross-CTA traffic at all.
//
//   warps 0-3  softmax warpgroup (thread r <-> query row r <-> TMEM lane r)
//   warp  4    tcgen05.mma issuer   warp 5  TMA producer   warp 6  TMEM owner
//
// Q (128 x DQ, DQ = D rounded up to 64) stays resident in smem as DQ/64 swizzled boxes when
// DQ <= 512; for 512 < D <= 1024 it does not fit beside the ring and its 64-column chunks
// are streamed (re-read from L2 once per KV tile, as the reference's FFPA kernel does), each
// just ahead of the K chunk it multiplies.  K and V stream through a ring of 16 KiB chunks in
// exactly the order the MMA warp consumes them:
//   K chunk  = {64 d x 128 keys}            -> 4 k16 steps of S += Q_c K_c^T (SS, N=128)
//   V chunk  = DV/64 boxes of {64 d x 32 keys} -> 2 k16 steps of O += P V   (TS, N=DV, V MN-major)
// S is double-buffered so QK(j+1) runs on the tensor pipe while the warpgroup is in the
// softmax of tile j:   QK(0) QK(1) | PV(0) QK(2) | PV(1) QK(3) | ...
#pragma once
#include <cuda.h>

#include "sm100_ptx.cuh"
#include "softmax_math.cuh"

namespace b200 {
namespace attn_slab {

constexpr int BR = 128;
constexpr int BC = 128;
constexpr int kThreads = 256;
constexpr int kRingMax = 12;     // ring slots when Q is streamed (6 when Q is resident)
constexpr int CHUNK_BYTES = 16384;
constexpr int kTmemCols = 512;
constexpr int kMaxQChunks = 8;   // DQ <= 512 resident
constexpr int kMaxDChunks = 16;  // DQ <= 1024 overall
constexpr float kRescaleThreshold = 8.0f;

// Q resident (nq <= 8, "wide" kernel): ring slots of 32 KiB = 8 MMAs per barrier round trip of the issuing warp (the
// 16 KiB / 4-MMA rounds of the first version left that warp's ~400 clk of serial latency per round exposed, see
// attn_pair_sm100.cuh); as many slots as fit beside Q, at most 5.  Q streamed (nq > 8): 12 slots of 16 KiB as before.
constexpr int WIDE_BYTES = 32768;
constexpr int kMaxDynSmem = 232448;
constexpr int ring_slots(int nq_chunks) {
  if (nq_chunks > kMaxQChunks) return kRingMax;
  const int fit = (kMaxDynSmem - 256 - 1024 - nq_chunks * CHUNK_BYTES) / WIDE_BYTES;
  return fit > 5 ? 5 : fit;
}
constexpr int smem_bytes(int nq_chunks) {
  return nq_chunks <= kMaxQChunks ? nq_chunks * CHUNK_BYTES + ring_slots(nq_chunks) * WIDE_BYTES + 256 + 1024
                                  : kRingMax * CHUNK_BYTES + 256 + 1024;
}

struct Params {
  int Nq;           // query rows (q, o, lse)
  int Nk;           // keys (k, v)
  int num_kv;       // ceil(Nk / BC)
  int causal;       // 1: query row i sees the keys j <= i + Nk - Nq (bottom-right aligned; host guarantees Nk >= Nq)
  int nq;           // DQ / 64: 64-wide d-chunks of Q/K
  int dv;           // output columns of this CTA's slab (multiple of 64, <= 256)
  int dsplit;       // slabs per query tile
  float scale_log2;
  float* lse;       // optional [B*H, Nq] fp32 log-sum-exp output (written by slab 0), nullptr = off
  float rms_g;      // > 0: fused RMS norm of the output rows (single-slab launches only, D <= 256); see attn_sm100.cuh
  int D;            // true head dim (mean of the RMS norm)
};

// kWide: Q resident, 32 KiB ring slots (K slot = two {64 d x 128 keys} boxes, V slot = 64 keys); else Q streamed, 16 KiB slots
// kCausal: the causal mask (Params::causal), a separate instantiation so that the full-attention kernel is unchanged
template <bool kWide, bool kCausal>
__global__ void __launch_bounds__(kThreads, 1)
attn_slab_fwd_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                   const __grid_constant__ CUtensorMap tmap_v, const __grid_constant__ CUtensorMap tmap_o,
                   const Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_u32 = smem_u32(smem_raw);
  const uint32_t smem_base = (raw_u32 + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - raw_u32);
  const int NQ = p.nq;
  constexpr bool q_stream = !kWide;                // Q chunks travel through the ring
  constexpr int SLOT = kWide ? WIDE_BYTES : CHUNK_BYTES;
  const int kRing = ring_slots(NQ);
  const int q_res_bytes = q_stream ? 0 : NQ * CHUNK_BYTES;
  const uint32_t q_base = smem_base;
  const uint32_t ring_base = smem_base + q_res_bytes;
  const uint32_t bar_base = ring_base + kRing * SLOT;
  auto ring_full = [&](int s) { return bar_base + 8u * s; };
  auto ring_empty = [&](int s) { return bar_base + 8u * (kRing + s); };
  auto s_full = [&](int b) { return bar_base + 8u * (2 * kRing + b); };
  auto p_full = [&](int b) { return bar_base + 8u * (2 * kRing + 2 + b); };
  const uint32_t o_done = bar_base + 8u * (2 * kRing + 4);
  const uint32_t q_full = bar_base + 8u * (2 * kRing + 5);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kRing + 6);
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(
      smem_gen + q_res_bytes + kRing * SLOT + 8 * (2 * kRing + 6));

  // shuffle-broadcast warp index: warp-uniform for ptxas -> convergent role branches and
  // uniform-datapath descriptor math in the MMA issue loop (no per-instruction R2UR waterfall)
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int bh = blockIdx.y;
  const int tile = blockIdx.x / p.dsplit;
  const int slab = blockIdx.x - tile * p.dsplit;
  // causal: the query tiles run in reverse, heaviest (longest KV extent) first
  const int qtile = kCausal ? static_cast<int>(gridDim.x) / p.dsplit - 1 - tile : tile;
  const int q0 = qtile * BR;
  const int d0 = slab * p.dv;          // first output column of this CTA
  const int T = kCausal ? attn_kv_tiles(1, p.num_kv, p.Nq, p.Nk, q0 + BR, BC) : p.num_kv;   // KV tiles of this query tile
  const int NVB = p.dv >> 6;           // 64-wide boxes per V chunk

  if (warp == 5 && lane == 0) {
    prefetch_tmap(&tmap_q);
    prefetch_tmap(&tmap_k);
    prefetch_tmap(&tmap_v);
    prefetch_tmap(&tmap_o);
  }
  if (warp == 4 && lane == 0) {
    for (int s = 0; s < kRing; ++s) {
      mbar_init(ring_full(s), 1);
      mbar_init(ring_empty(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(s_full(b), 1);
      mbar_init(p_full(b), 4);
    }
    mbar_init(o_done, 1);
    mbar_init(q_full, 1);
    fence_mbar_init();
  }
  if (warp == 6) tmem_alloc<1>(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_gen, 0);
  const uint32_t tmem_o = tmem_base + 256;

  if (warp == 5) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      if (!q_stream) {
        mbar_expect_tx(q_full, NQ * CHUNK_BYTES);
        for (int c = 0; c < NQ; ++c)
          tma_load_3d(q_base + c * CHUNK_BYTES, &tmap_q, q_full, c * 64, q0, bh, kEvictFirst);
      }
      int s = 0;
      uint32_t ph = 0;
      auto load_k_tile = [&](int j) {
        if constexpr (kWide) {
          for (int c = 0; c < NQ; c += 2) {      // two d-chunks per slot (one when NQ is odd and this is the last)
            const int nb = (c + 1 < NQ) ? 2 : 1;
            mbar_wait(ring_empty(s), ph ^ 1u, 100 + s);
            mbar_expect_tx(ring_full(s), nb * CHUNK_BYTES);
            for (int b = 0; b < nb; ++b)
              tma_load_3d(ring_base + s * SLOT + b * CHUNK_BYTES, &tmap_k, ring_full(s), (c + b) * 64, j * BC, bh, kEvictLast);
            if (++s == kRing) { s = 0; ph ^= 1u; }
          }
          return;
        }
        for (int c = 0; c < NQ; ++c) {
          if (q_stream) {   // Q chunk c goes through the ring right before K chunk c
            mbar_wait(ring_empty(s), ph ^ 1u, 120 + s);
            mbar_expect_tx(ring_full(s), CHUNK_BYTES);
            tma_load_3d(ring_base + s * CHUNK_BYTES, &tmap_q, ring_full(s), c * 64, q0, bh, kEvictLast);
            if (++s == kRing) { s = 0; ph ^= 1u; }
          }
          mbar_wait(ring_empty(s), ph ^ 1u, 100 + s);
          mbar_expect_tx(ring_full(s), CHUNK_BYTES);
          tma_load_3d(ring_base + s * CHUNK_BYTES, &tmap_k, ring_full(s), c * 64, j * BC, bh, kEvictLast);
          if (++s == kRing) { s = 0; ph ^= 1u; }
        }
      };
      auto load_v_tile = [&](int j) {
        if constexpr (kWide) {
          for (int r = 0; r < 2; ++r) {          // 64 keys per slot: NVB boxes {64 d x 64 keys}
            mbar_wait(ring_empty(s), ph ^ 1u, 110 + s);
            mbar_expect_tx(ring_full(s), NVB * 8192);
            for (int b = 0; b < NVB; ++b)
              tma_load_3d(ring_base + s * SLOT + b * 8192, &tmap_v, ring_full(s), d0 + b * 64, j * BC + r * 64, bh, kEvictLast);
            if (++s == kRing) { s = 0; ph ^= 1u; }
          }
          return;
        }
        for (int r = 0; r < 4; ++r) {
          mbar_wait(ring_empty(s), ph ^ 1u, 110 + s);
          mbar_expect_tx(ring_full(s), NVB * 4096);
          for (int b = 0; b < NVB; ++b)
            tma_load_3d(ring_base + s * CHUNK_BYTES + b * 4096, &tmap_v, ring_full(s), d0 + b * 64,
                        j * BC + r * 32, bh, kEvictLast);
          if (++s == kRing) { s = 0; ph ^= 1u; }
        }
      };
      load_k_tile(0);
      if (T > 1) load_k_tile(1);
      for (int j = 0; j < T; ++j) {
        load_v_tile(j);
        if (j + 2 < T) load_k_tile(j + 2);
      }
    }
  } else if (warp == 4) {
    // ============================== MMA issuer ==============================
    {
      // all 32 lanes run this loop (barrier waits are warp-wide); one elected lane issues
      const uint32_t idesc_qk = make_idesc_f16(BR, BC, false, false, true);
      const uint32_t idesc_pv = make_idesc_f16(BR, p.dv, false, true, true);
      int s = 0;
      uint32_t ph = 0;
      constexpr uint32_t kHi = desc_hi(1024);
      const uint32_t q_lo0 = desc_lo(q_base, 16);
      const uint32_t ring_lo_k = desc_lo(ring_base, 16);
      const uint32_t ring_lo_v = desc_lo(ring_base, kWide ? 8192 : 4096);   // LBO = one V box
      auto qk_tile = [&](int j) {
        const uint32_t d_tmem = tmem_base + (j & 1) * 128;
        if constexpr (kWide) {
          for (int c = 0; c < NQ; c += 2) {
            const bool two = (c + 1 < NQ);
            mbar_wait(ring_full(s), ph, 200 + s);
            tc_fence_after();
            const uint32_t qa = q_lo0 + c * (CHUNK_BYTES >> 4);
            const uint32_t kb = ring_lo_k + s * (SLOT >> 4);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_ss_lh<1>(d_tmem, qa + k * 2, kHi, kb + k * 2, kHi, idesc_qk, (c | k) != 0 ? 1u : 0u);
              if (two) {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  umma_ss_lh<1>(d_tmem, qa + (CHUNK_BYTES >> 4) + k * 2, kHi, kb + (CHUNK_BYTES >> 4) + k * 2, kHi, idesc_qk, 1u);
              }
              umma_commit(ring_empty(s));
              if (c + 2 >= NQ) umma_commit(s_full(j & 1));
            }
            __syncwarp();
            if (++s == kRing) { s = 0; ph ^= 1u; }
          }
          return;
        }
        for (int c = 0; c < NQ; ++c) {
          uint32_t qa = q_lo0 + c * (CHUNK_BYTES >> 4);
          int sq = -1;
          if (q_stream) {   // the Q chunk sits in the ring slot just before its K chunk
            mbar_wait(ring_full(s), ph, 190 + s);
            qa = ring_lo_k + s * (CHUNK_BYTES >> 4);
            sq = s;
            if (++s == kRing) { s = 0; ph ^= 1u; }
          }
          mbar_wait(ring_full(s), ph, 200 + s);
          tc_fence_after();
          const uint32_t kb = ring_lo_k + s * (CHUNK_BYTES >> 4);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_ss_lh<1>(d_tmem, qa + k * 2, kHi, kb + k * 2, kHi, idesc_qk, (c | k) != 0 ? 1u : 0u);
            if (sq >= 0) umma_commit(ring_empty(sq));
            umma_commit(ring_empty(s));
            if (c == NQ - 1) umma_commit(s_full(j & 1));
          }
          __syncwarp();
          if (++s == kRing) { s = 0; ph ^= 1u; }
        }
      };
      auto pv_tile = [&](int j) {
        const uint32_t p_tmem = tmem_base + (j & 1) * 128;
        mbar_wait(p_full(j & 1), (j >> 1) & 1, 240 + (j & 1));
        tc_fence_after();
        if constexpr (kWide) {
          for (int r = 0; r < 2; ++r) {
            mbar_wait(ring_full(s), ph, 210 + s);
            tc_fence_after();
            const uint32_t vb = ring_lo_v + s * (SLOT >> 4);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_ts_lh(tmem_o, p_tmem + (r * 4 + k) * 8, vb + k * (2048 >> 4), kHi, idesc_pv,
                           (j > 0 || (r | k) != 0) ? 1u : 0u);
              umma_commit(ring_empty(s));
              if (r == 1) umma_commit(o_done);
            }
            __syncwarp();
            if (++s == kRing) { s = 0; ph ^= 1u; }
          }
          return;
        }
        for (int r = 0; r < 4; ++r) {
          mbar_wait(ring_full(s), ph, 210 + s);
          tc_fence_after();
          const uint32_t vb = ring_lo_v + s * (CHUNK_BYTES >> 4);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 2; ++k)
              umma_ts_lh(tmem_o, p_tmem + (r * 2 + k) * 8, vb + k * (2048 >> 4), kHi, idesc_pv,
                         (j > 0 || (r | k) != 0) ? 1u : 0u);
            umma_commit(ring_empty(s));
            if (r == 3) umma_commit(o_done);
          }
          __syncwarp();
          if (++s == kRing) { s = 0; ph ^= 1u; }
        }
      };
      if (!q_stream) mbar_wait(q_full, 0, 250);
      tc_fence_after();
      qk_tile(0);
      if (T > 1) qk_tile(1);
      for (int j = 0; j < T; ++j) {
        pv_tile(j);
        if (j + 2 < T) qk_tile(j + 2);
      }
    }
  } else if (warp < 4) {
    // ============================== softmax warpgroup ==============================
    const int row = warp * 32 + lane;
    const uint32_t lane_field = static_cast<uint32_t>(warp * 32) << 16;
    const uint32_t tO = tmem_o + lane_field;
    const float c = p.scale_log2;
    float m_run = -INFINITY;
    float l_run = 0.f;
    const int key_end = kCausal ? attn_key_end(1, p.Nq, p.Nk, q0 + row) : p.Nk;   // keys past it are masked to -inf

    for (int j = 0; j < T; ++j) {
      const uint32_t tS = tmem_base + (j & 1) * 128 + lane_field;
      mbar_wait(s_full(j & 1), (j >> 1) & 1, 300 + (j & 1));
      tc_fence_after();
      uint32_t sreg[4][32];
      tmem_ld_x32(tS + 0, sreg[0]);
      tmem_ld_x32(tS + 32, sreg[1]);
      tmem_ld_x32(tS + 64, sreg[2]);
      tmem_ld_x32(tS + 96, sreg[3]);
      tmem_ld_wait();
      const int valid = key_end - j * BC;      // keys of this tile the row sees (the key tail / the diagonal)
      if (valid < BC) {
#pragma unroll
        for (int cb = 0; cb < 4; ++cb)
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (cb * 32 + i >= valid) sreg[cb][i] = 0xff800000u;
      }
      float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
      for (int cb = 0; cb < 4; ++cb) {
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          mx0 = fmaxf(mx0, __uint_as_float(sreg[cb][i + 0]));
          mx1 = fmaxf(mx1, __uint_as_float(sreg[cb][i + 1]));
          mx2 = fmaxf(mx2, __uint_as_float(sreg[cb][i + 2]));
          mx3 = fmaxf(mx3, __uint_as_float(sreg[cb][i + 3]));
        }
      }
      const float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
      const bool grow = (j == 0) || ((mx - m_run) * c > kRescaleThreshold);
      bool o_waited = false;
      if (__any_sync(0xffffffffu, grow)) {
        const float m_new = fmaxf(m_run, mx);
        const float alpha = (j == 0) ? 0.f : fast_exp2((m_run - m_new) * c);
        m_run = m_new;
        l_run *= alpha;
        if (j > 0) {
          mbar_wait(o_done, (j - 1) & 1, 310);
          o_waited = true;
          tc_fence_after();
          for (int cb = 0; cb < (p.dv >> 5); ++cb) {
            uint32_t o[32];
            tmem_ld_x32(tO + cb * 32, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st_x32(tO + cb * 32, o);
          }
        }
      }
      const float mc = m_run * c;
      // exp2 phase (softmax_math.cuh): packed FFMA2 / FADD2 around MUFU.EX2
      const uint64_t c2 = f2_pack(c, c);
      const uint64_t nmc2 = f2_pack(-mc, -mc);
      uint64_t acc[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
      for (int cb = 0; cb < 4; ++cb) {
        uint32_t pk[16];
        exp_chunk32(sreg[cb], c2, nmc2, pk, acc);
        tmem_st_x16(tS + cb * 16, pk);
      }
      l_run += f2_hsum4(acc);
      // S is double-buffered, so this warpgroup can run up to two P·V tiles ahead of the tensor pipe: it must
      // observe EVERY o_done phase in order, or a later parity wait would alias an older phase
      if (j > 0 && !o_waited) mbar_wait(o_done, (j - 1) & 1, 315);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full(j & 1));
    }

    // ---------------- epilogue: O / l -> fp16 -> swizzled smem (Q buffer) -> TMA store
    mbar_wait(o_done, (T - 1) & 1, 320);
    tc_fence_after();
    float inv_l = 1.0f / l_run;
    if (p.lse != nullptr && slab == 0 && (q0 + row) < p.Nq)
      p.lse[static_cast<size_t>(bh) * p.Nq + q0 + row] = 0.6931471805599453f * (m_run * c + log2f(l_run));
    if (p.rms_g > 0.f) {   // host guarantees dsplit == 1: the whole row is in this thread's lane
      float ss = 0.f;
      for (int cb = 0; cb < (p.dv >> 5); ++cb) {
        uint32_t o[32];
        tmem_ld_x32(tO + cb * 32, o);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) ss = fmaf(__uint_as_float(o[i]), __uint_as_float(o[i]), ss);
      }
      inv_l *= rsqrtf(ss * inv_l * inv_l / static_cast<float>(p.D) + 1e-5f) * p.rms_g;
    }
    for (int cb = 0; cb < (p.dv >> 5); ++cb) {
      uint32_t o[32];
      tmem_ld_x32(tO + cb * 32, o);
      tmem_ld_wait();
      // staging area = start of smem: the resident Q boxes, or the (now idle) ring when Q streamed
      uint8_t* box = smem_gen + (cb >> 1) * CHUNK_BYTES + row * 128;
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4) {
        uint4 v;
        v.x = pack_half2(__uint_as_float(o[q4 * 8 + 0]) * inv_l, __uint_as_float(o[q4 * 8 + 1]) * inv_l);
        v.y = pack_half2(__uint_as_float(o[q4 * 8 + 2]) * inv_l, __uint_as_float(o[q4 * 8 + 3]) * inv_l);
        v.z = pack_half2(__uint_as_float(o[q4 * 8 + 4]) * inv_l, __uint_as_float(o[q4 * 8 + 5]) * inv_l);
        v.w = pack_half2(__uint_as_float(o[q4 * 8 + 6]) * inv_l, __uint_as_float(o[q4 * 8 + 7]) * inv_l);
        const int chunk = (cb & 1) * 4 + q4;
        *reinterpret_cast<uint4*>(box + ((chunk ^ (row & 7)) << 4)) = v;
      }
    }
    fence_proxy_async_smem();
    named_bar_sync(1, 128);
    if (warp == 0 && lane == 0) {
      for (int b = 0; b < NVB; ++b)
        tma_store_3d(&tmap_o, smem_base + b * CHUNK_BYTES, d0 + b * 64, q0, bh);
      tma_store_commit();
      tma_store_wait<0>();
    }
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 6) tmem_dealloc<1>(tmem_base, kTmemCols);
}

}  // namespace attn_slab
}  // namespace b200
