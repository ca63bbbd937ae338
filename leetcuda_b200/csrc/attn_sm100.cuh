// attn_sm100.cuh — fused FlashAttention-2 forward for sm_100a, head dim <= 128.
//
//   O[b,h] = softmax(Q K^T * scale) V        fp16 in/out, fp32 statistics + accumulation
//
// Replaces the reference's flash_attn_mma_stages_* family
// (kernels/flash-attn/mma/basic/flash_attn_mma_share_qkv.cu:71-768 and siblings,
// SURVEY.md §8a rows a8-a12), which run one 256-thread CTA per 128 query rows
// with mma.sync m16n8k16 and keep S/P/O in registers.  Here instead one CTA
// owns TWO 128-row query tiles of one (batch, head) and the whole KV sequence:
//
//   warps 0-3  softmax warpgroup of query tile 0   (thread r <-> query row r, TMEM lane r)
//   warps 4-7  softmax warpgroup of query tile 1
//   warp  8    tcgen05.mma issuer (single thread)
//   warp  9    TMA producer (Q once, then the K/V ring)
//   warp  10   TMEM owner (alloc / dealloc)
//
//   TMEM (512 cols): S0 [0,128) S1 [128,256) O0 [256,256+DP) O1 [256+DP, 256+2DP)
//   P_t (fp16, 64 cols) aliases the first half of S_t.
//
//   per KV tile j (128 keys), per query tile t:
//     MMA   : S_t  = Q_t K_j^T            (SS, M=128 N=128 K=DP)          -> s_full[t]
//     WG t  : m,l update; P = exp2(S*c - m*c) -> fp16 -> TMEM             -> p_full[t]
//             (lazy rescale: O_t is touched only when the row max grew by > 2^8)
//     MMA   : O_t += P_t V_j               (TS, A from TMEM, M=128 N=DP K=128) -> o_done[t]
//   The two query tiles are software-pipelined against each other so that the
//   tensor pipe runs QK/PV of one tile while the other tile's warpgroup is in its
//   softmax (MUFU) phase.
//
// Shared memory: Q 2 x (128 x DP) fp16, K/V ring of kStages x (128 x DP) fp16, all
// as 128B-swizzled TMA boxes of 64 columns; the Q buffers are reused to stage O
// for the TMA store in the epilogue.
//
// Nq queries, Nk keys, causal (query row i sees the keys j <= i + Nk - Nq): a work item runs
// attn_kv_tiles(...) KV tiles, up to the tile holding the last key of its last real row (both
// query tiles run to tile 1's extent; tile 0 is fully masked on the last one), the per-row key
// end replaces the ragged-tail mask, and the items are dispatched heaviest first.
#pragma once
#include <cuda.h>

#include "sm100_ptx.cuh"
#include "softmax_math.cuh"

namespace b200 {
namespace attn {

constexpr int BR = 128;         // query rows per warpgroup / MMA M
constexpr int BC = 128;         // keys per KV tile / QK MMA N / PV MMA K
constexpr int kThreads = 384;   // 12 warps
constexpr int kStages = 4;      // K/V ring depth (K_j, V_j, K_j+1, V_j+1)
constexpr int kTmemCols = 512;

template <int DP>
struct Cfg {
  static constexpr int TILE_BYTES = BR * DP * 2;            // one Q / K / V tile
  static constexpr int BOX_BYTES = 128 * 128;               // one {64 x 128} swizzled box
  static constexpr int Q_BYTES = 2 * TILE_BYTES;
  static constexpr int KV_BYTES = kStages * TILE_BYTES;
  static constexpr int BAR_BYTES = 256;
  static constexpr int SMEM_BYTES = Q_BYTES + KV_BYTES + BAR_BYTES + 1024;
};

struct Params {
  int Nq;          // query rows (q, o, lse)
  int Nk;          // keys (k, v)
  int D;           // true head dim (<= DP)
  int num_kv;      // ceil(Nk / BC)
  int causal;      // 1: query row i sees the keys j <= i + Nk - Nq (bottom-right aligned; host guarantees Nk >= Nq)
  float scale_log2;  // softmax scale * log2(e)
  unsigned long long* trace;  // debug: clock64 timeline of CTA (0,0), nullptr = off (B200_FMHA_TRACE)
  float* lse;      // optional [B*H, Nq] fp32 output: ln sum_j exp(scale * q.k_j) per query row (the statistic
                   // merge_attn_states consumes, cuda_merge_attn_states.cu:19-95); nullptr = off
  float rms_g;     // > 0: RMS-normalise every output row over D in the epilogue (eps 1e-5) and scale by rms_g —
                   // the fused form of kernels/rms-norm/rms_norm.cu:55-110 applied to O; <= 0 = off
  // persistent launches (kPersist): one CTA per SM walks the (batch*head, query-tile-pair) work items
  __half* o_ptr;   // O base pointer: the epilogue stores rows straight from registers (no smem staging)
  int qpairs;      // ceil(Nq / 256): work items per (batch, head)
  int bhs;         // B * H
  int total_items; // qpairs * B * H
};

// timeline probe: role 0/1 = softmax warpgroup 0/1 (one lane), 2 = MMA issuer; 16 steps x 8 events.  Compiled in only
// with -DB200_ATTN_TRACE (side build, tools/gpu_probe_attn_variants.py --trace): the probes cost registers in every role
// (the MMA warp spilled its trace pointer inside the issue loop) and a predicate per probe in the hot loops.
#ifdef B200_ATTN_TRACE
#define B200_TRACE(role, step, ev)                                                      \
  do {                                                                                  \
    if (p.trace != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && (step) < 16)        \
      p.trace[((role) * 16 + (step)) * 8 + (ev)] = clock64();                           \
  } while (0)
#else
#define B200_TRACE(role, step, ev) do { } while (0)
#endif

// Pairs of every 32-score chunk whose exp2 runs on the FMA pipe instead of the MUFU pipe (softmax_math.cuh:
// exp_chunk32_mix; bit i = pair i; 0 = all on the MUFU pipe).  The classic softmax step is bound by the MUFU pipe
// (16 exp/clk/SM) with issue slots to spare.  A/B of the masks on one box, order-rotated over two rounds
// (profiles/r02_session2m.log; B4 H32 N4096, TFLOPS; cuDNN on that box 1445-1469 / 948-974):
//     mask                 D = 128        D = 64 (persistent grid)
//     0      (all MUFU)    1311-1319      648-739
//     0x4444 (4 of 16)     1332-1348      698-814
//     0x2492 (5 of 16)     1317-1336      760-822
//     0x5294 (6 of 16)     1319-1335      581-675
// At D = 64 a step has half the MMA work per exponential, so the softmax leg weighs more and a larger share pays.
#ifndef B200_ATTN_POLY_MASK
#define B200_ATTN_POLY_MASK 0x4444u       // head dims 65 .. 128
#endif
#ifndef B200_ATTN_POLY_MASK_D64
#define B200_ATTN_POLY_MASK_D64 0x2492u   // head dims <= 64
#endif

// lazy-rescale threshold in the log2 domain: P stays <= 2^8
constexpr float kRescaleThreshold = 8.0f;

// kPersist: persistent scheduling.  The one-shot launch runs (N/256) x B x H CTAs, one per SM at a time, and every
// CTA pays its prologue (TMEM allocation, barrier init, the latency of the first Q/K loads, the first Q.K^T) and
// its epilogue (O drain, conversion, store) with the tensor pipe idle — about 8 % of a CTA's life at N = 4096.
// Here one CTA per SM walks the work items w = blockIdx.x, blockIdx.x + gridDim.x, ...: all barriers simply keep
// counting phases, the K/V ring keeps streaming across items, Q.K^T of item i+1 is issued right behind the last
// P.V of item i (the tensor pipe executes in order, so S/P need no extra hand-shake), the softmax warpgroups drain
// O of item i while that runs, and two more barriers close the remaining hazards: q_empty (the Q buffer may be
// reloaded once the last Q.K^T of the item has retired) and o_free (the first P.V of the next item overwrites O
// only after the epilogue has read it).  The epilogue then stores from registers (Q's smem is busy being reloaded).
//
// kStep selects the softmax step (CTA timelines, profiles/r02_session2i.log: per 128-key row the classic step spends
// 67 clk reading S out of TMEM, 400 clk in the maximum scan and 1450 clk in the exp loop; the MUFU pipe alone needs 1024):
//   0  classic: read the 128 scores of the row, scan them for the maximum, exponentiate; P in two halves
//   (1: a speculative step with the maximum folded into the exp loop — exponentiate each half with the running maximum
//      while an FMNMX scan runs beside the MUFU work, redo on a miss — measured 1212 vs 1258, profiles/r02_session2b.log,
//      and removed: the scan instructions lengthen the exp loop by more than they take off the chain)
//   2  speculative, SUM-checked: no maximum scan at all.  The row is exponentiated with the RUNNING maximum; a stale
//      maximum only matters when P would leave the fp16 range, and the row sum that is accumulated anyway tells:
//      sum(P) <= 2^14 over 64 keys bounds every P by 2^14 (fp16 keeps its 11 bits up to 65504; O and l are fp32).
//      The check of the first half is evaluated one chunk late (behind the exps of chunk 2), so the drain of its
//      accumulator chain hides under MUFU work.  Only if some row of the warp exceeds the bound (or is inf / NaN) are
//      the raw scores re-read, the true maximum taken, O rescaled and the exps redone.
//   (3: the classic step on FOUR softmax warpgroups — two threads per query row, warps w and w+4 share 32 TMEM lanes —
//      was built, verified and measured 5 % slower, profiles/r02_session2l.log, and removed again: the exp loop is bound
//      by the MUFU pipe of the scheduler both warps sit on, tools/softmax_rate.cu, so a second warp adds nothing.)
//
// kCausal: the causal mask (Params::causal; the host instantiates it with kStep 0 only).  A separate instantiation keeps
// the per-row key end, the per-item extent and the reversed order out of the registers of the full-attention kernel.
template <int DP, bool kVT, int kStep, bool kPersist, bool kCausal>
__global__ void __launch_bounds__(kThreads, 1)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                const __grid_constant__ CUtensorMap tmap_v, const __grid_constant__ CUtensorMap tmap_o,
                const Params p) {
  using C_ = Cfg<DP>;
  constexpr int KSTEPS_QK = DP / 16;
  constexpr int KSTEPS_PV = BC / 16;
  constexpr int NBOX = DP / 64;  // 64-column boxes per tile
  constexpr bool kSumSpec = (kStep == 2);                    // sum-checked, no maximum scan
  static_assert(kStep == 0 || kStep == 2, "kStep: 0 classic, 2 sum-checked speculative");
  constexpr int W_MMA = 8, W_TMA = 9, W_TMEM = 10;           // warp indices of the service roles
  constexpr int kPArrivals = 4;                              // warps that arrive on p_full / p_hi of a tile
  constexpr int NP = 2;                                      // pieces P_t is handed to the MMA warp in
  extern __shared__ uint8_t smem_raw[];

  const uint32_t raw_u32 = smem_u32(smem_raw);
  const uint32_t smem_base = (raw_u32 + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - raw_u32);
  const uint32_t q_base = smem_base;
  const uint32_t kv_base = smem_base + C_::Q_BYTES;
  const uint32_t bar_base = kv_base + C_::KV_BYTES;
  auto q_full = [&](int t) { return bar_base + 8u * t; };
  auto kv_full = [&](int s) { return bar_base + 8u * (2 + s); };
  auto kv_empty = [&](int s) { return bar_base + 8u * (2 + kStages + s); };
  auto s_full = [&](int t) { return bar_base + 8u * (2 + 2 * kStages + t); };
  auto p_full = [&](int t) { return bar_base + 8u * (4 + 2 * kStages + t); };
  auto o_done = [&](int t) { return bar_base + 8u * (6 + 2 * kStages + t); };
  auto p_hi = [&](int t) { return bar_base + 8u * (8 + 2 * kStages + t); };   // second half of P_t
  auto pv_lo_done = [&](int t) { return bar_base + 8u * (11 + 2 * kStages + t); };   // kStep 2: first half of P_t.V retired
  auto q_empty = [&](int t) { return bar_base + 8u * (13 + 2 * kStages + t); };      // kPersist: last Q.K^T of the item retired
  auto o_free = [&](int t) { return bar_base + 8u * (15 + 2 * kStages + t); };       // kPersist: epilogue has read O_t
  auto p_part = [&](int t, int part) { return part == 0 ? p_full(t) : p_hi(t); };   // piece `part` of P_t is in TMEM
  const uint32_t tmem_slot = bar_base + 8u * (10 + 2 * kStages);
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(
      smem_gen + C_::Q_BYTES + C_::KV_BYTES + 8 * (10 + 2 * kStages));

  // shuffle-broadcast warp index: warp-uniform for ptxas -> convergent role branches and
  // uniform-datapath descriptor math in the MMA issue loop (no per-instruction R2UR waterfall)
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  // work items of this CTA: (batch*head, first query row); one-shot launches have exactly one.  Causal work items
  // are dispatched heaviest first: the one-shot grid runs its query-tile pairs in reverse; the persistent list is
  // ordered by descending KV extent (all heads of the last query-tile pair, then those of the one before, ...).
  const int w_first = kPersist ? static_cast<int>(blockIdx.x) : 0;
  const int w_step = kPersist ? static_cast<int>(gridDim.x) : 1;
  const int w_total = kPersist ? p.total_items : 1;
  auto item_coords = [&](int w, int& bh, int& q0) {
    if constexpr (kPersist) {
      if constexpr (kCausal) {
        const int r = w / p.bhs;
        bh = w - r * p.bhs;
        q0 = (p.qpairs - 1 - r) * (2 * BR);
      } else {
        bh = w / p.qpairs;
        q0 = (w - bh * p.qpairs) * (2 * BR);
      }
    } else {
      bh = blockIdx.y;
      q0 = (kCausal ? static_cast<int>(gridDim.x - 1u - blockIdx.x) : static_cast<int>(blockIdx.x)) * (2 * BR);
    }
  };
  // KV tiles of the item at q0: both query tiles run to the extent of tile 1 (tile 0 is masked on its last one)
  auto item_tiles = [&](int q0) { return kCausal ? attn_kv_tiles(1, p.num_kv, p.Nq, p.Nk, q0 + 2 * BR, BC) : p.num_kv; };

  if (warp == W_TMA && lane == 0) {
    prefetch_tmap(&tmap_q);
    prefetch_tmap(&tmap_k);
    prefetch_tmap(&tmap_v);
    prefetch_tmap(&tmap_o);
  }
  if (warp == W_MMA && lane == 0) {
    for (int t = 0; t < 2; ++t) {
      mbar_init(q_full(t), 1);
      mbar_init(s_full(t), 1);
      mbar_init(p_full(t), kPArrivals);
      mbar_init(p_hi(t), kPArrivals);
      mbar_init(o_done(t), 1);
      mbar_init(pv_lo_done(t), 1);
      mbar_init(q_empty(t), 1);
      mbar_init(o_free(t), 4);
    }
    for (int s = 0; s < kStages; ++s) {
      mbar_init(kv_full(s), 1);
      mbar_init(kv_empty(s), 1);
    }
    fence_mbar_init();
  }
  if (warp == W_TMEM) tmem_alloc<1>(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_gen, 0);
  const uint32_t tmem_s0 = tmem_base;            // S_t = tmem_s0 + t*128 ; P_t aliases S_t
  const uint32_t tmem_o0 = tmem_base + 256;      // O_t = tmem_o0 + t*DP

  // Register re-partition (setmaxnreg, first statement of each role branch): the two
  // softmax warpgroups hold a full S row (128 fp32) per thread; the producer/MMA
  // warpgroup needs almost nothing.  the launch allocation is 384 x 168 = 64512 = 256 x 208 + 128 x 88 (inc may only draw on
  // what dec released, otherwise the second warpgroup spins forever in TRY_ALLOC).
  if (warp >= W_MMA) {
   reg_dealloc<88>();
   if (warp == W_TMA) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      int bh = 0, q0 = 0, it = 0;
      auto load_q = [&](int t) {
        if (kPersist && it > 0) mbar_wait(q_empty(t), (it - 1) & 1, 120 + t);   // previous item's last Q.K^T retired
        mbar_expect_tx(q_full(t), C_::TILE_BYTES);
#pragma unroll
        for (int b = 0; b < NBOX; ++b)
          tma_load_3d(q_base + t * C_::TILE_BYTES + b * C_::BOX_BYTES, &tmap_q, q_full(t), b * 64,
                      q0 + t * BR, bh, kEvictFirst);
      };
      int s = 0;
      uint32_t ph = 0;
      auto load_k = [&](int j) {
        mbar_wait(kv_empty(s), ph ^ 1u, 100 + s);
        mbar_expect_tx(kv_full(s), C_::TILE_BYTES);
        const uint32_t dst = kv_base + s * C_::TILE_BYTES;
#pragma unroll
        for (int b = 0; b < NBOX; ++b)
          tma_load_3d(dst + b * C_::BOX_BYTES, &tmap_k, kv_full(s), b * 64, j * BC, bh, kEvictLast);
        if (++s == kStages) { s = 0; ph ^= 1u; }
      };
      auto load_v = [&](int j) {
        mbar_wait(kv_empty(s), ph ^ 1u, 110 + s);
        mbar_expect_tx(kv_full(s), C_::TILE_BYTES);
        const uint32_t dst = kv_base + s * C_::TILE_BYTES;
        if constexpr (kVT) {
          // V^T tile [DP d-rows x 128 keys], K-major: two boxes of 64 keys
#pragma unroll
          for (int b = 0; b < 2; ++b)
            tma_load_3d(dst + b * (DP * 128), &tmap_v, kv_full(s), j * BC + b * 64, 0, bh, kEvictLast);
        } else {
          // V tile [128 keys x DP], MN-major: NBOX boxes of 64 d-columns
#pragma unroll
          for (int b = 0; b < NBOX; ++b)
            tma_load_3d(dst + b * C_::BOX_BYTES, &tmap_v, kv_full(s), b * 64, j * BC, bh, kEvictLast);
        }
        if (++s == kStages) { s = 0; ph ^= 1u; }
      };
      for (int w = w_first; w < w_total; w += w_step, ++it) {
        item_coords(w, bh, q0);
        const int T = item_tiles(q0);
        load_q(0);
        load_k(0);
        load_q(1);
        load_v(0);
        for (int j = 1; j < T; ++j) {
          load_k(j);
          load_v(j);
        }
      }
    }
   } else if (warp == W_MMA) {
    // ============================== MMA issuer ==============================
    {
      // all 32 lanes run this loop (barrier waits are warp-wide); one elected lane issues
      constexpr uint32_t idesc_qk = make_idesc_f16(BR, BC, false, false, true);
      constexpr uint32_t idesc_pv = make_idesc_f16(BR, DP, false, !kVT, true);
      int s = 0;
      uint32_t ph = 0;
      auto advance = [&]() { if (++s == kStages) { s = 0; ph ^= 1u; } };
      // descriptors: constant high word (SBO 1024 B, SWIZZLE_128B) + linear low word
      constexpr uint32_t kHi = desc_hi(1024);
      auto issue_qk = [&](int t, uint32_t k_smem, bool last_of_item) {
        const uint32_t q_lo = desc_lo(q_base + t * C_::TILE_BYTES, 16);
        const uint32_t k_lo = desc_lo(k_smem, 16);
#pragma unroll
        for (int ks = 0; ks < KSTEPS_QK; ++ks) {
          const uint32_t off = (ks >> 2) * (C_::BOX_BYTES >> 4) + (ks & 3) * 2;
          umma_ss_lh<1>(tmem_s0 + t * 128, q_lo + off, kHi, k_lo + off, kHi, idesc_qk, ks != 0 ? 1u : 0u);
        }
        umma_commit(s_full(t));
        if (kPersist && last_of_item) umma_commit(q_empty(t));
      };
      // P_t arrives in NP pieces (halves: keys 0-63, 64-127; or quarters): the k16 steps of P.V over a piece
      // run on the tensor pipe while the warpgroup is still computing the exps of the next one
      auto issue_pv_part = [&](int t, int part, uint32_t v_smem, bool accumulate) {
        const uint32_t v_lo = desc_lo(v_smem, kVT ? 16 : C_::BOX_BYTES);
#pragma unroll
        for (int k4 = 0; k4 < KSTEPS_PV / NP; ++k4) {
          const int ks = part * (KSTEPS_PV / NP) + k4;
          const uint32_t off = kVT ? ((ks >> 2) * ((DP * 128) >> 4) + (ks & 3) * 2) : ks * (2048 >> 4);
          umma_ts_lh(tmem_o0 + t * DP, tmem_s0 + t * 128 + ks * 8, v_lo + off, kHi, idesc_pv,
                     (accumulate || ks != 0) ? 1u : 0u);
        }
        if (part == NP - 1) umma_commit(o_done(t));
        else if constexpr (kSumSpec) umma_commit(pv_lo_done(t));   // O_t may be rescaled behind this piece
      };
      int it = 0;
      uint32_t base = 0;   // phases the per-step barriers have completed: the KV extents of the previous items
      for (int w = w_first; w < w_total; w += w_step, ++it) {
      int bh, q0;
      item_coords(w, bh, q0);
      const int T = item_tiles(q0);
      // prologue: S_0(0), S_1(0)
      mbar_wait(q_full(0), it & 1, 200);
      mbar_wait(kv_full(s), ph, 210 + s);
      tc_fence_after();
      uint32_t k_smem = kv_base + s * C_::TILE_BYTES;
      if (elect_one()) issue_qk(0, k_smem, T == 1);
      __syncwarp();
      mbar_wait(q_full(1), it & 1, 201);
      tc_fence_after();
      if (elect_one()) {
        issue_qk(1, k_smem, T == 1);
        umma_commit(kv_empty(s));  // K_0 free once both QK retire
      }
      __syncwarp();
      advance();
      for (int j = 0; j < T; ++j) {
        const uint32_t par = (base + static_cast<uint32_t>(j)) & 1u;
        // V_j
        mbar_wait(kv_full(s), ph, 220 + s);
        tc_fence_after();
        const uint32_t v_smem = kv_base + s * C_::TILE_BYTES;
        const int sv = s;
        advance();
        const bool more = (j + 1 < T);
        const bool last_qk = (j + 2 == T);
        if (more) {
          mbar_wait(kv_full(s), ph, 230 + s);  // K_{j+1}
          tc_fence_after();
          k_smem = kv_base + s * C_::TILE_BYTES;
        }
        // tile 0, then tile 1: P.V piece by piece as the pieces of P arrive; behind the last piece the
        // next Q.K^T of the same tile (P aliases S, so it cannot go earlier)
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          B200_TRACE(2, j, 2 * t);
#pragma unroll
          for (int part = 0; part < NP; ++part) {
            mbar_wait(p_part(t, part), par, 240 + 4 * t + part);
            // the first P.V of an item overwrites O_t: the previous item's epilogue must have read it
            if (part == 0 && kPersist && j == 0 && it > 0) mbar_wait(o_free(t), (it - 1) & 1, 250 + t);
            if (part == 0) B200_TRACE(2, j, 2 * t + 1);
            tc_fence_after();
            if (elect_one()) {
              issue_pv_part(t, part, v_smem, j > 0);
              if (part == NP - 1) {
                if (t == 1) umma_commit(kv_empty(sv));  // V_j free
                if (more) {
                  issue_qk(t, k_smem, last_qk);
                  if (t == 1) umma_commit(kv_empty(s));  // K_{j+1} free
                }
              }
            }
            __syncwarp();
          }
        }
        if (more) advance();
        B200_TRACE(2, j, 4);
      }
      if constexpr (kPersist) base += static_cast<uint32_t>(T);
      }
    }
   }
  } else {
    // ============================== softmax warpgroups ==============================
    reg_alloc<208>();
    const int t = warp >> 2;                 // query tile of this warpgroup
    const int quarter = warp & 3;            // TMEM lane quarter of this warp
    const int row = quarter * 32 + lane;     // row inside the 128-row tile
    const uint32_t lane_field = static_cast<uint32_t>(quarter * 32) << 16;
    const uint32_t tS = tmem_s0 + t * 128 + lane_field;
    const uint32_t tO = tmem_o0 + t * DP + lane_field;
    const float c = p.scale_log2;
    const bool tracer = (quarter == 0 && lane == 0);
    uint32_t base = 0;   // phases the per-step barriers have completed: the KV extents of the previous items
    for (int w = w_first; w < w_total; w += w_step) {
    int bh, q0;
    item_coords(w, bh, q0);
    const int T = item_tiles(q0);
    float m_run = -INFINITY;  // running (possibly stale) row max of raw S
    float l_run = 0.f;        // running row sum of P

    for (int j = 0; j < T; ++j) {
      const uint32_t par = (base + static_cast<uint32_t>(j)) & 1u;
      if (tracer) B200_TRACE(t, j, 0);
      mbar_wait(s_full(t), par, 300 + t);
      if (tracer) B200_TRACE(t, j, 1);
      tc_fence_after();
      // keys of this tile the row sees (the key tail / the diagonal); the rest is masked to -inf
      const int valid = (kCausal ? attn_key_end(1, p.Nq, p.Nk, q0 + t * BR + row) : p.Nk) - j * BC;
      // O_t *= alpha in TMEM (lazy rescale; only ever called between two MMAs on O_t, see the callers)
      auto rescale_o = [&](float alpha) {
#pragma unroll
        for (int cb = 0; cb < DP / 32; ++cb) {
          uint32_t o[32];
          tmem_ld_x32(tO + cb * 32, o);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
          tmem_st_x32(tO + cb * 32, o);
        }
      };
      uint32_t sreg[4][32];
      tmem_ld_x32(tS + 0, sreg[0]);
      tmem_ld_x32(tS + 32, sreg[1]);
      tmem_ld_x32(tS + 64, sreg[2]);
      tmem_ld_x32(tS + 96, sreg[3]);
      tmem_ld_wait();
      if (tracer) B200_TRACE(t, j, 2);
      // mask the key tail of the last tile and, causal, the keys past the diagonal
      if (valid < BC) {
#pragma unroll
        for (int cb = 0; cb < 4; ++cb)
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (cb * 32 + i >= valid) sreg[cb][i] = 0xff800000u;  // -inf
      }
      if (kSumSpec && j > 0) {
        // ---------------- sum-checked speculative step (kStep 2, see the kernel comment)
        constexpr float kSumLimit = 16384.f;     // sum of P over 64 keys <= 2^14  =>  every P <= 2^14, fp16-safe
        float mc = m_run * c;
        const uint64_t c2 = f2_pack(c, c);
        uint64_t nmc2 = f2_pack(-mc, -mc);
        if (tracer) B200_TRACE(t, j, 3);
        // rare: some row of this warp left the fp16-safe range with the running maximum (or produced inf / NaN).
        // Take the true maximum of the raw scores of chunks [cb0, cb1) (re-read from TMEM where P has not
        // overwritten them: P chunks 0,1 live in the columns of score chunk 0, which the caller passes in
        // registers), rescale O and l, and redo the exps of those chunks.
        auto reload = [&](int cb, uint32_t (&sr)[32]) {
          tmem_ld_x32(tS + cb * 32, sr);
          tmem_ld_wait();
          if (valid < BC) {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (cb * 32 + i >= valid) sr[i] = 0xff800000u;
          }
        };
        auto rescale_to = [&](float hm, int piece) {
          const float m_new = fmaxf(m_run, hm);
          const float alpha = fast_exp2((m_run - m_new) * c);
          // O_t may only be touched between MMAs: after P.V of tile j-1 (first half) / after the P.V over the
          // first half of this tile (the second half is not issued before p_hi)
          if (piece == 0) mbar_wait(o_done(t), par ^ 1u, 310 + t);
          else mbar_wait(pv_lo_done(t), par, 312 + t);
          tc_fence_after();
          rescale_o(alpha);
          m_run = m_new;
          l_run *= alpha;
          mc = m_run * c;
          nmc2 = f2_pack(-mc, -mc);
        };
        uint64_t acc_lo[4] = {0ull, 0ull, 0ull, 0ull}, acc_hi[4] = {0ull, 0ull, 0ull, 0ull};
        uint32_t pk[16], pk2[16];
        exp_chunk32(sreg[0], c2, nmc2, pk, acc_lo);
        tmem_st_x16(tS + 0, pk);                 // P chunks 0,1 -> columns [0,32): the scores of chunk 0 stay in sreg[0]
        exp_chunk32(sreg[1], c2, nmc2, pk, acc_lo);
        tmem_st_x16(tS + 16, pk);
        exp_chunk32(sreg[2], c2, nmc2, pk2, acc_hi);  // held back: its columns [32,48) still carry the scores of chunk 1
        float hs = f2_hsum4(acc_lo);             // chain of the first half: resolved long ago, behind chunk 2's exps
        if (__any_sync(0xffffffffu, !(hs <= kSumLimit))) {
          uint32_t sr[32];
          float hm = -INFINITY;
#pragma unroll
          for (int i = 0; i < 32; ++i) hm = fmaxf(hm, __uint_as_float(sreg[0][i]));
          reload(1, sr);
#pragma unroll
          for (int i = 0; i < 32; ++i) hm = fmaxf(hm, __uint_as_float(sr[i]));
          rescale_to(hm, 0);
          acc_lo[0] = acc_lo[1] = acc_lo[2] = acc_lo[3] = 0ull;
          acc_hi[0] = acc_hi[1] = acc_hi[2] = acc_hi[3] = 0ull;
          uint32_t pkr[16];
          exp_chunk32(sr, c2, nmc2, pkr, acc_lo);
          tmem_st_x16(tS + 16, pkr);
          exp_chunk32(sreg[0], c2, nmc2, pkr, acc_lo);
          tmem_st_x16(tS + 0, pkr);
          exp_chunk32(sreg[2], c2, nmc2, pk2, acc_hi);
          hs = f2_hsum4(acc_lo);
        }
        l_run += hs;                             // folded per half: a rescale in the second half scales it too
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full(t));
        tmem_st_x16(tS + 32, pk2);
        exp_chunk32(sreg[3], c2, nmc2, pk, acc_hi);
        tmem_st_x16(tS + 48, pk);
        hs = f2_hsum4(acc_hi);
        if (tracer) B200_TRACE(t, j, 4);
        if (__any_sync(0xffffffffu, !(hs <= kSumLimit))) {
          uint32_t sr[32];
          float hm = -INFINITY;
          reload(2, sr);
#pragma unroll
          for (int i = 0; i < 32; ++i) hm = fmaxf(hm, __uint_as_float(sr[i]));
          reload(3, sr);
#pragma unroll
          for (int i = 0; i < 32; ++i) hm = fmaxf(hm, __uint_as_float(sr[i]));
          rescale_to(hm, 1);
          acc_hi[0] = acc_hi[1] = acc_hi[2] = acc_hi[3] = 0ull;
          uint32_t pkr[16];
          exp_chunk32(sr, c2, nmc2, pkr, acc_hi);      // sr holds chunk 3
          tmem_st_x16(tS + 48, pkr);
          reload(2, sr);
          exp_chunk32(sr, c2, nmc2, pkr, acc_hi);
          tmem_st_x16(tS + 32, pkr);
          hs = f2_hsum4(acc_hi);
        }
        l_run += hs;
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_hi(t));
        if (tracer) B200_TRACE(t, j, 5);
        continue;
      }
      {
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
#ifdef B200_EXPERIMENT_NO_MAX
        // perf experiment only (valid for small random scores): no maximum scan, exps relative to 0
        const float mx = 0.f;
#else
        const float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
#endif
        // lazy rescale decision (warp-uniform because tcgen05.ld/st are warp collectives)
        const bool grow = (j == 0) || ((mx - m_run) * c > kRescaleThreshold);
        if (__any_sync(0xffffffffu, grow)) {
          const float m_new = fmaxf(m_run, mx);
          const float alpha = (j == 0) ? 0.f : fast_exp2((m_run - m_new) * c);
          m_run = m_new;
          l_run *= alpha;
          if (j > 0) {
            // O_t must be complete (PV of tile j-1 retired) before it is rescaled
            mbar_wait(o_done(t), par ^ 1u, 310 + t);
            tc_fence_after();
  #pragma unroll
            for (int cb = 0; cb < DP / 32; ++cb) {
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
        if (tracer) B200_TRACE(t, j, 3);
        // exp2 phase (softmax_math.cuh): packed FFMA2 / FADD2 around MUFU.EX2
        const uint64_t c2 = f2_pack(c, c);
        const uint64_t nmc2 = f2_pack(-mc, -mc);
        uint64_t acc[4] = {0ull, 0ull, 0ull, 0ull};
  #pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
          uint32_t pk[16];
          constexpr uint32_t kPolyMask = (DP <= 64) ? B200_ATTN_POLY_MASK_D64 : B200_ATTN_POLY_MASK;
          if constexpr (kPolyMask != 0) exp_chunk32_mix<kPolyMask>(sreg[cb], c2, nmc2, pk, acc);
          else exp_chunk32(sreg[cb], c2, nmc2, pk, acc);
          tmem_st_x16(tS + cb * 16, pk);
          if (cb == 1) {   // first half of P_t (keys 0-63) complete: let P·V start on it (+7 %)
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(p_full(t));
          }
        }
        l_run += f2_hsum4(acc);
        if (tracer) B200_TRACE(t, j, 4);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_hi(t));
      }
      if (tracer) B200_TRACE(t, j, 5);
    }

    // ---------------- epilogue: O / l -> fp16 -> (one-shot) swizzled smem (Q_t buffer) -> TMA store
    //                                             (persistent) straight from registers to global memory
    mbar_wait(o_done(t), (base + static_cast<uint32_t>(T) - 1u) & 1u, 320 + t);
    if constexpr (kPersist) base += static_cast<uint32_t>(T);
    tc_fence_after();
    const int qrow = q0 + t * BR + row;
    float inv_l = 1.0f / l_run;
    if (p.lse != nullptr && qrow < p.Nq)
      p.lse[static_cast<size_t>(bh) * p.Nq + qrow] = 0.6931471805599453f * (m_run * c + log2f(l_run));
    if (p.rms_g > 0.f) {
      // fused RMS norm: the whole output row of this query sits in this thread's TMEM lane.  One extra
      // pass over the accumulator (TMEM reads are cheap) gives sum(o^2); columns beyond D are exactly 0.
      float ss = 0.f;
#pragma unroll
      for (int cb = 0; cb < DP / 32; ++cb) {
        uint32_t o[32];
        tmem_ld_x32(tO + cb * 32, o);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) ss = fmaf(__uint_as_float(o[i]), __uint_as_float(o[i]), ss);
      }
      inv_l *= rsqrtf(ss * inv_l * inv_l / static_cast<float>(p.D) + 1e-5f) * p.rms_g;
    }
    if constexpr (kPersist) {
      __half* orow = p.o_ptr + (static_cast<size_t>(bh) * p.Nq + qrow) * p.D;
#pragma unroll
      for (int cb = 0; cb < DP / 32; ++cb) {
        uint32_t o[32];
        tmem_ld_x32(tO + cb * 32, o);
        tmem_ld_wait();
        if (cb == DP / 32 - 1) {
          // O_t has been read: the next item's first P.V may overwrite it
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(o_free(t));
        }
        if (qrow < p.Nq) {
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            const int col = cb * 32 + q4 * 8;
            if (col < p.D) {
              uint4 v;
              v.x = pack_half2(__uint_as_float(o[q4 * 8 + 0]) * inv_l, __uint_as_float(o[q4 * 8 + 1]) * inv_l);
              v.y = pack_half2(__uint_as_float(o[q4 * 8 + 2]) * inv_l, __uint_as_float(o[q4 * 8 + 3]) * inv_l);
              v.z = pack_half2(__uint_as_float(o[q4 * 8 + 4]) * inv_l, __uint_as_float(o[q4 * 8 + 5]) * inv_l);
              v.w = pack_half2(__uint_as_float(o[q4 * 8 + 6]) * inv_l, __uint_as_float(o[q4 * 8 + 7]) * inv_l);
              *reinterpret_cast<uint4*>(orow + col) = v;
            }
          }
        }
      }
    } else {
    uint8_t* stage = smem_gen + t * C_::TILE_BYTES;
#pragma unroll
    for (int cb = 0; cb < DP / 32; ++cb) {
      uint32_t o[32];
      tmem_ld_x32(tO + cb * 32, o);
      tmem_ld_wait();
      uint8_t* box = stage + (cb >> 1) * C_::BOX_BYTES + row * 128;
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4) {
        uint4 v;
        v.x = pack_half2(__uint_as_float(o[q4 * 8 + 0]) * inv_l, __uint_as_float(o[q4 * 8 + 1]) * inv_l);
        v.y = pack_half2(__uint_as_float(o[q4 * 8 + 2]) * inv_l, __uint_as_float(o[q4 * 8 + 3]) * inv_l);
        v.z = pack_half2(__uint_as_float(o[q4 * 8 + 4]) * inv_l, __uint_as_float(o[q4 * 8 + 5]) * inv_l);
        v.w = pack_half2(__uint_as_float(o[q4 * 8 + 6]) * inv_l, __uint_as_float(o[q4 * 8 + 7]) * inv_l);
        const int chunk = (cb & 1) * 4 + q4;  // 16-byte chunk inside the 128-byte row
        *reinterpret_cast<uint4*>(box + ((chunk ^ (row & 7)) << 4)) = v;
      }
    }
    fence_proxy_async_smem();
    named_bar_sync(1 + t, 128);
    if (quarter == 0 && lane == 0 && (q0 + t * BR) < p.Nq) {
#pragma unroll
      for (int b = 0; b < NBOX; ++b)
        tma_store_3d(&tmap_o, q_base + t * C_::TILE_BYTES + b * C_::BOX_BYTES, b * 64, q0 + t * BR, bh);
      tma_store_commit();
      tma_store_wait<0>();
    }
    }
    }   // work items
  }

  // ============================== teardown ==============================
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == W_TMEM) tmem_dealloc<1>(tmem_base, kTmemCols);
}

}  // namespace attn
}  // namespace b200
