// attn_pair_sm100.cuh — fused attention forward for head dims 256 <= D <= 512 (D % 128 == 0) on a
// CTA PAIR: the FFPA / QKV-tiling configuration of BASELINE configs[3] (B2 H16 N2048 D512).
//
// Replaces ffpa-attn/csrc/cuffpa/ffpa_attn_templates_L1.cuh:7-590 (ffpa_mma_acc_{f16,f32}_L1) and
// kernels/flash-attn/mma/basic/flash_attn_mma_tiling_qkv.cu:77-797 for these head dims
// (SURVEY.md §8a rows a10, a13).
//
// The constraint is TMEM: 128 lanes x 512 fp32 columns per SM, and O[128 x 512] alone fills it.
// The column-slab kernel (attn_slab_sm100.cuh) answers with two sibling CTAs that both compute the
// whole S = Q K^T: a third of its tensor work is redundant.  Here the two CTAs of a cluster share
// ONE 128-row query tile through tcgen05.mma.cta_group::2 with M = 128: every CTA owns 64 query
// rows, and an M=128 pair instruction stores a CTA's 64 x N result as 128 lanes x N/2 columns
// (lanes 0-63: columns [0,N/2), lanes 64-127: columns [N/2,N) of the SAME rows).  Per CTA:
//
//   S = Q K^T  : N = 256 keys per KV tile           -> 128 lanes x 128 columns, double-buffered
//   O += P V   : two instructions, N = 256 and D-256 -> 128 lanes x (128 + (D-256)/2) columns
//   TMEM       : S0 [0,128)  S1 [128,256)  O_lo [256,384)  O_hi [384,384+(D-256)/2)
//
// Nothing is computed twice, the B operands (K rows / V columns) are split between the two CTAs'
// shared memory as cta_group::2 prescribes, and a query row lives entirely inside one CTA, so the
// softmax needs no cross-CTA exchange.  A row is spread over two TMEM lanes (r and 64+r) = two
// threads of different warps: they combine their row max (and, once, the row sum) through smem.
// P (fp16) cannot feed the MMA from TMEM here (the A operand of an M=128 pair instruction must be
// duplicated on lanes r and 64+r, and a warp only reaches its own 32 lanes), so it is staged in
// shared memory as the K-major A operand (64 rows x 256 keys, 32 KiB).
//
//   warps 0-3  softmax warpgroup: thread L <-> TMEM lane L, row L & 63, key half L >> 6
//   warp  4    tcgen05.mma issuer (leader CTA only)     warp 5  TMA producer     warp 6  TMEM owner
//
// Shared memory per CTA: Q resident (D/64 boxes {64 d x 64 rows}, 8 KiB each), P 32 KiB, a ring of
// 4 x 32 KiB chunks in MMA consumption order:
//   K chunk = two boxes {64 d x 128 keys} (this CTA's half of the 256 keys) -> 8 k16 steps of S += Q_c K_c^T
//   V chunk = {64 d x 64 keys} boxes of this CTA's d-columns (MN-major)     -> 4 k16 steps of O_lo/O_hi += P V
// A chunk is 8 MMAs = 512 tensor cycles per barrier round trip of the issuing warp: with 16 KiB chunks
// (4 MMAs, 256 cycles) that single warp's wait/elect/issue/commit latency (~400 clk) was the limiter
// (44 % tensor-active, profiles/r02_attn_pair_ncu_summary_v1.txt).
// Tensor work per KV tile and pair: 2 x 128 x 256 x 512 MACs = 4096 clk at 8192 MAC/clk, all useful;
// MUFU work per SM 64 x 256 / 16 = 1024 clk, so the softmax hides behind the MMAs.
#pragma once
#include <cuda.h>

#include "sm100_ptx.cuh"
#include "softmax_math.cuh"

namespace b200 {
namespace attn_pair {

constexpr int BR = 128;          // query rows per CTA pair
constexpr int ROWS = 64;         // query rows per CTA
constexpr int BC = 256;          // keys per KV tile
constexpr int kThreads = 256;
constexpr int kRing = 4;
constexpr int CHUNK_BYTES = 32768;
constexpr int KBOX_BYTES = 16384;  // {64 d x 128 keys} fp16
constexpr int VBOX_BYTES = 8192;   // {64 d x 64 keys} fp16
constexpr int QBOX_BYTES = 8192;   // {64 d x 64 rows} fp16
constexpr int P_BYTES = 32768;     // 64 rows x 256 keys fp16 = 4 boxes {64 keys x 64 rows}
constexpr int BAR_BYTES = 256;
constexpr int XCHG_BYTES = 2 * 128 * 4;   // row-max exchange, double-buffered by tile parity
constexpr int kTmemCols = 512;
constexpr float kRescaleThreshold = 8.0f;

constexpr int smem_bytes(int nq) {
  return nq * QBOX_BYTES + P_BYTES + kRing * CHUNK_BYTES + BAR_BYTES + XCHG_BYTES + 1024;
}

struct Params {
  int Nq;           // query rows (q, o, lse)
  int Nk;           // keys (k, v)
  int num_kv;       // ceil(Nk / BC)
  int causal;       // 1: query row i sees the keys j <= i + Nk - Nq (bottom-right aligned; host guarantees Nk >= Nq;
                    // one-shot launches only)
  int nq;           // D / 64: 64-wide d-chunks of Q / K (4, 6 or 8)
  int n_hi;         // D - 256: N of the second P.V instruction (0, 128 or 256)
  float scale_log2; // softmax scale * log2(e)
  float* lse;       // optional [B*H, Nq] fp32: log-sum-exp of the scaled scores (natural log); nullptr = off
  float rms_g;      // > 0: fused RMS norm of the output rows over D (eps 1e-5), scaled by rms_g; see attn_sm100.cuh
  // persistent launches (kPersist): one cluster per SM pair walks the (batch*head, query tile) work items
  __half* o_ptr;    // O base pointer: the epilogue stores rows straight from registers (Q's smem is being reloaded)
  int qtiles;       // ceil(Nq / 128): work items per (batch, head)
  int total_items;  // qtiles * B * H
};

// kPersist: at N = 2048 a pair runs only 8 KV tiles (33 k tensor cycles) per query tile, so the one-shot grid's
// prologue (TMEM allocation, barrier init, the first Q / K loads) and epilogue (O drain + store) with the tensor
// pipe idle cost ~15 % (1202 TFLOPS at N = 2048 against 1480 at N = 8192, profiles/r02_session2b.log).  The
// persistent form treats the KV tiles of all the work items of a cluster as ONE sequence g = 0, 1, 2, ...: the K/V
// ring, the double-buffered S and the single P buffer simply keep rotating across items; Q.K^T of the next item's
// first tiles is issued behind the P.V of this item's last tiles; Q is reloaded by a thread of its own (warp 7) as
// soon as the item's last Q.K^T has retired (q_empty); the softmax warpgroup drains O right after handing over the
// item's last P and releases it (o_free) before the next item's first P.V overwrites it; O goes to global memory
// straight from registers.  With kPersist = false the same code runs exactly one item per cluster.
template <bool kPersist>
__global__ void __launch_bounds__(kThreads, 1)
attn_pair_fwd_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                     const __grid_constant__ CUtensorMap tmap_v, const __grid_constant__ CUtensorMap tmap_o,
                     const Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_u32 = smem_u32(smem_raw);
  const uint32_t smem_base = (raw_u32 + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - raw_u32);
  const int NQ = p.nq;
  const int q_bytes = NQ * QBOX_BYTES;
  const uint32_t q_base = smem_base;
  const uint32_t p_base = q_base + q_bytes;
  const uint32_t ring_base = p_base + P_BYTES;
  const uint32_t bar_base = ring_base + kRing * CHUNK_BYTES;
  auto ring_full = [&](int s) { return bar_base + 8u * s; };               // leader's: both CTAs' loads land on it
  auto ring_empty = [&](int s) { return bar_base + 8u * (kRing + s); };    // per CTA, multicast commit
  auto s_full = [&](int b) { return bar_base + 8u * (2 * kRing + b); };    // per CTA, multicast commit
  const uint32_t p_full = bar_base + 8u * (2 * kRing + 2);                 // leader's: 8 softmax warps arrive
  const uint32_t o_done = bar_base + 8u * (2 * kRing + 3);                 // per CTA, multicast commit
  auto q_full = [&](int c2) { return bar_base + 8u * (2 * kRing + 8 + c2); };     // leader's, one per pair of Q boxes
  auto q_empty = [&](int c2) { return bar_base + 8u * (2 * kRing + 12 + c2); };   // per CTA, multicast commit (kPersist)
  const uint32_t o_free = bar_base + 8u * (2 * kRing + 7);                 // leader's: 8 softmax warps arrive (kPersist)
  const uint32_t tmem_slot = bar_base + 8u * (2 * kRing + 5);
  uint8_t* bar_gen = smem_gen + q_bytes + P_BYTES + kRing * CHUNK_BYTES;
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(bar_gen + 8 * (2 * kRing + 5));
  float* xchg = reinterpret_cast<float*>(bar_gen + BAR_BYTES);             // [2][128]

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = (rank == 0);
  // work items of this cluster; the KV tiles of all of them form one sequence g = it * T + j
  const int cid = static_cast<int>(blockIdx.x >> 1), ncl = static_cast<int>(gridDim.x >> 1);
  const int n_items = kPersist ? (p.total_items - cid + ncl - 1) / ncl : 1;
  // causal (one-shot only): the clusters run their query tiles in reverse, heaviest first
  const int qt0 = p.causal ? ncl - 1 - cid : cid;
  // KV tiles per item: the two CTAs share every MMA, so the extent follows the last row of the cluster's 128-row tile
  const int T = kPersist ? p.num_kv : attn_kv_tiles(p.causal, p.num_kv, p.Nq, p.Nk, qt0 * BR + BR, BC);
  const int total = n_items * T;
  auto item_coords = [&](int it, int& bh, int& q0) {     // q0: first query row of THIS CTA
    if constexpr (kPersist) {
      const int w = cid + it * ncl;
      bh = w / p.qtiles;
      q0 = (w - bh * p.qtiles) * BR + static_cast<int>(rank) * ROWS;
    } else {
      bh = blockIdx.y;
      q0 = qt0 * BR + static_cast<int>(rank) * ROWS;
    }
  };
  const int n_hi_cta = p.n_hi >> 1;           // d-columns of O_hi held by this CTA (64 or 128)
  const int NVB = 2 + (n_hi_cta >> 6);        // 64-wide V boxes per chunk (3 or 4)

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
    mbar_init(s_full(0), 1);
    mbar_init(s_full(1), 1);
    mbar_init(p_full, 8);
    mbar_init(o_done, 1);
    for (int c2 = 0; c2 < 4; ++c2) {
      mbar_init(q_full(c2), 1);
      mbar_init(q_empty(c2), 1);
    }
    mbar_init(o_free, 8);
    fence_mbar_init();
  }
  if (warp == 6) tmem_alloc<2>(tmem_slot, kTmemCols);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_gen, 0);
  const uint32_t tmem_o_lo = tmem_base + 256;
  const uint32_t tmem_o_hi = tmem_base + 384;

  if (warp == 7) {
    // ============================== Q producer (both CTAs): one load per work item ==============================
    if (lane == 0) {
      const uint32_t qfull0 = mapa(q_full(0), 0);
      for (int it = 0; it < n_items; ++it) {
        int bh, q0;
        item_coords(it, bh, q0);
        // Q is reloaded pair of boxes by pair of boxes, each as soon as the previous item's LAST Q.K^T tile has
        // consumed it: the reload then runs under that tile's remaining MMAs instead of after them
        for (int c2 = 0; c2 < NQ / 2; ++c2) {
          if (it > 0) mbar_wait(q_empty(c2), (it - 1) & 1, 130 + c2);
          if (leader) mbar_expect_tx(q_full(c2), 2 * 2 * QBOX_BYTES);
          tma_load_3d_cg2(q_base + (2 * c2) * QBOX_BYTES, &tmap_q, qfull0 + 8u * c2, c2 * 128, q0, bh, kEvictFirst);
          tma_load_3d_cg2(q_base + (2 * c2 + 1) * QBOX_BYTES, &tmap_q, qfull0 + 8u * c2, c2 * 128 + 64, q0, bh, kEvictFirst);
        }
      }
    }
  } else if (warp == 5) {
    // ============================== K/V producer (both CTAs, own halves) ==============================
    if (lane == 0) {
      const uint32_t full0 = mapa(ring_full(0), 0);      // the leader's barriers, as cluster addresses
      int s = 0;
      uint32_t ph = 0;
      auto load_k_tile = [&](int g) {
        int bh, q0;
        item_coords(g / T, bh, q0);
        const int key0 = (g % T) * BC + static_cast<int>(rank) * 128;
        for (int c2 = 0; c2 < NQ / 2; ++c2) {
          mbar_wait(ring_empty(s), ph ^ 1u, 100 + s);
          if (leader) mbar_expect_tx(ring_full(s), 2 * CHUNK_BYTES);
          const uint32_t dst = ring_base + s * CHUNK_BYTES;
          tma_load_3d_cg2(dst, &tmap_k, full0 + 8u * s, c2 * 128, key0, bh, kEvictLast);
          tma_load_3d_cg2(dst + KBOX_BYTES, &tmap_k, full0 + 8u * s, c2 * 128 + 64, key0, bh, kEvictLast);
          if (++s == kRing) { s = 0; ph ^= 1u; }
        }
      };
      auto load_v_tile = [&](int g) {
        int bh, q0;
        item_coords(g / T, bh, q0);
        const int d_lo = static_cast<int>(rank) * 128;
        const int d_hi = 256 + static_cast<int>(rank) * n_hi_cta;
        for (int r = 0; r < 4; ++r) {
          mbar_wait(ring_empty(s), ph ^ 1u, 110 + s);
          if (leader) mbar_expect_tx(ring_full(s), 2 * NVB * VBOX_BYTES);
          const uint32_t dst = ring_base + s * CHUNK_BYTES;
          const int key0 = (g % T) * BC + r * 64;
          for (int b = 0; b < NVB; ++b) {
            const int d = b < 2 ? d_lo + b * 64 : d_hi + (b - 2) * 64;
            tma_load_3d_cg2(dst + b * VBOX_BYTES, &tmap_v, full0 + 8u * s, d, key0, bh, kEvictLast);
          }
          if (++s == kRing) { s = 0; ph ^= 1u; }
        }
      };
      load_k_tile(0);
      if (total > 1) load_k_tile(1);
      for (int g = 0; g < total; ++g) {
        load_v_tile(g);
        if (g + 2 < total) load_k_tile(g + 2);
      }
    }
  } else if (warp == 4) {
    // ============================== MMA issuer (leader CTA) ==============================
    if (leader) {
      // all 32 lanes run the loop (barrier waits are warp-wide); one elected lane issues
      const uint32_t idesc_qk = make_idesc_f16(BR, BC, false, false, true);
      const uint32_t idesc_lo = make_idesc_f16(BR, 256, false, true, true);
      const uint32_t idesc_hi = make_idesc_f16(BR, p.n_hi > 0 ? p.n_hi : 256, false, true, true);
      constexpr uint32_t kHi = desc_hi(1024);
      const uint32_t q_lo0 = desc_lo(q_base, 16);
      const uint32_t p_lo0 = desc_lo(p_base, 16);
      const uint32_t ring_lo_k = desc_lo(ring_base, 16);
      const uint32_t ring_lo_v = desc_lo(ring_base, VBOX_BYTES);   // LBO = one {64 d x 64 keys} box
      int s = 0;
      uint32_t ph = 0;
      auto qk_tile = [&](int g) {
        const int it = g / T, j = g - it * T;
        const uint32_t d_tmem = tmem_base + (g & 1) * 128;
        for (int c2 = 0; c2 < NQ / 2; ++c2) {
          if (j == 0) mbar_wait(q_full(c2), it & 1, 250 + c2);   // first tile of a work item: this part of its Q must have landed
          mbar_wait(ring_full(s), ph, 200 + s);
          tc_fence_after();
          const uint32_t qa = q_lo0 + c2 * (2 * QBOX_BYTES >> 4);
          const uint32_t kb = ring_lo_k + s * (CHUNK_BYTES >> 4);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 8; ++k)     // two 64-wide d-chunks x four k16 steps
              umma_ss_lh<2>(d_tmem, qa + (k >> 2) * (QBOX_BYTES >> 4) + (k & 3) * 2, kHi,
                            kb + (k >> 2) * (KBOX_BYTES >> 4) + (k & 3) * 2, kHi, idesc_qk, (c2 | k) != 0 ? 1u : 0u);
            umma_commit_cg2(ring_empty(s), 0x3);
            if (kPersist && j == T - 1) umma_commit_cg2(q_empty(c2), 0x3);   // these Q boxes may be reloaded for the next item
            if (c2 == NQ / 2 - 1) umma_commit_cg2(s_full(g & 1), 0x3);
          }
          __syncwarp();
          if (++s == kRing) { s = 0; ph ^= 1u; }
        }
      };
      auto pv_tile = [&](int g) {
        const int it = g / T, j = g - it * T;
        mbar_wait(p_full, g & 1, 240);
        // the first P.V of an item overwrites O: the previous item's epilogue must have read it
        if (kPersist && j == 0 && it > 0) mbar_wait(o_free, (it - 1) & 1, 241);
        tc_fence_after();
        for (int r = 0; r < 4; ++r) {
          mbar_wait(ring_full(s), ph, 210 + s);
          tc_fence_after();
          const uint32_t vb = ring_lo_v + s * (CHUNK_BYTES >> 4);
          const uint32_t pa = p_lo0 + r * (QBOX_BYTES >> 4);              // P box r = keys [64r, 64r+64)
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {                                  // k16 steps inside the 64-key chunk
              const uint32_t acc = (j > 0 || (r | k) != 0) ? 1u : 0u;
              umma_ss_lh<2>(tmem_o_lo, pa + k * 2, kHi, vb + k * (2048 >> 4), kHi, idesc_lo, acc);
              if (p.n_hi > 0)     // D = 256 has no second column block
                umma_ss_lh<2>(tmem_o_hi, pa + k * 2, kHi, vb + (2 * VBOX_BYTES >> 4) + k * (2048 >> 4), kHi, idesc_hi, acc);
            }
            umma_commit_cg2(ring_empty(s), 0x3);
            if (r == 3) umma_commit_cg2(o_done, 0x3);
          }
          __syncwarp();
          if (++s == kRing) { s = 0; ph ^= 1u; }
        }
      };
      qk_tile(0);
      if (total > 1) qk_tile(1);
      for (int g = 0; g < total; ++g) {
        pv_tile(g);
        if (g + 2 < total) qk_tile(g + 2);
      }
    }
  } else if (warp < 4) {
    // ============================== softmax warpgroup ==============================
    const int L = warp * 32 + lane;          // TMEM lane of this thread
    const int row = L & 63;                  // query row inside this CTA's 64
    const int half = L >> 6;                 // which 128 keys of the 256-key tile / which column half of O
    const uint32_t lane_field = static_cast<uint32_t>(warp * 32) << 16;
    const float c = p.scale_log2;
    float m_run = -INFINITY;
    float l_run = 0.f;                       // partial row sum over this thread's key halves
    uint8_t* p_gen = smem_gen + q_bytes;
    int key_end = p.Nk;                      // one past the last key of this thread's row (keys past it: -inf)

    for (int g = 0; g < total; ++g) {
      const int it = g / T, j = g - it * T;
      if (j == 0) {                                         // a new work item
        m_run = -INFINITY;
        l_run = 0.f;
        int bh, q0;
        item_coords(it, bh, q0);
        key_end = attn_key_end(p.causal, p.Nq, p.Nk, q0 + row);
      }
      const uint32_t tS = tmem_base + (g & 1) * 128 + lane_field;
      mbar_wait(s_full(g & 1), (g >> 1) & 1, 300 + (g & 1));
      tc_fence_after();
      uint32_t sreg[4][32];
      tmem_ld_x32(tS + 0, sreg[0]);
      tmem_ld_x32(tS + 32, sreg[1]);
      tmem_ld_x32(tS + 64, sreg[2]);
      tmem_ld_x32(tS + 96, sreg[3]);
      tmem_ld_wait();
      const int valid = key_end - j * BC - half * 128;    // keys of this thread's half the row sees
      if (valid < 128) {
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
      float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
      // the other half of this row's keys sits on lane L ^ 64 (another warp): combine through smem
      float* xb = xchg + (g & 1) * 128;
      xb[L] = mx;
      named_bar_sync(1, 128);
      mx = fmaxf(mx, xb[L ^ 64]);
      // lazy rescale; the decision is identical in both threads of a row and warp-uniform
      const bool grow = (j == 0) || ((mx - m_run) * c > kRescaleThreshold);
      bool o_waited = false;
      if (__any_sync(0xffffffffu, grow)) {
        const float m_new = fmaxf(m_run, mx);
        const float alpha = (j == 0) ? 0.f : fast_exp2((m_run - m_new) * c);
        m_run = m_new;
        l_run *= alpha;
        if (j > 0) {
          mbar_wait(o_done, (g - 1) & 1, 310);
          o_waited = true;
          tc_fence_after();
          const int ncb = 4 + (n_hi_cta >> 5);    // 32-column blocks of O_lo (4) and O_hi (2 or 4)
          for (int cb = 0; cb < ncb; ++cb) {
            const uint32_t ta = (cb < 4 ? tmem_o_lo + cb * 32 : tmem_o_hi + (cb - 4) * 32) + lane_field;
            uint32_t o[32];
            tmem_ld_x32(ta, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st_x32(ta, o);
          }
          tmem_st_wait();
        }
      }
      const float mc = m_run * c;
      const uint64_t c2 = f2_pack(c, c);
      const uint64_t nmc2 = f2_pack(-mc, -mc);
      uint64_t acc[4] = {0ull, 0ull, 0ull, 0ull};
      uint32_t pk[4][16];
#pragma unroll
      for (int cb = 0; cb < 4; ++cb) exp_chunk32(sreg[cb], c2, nmc2, pk[cb], acc);
      l_run += f2_hsum4(acc);
      // the P buffer is single: P.V of the previous tile must have finished reading it.  (Every
      // o_done phase is observed in order, so a later parity wait cannot alias an older phase.)
      if (g > 0 && !o_waited) mbar_wait(o_done, (g - 1) & 1, 315);
      // P -> smem as the K-major A operand: box b = 64 keys, row pitch 128 B, 16-byte chunks XOR-swizzled
#pragma unroll
      for (int cb = 0; cb < 4; ++cb) {
        uint8_t* box = p_gen + (half * 2 + (cb >> 1)) * QBOX_BYTES + row * 128;
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          const uint4 v = make_uint4(pk[cb][q4 * 4 + 0], pk[cb][q4 * 4 + 1], pk[cb][q4 * 4 + 2], pk[cb][q4 * 4 + 3]);
          const int chunk = (cb & 1) * 4 + q4;
          *reinterpret_cast<uint4*>(box + ((chunk ^ (row & 7)) << 4)) = v;
        }
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(p_full, 0);
      if (j != T - 1) continue;

      // ---------------- epilogue of this work item: O / l -> fp16 -> global
      //   one-shot: swizzled smem (the Q boxes) -> TMA store;  persistent: straight from registers
      int bh, q0;
      item_coords(it, bh, q0);
      mbar_wait(o_done, g & 1, 320);
      tc_fence_after();
      float* xl = xchg + ((g + 1) & 1) * 128;      // the buffer tile g did not use
      xl[L] = l_run;
      const int ncb = 4 + (n_hi_cta >> 5);
      float ss = 0.f;
      float* xs = xchg + (g & 1) * 128;            // tile g's buffer: every thread is past its last use (p_full(g))
      if (p.rms_g > 0.f) {
        // fused RMS norm: this thread holds half of the row's columns, lane L ^ 64 the other half
        for (int cb = 0; cb < ncb; ++cb) {
          const uint32_t ta = (cb < 4 ? tmem_o_lo + cb * 32 : tmem_o_hi + (cb - 4) * 32) + lane_field;
          uint32_t o[32];
          tmem_ld_x32(ta, o);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) ss = fmaf(__uint_as_float(o[i]), __uint_as_float(o[i]), ss);
        }
        xs[L] = ss;
      }
      named_bar_sync(1, 128);
      const float l_row = l_run + xl[L ^ 64];
      float inv_l = 1.0f / l_row;
      if (p.lse != nullptr && half == 0 && (q0 + row) < p.Nq)
        p.lse[static_cast<size_t>(bh) * p.Nq + q0 + row] = 0.6931471805599453f * (m_run * c + log2f(l_row));
      if (p.rms_g > 0.f) {
        ss += xs[L ^ 64];
        inv_l *= rsqrtf(ss * inv_l * inv_l / static_cast<float>(NQ * 64) + 1e-5f) * p.rms_g;
      }
      for (int cb = 0; cb < ncb; ++cb) {
        const uint32_t ta = (cb < 4 ? tmem_o_lo + cb * 32 : tmem_o_hi + (cb - 4) * 32) + lane_field;
        // first head-dim column of these 32 accumulator columns
        const int d0 = cb < 4 ? half * 128 + cb * 32 : 256 + half * n_hi_cta + (cb - 4) * 32;
        uint32_t o[32];
        tmem_ld_x32(ta, o);
        tmem_ld_wait();
        if (kPersist && cb == ncb - 1) {
          // O has been read: the next item's first P.V may overwrite it
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(o_free, 0);
        }
        uint4 v[4];
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          v[q4].x = pack_half2(__uint_as_float(o[q4 * 8 + 0]) * inv_l, __uint_as_float(o[q4 * 8 + 1]) * inv_l);
          v[q4].y = pack_half2(__uint_as_float(o[q4 * 8 + 2]) * inv_l, __uint_as_float(o[q4 * 8 + 3]) * inv_l);
          v[q4].z = pack_half2(__uint_as_float(o[q4 * 8 + 4]) * inv_l, __uint_as_float(o[q4 * 8 + 5]) * inv_l);
          v[q4].w = pack_half2(__uint_as_float(o[q4 * 8 + 6]) * inv_l, __uint_as_float(o[q4 * 8 + 7]) * inv_l);
        }
        if constexpr (kPersist) {
          if ((q0 + row) < p.Nq) {
            __half* dst = p.o_ptr + (static_cast<size_t>(bh) * p.Nq + q0 + row) * (NQ * 64) + d0;
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) *reinterpret_cast<uint4*>(dst + q4 * 8) = v[q4];
          }
        } else {
          uint8_t* box = smem_gen + (d0 >> 6) * QBOX_BYTES + row * 128;
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            const int chunk = ((d0 & 63) >> 3) + q4;
            *reinterpret_cast<uint4*>(box + ((chunk ^ (row & 7)) << 4)) = v[q4];
          }
        }
      }
      if constexpr (kPersist) {
        // the exchange buffer used for the row sums is the next tile's row-max buffer: nobody may run ahead
        // into that tile before every partner has read its sum
        named_bar_sync(1, 128);
      } else {
        fence_proxy_async_smem();
        named_bar_sync(1, 128);
        if (warp == 0 && lane == 0 && q0 < p.Nq) {
          for (int b = 0; b < NQ; ++b)
            tma_store_3d(&tmap_o, smem_base + b * QBOX_BYTES, b * 64, q0, bh);
          tma_store_commit();
          tma_store_wait<0>();
        }
      }
    }
  }

  // ============================== teardown ==============================
  __syncwarp();
  tc_fence_before();
  cluster_sync_all();     // the peer's MMAs read this CTA's smem and commit onto its barriers until the end
  if (warp == 6) tmem_dealloc<2>(tmem_base, kTmemCols);
}

}  // namespace attn_pair
}  // namespace b200
