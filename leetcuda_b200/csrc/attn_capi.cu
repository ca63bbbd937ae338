// attn_capi.cu — C-ABI entry points of the attention path (include/leetcuda_b200.h).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "capi_common.cuh"
#include "attn_sm100.cuh"
#include "attn_slab_sm100.cuh"
#include "attn_pair_sm100.cuh"
#include "attn_cg2_sm100.cuh"

namespace b200 { namespace host {
int workspace(void** out, size_t bytes);
} }

#ifndef B200_ATTN_SPEC_DEFAULT
#define B200_ATTN_SPEC_DEFAULT 0
#endif
// Measured defaults (profiles/r02_session2b.log, r02_session2c.log; B4 H32 N4096, TFLOPS):
//   D = 128: single-CTA one-shot 1258-1279 | persistent 1236-1254 | speculative softmax 1212 (removed) | CTA pair (M=256) 946
//   D = 64 : single-CTA one-shot 600-730   | persistent 740-790
// The CTA-pair variant removes the shared-memory operand limit of Q.K^T (tools/umma_rate.cu) but every hand-shake of
// the softmax <-> MMA chain then crosses the cluster, and that chain — not a pipe — is what bounds the kernel.
#ifndef B200_ATTN_CG2_DEFAULT
#define B200_ATTN_CG2_DEFAULT 0
#endif
#ifndef B200_ATTN_PAIR_PERSIST_DEFAULT
#define B200_ATTN_PAIR_PERSIST_DEFAULT 0
#endif
#ifndef B200_ATTN_PERSIST_DEFAULT
#define B200_ATTN_PERSIST_DEFAULT 0
#endif

namespace {

using namespace b200;
using b200::host::fail;

template <int DP, bool kVT, int kStep, bool kPersist, bool kCausal>
int launch_fmha(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv,
                const CUtensorMap& to, const attn::Params& p, int BH, cudaStream_t stream) {
  // (the kernel is b200::attn::attn_fwd_kernel — the host-side names keep the C ABI's "fmha")
  using C_ = attn::Cfg<DP>;
  auto kern = attn::attn_fwd_kernel<DP, kVT, kStep, kPersist, kCausal>;
  static bool attr_set[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !attr_set[dev]) {
    B200_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      C_::SMEM_BYTES));
    attr_set[dev] = true;
  }
  dim3 grid((p.Nq + 2 * attn::BR - 1) / (2 * attn::BR), BH, 1);
  if (kPersist) {
    const int sms = host::sm_count();
    grid = dim3(static_cast<unsigned>(p.total_items < sms ? p.total_items : sms), 1, 1);
  }
  // debug: B200_FMHA_TRACE=<file> dumps the clock64 timeline of CTA (0,0) (synchronous!)
  const char* trace_path = getenv("B200_FMHA_TRACE");
  attn::Params pp = p;
  pp.trace = nullptr;
  if (trace_path && trace_path[0]) {
    const size_t n = 3 * 16 * 8;
    B200_CUDA_OK(cudaMalloc(&pp.trace, n * 8));
    B200_CUDA_OK(cudaMemset(pp.trace, 0, n * 8));
    kern<<<grid, attn::kThreads, C_::SMEM_BYTES, stream>>>(tq, tk, tv, to, pp);
    B200_CUDA_OK(cudaStreamSynchronize(stream));
    unsigned long long h[3 * 16 * 8];
    B200_CUDA_OK(cudaMemcpy(h, pp.trace, n * 8, cudaMemcpyDeviceToHost));
    cudaFree(pp.trace);
    if (FILE* f = fopen(trace_path, "w")) {
      for (int r = 0; r < 3; ++r)
        for (int j = 0; j < 16; ++j) {
          fprintf(f, "%d %d", r, j);
          for (int e = 0; e < 8; ++e) fprintf(f, " %llu", h[(r * 16 + j) * 8 + e]);
          fprintf(f, "\n");
        }
      fclose(f);
    }
    host::count_launch();
    return 0;
  }
  kern<<<grid, attn::kThreads, C_::SMEM_BYTES, stream>>>(tq, tk, tv, to, pp);
  B200_CUDA_OK(cudaGetLastError());
  host::count_launch();
  return 0;
}

// 64 < D <= 128 on CTA pairs (attn_cg2_sm100.cuh): cluster of two CTAs = 512 query rows, cta_group::2 MMAs with M = 256
template <bool kVT>
int launch_attn_cg2(const void* q, const void* k, const void* v, void* o, const attn2::Params& p, uint64_t BH, int N, int D,
                    cudaStream_t stream) {
  CUtensorMap tq, tk, tv, to;
  uint64_t dims[3] = {static_cast<uint64_t>(D), static_cast<uint64_t>(N), BH};
  uint64_t str[2] = {static_cast<uint64_t>(D) * 2, static_cast<uint64_t>(N) * D * 2};
  uint32_t qbox[3] = {64, 128, 1};
  uint32_t kbox[3] = {64, 64, 1};
  int rc;
  if ((rc = host::get_tmap(&tq, q, 3, dims, str, qbox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = host::get_tmap(&to, o, 3, dims, str, qbox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = host::get_tmap(&tk, k, 3, dims, str, kbox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if (kVT) {
    uint64_t vd[3] = {static_cast<uint64_t>(N), static_cast<uint64_t>(D), BH};
    uint64_t vs[2] = {static_cast<uint64_t>(N) * 2, static_cast<uint64_t>(N) * D * 2};
    if ((rc = host::get_tmap(&tv, v, 3, vd, vs, kbox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  } else {
    if ((rc = host::get_tmap(&tv, v, 3, dims, str, qbox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  auto kern = attn2::attn_cg2_fwd_kernel<kVT>;
  static bool attr_set[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !attr_set[dev]) {
    B200_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, attn2::SMEM_BYTES));
    attr_set[dev] = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(2u * static_cast<unsigned>((N + 4 * attn2::BR - 1) / (4 * attn2::BR)), static_cast<unsigned>(BH), 1);
  cfg.blockDim = dim3(attn2::kThreads, 1, 1);
  cfg.dynamicSmemBytes = attn2::SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attrs[1];
  attrs[0].id = cudaLaunchAttributeClusterDimension;
  attrs[0].val.clusterDim.x = 2;
  attrs[0].val.clusterDim.y = 1;
  attrs[0].val.clusterDim.z = 1;
  cfg.attrs = attrs;
  cfg.numAttrs = 1;
  B200_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, tq, tk, tv, to, p));
  host::count_launch();
  return 0;
}

// [BH, D, N] -> [BH, N, D] (fp16; N = the key length): the three reference ops that take V pre-transposed
// (flash_attn_mma.py:441-442) are served for D > 128 by restoring the natural layout first —
// an HBM-bound pre-pass (4*N*D bytes per head) in front of a tensor-bound kernel.
__global__ void transpose_dn_to_nd_kernel(const __half* __restrict__ in, __half* __restrict__ out, int D, int N) {
  __shared__ __half tile[32][33];
  const size_t head = static_cast<size_t>(blockIdx.z) * D * N;
  const int n0 = blockIdx.x * 32, d0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int d = d0 + i, n = n0 + threadIdx.x;
    if (d < D && n < N) tile[i][threadIdx.x] = in[head + static_cast<size_t>(d) * N + n];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int n = n0 + i, d = d0 + threadIdx.x;
    if (d < D && n < N) out[head + static_cast<size_t>(n) * D + d] = tile[threadIdx.x][i];
  }
}

// head dims 128 < D <= 1024: column-slab kernel (attn_slab_sm100.cuh)
// 256 <= D <= 512, D % 128 == 0: one 128-row query tile per CTA PAIR (attn_pair_sm100.cuh)
// Nq / Nk: query / key lengths (q, o, lse / k, v); causal: 0 | 1, validated by fmha_impl
int fmha_pair(const void* q, const void* k, const void* v, void* o, float* lse, float rms_g, int B, int H, int Nq, int Nk,
              int D, int causal, float scale, cudaStream_t stream) {
  const uint64_t BH = static_cast<uint64_t>(B) * H;
  attn_pair::Params p;
  p.Nq = Nq;
  p.Nk = Nk;
  p.num_kv = (Nk + attn_pair::BC - 1) / attn_pair::BC;
  p.causal = causal;
  p.nq = D / 64;
  p.n_hi = D - 256;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.lse = lse;
  p.rms_g = rms_g;

  CUtensorMap tq, tk, tv, to;
  uint64_t qdims[3] = {static_cast<uint64_t>(D), static_cast<uint64_t>(Nq), BH};
  uint64_t qstr[2] = {static_cast<uint64_t>(D) * 2, static_cast<uint64_t>(Nq) * D * 2};
  uint64_t kdims[3] = {static_cast<uint64_t>(D), static_cast<uint64_t>(Nk), BH};
  uint64_t kstr[2] = {static_cast<uint64_t>(D) * 2, static_cast<uint64_t>(Nk) * D * 2};
  uint32_t qbox[3] = {64, 64, 1};
  uint32_t kbox[3] = {64, 128, 1};
  uint32_t vbox[3] = {64, 64, 1};
  int rc;
  if ((rc = host::get_tmap(&tq, q, 3, qdims, qstr, qbox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = host::get_tmap(&to, o, 3, qdims, qstr, qbox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = host::get_tmap(&tk, k, 3, kdims, kstr, kbox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = host::get_tmap(&tv, v, 3, kdims, kstr, vbox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;

  // B200_ATTN_PAIR_PERSIST=0|1: one cluster per query tile / one cluster per SM pair walking the work items
  // (the persistent form runs every item over all KV tiles: causal or Nq != Nk always take the one-shot grid)
  static int persist_env = -1;
  if (persist_env < 0) {
    const char* e = getenv("B200_ATTN_PAIR_PERSIST");
    persist_env = (e && e[0] == '0') ? 0 : ((e && e[0] == '1') ? 1 : B200_ATTN_PAIR_PERSIST_DEFAULT);
  }
  const int persist = (persist_env && !causal && Nq == Nk) ? 1 : 0;
  p.o_ptr = static_cast<__half*>(o);
  p.qtiles = (Nq + attn_pair::BR - 1) / attn_pair::BR;
  p.total_items = p.qtiles * static_cast<int>(BH);
  const int smem = attn_pair::smem_bytes(p.nq);
  auto kern = persist ? attn_pair::attn_pair_fwd_kernel<true> : attn_pair::attn_pair_fwd_kernel<false>;
  static int attr_smem[64][2] = {{0}};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && attr_smem[dev][persist] < smem) {
    B200_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_smem[dev][persist] = smem;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(2u * static_cast<unsigned>(p.qtiles), static_cast<unsigned>(BH), 1);
  if (persist) {
    const int slots = host::sm_count() / 2;
    cfg.gridDim = dim3(2u * static_cast<unsigned>(p.total_items < slots ? p.total_items : slots), 1, 1);
  }
  cfg.blockDim = dim3(attn_pair::kThreads, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attrs[1];
  attrs[0].id = cudaLaunchAttributeClusterDimension;
  attrs[0].val.clusterDim.x = 2;
  attrs[0].val.clusterDim.y = 1;
  attrs[0].val.clusterDim.z = 1;
  cfg.attrs = attrs;
  cfg.numAttrs = 1;
  B200_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, tq, tk, tv, to, p));
  host::count_launch();
  return 0;
}

// B200_ATTN_LARGE_D=slab keeps the column-slab kernel for every D > 128 (A/B runs, bring-up)
bool pair_kernel_enabled() {
  static int cached = -1;
  if (cached < 0) {
    const char* e = getenv("B200_ATTN_LARGE_D");
    cached = (e && strcmp(e, "slab") == 0) ? 0 : 1;
  }
  return cached == 1;
}

int fmha_large_d(const void* q, const void* k, const void* v, void* o, float* lse, float rms_g, int B, int H, int Nq,
                 int Nk, int D, int causal, float scale, cudaStream_t stream) {
  // D = 256 also runs on the pair kernel (B200_ATTN_LARGE_D=pair256) but measured slower there than on one slab per CTA
  // (790 / 974 vs 912 / 1163 TFLOPS at N = 2048 / 4096, profiles/r02_session2d.log): with half the MMA work per key the
  // softmax of a 256-key tile is the longer leg
  static int pair256 = -1;
  if (pair256 < 0) { const char* e = getenv("B200_ATTN_LARGE_D"); pair256 = (e && strcmp(e, "pair256") == 0) ? 1 : 0; }
  if (D >= (pair256 ? 256 : 257) && D <= 512 && D % 128 == 0 && pair_kernel_enabled())
    return fmha_pair(q, k, v, o, lse, rms_g, B, H, Nq, Nk, D, causal, scale, stream);
  const uint64_t BH = static_cast<uint64_t>(B) * H;
  attn_slab::Params p;
  p.Nq = Nq;
  p.Nk = Nk;
  p.num_kv = (Nk + attn_slab::BC - 1) / attn_slab::BC;
  p.causal = causal;
  p.nq = (D + 63) / 64;
  p.dsplit = (D + 255) / 256;
  p.dv = (((D + p.dsplit - 1) / p.dsplit) + 63) / 64 * 64;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.lse = lse;
  p.rms_g = rms_g;
  p.D = D;
  if (rms_g > 0.f && p.dsplit > 1)
    return fail(B200_ENOTSUP, "fused rms_norm needs the whole output row in one CTA: D=%d is served by %d column slabs", D, p.dsplit);
  if (p.nq > attn_slab::kMaxDChunks) return fail(B200_ENOTSUP, "headdim not support! (D=%d > 1024)", D);

  CUtensorMap tq, tk, tv, to;
  uint64_t qdims[3] = {static_cast<uint64_t>(D), static_cast<uint64_t>(Nq), BH};
  uint64_t qstr[2] = {static_cast<uint64_t>(D) * 2, static_cast<uint64_t>(Nq) * D * 2};
  uint64_t kdims[3] = {static_cast<uint64_t>(D), static_cast<uint64_t>(Nk), BH};
  uint64_t kstr[2] = {static_cast<uint64_t>(D) * 2, static_cast<uint64_t>(Nk) * D * 2};
  const bool wide = p.nq <= attn_slab::kMaxQChunks;      // Q resident: 32 KiB ring slots, V boxes of 64 keys
  uint32_t box[3] = {64, 128, 1};
  uint32_t vbox[3] = {64, static_cast<uint32_t>(wide ? 64 : 32), 1};
  int rc;
  if ((rc = host::get_tmap(&tq, q, 3, qdims, qstr, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = host::get_tmap(&tk, k, 3, kdims, kstr, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = host::get_tmap(&to, o, 3, qdims, qstr, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = host::get_tmap(&tv, v, 3, kdims, kstr, vbox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;

  const int smem = attn_slab::smem_bytes(p.nq);
  auto kern = causal ? (wide ? attn_slab::attn_slab_fwd_kernel<true, true> : attn_slab::attn_slab_fwd_kernel<false, true>)
                     : (wide ? attn_slab::attn_slab_fwd_kernel<true, false> : attn_slab::attn_slab_fwd_kernel<false, false>);
  static int attr_smem[64][2][2] = {{{0}}};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && attr_smem[dev][wide][causal] < smem) {
    B200_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_smem[dev][wide][causal] = smem;
  }
  dim3 grid(((Nq + attn_slab::BR - 1) / attn_slab::BR) * p.dsplit, static_cast<unsigned>(BH), 1);
  kern<<<grid, attn_slab::kThreads, smem, stream>>>(tq, tk, tv, to, p);
  B200_CUDA_OK(cudaGetLastError());
  host::count_launch();
  return 0;
}

// Nq query rows (q, o, lse) against Nk keys (k, v).  causal = 1: query row i sees the keys j <= i + Nk - Nq.  The
// entries without the two lengths / the mask call this with Nq = Nk = N, causal = 0.
int fmha_impl(const void* q, const void* k, const void* v, void* o, float* lse, int B, int H, int Nq, int Nk, int D,
              int v_transposed, int causal, float scale, void* stream_, float rms_g = 0.f) {
  if (!q || !k || !v || !o) return fail(B200_EINVAL, "fmha: null pointer");
  if (B <= 0 || H <= 0 || Nq <= 0 || Nk <= 0 || D <= 0)
    return fail(B200_EINVAL, "fmha: bad shape B=%d H=%d Nq=%d Nk=%d D=%d", B, H, Nq, Nk, D);
  if (causal != 0 && causal != 1) return fail(B200_EINVAL, "fmha: causal must be 0 or 1 (got %d)", causal);
  if (causal && Nk < Nq)
    return fail(B200_EINVAL, "fmha: causal attention needs Nk >= Nq (Nq=%d, Nk=%d): every query row must see a key", Nq, Nk);
  if (static_cast<long long>(B) * H > 65535)
    return fail(B200_EINVAL, "fmha: B*H = %lld exceeds the grid limit 65535", static_cast<long long>(B) * H);
  if (D % 8 != 0) return fail(B200_ENOTSUP, "headdim not support! (D=%d must be a multiple of 8)", D);
  if (D > 1024) return fail(B200_ENOTSUP, "headdim not support! (D=%d > 1024)", D);
  if (v_transposed && (Nk % 8) != 0) {
    if (Nq == Nk) return fail(B200_EINVAL, "fmha: N (%d) must be a multiple of 8 for transposed V", Nk);
    return fail(B200_EINVAL, "fmha: Nk (%d) must be a multiple of 8 for transposed V", Nk);
  }
  // the variants that run every work item over all KV tiles (B200_ATTN_CG2=1, B200_ATTN_SPEC=2) serve only full
  // attention with Nq == Nk; everything else takes the default kernels
  const bool full_square = !causal && Nq == Nk;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (!(scale > 0.f)) scale = 1.0f / sqrtf(static_cast<float>(D));
  if (D > 128) {
    if (v_transposed) {
      // the restored V lives in a stream-ordered allocation: calls on different streams never share
      // scratch, nothing stays pinned between calls, and neither the allocation nor the free
      // synchronises the device (the memory returns to the pool once this stream passes the free)
      void* ws = nullptr;
      const size_t bytes = static_cast<size_t>(B) * H * Nk * D * 2;
      B200_CUDA_OK(cudaMallocAsync(&ws, bytes, stream));
      dim3 grid((Nk + 31) / 32, (D + 31) / 32, B * H), block(32, 8, 1);
      transpose_dn_to_nd_kernel<<<grid, block, 0, stream>>>(static_cast<const __half*>(v),
                                                            static_cast<__half*>(ws), D, Nk);
      cudaError_t le = cudaGetLastError();
      int rc = 0;
      if (le != cudaSuccess) rc = fail(B200_ECUDA, "transpose launch failed: %s", cudaGetErrorString(le));
      else {
        host::count_launch();
        rc = fmha_large_d(q, k, ws, o, lse, rms_g, B, H, Nq, Nk, D, causal, scale, stream);
      }
      cudaFreeAsync(ws, stream);
      return rc;
    }
    return fmha_large_d(q, k, v, o, lse, rms_g, B, H, Nq, Nk, D, causal, scale, stream);
  }
  const int DP = D <= 64 ? 64 : 128;
  const uint64_t BH = static_cast<uint64_t>(B) * H;
  {
    // CTA-pair kernel for 64 < D <= 128 whenever a pair's 512 query rows are (mostly) real rows;
    // B200_ATTN_CG2=0|1 overrides (A/B runs)
    static int cg2 = -1;
    if (cg2 < 0) {
      const char* e = getenv("B200_ATTN_CG2");
      cg2 = (e && e[0] == '0') ? 0 : ((e && e[0] == '1') ? 1 : B200_ATTN_CG2_DEFAULT);
    }
    const int N = Nq;
    if (cg2 && full_square && DP == 128 && (N % 512 == 0 || N >= 2048)) {
      attn2::Params p2;
      p2.N = N;
      p2.D = D;
      p2.num_kv = (N + attn2::BC - 1) / attn2::BC;
      p2.scale_log2 = scale * 1.4426950408889634f;
      p2.lse = lse;
      p2.rms_g = rms_g;
      return v_transposed ? launch_attn_cg2<true>(q, k, v, o, p2, BH, N, D, stream)
                          : launch_attn_cg2<false>(q, k, v, o, p2, BH, N, D, stream);
    }
  }

  attn::Params p;
  p.Nq = Nq;
  p.Nk = Nk;
  p.D = D;
  p.num_kv = (Nk + attn::BC - 1) / attn::BC;
  p.causal = causal;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.lse = lse;
  p.rms_g = rms_g;

  CUtensorMap tq, tk, tv, to;
  uint64_t qdims[3] = {static_cast<uint64_t>(D), static_cast<uint64_t>(Nq), BH};
  uint64_t qstr[2] = {static_cast<uint64_t>(D) * 2, static_cast<uint64_t>(Nq) * D * 2};
  uint64_t kdims[3] = {static_cast<uint64_t>(D), static_cast<uint64_t>(Nk), BH};
  uint64_t kstr[2] = {static_cast<uint64_t>(D) * 2, static_cast<uint64_t>(Nk) * D * 2};
  uint32_t box[3] = {64, 128, 1};
  int rc;
  if ((rc = host::get_tmap(&tq, q, 3, qdims, qstr, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = host::get_tmap(&tk, k, 3, kdims, kstr, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = host::get_tmap(&to, o, 3, qdims, qstr, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if (v_transposed) {
    uint64_t vd[3] = {static_cast<uint64_t>(Nk), static_cast<uint64_t>(D), BH};
    uint64_t vs[2] = {static_cast<uint64_t>(Nk) * 2, static_cast<uint64_t>(Nk) * D * 2};
    uint32_t vb[3] = {64, static_cast<uint32_t>(DP), 1};
    if ((rc = host::get_tmap(&tv, v, 3, vd, vs, vb, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  } else {
    if ((rc = host::get_tmap(&tv, v, 3, kdims, kstr, box, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  }
  const int bh = static_cast<int>(BH);
  // B200_ATTN_SPEC=0|2 picks the softmax step (attn_sm100.cuh, kStep: 0 classic, 2 sum-checked speculative);
  // B200_ATTN_PERSIST=0|1: one CTA per work item / one CTA per SM walking the work items
  static int spec = -1, persist = -1;
  if (spec < 0) {
    const char* e = getenv("B200_ATTN_SPEC");
    spec = (e && e[0] == '2') ? 2 : ((e && e[0] == '0') ? 0 : B200_ATTN_SPEC_DEFAULT);
    const char* f = getenv("B200_ATTN_PERSIST");
    persist = (f && f[0] == '0') ? 0 : ((f && f[0] == '1') ? 1 : -1);   // -1: per head dim (below)
  }
  const int use_persist = persist >= 0 ? persist : (DP == 64 ? 1 : B200_ATTN_PERSIST_DEFAULT);
  const int use_spec = full_square ? spec : 0;
  p.o_ptr = static_cast<__half*>(o);
  p.qpairs = (Nq + 2 * attn::BR - 1) / (2 * attn::BR);
  p.bhs = bh;
  p.total_items = p.qpairs * bh;
  if (causal) {
    switch ((DP == 64 ? 0 : 4) + (v_transposed ? 2 : 0) + (use_persist ? 1 : 0)) {
#define B200_ATTN_CAUSAL_CASE(n, dp, vt, pe) \
      case n: return launch_fmha<dp, vt, 0, pe, true>(tq, tk, tv, to, p, bh, stream);
      B200_ATTN_CAUSAL_CASE(0, 64, false, false) B200_ATTN_CAUSAL_CASE(1, 64, false, true)
      B200_ATTN_CAUSAL_CASE(2, 64, true, false) B200_ATTN_CAUSAL_CASE(3, 64, true, true)
      B200_ATTN_CAUSAL_CASE(4, 128, false, false) B200_ATTN_CAUSAL_CASE(5, 128, false, true)
      B200_ATTN_CAUSAL_CASE(6, 128, true, false) B200_ATTN_CAUSAL_CASE(7, 128, true, true)
#undef B200_ATTN_CAUSAL_CASE
    }
    return fail(B200_EINVAL, "fmha: internal dispatch error");
  }
  switch ((DP == 64 ? 0 : 8) + (v_transposed ? 4 : 0) + use_spec + (use_persist ? 1 : 0)) {   // use_spec is 0 or 2
#define B200_ATTN_CASE(n, dp, vt, sp, pe) \
    case n: return launch_fmha<dp, vt, sp, pe, false>(tq, tk, tv, to, p, bh, stream);
#define B200_ATTN_CASES(n0, dp, vt)                                                             \
    B200_ATTN_CASE(n0 + 0, dp, vt, 0, false) B200_ATTN_CASE(n0 + 1, dp, vt, 0, true)            \
    B200_ATTN_CASE(n0 + 2, dp, vt, 2, false) B200_ATTN_CASE(n0 + 3, dp, vt, 2, true)
    B200_ATTN_CASES(0, 64, false)
    B200_ATTN_CASES(4, 64, true)
    B200_ATTN_CASES(8, 128, false)
    B200_ATTN_CASES(12, 128, true)
#undef B200_ATTN_CASES
#undef B200_ATTN_CASE
  }
  return fail(B200_EINVAL, "fmha: internal dispatch error");
}

}  // namespace

extern "C" {

int b200_fmha_fwd_f16(const void* q, const void* k, const void* v, void* o, int B, int H, int N,
                      int D, int v_transposed, float scale, void* stream) {
  return fmha_impl(q, k, v, o, nullptr, B, H, N, N, D, v_transposed, 0, scale, stream);
}

int b200_fmha_fwd_f16_lse(const void* q, const void* k, const void* v, void* o, float* lse, int B, int H,
                          int N, int D, int v_transposed, float scale, void* stream) {
  if (!lse) return fail(B200_EINVAL, "fmha_lse: null lse pointer");
  return fmha_impl(q, k, v, o, lse, B, H, N, N, D, v_transposed, 0, scale, stream);
}

int b200_fmha_fwd_f16_ex(const void* q, const void* k, const void* v, void* o, float* lse, int B, int H, int Nq, int Nk,
                         int D, int v_transposed, int causal, float scale, void* stream) {
  return fmha_impl(q, k, v, o, lse, B, H, Nq, Nk, D, v_transposed, causal, scale, stream);
}

int b200_fmha_fwd_f16_rmsnorm(const void* q, const void* k, const void* v, void* o, float* lse, int B, int H,
                              int N, int D, int v_transposed, float scale, float rms_g, void* stream) {
  return fmha_impl(q, k, v, o, lse, B, H, N, N, D, v_transposed, 0, scale, stream, rms_g > 0.f ? rms_g : 0.f);
}

int b200_fmha_fwd_f16_host(const void* q, const void* k, const void* v, void* o, int B, int H,
                           int N, int D, int v_transposed, float scale, void* stream_) {
  if (!q || !k || !v || !o || B <= 0 || H <= 0 || N <= 0 || D <= 0)
    return fail(B200_EINVAL, "fmha_host: bad args");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int BH = B * H;
  const size_t head = static_cast<size_t>(N) * D * 2;            // bytes of one (b,h) slice
  const size_t bytes = head * BH;
  const size_t slot = (bytes + 255) & ~static_cast<size_t>(255);
  void* ws = nullptr;
  int rc = b200::host::workspace(&ws, 4 * slot);
  if (rc) return rc;
  char* dq = static_cast<char*>(ws);
  char* dk = dq + slot;
  char* dv = dk + slot;
  char* dout = dv + slot;
  // (batch x head) units are independent: pipeline chunks of heads through the copy engines
  // (H2D of chunk i+1 and D2H of chunk i-1 overlap the kernel of chunk i)
  host::HostPipe* pp = nullptr;
  if ((rc = host::host_pipe(&pp))) return rc;
  host::HostPipe& pipe = *pp;
  int chunks = BH < 16 ? BH : 16;
  const int per = (BH + chunks - 1) / chunks;
  cudaEvent_t ev_start = pipe.ev[host::kPipeEvents - 1];
  B200_CUDA_OK(cudaEventRecord(ev_start, stream));
  B200_CUDA_OK(cudaStreamWaitEvent(pipe.in, ev_start, 0));
  B200_CUDA_OK(cudaStreamWaitEvent(pipe.out, ev_start, 0));
  int ci = 0;
  for (int h0 = 0; h0 < BH; h0 += per, ++ci) {
    const int nh = (BH - h0 < per) ? (BH - h0) : per;
    const size_t off = head * h0, len = head * nh;
    B200_CUDA_OK(cudaMemcpyAsync(dq + off, static_cast<const char*>(q) + off, len, cudaMemcpyHostToDevice, pipe.in));
    B200_CUDA_OK(cudaMemcpyAsync(dk + off, static_cast<const char*>(k) + off, len, cudaMemcpyHostToDevice, pipe.in));
    B200_CUDA_OK(cudaMemcpyAsync(dv + off, static_cast<const char*>(v) + off, len, cudaMemcpyHostToDevice, pipe.in));
    B200_CUDA_OK(cudaEventRecord(pipe.ev[2 * ci], pipe.in));
    B200_CUDA_OK(cudaStreamWaitEvent(stream, pipe.ev[2 * ci], 0));
    rc = fmha_impl(dq + off, dk + off, dv + off, dout + off, nullptr, 1, nh, N, N, D, v_transposed, 0, scale, stream);
    if (rc) return rc;
    B200_CUDA_OK(cudaEventRecord(pipe.ev[2 * ci + 1], stream));
    B200_CUDA_OK(cudaStreamWaitEvent(pipe.out, pipe.ev[2 * ci + 1], 0));
    B200_CUDA_OK(cudaMemcpyAsync(static_cast<char*>(o) + off, dout + off, len, cudaMemcpyDeviceToHost, pipe.out));
  }
  B200_CUDA_OK(cudaStreamSynchronize(pipe.out));
  B200_CUDA_OK(cudaStreamSynchronize(stream));
  return 0;
}

}  // extern "C"
