/* leetcuda_b200.h — C ABI of the B200-native (sm_100a) replacement for LeetCUDA's
 * two dense-contraction hot paths.  Plain pointers and sizes only: no torch
 * types cross this boundary.  All device pointers must live on the CUDA device
 * that is current on the calling thread; `stream` is a cudaStream_t (NULL = the
 * legacy default stream, which is what the reference launches on).
 *
 * Every entry point returns 0 on success or a negative B200_E* code; the text of
 * the last failure on the calling thread is returned by b200_last_error().
 * The reference's ops throw std::runtime_error for the same conditions
 * (kernels/hgemm/utils/utils.h:137-147, kernels/flash-attn/utils/utils.h) and
 * never check CUDA errors; the Python mirror in leetcuda_b200/ turns a non-zero
 * status into RuntimeError so callers see the reference's behaviour.
 */
#ifndef LEETCUDA_B200_H_
#define LEETCUDA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_EINVAL (-1)  /* bad shape / alignment / null pointer            */
#define B200_ECUDA (-2)   /* CUDA runtime or driver error (text in last_error) */
#define B200_ENOTSUP (-3) /* e.g. head dim outside the dispatch set          */

/* Layout of the B operand of b200_hgemm_f16. */
#define B200_B_ROW_MAJOR_KN 0 /* "NN": b is [K,N] row-major (N contiguous)           */
#define B200_B_ROW_MAJOR_NK 1 /* "TN": b storage is [N,K] row-major (K contiguous)   */

/* ABI version of this header (major*1000 + minor). */
int b200_version(void);

/* Text of the last error raised on the calling thread ("" if none). */
const char* b200_last_error(void);

/* Number of kernels this library has launched in the calling process (all
 * threads).  Used by bench.py to report `gpu_launches`. */
uint64_t b200_launch_count(void);

/* C[M,N] = A[M,K] x B, fp16 in / fp16 out, fp32 accumulation in TMEM.
 *
 * Replaces every `void hgemm_*(torch::Tensor a, torch::Tensor b, torch::Tensor c
 * [, int stages, bool swizzle, int swizzle_stride])` bound in the reference's
 * kernels/hgemm/pybind/hgemm.cc:124-182 (host launchers e.g.
 * kernels/hgemm/mma/swizzle/hgemm_mma_stage_swizzle.cu:808-887 for NN and
 * kernels/hgemm/mma/basic/hgemm_mma_stage_tn.cu:555-629 for TN).  The reference's
 * stages/swizzle/swizzle_stride arguments are tuning hints of its own tiling and
 * have no counterpart here.
 *
 * a: [M,K] row-major.  b: see b_layout.  c: [M,N] row-major, written in place.
 * Constraints: M,N,K > 0; K % 8 == 0 and N % 8 == 0 (16-byte TMA strides);
 * pointers 16-byte aligned.  Unlike the reference (M,N % 128 == 0, K % 32 == 0,
 * hgemm_mma_stage.cu:675-676) ragged M/N/K tiles are handled.
 */
int b200_hgemm_f16(const void* a, const void* b, void* c, int M, int N, int K, int b_layout,
                   void* stream);

/* Same as b200_hgemm_f16 with explicit tuning/debug knobs (0 = default):
 *   cta_group  1 | 2      tcgen05 cta_group (2 = CTA pair, 256x256 tile)
 *              3          CTA pair, 512x256 macro tile (two accumulators sharing B); 30..33 = the
 *                         same with accumulator 1 trailing accumulator 0 by 0|1|2 k-blocks
 *   group_m    >0         m-tiles per rasterisation group
 *   max_ctas   >0         cap on the persistent grid
 *   b_lbo,b_sbo,b_kstep   UMMA descriptor byte offsets of the MN-major B operand; the top byte of
 *                         b_lbo carries two more debug overrides: bits [28,32) the UMMA layout type of
 *                         that descriptor, bits [24,28) the CUtensorMapSwizzle of the B tensor map
 */
int b200_hgemm_f16_ex(const void* a, const void* b, void* c, int M, int N, int K, int b_layout,
                      int cta_group, int group_m, int max_ctas, uint32_t b_lbo, uint32_t b_sbo,
                      uint32_t b_kstep, void* stream);

/* Reference-accumulation parity mode: same as b200_hgemm_f16 but the tensor core accumulates in
 * fp16 (tcgen05 D format f16, one rounding per k16 instruction) exactly like the reference's
 * HMMA.16816.F16 kernels (mma/basic/hgemm_mma.cu:67-73) and its cuBLAS CUBLAS_COMPUTE_16F op
 * (cublas/hgemm_cublas.cu:50-52).  Less accurate than the default fp32 accumulation; provided so
 * that outputs can be compared with the reference's bit for bit.  Select it for every mirror op
 * with LEETCUDA_B200_HGEMM_ACC=f16. */
int b200_hgemm_f16_acc16(const void* a, const void* b, void* c, int M, int N, int K, int b_layout,
                         void* stream);

/* Row-sharded variant used by the multi-GPU path (SURVEY.md §8e): computes the
 * rows [row0, row0+rows) of C = A_shard x B where a_shard is [rows,K] and writes
 * them into c_full (an [M_total,N] buffer) at row offset row0.  c_full may be a
 * peer-mapped pointer of another GPU (NVLink P2P store from the epilogue). */
int b200_hgemm_f16_rows(const void* a_shard, const void* b, void* c_full, int rows, int N, int K,
                        int b_layout, int row0, void* stream);

/* Fused GEMM + all-gather of C: like b200_hgemm_f16_rows, but the epilogue also delivers every
 * finished tile to the other GPUs while the remaining tiles are still being computed.  At least one
 * of the two target descriptions must be given (else B200_EINVAL):
 *   c_full_peers / n_peers (1..7) : peer-mapped C buffers of the other GPUs.  This is the default
 *                              transport: each finished 64x32 box is staged in shared memory and
 *                              TMA-stored to c_full and to every peer (NVLink P2P).
 *   c_full_multicast         : an NVLS multicast mapping of the symmetric C buffer.  Used when no
 *                              peers are given (one multimem.st per 16 bytes reaches every GPU, this
 *                              one included), or when B200_FUSED_EPILOGUE=direct|mc selects it.
 * n_peers > 0 with c_full_peers == NULL is rejected.  The caller closes the step with a cross-GPU
 * barrier and must not let a peer overwrite a C buffer that is still being read (leetcuda_b200/dist.py
 * alternates two symmetric buffers). */
int b200_hgemm_f16_rows_fused(const void* a_shard, const void* b, void* c_full, void* c_full_multicast,
                              void* const* c_full_peers, int n_peers, int rows, int N, int K,
                              int b_layout, int row0, void* stream);

/* O = softmax(Q K^T * scale) V per (batch, head); fp16 in/out, fp32 softmax
 * statistics and fp32 accumulation; non-causal, no mask, no dropout, equal query and key lengths
 * (b200_fmha_fwd_f16_ex below adds the causal mask and separate lengths).
 *
 * Replaces every `void flash_attn_mma_stages_*(Q,K,V,O,int stages)` bound in
 * kernels/flash-attn/pybind/flash_attn.cc:168-224 (e.g. the shared-QKV launcher
 * kernels/flash-attn/mma/basic/flash_attn_mma_share_qkv.cu:770-921), the CuTe op
 * flash_attn_cute (cutlass/flash_attn_cute.cu:496-524) and ffpa-attn's
 * ffpa_mma_acc_{f16,f32}_L1 (ffpa-attn/csrc/pybind/ffpa_attn_api.cc:8-16).
 *
 * q,k,o: [B,H,N,D] contiguous.  v: [B,H,N,D] (v_transposed = 0) or [B,H,D,N]
 * (v_transposed = 1, the reference's *_swizzle_qkv ops).  scale <= 0 selects the
 * reference's 1/sqrt(D) (flash_attn_mma_split_q.cu:79).
 * Constraints: D % 8 == 0 and D <= 1024; any N >= 1 (N % 8 == 0 for v_transposed).  For
 * v_transposed with D > 128 V is first restored to [B,H,N,D] in a stream-ordered scratch
 * allocation (cudaMallocAsync / cudaFreeAsync on `stream`).
 * Kernels: D <= 128 the single-CTA two-query-tile kernel (persistent scheduling for D <= 64; a CTA-pair
 * variant with cta_group::2 M = 256 exists behind B200_ATTN_CG2=1 and measured slower); D = 256, 384, 512
 * the CTA-pair kernel with one 128-row query tile per cluster (cta_group::2, M = 128); every other
 * D <= 1024 the column-slab kernel.
 * Numerics: S, the softmax statistics and O in fp32, P rounded to fp16 before P.V (as the reference); the
 * exponentials are ex2.approx (MUFU) except, for D <= 128, a fixed quarter to third of the score pairs, which a
 * degree-3 polynomial on the FMA pipe evaluates with max. relative error 7.6e-5 — below the fp16 rounding P
 * receives next (tests/test_softmax_math.py).  Measured max |error| 2-3e-3 on adversarial inputs, 2e-4
 * typical, against the reference's own tolerance allclose(1e-2, 1e-2).
 */
int b200_fmha_fwd_f16(const void* q, const void* k, const void* v, void* o, int B, int H, int N,
                      int D, int v_transposed, float scale, void* stream);

/* Same, and also writes lse[b,h,i] = ln sum_j exp(scale * q_i . k_j) (fp32, [B,H,N] contiguous):
 * the per-row statistic that b200_merge_attn_states consumes (as [num_heads, num_tokens] when B = 1)
 * to combine partial results over disjoint key ranges (split-KV).  The reference's attention ops
 * have no such output (its merge test feeds synthetic LSEs,
 * kernels/openai-triton/merge-attn-states/test_merge_attn_states.py:100-152). */
int b200_fmha_fwd_f16_lse(const void* q, const void* k, const void* v, void* o, float* lse, int B,
                          int H, int N, int D, int v_transposed, float scale, void* stream);

/* Attention with separate query / key lengths and an optional causal mask:
 *   o[b,h,i] = sum_{allowed j} softmax_j(scale * q_i . k_j) v_j
 * q, o: [B,H,Nq,D].  k: [B,H,Nk,D].  v: [B,H,Nk,D], or [B,H,D,Nk] with v_transposed.  lse: [B,H,Nq] fp32, may be
 * NULL.  All of them fp16 (lse fp32), contiguous.
 *   causal = 0: every query row attends to all Nk keys; any Nq, Nk >= 1.
 *   causal = 1: query row i attends to the keys j <= i + (Nk - Nq): the BOTTOM-RIGHT alignment of FlashAttention-2
 *               >= 2.1 (the last query row sees every key).  It equals the top-left alignment when Nq == Nk, and is
 *               NOT what torch's scaled_dot_product_attention(is_causal=True) computes for Nq != Nk (top-left).
 *               Requires Nk >= Nq, so that every row sees at least one key.
 *   lse[b,h,i] = ln sum_{allowed j} exp(scale * q_i . k_j): the statistic of b200_fmha_fwd_f16_lse restricted to the
 *   allowed keys, so two calls over disjoint key ranges can be combined with b200_merge_attn_states.
 * B200_EINVAL for a null q/k/v/o, B, H, Nq, Nk or D <= 0, causal outside {0, 1}, causal with Nk < Nq, and
 * v_transposed with Nk % 8 != 0; B200_ENOTSUP for the head dims b200_fmha_fwd_f16 rejects.  Numerics as
 * b200_fmha_fwd_f16.  With causal = 0 and Nq == Nk the result is bit-identical to b200_fmha_fwd_f16{,_lse}.
 * Kernels: those of b200_fmha_fwd_f16.  A causal work item (query tile) runs only the KV tiles up to its last
 * row's diagonal and masks the keys past the diagonal, and the longest items are dispatched first.  The opt-in
 * variants B200_ATTN_CG2=1, B200_ATTN_SPEC=2 and B200_ATTN_PAIR_PERSIST=1 are not taken when causal = 1 or
 * Nq != Nk: the default kernel for the head dim runs instead. */
int b200_fmha_fwd_f16_ex(const void* q, const void* k, const void* v, void* o, float* lse, int B, int H,
                         int Nq, int Nk, int D, int v_transposed, int causal, float scale, void* stream);

/* ------------------------------------------------------------------ SGEMM (TF32)
 * C[M,N] (fp32) = A[M,K] (fp32) x B on the tensor cores through tcgen05 kind::tf32 with fp32
 * accumulation — the sibling of the HGEMM path (SURVEY §8f-2).  Replaces
 *   sgemm_wmma_m16n16k8_mma4x2_warp2x4_stages{,_dsmem}(a,b,c,stages,swizzle,swizzle_stride)
 *   (kernels/sgemm/sgemm_wmma_tf32_stage.cu:573-742, bound in kernels/sgemm/sgemm.cu:762-764).
 * Like the reference (sgemm_wmma_tf32_stage.cu:586-592: f32x4_tf32x4_kernel over a and b IN PLACE),
 * round_inputs_in_place != 0 first rewrites a and b with their TF32 roundings (cvt.rna.tf32.f32);
 * with 0 the inputs are left untouched and the tensor core reads the upper 19 bits of each fp32
 * (truncation).  b_layout as for b200_hgemm_f16 (the reference has only the [K,N] form).
 * Constraints: M,N,K > 0; K % 4 == 0 and N % 4 == 0; pointers 16-byte aligned.
 */
int b200_sgemm_tf32(float* a, float* b, float* c, int M, int N, int K, int b_layout,
                    int round_inputs_in_place, void* stream);

/* fp32 product on the TF32 tensor cores through the 3xTF32 split: every operand is split into two TF32 numbers
 * (x = hi + lo, both exactly representable) and C = hi_a hi_b + hi_a lo_b + lo_a hi_b is evaluated by ONE tf32 GEMM
 * over concatenated operands (K' = 3K, scratch from cudaMallocAsync on `stream`).  The operand rounding of a plain
 * TF32 product (1e-3 relative) is gone; what remains is the tensor core's truncating fp32 accumulation: measured
 * 5e-5 relative at K = 1024..4096, against 2e-6 for an FFMA kernel.  That is why the reference's 13 CUDA-core fp32
 * ops (kernels/sgemm/sgemm.cu:743-760, kernels/sgemm/sgemm_async.cu) stay vendor fp32 rows in the Python mirror by
 * default and use this entry only under LEETCUDA_B200_SGEMM_FP32=3xtf32.
 * a: [M,K], b: [K,N], c: [M,N] row-major fp32; a and b are not modified.  K % 4 == 0, N % 4 == 0. */
int b200_sgemm_3xtf32(const float* a, const float* b, float* c, int M, int N, int K, void* stream);

/* b200_sgemm_tf32 without the rounding pass, with the tuning/debug knobs of b200_hgemm_f16_ex. */
int b200_sgemm_tf32_ex(const float* a, const float* b, float* c, int M, int N, int K, int b_layout,
                       int cta_group, int group_m, int max_ctas, uint32_t b_lbo, uint32_t b_sbo,
                       uint32_t b_kstep, void* stream);

/* x[i] <- tf32(x[i]) (round to nearest, ties away), in place, n elements; x 16-byte aligned. */
int b200_tf32_round_inplace(float* x, size_t n, void* stream);

/* ------------------------------------------------------------------ merge_attn_states
 * Combine two partial attention results over disjoint key ranges (split-KV), SURVEY §8f-3.  Replaces
 *   merge_attn_states_cuda(output, output_lse?, prefix_output, prefix_lse, suffix_output, suffix_lse)
 *   (kernels/openai-triton/merge-attn-states/cuda_merge_attn_states.cu:19-95, 158-166).
 * output / prefix_output / suffix_output: [num_tokens, num_heads, head_size] of `dtype`, contiguous;
 * the lse tensors: [num_heads, num_tokens] fp32; output_lse may be NULL.  A +inf lse marks an empty
 * part and is treated as -inf, as in the reference.  head_size must be a multiple of 16/sizeof(T).
 */
#define B200_DTYPE_F32 0
#define B200_DTYPE_F16 1
#define B200_DTYPE_BF16 2
int b200_merge_attn_states(void* output, float* output_lse, const void* prefix_output,
                           const float* prefix_lse, const void* suffix_output, const float* suffix_lse,
                           int num_tokens, int num_heads, int head_size, int dtype, void* stream);

/* ------------------------------------------------------------------ rope / rms_norm (SURVEY §8f-4)
 * The element-wise steps either side of attention in the reference's catalogue.
 *
 * b200_rope_f32: rotary position embedding.  Replaces rope_f32 / rope_f32_v2 / rope_f32x4_pack(x, out)
 *   (kernels/rope/rope.cu:20-71, host :88-125).  x, out: [seq_len, hidden] fp32 contiguous; the pair
 *   (x[p,2i], x[p,2i+1]) is rotated by the angle p * theta^(-2i/hidden), theta = 10000.  hidden % 4 == 0.
 *
 * b200_rms_norm: y = x * rsqrt(mean(x^2, row) + 1e-5) * g.  Replaces rms_norm_f32{,x4}(x, y, g) and the
 *   seven rms_norm_f16* ops (kernels/rms-norm/rms_norm.cu:55-110, 161-415, host :493-771).  x, y:
 *   [rows, K] of `dtype` (B200_DTYPE_F32 or B200_DTYPE_F16), statistics always in fp32.  K must be a
 *   multiple of 16/sizeof(T) and at most 16384 (fp16) / 8192 (fp32).
 */
int b200_rope_f32(const float* x, float* out, int seq_len, int hidden, void* stream);

/* The same rotation on the attention operands: q, k fp16 [B,H,N,D] contiguous, the position of a row is its
 * sequence index n, pairs are (d = 2i, 2i+1), angle n * theta^(-2i/D); fp32 arithmetic, one rounding to fp16.
 * One launch rotates both tensors; q_out / k_out may alias q / k.  It is a pre-pass, not a fusion into the
 * attention main loop, on purpose: there K would be re-rotated once per query tile (N/256 times) with its
 * sin/cos on the MUFU pipe that already bounds the kernel; rotated once it costs one extra read + write of
 * q and k (HBM-bound).  D % 8 == 0. */
int b200_rope_qk_f16(const void* q, const void* k, void* q_out, void* k_out, int B, int H, int N, int D,
                     void* stream);
int b200_rms_norm(const void* x, void* y, float g, int rows, int K, int dtype, void* stream);

/* Attention with the RMS normalisation of every output row fused into the epilogue:
 *   o[b,h,i,:] = rms_norm(softmax(q_i K^T * scale) V) * rms_g     (eps 1e-5, statistics in fp32 over D)
 * i.e. b200_fmha_fwd_f16 followed by b200_rms_norm over rows of length D, without the round trip of O
 * through HBM (the row already sits in the registers of one thread when the epilogue runs).  rms_g <= 0
 * disables the normalisation (then identical to b200_fmha_fwd_f16_lse with an optional lse).  lse may be
 * NULL.  Supported for D <= 256 and for the CTA-pair kernel's head dims (384, 512); B200_ENOTSUP otherwise. */
int b200_fmha_fwd_f16_rmsnorm(const void* q, const void* k, const void* v, void* o, float* lse, int B,
                              int H, int N, int D, int v_transposed, float scale, float rms_g, void* stream);

/* Host-buffer convenience wrappers used for end-to-end timing: inputs are host
 * pointers (pinned or pageable); the call copies them to a cached device
 * workspace, runs the kernel and copies the result back, all on `stream`, and
 * returns after the stream has drained. */
int b200_hgemm_f16_host(const void* a, const void* b, void* c, int M, int N, int K, int b_layout,
                        void* stream);
int b200_fmha_fwd_f16_host(const void* q, const void* k, const void* v, void* o, int B, int H,
                           int N, int D, int v_transposed, float scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LEETCUDA_B200_H_ */
