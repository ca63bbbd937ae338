"""Fusions of the element-wise steps around attention (SURVEY §8f-4) and their bench rows.

* ``attn_rmsnorm(q, k, v, o, g)`` — attention whose epilogue RMS-normalises every output row over the head
  dim (``b200_fmha_fwd_f16_rmsnorm``): the result of ``rms_norm(attention(q, k, v)) * g`` without the round
  trip of O through HBM.  The unfused composition (``flash_attn`` op + ``rms_norm`` op) is the reference's
  way of doing it: kernels/flash-attn ops followed by kernels/rms-norm/rms_norm.cu ops on ``O.view(-1, D)``.
* RoPE.  The reference's rope ops are position-wise rotations of fp32 rows (kernels/rope/rope.cu).  Inside
  the attention main loop the K side of a fused rope would be re-rotated once per query tile (N/256 times)
  and its sin/cos would land on the MUFU pipe that already bounds the kernel, so the rotation stays a
  streaming op of its own here (``leetcuda_b200.rope``, HBM-bound).
"""
from __future__ import annotations

import torch

from . import _capi
from .flash_attn import _check


def attn_rmsnorm(Q, K, V, O, g: float = 1.0, *, v_transposed: bool = False, scale: float = 0.0, lse=None) -> None:
    """``O = rms_norm(softmax(Q K^T * scale) V, dim=-1, eps=1e-5) * g`` in one kernel."""
    B, H, N, D = _check(Q, K, V, O, v_transposed)
    if not g > 0.0:
        raise RuntimeError("attn_rmsnorm: g must be > 0")
    lse_ptr = None
    if lse is not None:
        if lse.dtype != torch.float32 or tuple(lse.shape) != (B, H, N) or not lse.is_cuda or not lse.is_contiguous():
            raise RuntimeError("attn_rmsnorm: lse must be a contiguous fp32 CUDA tensor [B,H,N]")
        lse_ptr = lse.data_ptr()
    idx = Q.device.index
    with torch.cuda.device(idx):
        rc = _capi.lib().b200_fmha_fwd_f16_rmsnorm(Q.data_ptr(), K.data_ptr(), V.data_ptr(), O.data_ptr(), lse_ptr,
                                                   B, H, N, D, int(v_transposed), float(scale), float(g),
                                                   _capi.raw_stream(idx))
    if rc == -3:
        raise RuntimeError(_capi.last_error())
    _capi.check(rc, "attn_rmsnorm")


def rope_qk(Q, K, Q_out=None, K_out=None) -> None:
    """Rotary embedding of the attention operands (fp16 ``[B,H,N,D]``, position = sequence index), both tensors
    in one launch (``b200_rope_qk_f16``); in place when no outputs are given."""
    Q_out = Q if Q_out is None else Q_out
    K_out = K if K_out is None else K_out
    for t in (Q, K, Q_out, K_out):
        if t.dtype != torch.float16:
            raise RuntimeError("values must be torch::kHalf")
        if not (t.is_cuda and t.is_contiguous()):
            raise RuntimeError("leetcuda_b200.rope_qk: tensors must be contiguous CUDA tensors")
    if Q.dim() != 4 or tuple(K.shape) != tuple(Q.shape) or tuple(Q_out.shape) != tuple(Q.shape) \
            or tuple(K_out.shape) != tuple(Q.shape):
        raise RuntimeError("Tensor size mismatch!")
    B, H, N, D = Q.shape
    idx = Q.device.index
    with torch.cuda.device(idx):
        rc = _capi.lib().b200_rope_qk_f16(Q.data_ptr(), K.data_ptr(), Q_out.data_ptr(), K_out.data_ptr(), B, H, N, D,
                                          _capi.raw_stream(idx))
    _capi.check(rc, "rope_qk")


def attn_rope(Q, K, V, O, *, rms_g: float = 0.0, lse=None, causal: bool = False) -> None:
    """``O = attention(rope(Q), rope(K), V)`` (optionally RMS-normalised): the rope pre-pass into scratch copies of
    Q and K, then the fused attention kernel — two launches.  ``causal`` is passed to ``fmha_fwd``; the causal mask
    with the fused RMS-norm epilogue is not supported."""
    if causal and rms_g > 0.0:
        raise RuntimeError("attn_rope: causal attention with the fused RMS-norm epilogue (rms_g > 0) is not supported")
    q_r, k_r = torch.empty_like(Q), torch.empty_like(K)
    rope_qk(Q, K, q_r, k_r)
    if rms_g > 0.0:
        attn_rmsnorm(q_r, k_r, V, O, rms_g, lse=lse)
    else:
        from .flash_attn import fmha_fwd
        fmha_fwd(q_r, k_r, V, O, lse=lse, causal=causal)


def bench_rows(torch_mod, dev, steps, peak_hbm, peak_src, cuda_time_ms):
    """bench.py rows of §8f-4: rope and rms_norm against the HBM roofline, and the fused attention epilogue
    against attention + a separate rms_norm pass."""
    from . import flash_attn, rms_norm as RN, rope as RP
    t = torch_mod
    sync = lambda: t.cuda.synchronize()
    rows = []
    # rope: fp32 [seq, hidden], 2 sets x (read + write) 512 MB: far beyond L2
    S, Hd = 65536, 2048
    xs = [t.randn(S, Hd, device=dev) for _ in range(2)]
    ys = [t.empty(S, Hd, device=dev) for _ in range(2)]
    for i in range(3):
        RP.rope_f32x4_pack(xs[i % 2], ys[i % 2])
    ms = cuda_time_ms(lambda i: RP.rope_f32x4_pack(xs[i % 2], ys[i % 2]), steps, sync) / steps
    nbytes = 2 * S * Hd * 4
    rows.append({"metric": "rope GB/s @seq65536 hidden2048 fp32 (read + write)", "value": nbytes / ms / 1e6, "unit": "GB/s",
                 "ms_per_step": ms, "config": {"workload": "rope_seq65536_hidden2048_fp32", "op": "rope_f32x4_pack"},
                 "roofline": {"bound": "hbm", "achieved": nbytes / ms / 1e6, "peak": peak_hbm, "unit": "GB/s",
                              "frac": nbytes / ms / 1e6 / peak_hbm, "traffic": None, "peak_source": peak_src,
                              "kernel": "rope_f32_kernel", "kernel_ms": ms, "algorithmic_bytes": nbytes}})
    del xs, ys
    # rms_norm: fp16 [rows, K]
    R, Kk = 131072, 2048
    xs = [t.randn(R, Kk, device=dev, dtype=t.half) for _ in range(2)]
    ys = [t.empty(R, Kk, device=dev, dtype=t.half) for _ in range(2)]
    for i in range(3):
        RN.rms_norm_f16x8_pack_f32(xs[i % 2], ys[i % 2], 1.0)
    ms = cuda_time_ms(lambda i: RN.rms_norm_f16x8_pack_f32(xs[i % 2], ys[i % 2], 1.0), steps, sync) / steps
    nbytes = 2 * R * Kk * 2
    rows.append({"metric": "rms_norm GB/s @rows131072 K2048 fp16 (read + write)", "value": nbytes / ms / 1e6, "unit": "GB/s",
                 "ms_per_step": ms, "config": {"workload": "rms_norm_rows131072_K2048_fp16", "op": "rms_norm_f16x8_pack_f32"},
                 "roofline": {"bound": "hbm", "achieved": nbytes / ms / 1e6, "peak": peak_hbm, "unit": "GB/s",
                              "frac": nbytes / ms / 1e6 / peak_hbm, "traffic": None, "peak_source": peak_src,
                              "kernel": "rms_norm_kernel<half, warp per row>", "kernel_ms": ms, "algorithmic_bytes": nbytes}})
    del xs, ys
    # rope pre-pass of the attention operands (B4 H32 N4096 D128): q and k, read + write
    B, H, N, D = 4, 32, 4096, 128
    sets = [[t.randn(B, H, N, D, device=dev, dtype=t.half) for _ in range(3)] for _ in range(2)]
    qr, kr = t.empty(B, H, N, D, device=dev, dtype=t.half), t.empty(B, H, N, D, device=dev, dtype=t.half)
    for i in range(3):
        rope_qk(sets[i % 2][0], sets[i % 2][1], qr, kr)
    ms = cuda_time_ms(lambda i: rope_qk(sets[i % 2][0], sets[i % 2][1], qr, kr), steps, sync) / steps
    nbytes = 4 * B * H * N * D * 2
    rows.append({"metric": "rope of q,k GB/s @B4H32N4096D128 fp16 (read + write)", "value": nbytes / ms / 1e6, "unit": "GB/s",
                 "ms_per_step": ms, "config": {"workload": "rope_qk_B4_H32_N4096_D128_fp16", "op": "rope_qk"},
                 "roofline": {"bound": "hbm", "achieved": nbytes / ms / 1e6, "peak": peak_hbm, "unit": "GB/s",
                              "frac": nbytes / ms / 1e6 / peak_hbm, "traffic": None, "peak_source": peak_src,
                              "kernel": "rope_qk_f16_kernel", "kernel_ms": ms, "algorithmic_bytes": nbytes}})
    del qr, kr
    # fused epilogue vs attention + separate rms_norm pass (same shape)
    o = t.empty(B, H, N, D, device=dev, dtype=t.half)
    o2 = t.empty(B, H, N, D, device=dev, dtype=t.half)
    for i in range(3):
        attn_rmsnorm(*sets[i % 2], o, 1.0)
    f_ms = cuda_time_ms(lambda i: attn_rmsnorm(*sets[i % 2], o, 1.0), steps, sync) / steps

    def unfused(i):
        flash_attn.fmha_fwd(*sets[i % 2], o)
        RN.rms_norm(o.view(-1, D), o2.view(-1, D), 1.0)
    for i in range(3):
        unfused(i)
    u_ms = cuda_time_ms(unfused, steps, sync) / steps
    fl = 4.0 * B * H * N * N * D
    rows.append({"metric": "attention + fused RMS-norm epilogue TFLOPS @B4H32N4096D128", "value": fl / f_ms / 1e9, "unit": "TFLOPS",
                 "ms_per_step": f_ms, "config": {"workload": "attn_rmsnorm_B4_H32_N4096_D128_fp16", "op": "attn_rmsnorm"},
                 "unfused": {"ms_per_step": u_ms, "tflops": fl / u_ms / 1e9,
                             "what": "attention kernel + rms_norm kernel over O (one extra read + write of O)"}})
    return rows
