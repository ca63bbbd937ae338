"""Drop-in mirror of the reference's FlashAttention extension module (`flash_attn_lib`).

Every name bound in /root/reference/kernels/flash-attn/pybind/flash_attn.cc:168-224
exists here with the same signature and error behaviour:

* 28 ops  ``op(Q, K, V, O, stages) -> None``  (6 basic, 4 acc_f32, 15 swizzle, 3 "others")
* ``flash_attn_cute(Q, K, V, O) -> None``

Q, K, O are fp16 contiguous ``[B,H,N,D]``; V is ``[B,H,N,D]`` except for the three
``*_swizzle_qkv`` ops of the share-kv / share-qkv / tiling-qk families, which take V
pre-transposed ``[B,H,D,N]`` (flash_attn_mma.py:441-442,716,807,898).  O is written
in place.  Non-causal, scale = 1/sqrt(D) (flash_attn_mma_split_q.cu:79).

All of them run the same fused sm_100a kernel through ``b200_fmha_fwd_f16``;
``stages`` is a hint of the reference's cp.async pipeline and is ignored.  The
reference's family differences (which of Q/K/V share smem, fp16 vs fp32 MMA
accumulators) are implementation details of its mma.sync kernels: here S and O
always accumulate in fp32 in TMEM, which is at least as accurate as every variant.
"""
from __future__ import annotations

import torch

from . import _capi

_BASIC = [
    "flash_attn_mma_stages_split_kv", "flash_attn_mma_stages_split_q",
    "flash_attn_mma_stages_split_q_shared_kv", "flash_attn_mma_stages_split_q_shared_qkv",
    "flash_attn_mma_stages_split_q_tiling_qk", "flash_attn_mma_stages_split_q_tiling_qkv",
]
_ACC_F32 = [
    "flash_attn_mma_stages_split_q_shared_kv_acc_f32",
    "flash_attn_mma_stages_split_q_shared_qkv_acc_f32",
    "flash_attn_mma_stages_split_q_tiling_qk_acc_f32",
    "flash_attn_mma_stages_split_q_tiling_qkv_acc_f32",
]
_SWIZZLE = [
    "flash_attn_mma_stages_split_q_shared_kv_swizzle_q",
    "flash_attn_mma_stages_split_q_shared_kv_swizzle_qk",
    "flash_attn_mma_stages_split_q_shared_kv_swizzle_qkv",
    "flash_attn_mma_stages_split_q_shared_qkv_swizzle_q",
    "flash_attn_mma_stages_split_q_shared_qkv_swizzle_qk",
    "flash_attn_mma_stages_split_q_shared_qkv_swizzle_qkv",
    "flash_attn_mma_stages_split_q_tiling_qk_swizzle_q",
    "flash_attn_mma_stages_split_q_tiling_qk_swizzle_qk",
    "flash_attn_mma_stages_split_q_tiling_qk_swizzle_qkv",
    "flash_attn_mma_stages_split_q_tiling_qkv_swizzle_q",
    "flash_attn_mma_stages_split_q_tiling_qkv_swizzle_qk",
    "flash_attn_mma_stages_split_q_tiling_qkv_swizzle_qkv",
    "flash_attn_mma_stages_split_q_tiling_qkv_acc_f32_swizzle_q",
    "flash_attn_mma_stages_split_q_tiling_qkv_acc_f32_swizzle_qk",
    "flash_attn_mma_stages_split_q_tiling_qkv_acc_f32_swizzle_qkv",
]
_OTHERS = [  # only under -DBUILD_FLASH_ATTN_MMA_OTHERS in the reference (flash_attn.cc:217-223)
    "flash_attn_mma_stages_split_q_shared_qkv_Os2g",
    "flash_attn_mma_stages_split_q_shared_kv_acc_f32_rr",
    "flash_attn_mma_stages_split_q_shared_qkv_acc_f32_rr",
]
# ops whose V argument is [B,H,D,N]
V_TRANSPOSED_OPS = {
    "flash_attn_mma_stages_split_q_shared_kv_swizzle_qkv",
    "flash_attn_mma_stages_split_q_shared_qkv_swizzle_qkv",
    "flash_attn_mma_stages_split_q_tiling_qk_swizzle_qkv",
}
OP_NAMES = _BASIC + _ACC_F32 + _SWIZZLE + _OTHERS


def _check(Q, K, V, O, v_transposed):
    # reference: CHECK_TORCH_TENSOR_DTYPE / _SHAPE (kernels/flash-attn/utils/utils.h:137-147)
    for t in (Q, K, V, O):
        if t.dtype != torch.float16:
            raise RuntimeError("values must be torch::kHalf")
    if Q.dim() != 4:
        raise RuntimeError("Tensor size mismatch!")
    B, H, N, D = Q.shape
    if tuple(K.shape) != (B, H, N, D) or tuple(O.shape) != (B, H, N, D):
        raise RuntimeError("Tensor size mismatch!")
    want_v = (B, H, D, N) if v_transposed else (B, H, N, D)
    if tuple(V.shape) != want_v:
        raise RuntimeError("Tensor size mismatch!")
    for t in (Q, K, V, O):
        if not t.is_cuda:
            raise RuntimeError("leetcuda_b200.flash_attn: tensors must be CUDA tensors (no CPU path)")
        if not t.is_contiguous():
            raise RuntimeError("leetcuda_b200.flash_attn: tensors must be contiguous")
    return B, H, N, D


def _check_ex(Q, K, V, O, v_transposed, causal, lse):
    """Shapes of fmha_fwd: Q, O [B,H,Nq,D]; K [B,H,Nk,D]; V [B,H,Nk,D] or [B,H,D,Nk]; lse fp32 [B,H,Nq]."""
    for t in (Q, K, V, O):
        if t.dtype != torch.float16:
            raise RuntimeError("values must be torch::kHalf")
    if Q.dim() != 4 or K.dim() != 4:
        raise RuntimeError("Tensor size mismatch!")
    B, H, Nq, D = Q.shape
    Nk = K.shape[2]
    if tuple(K.shape) != (B, H, Nk, D):
        raise RuntimeError(f"fmha_fwd: K must be [B,H,Nk,D] = [{B},{H},Nk,{D}], got {list(K.shape)}")
    if tuple(O.shape) != (B, H, Nq, D):
        raise RuntimeError(f"fmha_fwd: O must have Q's shape {list(Q.shape)}, got {list(O.shape)}")
    want_v = (B, H, D, Nk) if v_transposed else (B, H, Nk, D)
    if tuple(V.shape) != want_v:
        raise RuntimeError(f"fmha_fwd: V must be {list(want_v)} ({'[B,H,D,Nk]' if v_transposed else '[B,H,Nk,D]'}), "
                           f"got {list(V.shape)}")
    if causal and Nk < Nq:
        raise RuntimeError(f"fmha_fwd: causal attention needs at least as many keys as queries (Nq={Nq}, Nk={Nk}): "
                           "query row i sees the keys j <= i + Nk - Nq")
    if lse is not None:
        if lse.dtype != torch.float32 or tuple(lse.shape) != (B, H, Nq) or not lse.is_cuda or not lse.is_contiguous():
            raise RuntimeError(f"fmha_fwd: lse must be a contiguous fp32 CUDA tensor [B,H,Nq] = [{B},{H},{Nq}], got "
                               f"{lse.dtype} {list(lse.shape)}")
    for t in (Q, K, V, O):
        if not t.is_cuda:
            raise RuntimeError("leetcuda_b200.flash_attn: tensors must be CUDA tensors (no CPU path)")
        if not t.is_contiguous():
            raise RuntimeError("leetcuda_b200.flash_attn: tensors must be contiguous")
    return B, H, Nq, Nk, D


def fmha_fwd(Q, K, V, O, *, v_transposed: bool = False, scale: float = 0.0, lse=None, causal: bool = False) -> None:
    """``O = softmax(Q K^T * scale) V`` on the current CUDA stream of ``Q``'s device.

    Q, O: ``[B,H,Nq,D]``; K: ``[B,H,Nk,D]``; V: ``[B,H,Nk,D]`` (``[B,H,D,Nk]`` with ``v_transposed``).
    ``causal=True``: query row i attends to the keys ``j <= i + Nk - Nq`` (bottom-right alignment, as
    FlashAttention-2 >= 2.1; top-left, i.e. ``scaled_dot_product_attention(is_causal=True)``, only when Nq == Nk)
    and needs ``Nk >= Nq``.
    ``lse`` (optional, fp32 ``[B,H,Nq]`` CUDA tensor) receives ``ln sum_j exp(scale * q_i . k_j)`` over the keys the
    row attends to — the statistic ``merge_attn_states`` needs to combine results over disjoint key ranges."""
    B, H, Nq, Nk, D = _check_ex(Q, K, V, O, v_transposed, causal, lse)
    idx = Q.device.index
    args = [Q.data_ptr(), K.data_ptr(), V.data_ptr(), O.data_ptr()]
    if causal or Nq != Nk:
        fn = _capi.lib().b200_fmha_fwd_f16_ex
        args += [None if lse is None else lse.data_ptr(), B, H, Nq, Nk, D, int(v_transposed), int(bool(causal)),
                 float(scale)]
    else:
        if lse is not None:
            fn = _capi.lib().b200_fmha_fwd_f16_lse
            args.append(lse.data_ptr())
        else:
            fn = _capi.lib().b200_fmha_fwd_f16
        args += [B, H, Nq, D, int(v_transposed), float(scale)]
    if torch.cuda.current_device() != idx:
        with torch.cuda.device(idx):
            rc = fn(*args, _capi.raw_stream(idx))
    else:
        rc = fn(*args, _capi.raw_stream(idx))
    if rc == -3:  # B200_ENOTSUP: the reference throws exactly this text (flash_attn_mma_split_q.cu:793)
        raise RuntimeError("headdim not support!")
    _capi.check(rc, "fmha_fwd")


def fmha_host(Q, K, V, O, *, v_transposed: bool = False, scale: float = 0.0) -> None:
    """Host-buffer entry point (``b200_fmha_fwd_f16_host``): ``Q``, ``K``, ``V``, ``O`` are CPU fp16 tensors
    (pinned for full PCIe bandwidth).  The call uploads the inputs, runs the kernel on the current device and
    downloads ``O``, pipelined over (batch x head) chunks; it returns when ``O`` is complete."""
    for t in (Q, K, V, O):
        if t.dtype != torch.float16:
            raise RuntimeError("values must be torch::kHalf")
        if t.is_cuda or not t.is_contiguous():
            raise RuntimeError("leetcuda_b200.fmha_host: tensors must be contiguous host tensors")
    B, H, N, D = Q.shape
    want_v = (B, H, D, N) if v_transposed else (B, H, N, D)
    if tuple(K.shape) != (B, H, N, D) or tuple(O.shape) != (B, H, N, D) or tuple(V.shape) != want_v:
        raise RuntimeError("Tensor size mismatch!")
    idx = torch.cuda.current_device()
    rc = _capi.lib().b200_fmha_fwd_f16_host(Q.data_ptr(), K.data_ptr(), V.data_ptr(), O.data_ptr(), B, H, N, D,
                                            int(v_transposed), float(scale), _capi.raw_stream(idx))
    if rc == -3:
        raise RuntimeError("headdim not support!")
    _capi.check(rc, "fmha_host")


def _fmha_ref(Q, K, V, O, v_transposed: bool = False) -> None:
    """The reference-named ops: equal query / key lengths, full attention, the reference's shape checks."""
    _check(Q, K, V, O, v_transposed)
    fmha_fwd(Q, K, V, O, v_transposed=v_transposed)


def _make(name: str):
    vt = name in V_TRANSPOSED_OPS

    def op(Q, K, V, O, stages: int = 1) -> None:
        _fmha_ref(Q, K, V, O, vt)
    op.__name__ = op.__qualname__ = name
    op.__doc__ = (f"{name}(Q, K, V, O, stages) -> None  "
                  f"[V is {'[B,H,D,N]' if vt else '[B,H,N,D]'}; stages ignored; sm_100a fused kernel]")
    return op


for _n in OP_NAMES:
    globals()[_n] = _make(_n)


def flash_attn_cute(Q, K, V, O) -> None:
    """reference: kernels/flash-attn/cutlass/flash_attn_cute.cu:496-524."""
    _fmha_ref(Q, K, V, O)


__all__ = OP_NAMES + ["flash_attn_cute", "fmha_fwd", "fmha_host", "OP_NAMES", "V_TRANSPOSED_OPS"]
