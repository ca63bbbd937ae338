"""Drop-in mirror of ffpa-attn's python package (`ffpa_attn`) and extension (`pyffpa_cuda`).

reference: /root/reference/ffpa-attn/ffpa_attn/interface.py:1-68,
           /root/reference/ffpa-attn/ffpa_attn/__init__.py,
           /root/reference/ffpa-attn/csrc/pybind/ffpa_attn_api.cc:8-16

``ffpa(q, k, v, o=None, num_stages=2, level=L1, acc=FP32) -> o`` and the two raw ops
``ffpa_mma_acc_{f16,f32}_L1(Q, K, V, O, stages)``; Q,K,V,O fp16 ``[B,H,N,D]``.
"""
from __future__ import annotations

from enum import Enum
from functools import partial
from typing import Optional

import torch

from .flash_attn import _fmha_ref

__version__ = "0.0.2.b200"


class LevelType(Enum):
    L1 = 0
    L2 = 1
    L3 = 2


class MMAAccType(Enum):
    FP32 = 0
    FP16 = 1


def ffpa_mma_acc_f32_L1(Q, K, V, O, stages: int = 2) -> None:
    """reference: ffpa-attn/csrc/cuffpa/ffpa_attn_F16F16F32_L1.cu:43-84."""
    _fmha_ref(Q, K, V, O)


def ffpa_mma_acc_f16_L1(Q, K, V, O, stages: int = 2) -> None:
    """reference: ffpa-attn/csrc/cuffpa/ffpa_attn_F16F16F16_L1.cu:5-38 (fp32 accumulation here)."""
    _fmha_ref(Q, K, V, O)


def faster_prefill_attn_func(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor,
                             o: Optional[torch.Tensor] = None, num_stages: int = 2,
                             level: LevelType = LevelType.L1, acc: MMAAccType = MMAAccType.FP32):
    # Q, K, V, O: [B, H, N, D] layout (interface.py:30-40)
    if not isinstance(o, torch.Tensor) or o is None:
        o = torch.zeros_like(q)
    assert level == LevelType.L1, "only support FFPA L1 level now."
    if acc == MMAAccType.FP32:
        ffpa_mma_acc_f32_L1(q, k, v, o, num_stages)
    else:
        ffpa_mma_acc_f16_L1(q, k, v, o, num_stages)
    return o


ffpa = faster_prefill_attn_func
ffpa_acc_f32_L1 = partial(faster_prefill_attn_func, level=LevelType.L1, acc=MMAAccType.FP32)
ffpa_acc_f16_L1 = partial(faster_prefill_attn_func, level=LevelType.L1, acc=MMAAccType.FP16)

L1, L2, L3 = LevelType.L1, LevelType.L2, LevelType.L3
FP32, FP16 = MMAAccType.FP32, MMAAccType.FP16
