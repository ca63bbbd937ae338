"""ctypes loader for the C ABI declared in include/leetcuda_b200.h.

The shared library is the product: if it is missing this module raises — no op of
the package silently falls back to a CPU or PyTorch implementation (the oracle under
oracle/ is test infrastructure only and is never imported from here).  The only ops
that deliberately call the vendor library are the reference's own vendor rows, and
their docstrings say so: hgemm_cublas_tensor_op_{nn,tn}, sgemm_cublas{,_tf32}, and the
13 full-precision fp32 SGEMM names (cuBLAS fp32 unless LEETCUDA_B200_SGEMM_FP32=3xtf32).
"""
from __future__ import annotations

import ctypes
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libleetcuda_b200.so"

B200_OK = 0
B_ROW_MAJOR_KN = 0  # "NN"
B_ROW_MAJOR_NK = 1  # "TN"

_lib = None

_vp = ctypes.c_void_p
_i = ctypes.c_int
_u32 = ctypes.c_uint32
_f = ctypes.c_float

# name -> (restype, argtypes); mirrors include/leetcuda_b200.h one to one
SIGNATURES = {
    "b200_version": (_i, []),
    "b200_last_error": (ctypes.c_char_p, []),
    "b200_launch_count": (ctypes.c_uint64, []),
    "b200_hgemm_f16": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "b200_hgemm_f16_ex": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _u32, _u32, _u32, _vp]),
    "b200_hgemm_f16_acc16": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "b200_hgemm_f16_rows": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200_hgemm_f16_rows_fused": (_i, [_vp, _vp, _vp, _vp, ctypes.POINTER(ctypes.c_void_p), _i, _i, _i, _i, _i, _i, _vp]),
    "b200_fmha_fwd_f16": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp]),
    "b200_fmha_fwd_f16_lse": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp]),
    "b200_fmha_fwd_f16_ex": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "b200_fmha_fwd_f16_rmsnorm": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _f, _vp]),
    "b200_rope_f32": (_i, [_vp, _vp, _i, _i, _vp]),
    "b200_rope_qk_f16": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "b200_rms_norm": (_i, [_vp, _vp, _f, _i, _i, _i, _vp]),
    "b200_sgemm_tf32": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200_sgemm_3xtf32": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "b200_sgemm_tf32_ex": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _u32, _u32, _u32, _vp]),
    "b200_tf32_round_inplace": (_i, [_vp, ctypes.c_size_t, _vp]),
    "b200_merge_attn_states": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "b200_hgemm_f16_host": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "b200_fmha_fwd_f16_host": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp]),
}


def lib() -> ctypes.CDLL:
    """Load (once) and return the shared library; raise loudly if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("LEETCUDA_B200_LIB", LIB_PATH))
    if not path.exists():
        raise RuntimeError(
            f"{path} not found: build it with `python -m leetcuda_b200.build` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`). "
            "leetcuda_b200 has no fallback path."
        )
    handle = ctypes.CDLL(str(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)  # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    _lib = handle
    return handle


def last_error() -> str:
    return lib().b200_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    """Map a C-ABI status onto the reference's error behaviour (RuntimeError)."""
    if rc != B200_OK:
        raise RuntimeError(f"{what}: {last_error()} (status {rc})")


def launch_count() -> int:
    return int(lib().b200_launch_count())


def raw_stream(device_index: int) -> int:
    """cudaStream_t of torch's current stream on `device_index` (fast path: no Stream object)."""
    import torch
    try:
        return torch._C._cuda_getCurrentRawStream(device_index)
    except AttributeError:  # older/newer torch without the private helper
        return torch.cuda.current_stream(device_index).cuda_stream
