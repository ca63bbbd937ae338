"""Argument checks of the causal / separate-length attention entry (b200_fmha_fwd_f16_ex) and of fmha_fwd's shape
validation: all rejected before any CUDA call, so they run without a GPU."""
import pytest
import torch

from leetcuda_b200 import _capi, flash_attn, fused_ops

EINVAL, ENOTSUP = -1, -3
P = 16   # a non-null dummy pointer: the call must fail before it is dereferenced


def _ex(lib, q=P, k=P, v=P, o=P, lse=None, B=1, H=1, Nq=128, Nk=128, D=64, vt=0, causal=0):
    return lib.b200_fmha_fwd_f16_ex(q, k, v, o, lse, B, H, Nq, Nk, D, vt, causal, 0.0, None)


@pytest.mark.parametrize("which", ["q", "k", "v", "o"])
def test_ex_rejects_null_pointers(built_lib, which):
    assert _ex(built_lib, **{which: None}) == EINVAL
    assert "null" in _capi.last_error()


@pytest.mark.parametrize("Nq,Nk", [(0, 128), (128, 0), (-1, 128), (128, -5)])
def test_ex_rejects_empty_lengths(built_lib, Nq, Nk):
    assert _ex(built_lib, Nq=Nq, Nk=Nk) == EINVAL
    assert "bad shape" in _capi.last_error()


def test_ex_rejects_causal_with_fewer_keys_than_queries(built_lib):
    assert _ex(built_lib, Nq=256, Nk=255, causal=1) == EINVAL
    assert "Nk >= Nq" in _capi.last_error()
    # without the mask the same lengths pass the argument checks (and stop here at the unsupported head dim)
    assert _ex(built_lib, Nq=256, Nk=255, causal=0, D=100) == ENOTSUP


@pytest.mark.parametrize("causal", [2, -1, 7])
def test_ex_rejects_causal_outside_0_1(built_lib, causal):
    assert _ex(built_lib, causal=causal) == EINVAL
    assert "causal must be 0 or 1" in _capi.last_error()


def test_ex_rejects_transposed_v_with_ragged_key_length(built_lib):
    assert _ex(built_lib, Nq=64, Nk=100, vt=1) == EINVAL
    assert "multiple of 8" in _capi.last_error()
    assert _ex(built_lib, Nq=100, Nk=100, vt=1, causal=1) == EINVAL
    assert "multiple of 8" in _capi.last_error()


@pytest.mark.parametrize("D", [100, 2048])
def test_ex_unsupported_headdim_matches_plain_entry(built_lib, D):
    rc_plain = built_lib.b200_fmha_fwd_f16(P, P, P, P, 1, 1, 128, D, 0, 0.0, None)
    err_plain = _capi.last_error()
    rc_ex = _ex(built_lib, D=D, causal=1)
    assert rc_plain == rc_ex == ENOTSUP
    assert _capi.last_error() == err_plain and "headdim not support" in err_plain


def _t(*shape, dtype=torch.float16):
    return torch.zeros(*shape, dtype=dtype)


def test_fmha_fwd_shape_errors_raise_before_the_library(monkeypatch):
    """Mismatched shapes raise a RuntimeError that names the problem, and the library is never touched."""
    def no_lib():
        raise AssertionError("the library must not be reached")
    monkeypatch.setattr(_capi, "lib", no_lib)
    q, k, v, o = _t(1, 2, 64, 32), _t(1, 2, 96, 32), _t(1, 2, 96, 32), _t(1, 2, 64, 32)
    with pytest.raises(RuntimeError, match="causal attention needs at least as many keys"):
        flash_attn.fmha_fwd(_t(1, 2, 128, 32), k, v, _t(1, 2, 128, 32), causal=True)
    with pytest.raises(RuntimeError, match=r"lse must be a contiguous fp32 CUDA tensor \[B,H,Nq\]"):
        flash_attn.fmha_fwd(q, k, v, o, lse=torch.zeros(1, 2, 96))
    with pytest.raises(RuntimeError, match="K must be"):
        flash_attn.fmha_fwd(q, _t(1, 2, 96, 16), v, o)
    with pytest.raises(RuntimeError, match="V must be"):
        flash_attn.fmha_fwd(q, k, _t(1, 2, 64, 32), o)
    with pytest.raises(RuntimeError, match="V must be"):
        flash_attn.fmha_fwd(q, k, v, o, v_transposed=True)
    with pytest.raises(RuntimeError, match="O must have Q's shape"):
        flash_attn.fmha_fwd(q, k, v, _t(1, 2, 96, 32))
    # well-formed shapes get as far as the device check (CPU tensors: no CPU path)
    with pytest.raises(RuntimeError, match="no CPU path"):
        flash_attn.fmha_fwd(q, k, v, o, causal=True)
    with pytest.raises(RuntimeError, match="no CPU path"):
        flash_attn.fmha_fwd(q, k, v.transpose(-2, -1).contiguous(), o, v_transposed=True)


def test_reference_ops_keep_equal_lengths():
    """The reference-named ops still demand K, V of Q's shape, and raise the reference's text."""
    q, k = _t(1, 1, 64, 32), _t(1, 1, 96, 32)
    with pytest.raises(RuntimeError, match="Tensor size mismatch!"):
        flash_attn.flash_attn_mma_stages_split_q(q, k, k, q.clone(), 1)
    with pytest.raises(RuntimeError, match="Tensor size mismatch!"):
        flash_attn.flash_attn_cute(q, k, k, q.clone())


def test_attn_rope_causal_with_rms_norm_is_rejected():
    q = _t(1, 1, 64, 32)
    with pytest.raises(RuntimeError, match="causal attention with the fused RMS-norm epilogue"):
        fused_ops.attn_rope(q, q, q, q.clone(), rms_g=1.0, causal=True)
