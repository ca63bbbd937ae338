"""GPU tests of causal attention and of separate query / key lengths (b200_fmha_fwd_f16_ex through fmha_fwd), on
every default kernel: the two-tile kernel (D <= 128; persistent at D <= 64), the column-slab kernel and the CTA-pair
kernel (D = 256 .. 512, D % 128 == 0).

Truth: fp32 torch on the GPU with the bottom-right mask built explicitly, ones(Nq, Nk).tril(Nk - Nq): query row i
sees the keys j <= i + Nk - Nq.  Tolerance as test_fmha_gpu.py: allclose(1e-2, 1e-2) and max |err| < 2e-3; the LSE
within 2e-3 of logsumexp over the allowed scores.
"""
import math

import pytest
import torch
import torch.nn.functional as F

from leetcuda_b200 import _capi, flash_attn

pytestmark = pytest.mark.gpu
RTOL = ATOL = 1e-2


def _randn(shape, g):
    return torch.randn(*shape, device="cuda", dtype=torch.half, generator=g)


def _inputs(B, H, Nq, Nk, D, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return _randn((B, H, Nq, D), g), _randn((B, H, Nk, D), g), _randn((B, H, Nk, D), g)


def _truth(q, k, v, causal):
    """fp32 softmax(Q K^T / sqrt(D)) V over the allowed keys, and the row log-sum-exp."""
    Nq, Nk, D = q.shape[2], k.shape[2], q.shape[3]
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        s = torch.matmul(q.float(), k.float().transpose(-2, -1)) * (1.0 / math.sqrt(D))
        if causal:
            allowed = torch.ones(Nq, Nk, dtype=torch.bool, device=q.device).tril(Nk - Nq)
            s = s.masked_fill(~allowed, float("-inf"))
        lse = torch.logsumexp(s, dim=-1)
        o = torch.matmul(torch.softmax(s, dim=-1), v.float())
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return o, lse


def _run(q, k, v, causal, vt=False, lse=True):
    B, H, Nq, D = q.shape
    o = torch.full_like(q, float("nan"))
    l = torch.full((B, H, Nq), float("nan"), device="cuda") if lse else None
    flash_attn.fmha_fwd(q, k, v.transpose(-2, -1).contiguous() if vt else v, o, v_transposed=vt, lse=l, causal=causal)
    torch.cuda.synchronize()
    return o, l


def _assert_close(q, k, v, causal, o, lse):
    want, want_lse = _truth(q, k, v, causal)
    got = o.float()
    assert torch.allclose(got, want, rtol=RTOL, atol=ATOL)
    assert (got - want).abs().max().item() < 2e-3
    if lse is not None:
        assert (lse - want_lse).abs().max().item() < 2e-3


# ------------------------------------------------------------------ causal, Nq == Nk
@pytest.mark.parametrize("N", [8, 128, 200, 256, 300, 1024])
@pytest.mark.parametrize("D", [32, 64, 96, 128, 192, 256, 320, 512, 640])
def test_causal_square(D, N):
    q, k, v = _inputs(1, 2, N, N, D, seed=D * 7 + N)
    o, lse = _run(q, k, v, causal=True)
    _assert_close(q, k, v, True, o, lse)


@pytest.mark.parametrize("N", [8, 128, 200, 256, 1024])
@pytest.mark.parametrize("D", [64, 128, 320])
def test_causal_square_transposed_v(D, N):
    q, k, v = _inputs(1, 2, N, N, D, seed=D * 5 + N)
    o, lse = _run(q, k, v, causal=True, vt=True)
    _assert_close(q, k, v, True, o, lse)


# ------------------------------------------------------------------ causal, Nq < Nk (bottom-right)
@pytest.mark.parametrize("D", [64, 128, 512])
@pytest.mark.parametrize("Nq,Nk", [(1, 4096), (7, 1000), (256, 1000), (1024, 4096)])
def test_causal_fewer_queries(Nq, Nk, D):
    q, k, v = _inputs(1, 2, Nq, Nk, D, seed=Nq + Nk + D)
    o, lse = _run(q, k, v, causal=True)
    _assert_close(q, k, v, True, o, lse)


@pytest.mark.parametrize("shape", [(4, 32, 1024, 1024, 64), (2, 64, 700, 1500, 64), (4, 32, 520, 520, 32)])
def test_causal_persistent_many_items(shape):
    """D <= 64 runs the persistent grid: more work items than SMs, of different KV extents, walked heaviest first."""
    B, H, Nq, Nk, D = shape
    q, k, v = _inputs(B, H, Nq, Nk, D, seed=Nq + Nk)
    o, lse = _run(q, k, v, causal=True)
    _assert_close(q, k, v, True, o, lse)


# ------------------------------------------------------------------ full attention, Nq != Nk
@pytest.mark.parametrize("D", [64, 128, 512])
@pytest.mark.parametrize("Nq,Nk", [(512, 1024), (1000, 300), (1, 777)])
def test_full_separate_lengths(Nq, Nk, D):
    q, k, v = _inputs(1, 2, Nq, Nk, D, seed=3 * Nq + Nk + D)
    o, lse = _run(q, k, v, causal=False)
    _assert_close(q, k, v, False, o, lse)


# ------------------------------------------------------------------ bit identity
@pytest.mark.parametrize("D", [64, 128, 256, 512])
def test_ex_full_square_is_bit_identical_to_plain_entries(D):
    B, H, N = 2, 3, 1000
    q, k, v = _inputs(B, H, N, N, D, seed=D)
    lib = _capi.lib()
    stream = _capi.raw_stream(torch.cuda.current_device())
    o_plain, o_lse, o_ex = (torch.full_like(q, float("nan")) for _ in range(3))
    lse_plain, lse_ex = (torch.full((B, H, N), float("nan"), device="cuda") for _ in range(2))
    ptrs = (q.data_ptr(), k.data_ptr(), v.data_ptr())
    assert lib.b200_fmha_fwd_f16(*ptrs, o_plain.data_ptr(), B, H, N, D, 0, 0.0, stream) == 0
    assert lib.b200_fmha_fwd_f16_lse(*ptrs, o_lse.data_ptr(), lse_plain.data_ptr(), B, H, N, D, 0, 0.0, stream) == 0
    assert lib.b200_fmha_fwd_f16_ex(*ptrs, o_ex.data_ptr(), lse_ex.data_ptr(), B, H, N, N, D, 0, 0, 0.0, stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(o_ex, o_plain) and torch.equal(o_ex, o_lse)
    assert torch.equal(lse_ex, lse_plain)


@pytest.mark.parametrize("D", [64, 128])
def test_causal_prefix_invariance(D):
    """Causal attention over the first m tokens equals rows [:m] of causal attention over all N, bit for bit: the
    work item of a row runs the same KV tiles with the same mask either way."""
    B, H, N = 1, 4, 4096
    q, k, v = _inputs(B, H, N, N, D, seed=41 + D)
    full, full_lse = _run(q, k, v, causal=True)
    for m in (256, 1024, 2816):
        sub = lambda t: t[:, :, :m].contiguous()
        o, lse = _run(sub(q), sub(k), sub(v), causal=True)
        assert torch.equal(o, full[:, :, :m]), m
        assert torch.equal(lse, full_lse[:, :, :m]), m


# ------------------------------------------------------------------ split-KV end to end
@pytest.mark.parametrize("D", [128, 512])
@pytest.mark.parametrize("Nq", [512, 300])
def test_split_kv_merge_causal(D, Nq):
    """Keys [0, Nk1) without a mask, keys [Nk1, Nk) causal (the Nq newest queries sit at the end of the cache), merged
    with merge_attn_states from the kernels' own LSEs == causal attention over all Nk keys."""
    from leetcuda_b200 import merge_attn_states as MA
    H, Nk, Nk1 = 8, 1024, 512
    q, k, v = _inputs(1, H, Nq, Nk, D, seed=Nq + D)
    parts = []
    for ks, causal in ((slice(0, Nk1), False), (slice(Nk1, Nk), True)):
        o, lse = _run(q, k[:, :, ks].contiguous(), v[:, :, ks].contiguous(), causal=causal)
        parts.append((o[0].transpose(0, 1).contiguous(), lse[0].contiguous()))   # [T,H,D], [H,T]
    merged = torch.empty_like(parts[0][0])
    merged_lse = torch.empty_like(parts[0][1])
    MA.merge_attn_states_cuda(merged, parts[0][0], parts[0][1], parts[1][0], parts[1][1], merged_lse)
    torch.cuda.synchronize()
    want, want_lse = _truth(q, k, v, causal=True)
    want = want[0].transpose(0, 1)
    assert torch.allclose(merged.float(), want, rtol=RTOL, atol=ATOL)
    assert (merged.float() - want).abs().max().item() < 3e-3
    assert (merged_lse - want_lse[0]).abs().max().item() < 2e-3


# ------------------------------------------------------------------ full size
def test_full_size_causal_vs_sdpa():
    """B4 H32 N4096 D128: at Nq == Nk the bottom-right mask is SDPA's is_causal=True (tolerance of
    test_full_size_vs_sdpa)."""
    g = torch.Generator(device="cuda").manual_seed(4096)
    q, k, v = (_randn((4, 32, 4096, 128), g) for _ in range(3))
    got, _ = _run(q, k, v, causal=True, lse=False)
    want = F.scaled_dot_product_attention(q, k, v, is_causal=True).float()
    assert torch.allclose(got.float(), want, atol=ATOL, rtol=RTOL)
    assert (got.float() - want).abs().max().item() < 3e-3
