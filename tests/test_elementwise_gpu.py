"""GPU parity tests of the element-wise steps around attention (SURVEY §8f-4): rope, rms_norm and the
RMS-norm epilogue fused into the attention kernels, through the C ABI.

Checker: the CPU oracle (oracle.c: oracle_rope_f32 restates kernels/rope/rope.cu:20-34, oracle_rms_norm
restates kernels/rms-norm/rms_norm.cu:55-73 / :319-338).  Tolerances: rope |err| <= 3e-7 * seq_len * max|x| + 1e-5
— the angle p * theta^(-2i/hidden) is an fp32 product of a position up to seq_len with a frequency that carries
~1 ulp (6e-8 relative) of evaluation error whichever way it is computed (powf + division in the reference, exp2f
here), i.e. up to seq_len * 6e-8 rad on the fastest pair; rms_norm fp32 1e-5 relative, fp16 one fp16 ulp.
"""
import numpy as np
import pytest
import torch

from leetcuda_b200 import _capi, flash_attn, fused_ops, rms_norm, rope
from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("shape", [(64, 128), (4096, 512), (1000, 96), (33, 2048), (7, 4)])
def test_rope_vs_oracle(shape):
    S, Hd = shape
    x_np = np.random.default_rng(S + Hd).standard_normal((S, Hd), dtype=np.float32)
    want = O.rope_f32(x_np)
    x = torch.from_numpy(x_np).cuda()
    for name in rope.OP_NAMES:
        out = torch.full_like(x, float("nan"))
        getattr(rope, name)(x, out)
        torch.cuda.synchronize()
        np.testing.assert_allclose(out.cpu().numpy(), want, rtol=0, atol=3e-7 * S * np.abs(x_np).max() + 1e-5, err_msg=name)
    # rotation preserves the norm of every pair
    n_in = (x[:, 0::2] ** 2 + x[:, 1::2] ** 2)
    n_out = (out[:, 0::2] ** 2 + out[:, 1::2] ** 2)
    assert torch.allclose(n_in, n_out, rtol=1e-5, atol=1e-6)
    # position 0 is the identity
    assert torch.equal(out[0], x[0])


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("shape", [(4096, 512), (1000, 1024), (17, 64), (512, 4096), (3, 8192), (64, 2048)])
def test_rms_norm_vs_oracle(shape, dtype):
    R, K = shape
    x_np = np.random.default_rng(R + K).standard_normal((R, K), dtype=np.float32)
    x_np = x_np.astype(np.float16 if dtype == torch.float16 else np.float32)
    g = 1.25
    want = O.rms_norm(x_np, g).astype(np.float32)
    x = torch.from_numpy(x_np).cuda()
    names = [n for n in rms_norm.OP_NAMES if ("f32" == n.split("_")[2][:3]) == (dtype == torch.float32)]
    assert names
    for name in names:
        y = torch.full_like(x, float("nan"))
        getattr(rms_norm, name)(x, y, g)
        torch.cuda.synchronize()
        got = y.cpu().numpy().astype(np.float32)
        if dtype == torch.float32:
            np.testing.assert_allclose(got, want, rtol=2e-5, atol=1e-6, err_msg=name)
        else:
            # within one fp16 ulp of the oracle (the row sum is accumulated in a different order)
            np.testing.assert_allclose(got, want, rtol=1e-3, atol=1e-3, err_msg=name)
            assert np.mean(got == want) > 0.98, name
    with pytest.raises(RuntimeError):
        getattr(rms_norm, names[0])(x.double(), x.double(), g)


@pytest.mark.parametrize("shape", [(1, 2, 512, 128), (2, 2, 300, 64), (1, 1, 256, 96), (1, 2, 512, 256), (1, 2, 512, 512),
                                   (1, 1, 384, 384)])
def test_fused_rmsnorm_epilogue(shape):
    """attn_rmsnorm == rms_norm(attention) to fp16 rounding: the fused path normalises the fp32 row before
    the single rounding to fp16, the composition rounds twice."""
    B, H, N, D = shape
    g_ = torch.Generator(device="cuda").manual_seed(N + D)
    q, k, v = (torch.randn(B, H, N, D, device="cuda", dtype=torch.half, generator=g_) for _ in range(3))
    o = torch.zeros_like(q)
    flash_attn.fmha_fwd(q, k, v, o)
    fused = torch.full_like(q, float("nan"))
    lse = torch.zeros(B, H, N, device="cuda")
    before = _capi.launch_count()
    fused_ops.attn_rmsnorm(q, k, v, fused, 0.75, lse=lse)
    torch.cuda.synchronize()
    assert _capi.launch_count() - before == 1
    # truth from the fp32 attention result
    s = (q.float() @ k.float().transpose(-2, -1)) / (D ** 0.5)
    of = torch.softmax(s, dim=-1) @ v.float()
    want = of * torch.rsqrt((of * of).mean(dim=-1, keepdim=True) + 1e-5) * 0.75
    assert torch.allclose(fused.float(), want, rtol=1e-2, atol=1e-2)
    assert (fused.float() - want).abs().max().item() < 4e-3
    assert (lse - torch.logsumexp(s, dim=-1)).abs().max().item() < 2e-3
    # and the unfused composition through the two ops agrees
    y = torch.empty_like(o)
    rms_norm.rms_norm(o.view(-1, D), y.view(-1, D), 0.75)
    torch.cuda.synchronize()
    assert torch.allclose(fused.float(), y.float(), rtol=1e-2, atol=1e-2)


def test_fused_rmsnorm_unsupported_head_dim_is_an_error():
    q = torch.randn(1, 1, 128, 640, device="cuda", dtype=torch.half)
    with pytest.raises(RuntimeError):
        fused_ops.attn_rmsnorm(q, q, q, torch.empty_like(q), 1.0)


@pytest.mark.parametrize("shape", [(1, 2, 512, 128), (2, 3, 300, 64), (1, 1, 1024, 96), (1, 2, 256, 512)])
def test_rope_qk_and_attention(shape):
    """rope_qk (fp16 attention layout) against the fp32 rope oracle applied per head, and attention on the
    rotated operands against the fp32 truth."""
    B, H, N, D = shape
    g_ = torch.Generator(device="cuda").manual_seed(N + D)
    q, k, v = (torch.randn(B, H, N, D, device="cuda", dtype=torch.half, generator=g_) for _ in range(3))
    q_r, k_r = torch.empty_like(q), torch.empty_like(k)
    fused_ops.rope_qk(q, k, q_r, k_r)
    torch.cuda.synchronize()
    for src, got in ((q, q_r), (k, k_r)):
        for b in range(B):
            for h in range(H):
                want = O.rope_f32(src[b, h].float().cpu().numpy())
                np.testing.assert_allclose(got[b, h].float().cpu().numpy(), want, rtol=2e-3, atol=2e-3)
    # in place == out of place
    q2, k2 = q.clone(), k.clone()
    fused_ops.rope_qk(q2, k2)
    torch.cuda.synchronize()
    assert torch.equal(q2, q_r) and torch.equal(k2, k_r)
    o = torch.zeros_like(q)
    fused_ops.attn_rope(q, k, v, o)
    torch.cuda.synchronize()
    s = (q_r.float() @ k_r.float().transpose(-2, -1)) / (D ** 0.5)
    want = torch.softmax(s, dim=-1) @ v.float()
    assert torch.allclose(o.float(), want, rtol=1e-2, atol=1e-2)


# ---------------------------------------------------------------------------------------------------------------
# against the recorded outputs of the reference's own kernels (oracle/_ref rebuilt for sm_100a with the reference's
# flags, --use_fast_math included; oracle/gen_golden.py on a B200)
# ---------------------------------------------------------------------------------------------------------------
import json  # noqa: E402
from pathlib import Path  # noqa: E402

from oracle.gen_golden import RMSNORM_CASES, ROPE_CASES, rowwise_inputs  # noqa: E402

GOLDEN = Path(__file__).parent / "golden"


@pytest.mark.parametrize("case", ROPE_CASES)
def test_rope_vs_reference_golden(case):
    S, Hd, seed = case
    f = GOLDEN / f"rope_{S}x{Hd}_s{seed}.npz"
    if not f.exists():
        pytest.skip("golden file not generated yet")
    g = np.load(f)
    x_np = rowwise_inputs(S, Hd, seed)
    x = torch.from_numpy(x_np).cuda()
    out = torch.empty_like(x)
    rope.rope_f32x4_pack(x, out)
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    # the reference's build evaluates sin / cos / pow with fast-math intrinsics: |err| ~ 2^-21.4 * angle on top of the
    # fp32 angle itself, i.e. up to ~5e-7 * seq_len per unit of |x|
    tol = 5e-7 * S * np.abs(x_np).max() + 1e-5
    for name in ("rope_f32", "rope_f32_v2", "rope_f32x4_pack"):
        if name in g.files:
            np.testing.assert_allclose(got[::4], g[name], rtol=0, atol=tol, err_msg=name)
    # and this library's result is at least as close to the IEEE restatement as the reference's own kernel is
    want = O.rope_f32(x_np)
    assert np.abs(got - want)[::4].max() <= np.abs(g["rope_f32"] - want[::4]).max() + 1e-6


@pytest.mark.parametrize("case", RMSNORM_CASES)
def test_rms_norm_vs_reference_golden(case):
    R, K, seed = case
    f = GOLDEN / f"rmsnorm_{R}x{K}_s{seed}.npz"
    if not f.exists():
        pytest.skip("golden file not generated yet")
    g = np.load(f)
    gain = 1.25
    sub = json.loads(str(g["meta"]))["subsample"]          # the goldens keep every sub-th row
    x32 = torch.from_numpy(rowwise_inputs(R, K, seed)).cuda()
    x16 = x32.half()
    y32, y16 = torch.empty_like(x32), torch.empty_like(x16)
    rms_norm.rms_norm_f32x4(x32, y32, gain)
    rms_norm.rms_norm_f16x8_pack_f32(x16, y16, gain)
    torch.cuda.synchronize()
    for name in ("rms_norm_f32", "rms_norm_f32x4"):
        np.testing.assert_allclose(y32.cpu().numpy()[::sub], g[name], rtol=1e-5, atol=1e-6, err_msg=name)
    got16 = y16.cpu().numpy().astype(np.float32)[::sub]
    for name in ("rms_norm_f16x8_f32", "rms_norm_f16x8_pack_f32", "rms_norm_f16_f32"):      # fp32 statistics: one fp16 ulp
        np.testing.assert_allclose(got16, g[name].astype(np.float32), rtol=1e-3, atol=1e-3, err_msg=name)
    for name in ("rms_norm_f16_f16", "rms_norm_f16x2_f16", "rms_norm_f16x8_f16", "rms_norm_f16x8_pack_f16"):
        # the reference accumulates these variants' statistics in fp16: they sit within ~1 % of the fp32-statistics result
        np.testing.assert_allclose(got16, g[name].astype(np.float32), rtol=3e-2, atol=3e-2, err_msg=name)
