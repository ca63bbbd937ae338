"""Pins the CPU oracle against outputs of the reference's OWN kernels (tests/golden/*.npz,
recorded on a B200 from the unmodified reference sources by oracle/gen_golden.py), and checks
the oracle's internal consistency.  Runs without a GPU."""
import json
from pathlib import Path

import numpy as np
import pytest

from oracle import oracle as O
from oracle.gen_golden import (ATTN_CASES, FFPA_CASES, HGEMM_CASES, MERGE_CASES, SGEMM_CASES, attn_inputs,
                               hgemm_inputs, merge_inputs, sgemm_inputs)

GOLD = Path(__file__).parent / "golden"


def _load(name):
    f = GOLD / name
    if not f.exists():
        pytest.skip(f"{name} not generated yet")
    g = np.load(f)
    return g, json.loads(str(g["meta"]))


@pytest.mark.parametrize("case", HGEMM_CASES)
def test_hgemm_f16acc_restatement_reproduces_reference_kernels(case):
    """oracle_hgemm_f16acc (one fp16-rounded accumulation per k16 MMA) IS the reference's
    arithmetic: >= 99.5 % of the outputs of every reference tensor-core kernel (mma.sync, WMMA,
    CuTe, cuBLAS COMPUTE_16F) are reproduced bit for bit, the rest within one fp16 ulp."""
    M, N, K, seed = case
    g, meta = _load(f"hgemm_{M}x{N}x{K}_s{seed}.npz")
    sub = meta.get("subsample", 1)
    a, b = hgemm_inputs(M, N, K, seed)
    o16 = O.hgemm_f16acc(a, b, k_chunk=16)[::sub, ::sub]
    names = [k for k in g.files if k != "meta"]
    assert len(names) >= 6
    for name in names:
        ref = g[name]
        assert ref.dtype == np.float16 and ref.shape == o16.shape
        exact = np.mean(ref == o16)
        assert exact >= 0.995, (name, exact)
        # a one-ulp difference in an intermediate fp16 accumulator can survive cancellation,
        # so the residual is bounded by one ulp at the magnitude of the largest outputs
        ulp = 2.0 ** (np.floor(np.log2(np.abs(o16.astype(np.float64)).max())) - 10)
        assert np.abs(ref.astype(np.float64) - o16.astype(np.float64)).max() <= ulp, name


@pytest.mark.parametrize("case", HGEMM_CASES)
def test_hgemm_f32acc_is_closer_to_truth_than_the_reference(case):
    M, N, K, seed = case
    g, meta = _load(f"hgemm_{M}x{N}x{K}_s{seed}.npz")
    sub = meta.get("subsample", 1)
    a, b = hgemm_inputs(M, N, K, seed)
    truth = O.hgemm_f64(a, b)[::sub, ::sub]
    o32 = O.hgemm_f32acc(a, b)[::sub, ::sub].astype(np.float64)
    e32 = np.abs(o32 - truth).max()
    for name in (k for k in g.files if k != "meta"):
        eref = np.abs(g[name].astype(np.float64) - truth).max()
        assert e32 < eref, (name, e32, eref)
        # north_star tolerance holds between the two accumulation modes at these sizes
        np.testing.assert_allclose(o32, g[name].astype(np.float64), rtol=1e-2, atol=1e-2 * max(1, K // 64))


def test_hgemm_layouts_and_exactness():
    rng = np.random.default_rng(0)
    a = rng.integers(-3, 4, (64, 96)).astype(np.float16)
    b = rng.integers(-3, 4, (96, 40)).astype(np.float16)
    want = a.astype(np.int64) @ b.astype(np.int64)
    for fn in (O.hgemm_f32acc, O.hgemm_f16acc):
        assert np.array_equal(fn(a, b).astype(np.int64), want)
        assert np.array_equal(fn(a, np.ascontiguousarray(b.T), tn=True).astype(np.int64), want)
    assert np.array_equal(O.hgemm_f64(a, b), want.astype(np.float64))


@pytest.mark.parametrize("case", ATTN_CASES)
def test_attention_oracle_vs_reference_kernels(case):
    B, H, N, D, seed = case
    g, meta = _load(f"attn_B{B}H{H}N{N}D{D}_s{seed}.npz")
    q, k, v = attn_inputs(B, H, N, D, seed)
    truth = O.attn_f32(q, k, v).astype(np.float32)
    online = O.attn_online(q, k, v, Bc=64, s_f16=True).astype(np.float32)
    for name in (x for x in g.files if x != "meta"):
        ref = g[name].astype(np.float32)
        # the reference's own --check criterion (flash_attn_mma.py:465-494)
        np.testing.assert_allclose(ref, truth, atol=1e-2, rtol=1e-2, err_msg=name)
        np.testing.assert_allclose(ref, online, atol=1e-2, rtol=1e-2, err_msg=name)


@pytest.mark.parametrize("case", FFPA_CASES)
def test_ffpa_oracle_vs_reference_kernels(case):
    B, H, N, D, seed = case
    g, meta = _load(f"ffpa_B{B}H{H}N{N}D{D}_s{seed}.npz")
    q, k, v = attn_inputs(B, H, N, D, seed)
    truth = O.attn_f32(q, k, v).astype(np.float32)
    for name in (x for x in g.files if x != "meta"):
        np.testing.assert_allclose(g[name].astype(np.float32), truth, atol=1e-2, rtol=1e-2, err_msg=name)


def test_attention_oracles_agree_and_handle_edges():
    rng = np.random.default_rng(1)
    for (B, H, N, D) in [(1, 1, 8, 32), (2, 1, 200, 64), (1, 2, 130, 128)]:   # ragged N
        q, k, v = (rng.standard_normal((B, H, N, D), dtype=np.float32).astype(np.float16) for _ in range(3))
        ref = O.attn_f32(q, k, v).astype(np.float32)
        for Bc in (16, 64, 128):
            np.testing.assert_allclose(O.attn_online(q, k, v, Bc=Bc).astype(np.float32), ref, atol=2e-3, rtol=1e-2)
        vt = np.ascontiguousarray(np.swapaxes(v, -1, -2))
        assert np.array_equal(O.attn_f32(q, k, vt, v_transposed=True), O.attn_f32(q, k, v))
    ones = np.ones((1, 1, 64, 32), np.float16)
    q = rng.standard_normal((1, 1, 64, 32), dtype=np.float32).astype(np.float16)
    assert np.allclose(O.attn_f32(q, q, ones).astype(np.float32), 1.0, atol=1e-3)


def test_flop_counts_match_reference_definitions():
    # hgemm.py:282 and flash_attn_mma.py:241-278 evaluated by hand for the BASELINE shapes
    assert O.hgemm_flops(8192, 8192, 8192) == 2 * 8192 ** 3
    B, H, N, D = 4, 32, 4096, 128
    mm = O.mha_flops(B, H, N, D, only_matmul=True)
    assert mm == B * H * N * N * (2 * D - 1) + B * H * N * D * (2 * N - 1)
    assert abs(mm / (4 * B * H * N * N * D) - 1) < 1e-2
    assert O.mha_flops(B, H, N, D) - mm == B * H * N * N + 2 * B * H * N * (N - 1) + 3 * B * H * N * N


@pytest.mark.parametrize("case", SGEMM_CASES)
def test_sgemm_tf32_restatement_vs_reference_kernels(case):
    """The TF32 restatement is pinned on the reference's own kernels: (1) the in-place rounding of
    the operands (sgemm_wmma_tf32_stage.cu:44-60, 586-592) is reproduced BIT FOR BIT by
    oracle_tf32_round (rna, not truncation); (2) the three recorded wmma kernels agree with each
    other bit for bit and with the oracle's fp32-accumulated product within the bound of one
    truncated fp32 addition per k (the tensor core's internal accumulation is not architected)."""
    M, N, K, seed = case
    g, meta = _load(f"sgemm_{M}x{N}x{K}_s{seed}.npz")
    sub = meta["subsample"]
    a, b = sgemm_inputs(M, N, K, seed)
    assert np.array_equal(g["a_after"], O.tf32_round(a)[:8])
    assert np.array_equal(g["b_after"], O.tf32_round(b)[:8])
    assert not np.array_equal(g["a_after"], O.tf32_round(a, truncate=True)[:8])
    o = O.sgemm_tf32(a, b, mode="rna")[::sub, ::sub].astype(np.float64)
    truth = O.sgemm_f64(a, b, mode="rna")[::sub, ::sub]
    bound = K * 2.0 ** -23 * np.abs(truth).max()
    assert np.abs(o - truth).max() <= bound / 8          # the oracle itself: round-to-nearest sums
    refs = [g[k] for k in g.files if k.startswith("sgemm_wmma")]
    assert len(refs) == 3
    for r in refs:
        assert r.dtype == np.float32 and np.array_equal(r, refs[0])
        assert np.abs(r.astype(np.float64) - o).max() <= bound
    # the vendor TF32 GEMM (called on the unrounded a, b) lands within TF32 operand precision of it
    np.testing.assert_allclose(g["sgemm_cublas_tf32"].astype(np.float64), truth, rtol=1e-2, atol=1e-2)


def test_tf32_round_restatement_known_answers():
    x = np.array([1.0, 1.0 + 2.0 ** -11, 1.0 + 2.0 ** -11 + 2.0 ** -20, 1.0 + 2.0 ** -10,
                  -1.0 - 2.0 ** -11, np.inf, -np.inf], dtype=np.float32)
    want_rna = np.array([1.0, 1.0 + 2.0 ** -10, 1.0 + 2.0 ** -10, 1.0 + 2.0 ** -10,
                         -1.0 - 2.0 ** -10, np.inf, -np.inf], dtype=np.float32)   # ties away from zero
    want_trunc = np.array([1.0, 1.0, 1.0, 1.0 + 2.0 ** -10, -1.0, np.inf, -np.inf], dtype=np.float32)
    assert np.array_equal(O.tf32_round(x), want_rna)
    assert np.array_equal(O.tf32_round(x, truncate=True), want_trunc)
    assert np.all((O.tf32_round(np.random.default_rng(0).standard_normal(1000).astype(np.float32))
                   .view(np.uint32) & 0x1FFF) == 0)


def test_sgemm_oracle_layouts_and_exactness():
    rng = np.random.default_rng(1)
    a = rng.integers(-5, 6, (48, 72)).astype(np.float32)
    b = rng.integers(-5, 6, (72, 40)).astype(np.float32)
    want = a.astype(np.int64) @ b.astype(np.int64)
    for mode in ("rna", "trunc", "asis"):
        assert np.array_equal(O.sgemm_tf32(a, b, mode=mode).astype(np.int64), want)
        assert np.array_equal(O.sgemm_tf32(a, np.ascontiguousarray(b.T), tn=True, mode=mode).astype(np.int64), want)
    assert np.array_equal(O.sgemm_f64(a, b), want.astype(np.float64))


def _unbits(x, dt):
    if dt == "f32":
        return x.astype(np.float64)
    if dt == "f16":
        return x.view(np.float16).astype(np.float64)
    return (x.astype(np.uint32) << 16).view(np.float32).astype(np.float64)


@pytest.mark.parametrize("case", MERGE_CASES)
def test_merge_attn_states_restatement_vs_reference_kernel(case):
    """oracle_merge_attn_states against the recorded outputs of the reference's CUDA kernel: same
    formula in fp32; glibc's expf/logf and CUDA's differ in the last place, so >= 99.9 % of the
    16-bit outputs are bit-identical (the rest one rounding step away) and the fp32 outputs agree to ~1e-6."""
    T, H, D, dt, seed = case
    g, meta = _load(f"merge_T{T}H{H}D{D}_{dt}_s{seed}.npz")
    sub = meta["subsample"]
    p, p_lse, s, s_lse = merge_inputs(T, H, D, dt, seed)
    out, out_lse = O.merge_attn_states(p, p_lse, s, s_lse, dt)
    ref, got = _unbits(g["out"], dt), _unbits(out[::sub], dt)
    assert not np.isnan(ref).any()
    if dt == "f32":   # keeps every last-place difference of its row's scale (absolute: the terms may cancel)
        assert np.all(np.abs(ref - got) <= 2.0 ** -20 * np.maximum(np.abs(ref), 1.0))
        assert np.mean(ref == got) >= 0.8
    else:
        ulp = {"f16": 2.0 ** -10, "bf16": 2.0 ** -7}[dt]
        assert np.all(np.abs(ref - got) <= 1.01 * ulp * np.maximum(np.abs(ref), 0.25))
        assert np.mean(ref == got) >= 0.999
    assert np.abs(g["out_lse"] - out_lse).max() <= 4e-7 * max(1.0, np.abs(out_lse).max())


def test_merge_attn_states_oracle_properties():
    T, H, D = 33, 3, 16
    p, p_lse, s, s_lse = merge_inputs(T, H, D, "f32", seed=1)
    out, lse = O.merge_attn_states(p, p_lse, s, s_lse, "f32")
    # a part whose lse is +inf (empty key range) contributes nothing
    emp = np.isinf(p_lse)
    assert emp.any()
    hh, tt = np.nonzero(emp)
    assert np.array_equal(out[tt, hh], s[tt, hh]) and np.array_equal(lse[hh, tt], s_lse[hh, tt])
    # symmetric in its two parts
    out2, lse2 = O.merge_attn_states(s, s_lse, p, p_lse, "f32")
    np.testing.assert_allclose(out, out2, rtol=1e-6, atol=1e-7)
    assert np.array_equal(lse, lse2)
    # merging a part with itself returns it, lse + log 2
    out3, lse3 = O.merge_attn_states(s, s_lse.clip(max=10), s, s_lse.clip(max=10), "f32")
    np.testing.assert_allclose(out3, s, rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(lse3, s_lse.clip(max=10) + np.log(2.0), rtol=1e-6)


# ------------------------------------------------------------------ rope / rms_norm (SURVEY §8f-4)
from oracle.gen_golden import RMSNORM_CASES, ROPE_CASES, rowwise_inputs  # noqa: E402


@pytest.mark.parametrize("case", ROPE_CASES)
def test_rope_restatement_vs_reference_kernels(case):
    """oracle_rope_f32 (IEEE powf / sinf / cosf) against the recorded outputs of the reference's rope kernels, which were
    built with --use_fast_math (kernels/rope/rope.py:21): agreement within the fast-math error of the angle's sin / cos,
    ~5e-7 * seq_len per unit of |x|; the three reference kernels agree with each other to the same bound."""
    S, Hd, seed = case
    f = Path(__file__).parent / "golden" / f"rope_{S}x{Hd}_s{seed}.npz"
    if not f.exists():
        pytest.skip("golden file not generated yet")
    g = np.load(f)
    x = rowwise_inputs(S, Hd, seed)
    want = O.rope_f32(x)
    tol = 5e-7 * S * np.abs(x).max() + 1e-5
    for name in g.files:
        if name != "meta":
            np.testing.assert_allclose(want[::4], g[name], rtol=0, atol=tol, err_msg=name)
    # rotation: position 0 untouched, pair norms preserved
    assert np.array_equal(want[0], x[0])
    np.testing.assert_allclose(want[:, 0::2] ** 2 + want[:, 1::2] ** 2, x[:, 0::2] ** 2 + x[:, 1::2] ** 2, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("case", RMSNORM_CASES)
def test_rms_norm_restatement_vs_reference_kernels(case):
    R, K, seed = case
    f = Path(__file__).parent / "golden" / f"rmsnorm_{R}x{K}_s{seed}.npz"
    if not f.exists():
        pytest.skip("golden file not generated yet")
    g = np.load(f)
    x = rowwise_inputs(R, K, seed)
    meta = json.loads(str(g["meta"]))
    gain, sub = meta["g"], meta["subsample"]                                    # the goldens keep every sub-th row
    want32 = O.rms_norm(x, gain)
    for name in ("rms_norm_f32", "rms_norm_f32x4"):
        np.testing.assert_allclose(want32[::sub], g[name], rtol=1e-5, atol=1e-6, err_msg=name)
    want16 = O.rms_norm(x.astype(np.float16), gain).astype(np.float32)[::sub]
    for name in ("rms_norm_f16x8_f32", "rms_norm_f16x8_pack_f32", "rms_norm_f16_f32"):
        ref = g[name].astype(np.float32)
        np.testing.assert_allclose(want16, ref, rtol=1e-3, atol=1e-3, err_msg=name)
        assert np.mean(want16 == ref) > 0.97, (name, np.mean(want16 == ref))
    for name in ("rms_norm_f16_f16", "rms_norm_f16x2_f16", "rms_norm_f16x8_f16", "rms_norm_f16x8_pack_f16"):
        np.testing.assert_allclose(want16, g[name].astype(np.float32), rtol=3e-2, atol=3e-2, err_msg=name)
