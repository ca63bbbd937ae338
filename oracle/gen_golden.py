"""TEST INFRASTRUCTURE — generate golden vectors from the reference's own kernels.

Runs ON THE GPU BOX (under gpurun) with the prebuilt oracle/_ref modules (the
UNMODIFIED reference kernels compiled for sm_100a by oracle/build_ref.py) and writes
their outputs for seeded inputs to gpurun_out/golden/*.npz; the files are then
committed under tests/golden/.  Inputs are NOT stored: they are regenerated from
the numpy seed by `golden_inputs()` below (also imported by the tests), so a
fixture is {meta, reference outputs}.

    python oracle/gen_golden.py [outdir [family ...]]     family in {sgemm, merge, rope, rmsnorm, hgemm, fa, ffpa}
"""
from __future__ import annotations

import json
import os
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent))

HGEMM_CASES = [  # (M, N, K, seed)
    (256, 256, 128, 11),
    (512, 512, 512, 12),
]
ATTN_CASES = [  # (B, H, N, D, seed)
    (1, 2, 256, 64, 21),
    (1, 2, 256, 128, 22),
]
SGEMM_CASES = [  # (M, N, K, seed)
    (256, 256, 128, 41),
    (512, 512, 512, 42),
]
MERGE_CASES = [  # (num_tokens, num_heads, head_size, dtype, seed): test_merge_attn_states.py:47-50 shapes
    (613, 16, 128, "f32", 51),
    (613, 16, 128, "f16", 52),
    (613, 16, 128, "bf16", 53),
    (512, 16, 128, "f16", 54),
]
ROPE_CASES = [  # (seq_len, hidden, seed): small positions, where the reference's fast-math sin/cos is still tight
    (256, 512, 61),
    (1024, 128, 62),
]
RMSNORM_CASES = [  # (rows, K, seed): kernels/rms-norm/rms_norm.py shapes (N x K, K <= 1024 for the block-per-row kernels)
    (512, 512, 71),
    (256, 1024, 72),
]
FFPA_CASES = [  # (B, H, N, D, seed)
    (1, 2, 256, 256, 31),
    (1, 1, 256, 512, 32),
]


def hgemm_inputs(M, N, K, seed):
    """Same distribution as the reference scripts (torch.randn fp16, hgemm.py:444-446)."""
    rng = np.random.default_rng(seed)
    a = rng.standard_normal((M, K), dtype=np.float32).astype(np.float16)
    b = rng.standard_normal((K, N), dtype=np.float32).astype(np.float16)
    return a, b


def sgemm_inputs(M, N, K, seed):
    """torch.randn fp32 like kernels/sgemm/sgemm.py:128-131."""
    rng = np.random.default_rng(seed)
    a = rng.standard_normal((M, K), dtype=np.float32)
    b = rng.standard_normal((K, N), dtype=np.float32)
    return a, b


def rowwise_inputs(rows, cols, seed):
    """torch.randn fp32 [rows, cols] like kernels/rope/rope.py:101 and kernels/rms-norm/rms_norm.py:79."""
    return np.random.default_rng(seed).standard_normal((rows, cols), dtype=np.float32)


def merge_inputs(T, H, D, dtype, seed):
    """Inputs as test_merge_attn_states.py:126-152: randn lse with ~10 % +inf entries (never both
    parts of one position), randn partial outputs.  Returns (p_out, p_lse, s_out, s_lse); the outputs
    are float32 arrays for "f32" and uint16 bit patterns for "f16" / "bf16"."""
    rng = np.random.default_rng(seed)
    p_lse = rng.standard_normal((H, T), dtype=np.float32)
    s_lse = rng.standard_normal((H, T), dtype=np.float32)
    mp = rng.random((H, T)) < 0.1
    ms = rng.random((H, T)) < 0.1
    both = mp & ms
    p_lse[mp & ~both] = np.inf
    s_lse[ms & ~both] = np.inf
    p = rng.standard_normal((T, H, D), dtype=np.float32)
    s = rng.standard_normal((T, H, D), dtype=np.float32)
    if dtype == "f16":
        p, s = p.astype(np.float16).view(np.uint16), s.astype(np.float16).view(np.uint16)
    elif dtype == "bf16":
        def bf(x):   # round to nearest even
            u = x.view(np.uint32)
            return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)
        p, s = bf(p), bf(s)
    return p, p_lse, s, s_lse


def attn_inputs(B, H, N, D, seed):
    """randn q,k,v as flash_attn_mma.py:417-435."""
    rng = np.random.default_rng(seed)
    q = rng.standard_normal((B, H, N, D), dtype=np.float32).astype(np.float16)
    k = rng.standard_normal((B, H, N, D), dtype=np.float32).astype(np.float16)
    v = rng.standard_normal((B, H, N, D), dtype=np.float32).astype(np.float16)
    return q, k, v


def main(outdir: Path, only=()):
    import torch
    from oracle.build_ref import load_prebuilt
    outdir.mkdir(parents=True, exist_ok=True)
    dev = "cuda"
    meta = {"device": torch.cuda.get_device_name(0), "torch": torch.__version__}
    want = lambda fam: not only or fam in only

    rs = load_prebuilt("ref_sgemm") if want("sgemm") else None
    if rs is not None:
        for (M, N, K, seed) in SGEMM_CASES:
            a_np, b_np = sgemm_inputs(M, N, K, seed)
            out = {}
            for name, stages in [("sgemm_wmma_m16n16k8_mma4x2_warp2x4_stages", 2),
                                 ("sgemm_wmma_m16n16k8_mma4x2_warp2x4_stages", 3),
                                 ("sgemm_wmma_m16n16k8_mma4x2_warp2x4_stages_dsmem", 2)]:
                a = torch.from_numpy(a_np).to(dev)   # fresh copies: the op rounds a and b in place
                b = torch.from_numpy(b_np).to(dev)
                c = torch.zeros(M, N, dtype=torch.float32, device=dev)
                getattr(rs, name)(a, b, c, stages, False, 1)
                torch.cuda.synchronize()
                out[f"{name}__s{stages}"] = c.cpu().numpy()
                if "a_after" not in out:       # the in-place side effect on the inputs (first 8 rows)
                    out["a_after"] = a[:8].cpu().numpy()
                    out["b_after"] = b[:8].cpu().numpy()
            a = torch.from_numpy(a_np).to(dev)
            b = torch.from_numpy(b_np).to(dev)
            c = torch.zeros(M, N, dtype=torch.float32, device=dev)
            rs.sgemm_cublas_tf32(a, b, c)
            torch.cuda.synchronize()
            out["sgemm_cublas_tf32"] = c.cpu().numpy()
            sub = 4 if M >= 512 else 1
            out = {k_: (v_ if k_.endswith("_after") else v_[::sub, ::sub].copy()) for k_, v_ in out.items()}
            np.savez_compressed(outdir / f"sgemm_{M}x{N}x{K}_s{seed}.npz",
                                meta=json.dumps({**meta, "M": M, "N": N, "K": K, "seed": seed,
                                                 "subsample": sub}), **out)
            print("golden sgemm", M, N, K, list(out))

    rm = load_prebuilt("ref_merge") if want("merge") else None
    if rm is not None:
        tdt = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
        for (T, H, D, dt, seed) in MERGE_CASES:
            p, p_lse, s, s_lse = merge_inputs(T, H, D, dt, seed)
            as_t = lambda x: (torch.from_numpy(x) if dt == "f32" else torch.from_numpy(x.view(np.int16)).view(tdt[dt])).to(dev)
            tp, ts = as_t(p), as_t(s)
            tpl, tsl = torch.from_numpy(p_lse).to(dev), torch.from_numpy(s_lse).to(dev)
            out = torch.zeros_like(tp)
            out_lse = torch.zeros(H, T, dtype=torch.float32, device=dev)
            rm.merge_attn_states_cuda(out, out_lse, tp, tpl, ts, tsl)
            torch.cuda.synchronize()
            o_np = out.cpu().numpy() if dt == "f32" else out.view(torch.int16).cpu().numpy().view(np.uint16)
            sub = 8 if dt == "f32" else 4       # every committed file stays under 1 MB
            np.savez_compressed(outdir / f"merge_T{T}H{H}D{D}_{dt}_s{seed}.npz",
                                meta=json.dumps({**meta, "T": T, "H": H, "D": D, "dtype": dt, "seed": seed,
                                                 "subsample": sub}),
                                out=o_np[::sub].copy(), out_lse=out_lse.cpu().numpy())
            print("golden merge", T, H, D, dt)

    rr = load_prebuilt("ref_rope") if want("rope") else None
    if rr is not None:
        for (S, Hd, seed) in ROPE_CASES:
            x = torch.from_numpy(rowwise_inputs(S, Hd, seed)).to(dev)
            out = {}
            for name in ("rope_f32", "rope_f32_v2", "rope_f32x4_pack"):
                if name == "rope_f32_v2" and Hd // 2 > 1024:
                    continue                      # one thread per pair, one block per row (rope.cu:101-112)
                y = torch.zeros_like(x)
                getattr(rr, name)(x, y)
                torch.cuda.synchronize()
                out[name] = y.cpu().numpy()
            np.savez_compressed(outdir / f"rope_{S}x{Hd}_s{seed}.npz",
                                meta=json.dumps({**meta, "seq_len": S, "hidden": Hd, "seed": seed, "flags": "--use_fast_math",
                                                 "subsample": 4}), **{k_: v_[::4].copy() for k_, v_ in out.items()})
            print("golden rope", S, Hd, list(out))

    rn = load_prebuilt("ref_rmsnorm") if want("rmsnorm") else None
    if rn is not None:
        for (R, K, seed) in RMSNORM_CASES:
            x32 = torch.from_numpy(rowwise_inputs(R, K, seed)).to(dev)
            x16 = x32.half()
            g = 1.25
            out = {}
            for name in ("rms_norm_f32", "rms_norm_f32x4"):
                y = torch.zeros_like(x32)
                getattr(rn, name)(x32, y, g)
                torch.cuda.synchronize()
                out[name] = y.cpu().numpy()
            for name in ("rms_norm_f16_f16", "rms_norm_f16x2_f16", "rms_norm_f16x8_f16", "rms_norm_f16x8_pack_f16",
                         "rms_norm_f16x8_f32", "rms_norm_f16x8_pack_f32", "rms_norm_f16_f32"):
                y = torch.zeros_like(x16)
                getattr(rn, name)(x16, y, g)
                torch.cuda.synchronize()
                out[name] = y.cpu().numpy()
            np.savez_compressed(outdir / f"rmsnorm_{R}x{K}_s{seed}.npz",
                                meta=json.dumps({**meta, "rows": R, "K": K, "seed": seed, "g": g, "flags": "--use_fast_math",
                                                 "subsample": 8}), **{k_: v_[::8].copy() for k_, v_ in out.items()})
            print("golden rmsnorm", R, K, list(out))

    rh = load_prebuilt("ref_hgemm") if want("hgemm") else None
    if rh is not None:
        for (M, N, K, seed) in HGEMM_CASES:
            a_np, b_np = hgemm_inputs(M, N, K, seed)
            a = torch.from_numpy(a_np).to(dev)
            b = torch.from_numpy(b_np).to(dev)
            b_col = b.t().contiguous().view(K, N)  # as_col_major (tools/utils.py:151-156)
            out = {}
            staged_nn = ["hgemm_mma_m16n8k16_mma2x4_warp4x4x2_stages_dsmem_swizzle",
                         "hgemm_mma_m16n8k16_mma2x4_warp4x4x2_stages_dsmem",
                         "hgemm_mma_m16n8k16_mma2x4_warp4x4_stages",
                         "hgemm_wmma_m16n16k16_mma4x2_warp2x4_stages"]
            staged_tn = ["hgemm_mma_m16n8k16_mma2x4_warp4x4_stages_dsmem_tn",
                         "hgemm_mma_stages_block_swizzle_tn_cute"]
            for name in staged_nn:
                c = torch.zeros(M, N, dtype=torch.half, device=dev)
                getattr(rh, name)(a, b, c, 2, False, 1)
                torch.cuda.synchronize()
                out[name] = c.cpu().numpy()
            for name in staged_tn:
                if "cute" in name and (N % 256 or M % 128):
                    continue
                c = torch.zeros(M, N, dtype=torch.half, device=dev)
                getattr(rh, name)(a, b_col, c, 2, False, 1)
                torch.cuda.synchronize()
                out[name] = c.cpu().numpy()
            c = torch.zeros(M, N, dtype=torch.half, device=dev)
            rh.hgemm_mma_m16n8k16_mma2x4_warp4x4(a, b, c)
            torch.cuda.synchronize()
            out["hgemm_mma_m16n8k16_mma2x4_warp4x4"] = c.cpu().numpy()
            rh.init_cublas_handle()
            c = torch.zeros(M, N, dtype=torch.half, device=dev)
            rh.hgemm_cublas_tensor_op_nn(a, b, c)
            torch.cuda.synchronize()
            out["hgemm_cublas_tensor_op_nn"] = c.cpu().numpy()
            rh.destroy_cublas_handle()
            sub = 4 if M >= 512 else 1   # keep fixtures small: every 4th row/column of the big case
            out = {k_: v_[::sub, ::sub].copy() for k_, v_ in out.items()}
            np.savez_compressed(outdir / f"hgemm_{M}x{N}x{K}_s{seed}.npz",
                                meta=json.dumps({**meta, "M": M, "N": N, "K": K, "seed": seed,
                                                 "subsample": sub}), **out)
            print("golden hgemm", M, N, K, list(out))

    rf = load_prebuilt("ref_fa") if want("fa") else None
    if rf is not None:
        for (B, H, N, D, seed) in ATTN_CASES:
            q_np, k_np, v_np = attn_inputs(B, H, N, D, seed)
            q, k, v = (torch.from_numpy(x).to(dev) for x in (q_np, k_np, v_np))
            tv = v.transpose(-2, -1).contiguous()
            out = {}
            for name, vv in [("flash_attn_mma_stages_split_q", v),
                             ("flash_attn_mma_stages_split_q_shared_qkv", v),
                             ("flash_attn_mma_stages_split_q_shared_qkv_acc_f32", v),
                             ("flash_attn_mma_stages_split_q_tiling_qkv", v),
                             ("flash_attn_mma_stages_split_q_shared_qkv_swizzle_qkv", tv)]:
                o = torch.zeros_like(q)
                try:
                    getattr(rf, name)(q, k, vv, o, 1)
                    torch.cuda.synchronize()
                    out[name] = o.cpu().numpy()
                except Exception as e:  # headdim outside that op's dispatch set
                    print("skip", name, D, e)
            np.savez_compressed(outdir / f"attn_B{B}H{H}N{N}D{D}_s{seed}.npz",
                                meta=json.dumps({**meta, "B": B, "H": H, "N": N, "D": D, "seed": seed}), **out)
            print("golden attn", B, H, N, D, list(out))

    rp = load_prebuilt("ref_ffpa") if want("ffpa") else None
    if rp is not None:
        for (B, H, N, D, seed) in FFPA_CASES:
            q_np, k_np, v_np = attn_inputs(B, H, N, D, seed)
            q, k, v = (torch.from_numpy(x).to(dev) for x in (q_np, k_np, v_np))
            out = {}
            for name in ["ffpa_mma_acc_f32_L1", "ffpa_mma_acc_f16_L1"]:
                o = torch.zeros_like(q)
                try:
                    getattr(rp, name)(q, k, v, o, 2)
                    torch.cuda.synchronize()
                    out[name] = o.cpu().numpy()
                except Exception as e:
                    print("skip", name, D, e)
            np.savez_compressed(outdir / f"ffpa_B{B}H{H}N{N}D{D}_s{seed}.npz",
                                meta=json.dumps({**meta, "B": B, "H": H, "N": N, "D": D, "seed": seed}), **out)
            print("golden ffpa", B, H, N, D, list(out))


if __name__ == "__main__":
    main(Path(sys.argv[1]) if len(sys.argv) > 1 else HERE.parent / "gpurun_out" / "golden",
         only=tuple(sys.argv[2:]))
