"""Causal attention against full attention at the same shape, and against torch SDPA (is_causal=True).

    python tools/bench_causal.py [--steps 20] [--warmup 3] [--rounds 3]

Prints one JSON line per shape.  Timing practice of bench.py: CUDA events around `steps` back-to-back calls, at
least 3 warm-up calls per variant, two operand sets that rotate call by call (each set larger than the 126 MB L2),
and the card's name and power limit read in the same run.  The causal call, the full (non-causal) call and SDPA run
on the same inputs, alternated inside one process for `rounds` rounds; the median round is reported.

FLOPs: 4 * B * H * D * pairs, pairs = Nq (Nq + 1) / 2 + Nq (Nk - Nq) for the causal mask (query row i sees the keys
j <= i + Nk - Nq) and Nq * Nk without it.  `ratio` = causal time / full time; `gate` is the ratio the causal
schedule is expected to reach at that head dim (DESIGN.md §3, causal paragraph).
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

# (B, H, Nq, Nk, D, gate on causal / full time)
ROWS = [
    (4, 32, 4096, 4096, 128, 0.62),
    (4, 32, 4096, 4096, 64, 0.65),
    (2, 16, 4096, 4096, 256, 0.65),
    (2, 16, 2048, 2048, 512, 0.70),
    (1, 32, 1024, 8192, 128, None),      # chunked prefill: 1024 new queries against an 8192-key cache (reported only)
]


def card_info(torch):
    name = torch.cuda.get_device_name(0)
    limit_w = None
    try:
        import pynvml as nv
        nv.nvmlInit()
        limit_w = nv.nvmlDeviceGetEnforcedPowerLimit(nv.nvmlDeviceGetHandleByIndex(0)) / 1000.0
    except Exception:
        try:
            out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                                 capture_output=True, text=True, timeout=30).stdout.strip()
            limit_w = float(out.splitlines()[0])
        except Exception:
            pass
    return name, limit_w


def time_ms(torch, fn, steps):
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import torch
    import torch.nn.functional as F
    from leetcuda_b200 import flash_attn

    if not torch.cuda.is_available():
        raise SystemExit("bench_causal: needs a CUDA device")
    warmup = max(3, args.warmup)
    name, limit_w = card_info(torch)
    for (B, H, Nq, Nk, D, gate) in ROWS:
        g = torch.Generator(device="cuda").manual_seed(Nq + Nk + D)
        sets = [[torch.randn(B, H, n, D, device="cuda", dtype=torch.half, generator=g) for n in (Nq, Nk, Nk)]
                for _ in range(2)]
        o = torch.empty(B, H, Nq, D, device="cuda", dtype=torch.half)
        if Nq == Nk:
            sdpa_what = "F.scaled_dot_product_attention(is_causal=True)"
            sdpa = lambda i: F.scaled_dot_product_attention(*sets[i % 2], is_causal=True)
        else:   # is_causal=True is top-left aligned for Nq != Nk: give SDPA the bottom-right mask explicitly
            mask = torch.ones(Nq, Nk, dtype=torch.bool, device="cuda").tril(Nk - Nq)
            sdpa_what = "F.scaled_dot_product_attention(attn_mask=ones(Nq, Nk).tril(Nk - Nq))"
            sdpa = lambda i: F.scaled_dot_product_attention(*sets[i % 2], attn_mask=mask)
        variants = {
            "causal": lambda i: flash_attn.fmha_fwd(*sets[i % 2], o, causal=True),
            "full": lambda i: flash_attn.fmha_fwd(*sets[i % 2], o),
            "sdpa_causal": sdpa,
        }
        for fn in variants.values():
            for i in range(warmup):
                fn(i)
        torch.cuda.synchronize()
        ms = {k: [] for k in variants}
        for _ in range(args.rounds):
            for k, fn in variants.items():
                ms[k].append(time_ms(torch, fn, args.steps))
        med = {k: statistics.median(v) for k, v in ms.items()}
        pairs_causal = Nq * (Nq + 1) // 2 + Nq * (Nk - Nq)
        fl_causal = 4.0 * B * H * D * pairs_causal
        fl_full = 4.0 * B * H * D * Nq * Nk
        ratio = med["causal"] / med["full"]
        row = {
            "shape": {"B": B, "H": H, "Nq": Nq, "Nk": Nk, "D": D},
            "causal_ms": med["causal"], "full_ms": med["full"], "sdpa_causal_ms": med["sdpa_causal"],
            "causal_tflops": fl_causal / med["causal"] / 1e9, "full_tflops": fl_full / med["full"] / 1e9,
            "sdpa_causal_tflops": fl_causal / med["sdpa_causal"] / 1e9,
            "ratio_causal_over_full": ratio, "ideal_work_ratio": pairs_causal / (Nq * Nk),
            "gate": gate, "gate_met": (ratio <= gate) if gate is not None else None,
            "rounds_ms": ms, "steps": args.steps, "warmup": warmup,
            "sdpa": sdpa_what, "device": name, "power_limit_w": limit_w,
        }
        print(json.dumps(row), flush=True)
        del sets, o
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
