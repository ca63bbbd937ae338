#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native LeetCUDA hot paths.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Primary line (BASELINE.json configs[1]): HGEMM fp16 M=N=K=8192 through the reference-facing op
`hgemm_mma_m16n8k16_mma2x4_warp4x4x2_stages_dsmem_swizzle` (NN layout).  One "step" = one GEMM
launch.  The same JSON line carries the other two single-GPU BASELINE configs:

* "secondary"  FA-2 forward B4 H32 N4096 D128 (configs[2]) through `flash_attn_mma_stages_split_q_shared_qkv`
* "config4"    FFPA large-D forward B2 H16 N2048 D512 (configs[3]) through `ffpa_mma_acc_f32_L1`

each with its own roofline, end-to-end figure (host buffers through the C-ABI *_host entry) and
vendor / CPU numbers from the same run, plus "next_rows" (SURVEY §8f: TF32 SGEMM, merge_attn_states,
the fused rope / rms-norm steps around attention).

* value      whole-job TFLOPS, inputs resident in HBM, CUDA-event timed, max over ranks
* e2e        same metric through the public host-buffer call: H2D of the inputs and D2H of the
             result inside the timed region, every step
* roofline   tensor-bound: algorithmic FLOPs / measured kernel time vs MEASURED_PEAKS.json
* cpu_baseline  torch.matmul / SDPA on the host cores (north_star's CPU path), bounded sample

N > 1 (torchrun, one rank per GPU): BASELINE configs[4], HGEMM 16384^3 row-sharded over the ranks
(strong scaling, SURVEY §8e) — rank r owns 16384/N rows of A and C, B replicated, and every rank
ends with the full [16384, 16384] C: the GEMM epilogue pushes each finished box of C to all peers
with TMA stores over NVLink (fused all-gather, leetcuda_b200/dist.py), closed by a symmetric-memory
barrier.  The same run also times the stated baseline, GEMM + ncclAllGather (`nccl_baseline`).
B200_DIST_TRANSPORT=nccl makes that baseline the headline transport.  The N = 1 line carries the
single-GPU 16384^3 figure (`strong_scaling_n1`) the N > 1 values are to be compared with.

--impl reference times the reference's CPU path (torch.matmul on the host cores, all threads) on
the same workload as this arm at the same N; rank 0 only.

--dump-outputs DIR (N = 1) writes, after the timed steps, what the last timed step of the HGEMM line and of
each attention row returned to its caller: a fixed, seeded sample of rows as float32 DIR/<name>.npy (44 MB in
all).  The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

S = 8192                       # HGEMM M=N=K at N=1 (BASELINE configs[1])
S16 = 16384                    # HGEMM M=N=K at N>1 (BASELINE configs[4], row-sharded)
FA = (4, 32, 4096, 128)        # B, H, N, D   (BASELINE configs[2])
FF = (2, 16, 2048, 512)        # B, H, N, D   (BASELINE configs[3])
OP = "hgemm_mma_m16n8k16_mma2x4_warp4x4x2_stages_dsmem_swizzle"


def line_config(world: int, transport: str) -> dict:
    """`config` of the JSON line — identical in both arms (--impl ours / reference)."""
    if world == 1:
        return {"workload": "hgemm_nn_8192x8192x8192_fp16", "op": OP, "accumulate": "fp32",
                "parallelism": "single GPU",
                "l2": "operands rotate over 3 sets, each > 126 MB L2: no flush needed"}
    return {"workload": f"hgemm_nn_16384x16384x16384_fp16_rowsharded_x{world}_allgatherC", "op": OP,
            "accumulate": "fp32", "parallelism": f"row-shard x{world}, transport {transport}",
            "l2": "operands rotate over 2 sets, each > 126 MB L2: no flush needed"}


def line_metric(world: int) -> str:
    return "HGEMM fp16 TFLOPS @8192^3" if world == 1 else "HGEMM fp16 TFLOPS @16384^3 row-sharded, all-gather of C"


def measured_peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        try:
            d = json.loads(f.read_text())
            return float(d["bf16_tflops"]), float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst)"
        except Exception:
            pass
    return 1590.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clock / throttle reasons with NVML while the timed region runs (NVML is
    initialised before the region starts; the thread only reads)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None
        self._nv = None
        self._h = None
        try:
            import pynvml as nv
            nv.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = index
            try:
                ids = [int(x) for x in vis.split(",") if x.strip() != ""]
                if ids:
                    phys = ids[index]
            except ValueError:
                pass
            self._h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)
            self._nv = nv
        except Exception as e:  # NVML missing: record that rather than fail the bench
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def _sample(self):
        nv = self._nv
        self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        for bit, nm in self.REASONS.items():
            if r & bit:
                self.reasons.add(nm)

    def _run(self):
        while not self._stop.is_set():
            try:
                self._sample()
            except Exception as e:
                self.reasons.add(f"nvml_error:{type(e).__name__}")
                return
            time.sleep(0.0005)

    def __enter__(self):
        if self._nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=2)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def settle(seconds: float = 0.75):
    """Untimed pause between rows: the board's power controller averages over a window, and a row that starts right
    behind a burst of tensor-bound GEMMs was seen running at ~60 % (sw_power_cap, SM clock well below max) for its whole
    18 ms timed region.  Every row therefore starts from an idle chip like the primary line does, and reports its own
    clocks."""
    import torch
    torch.cuda.synchronize()
    time.sleep(seconds)


def sample_rows(t, n: int, seed: int):
    """A fixed, seeded sample of n rows of t (viewed as [rows, last dim]), as float32 on the host."""
    import numpy as np
    import torch
    flat = t.reshape(-1, t.shape[-1])
    idx = np.sort(np.random.default_rng(seed).choice(flat.shape[0], min(n, flat.shape[0]), replace=False))
    return flat[torch.from_numpy(idx).to(t.device)].float().cpu().numpy()


def cuda_time_ms(fn, steps, sync):
    import torch
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    sync()
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    sync()
    return e0.elapsed_time(e1)


# ------------------------------------------------------------------------------------------------
# reference arm: north_star's CPU path, same workload as this arm at the same N
# ------------------------------------------------------------------------------------------------
def run_reference(args):
    """torch.matmul on fp16 host tensors over the WHOLE problem of the `ours` arm at this N
    (8192^3 at N=1, 16384^3 at N>1) — every step is the full GEMM.  Only when K steps of the full
    problem would not end within a few minutes is a step cut down to a row slab of A (stated in
    cpu_baseline.sample); the per-flop rate of a slab is lower than that of the whole problem, so the
    full problem is the default."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    size = S if world == 1 else S16
    torch.manual_seed(0)
    a = torch.randn(size, size, dtype=torch.half)
    b = torch.randn(size, size, dtype=torch.half)
    cores = torch.get_num_threads()
    # one untimed probe on a 1024-row slab to size the steps (also first-touch of a and b)
    t0 = time.perf_counter()
    torch.matmul(a[:1024], b)
    est_full = (time.perf_counter() - t0) * size / 1024
    budget = 240.0
    warm = max(1, min(args.warmup, 2))
    rows = size
    if est_full * (args.steps + warm) > budget:
        rows = int(size * budget / (est_full * (args.steps + warm))) // 1024 * 1024
        rows = max(1024, min(size, rows))
    av = a[:rows]
    for _ in range(warm):
        torch.matmul(av, b)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        torch.matmul(av, b)
    dt = (time.perf_counter() - t0) / args.steps
    tflops = 2.0 * rows * size * size / dt / 1e12
    sample = (f"torch.matmul fp16 on {cores} host threads, the whole {size}^3 problem per step" if rows == size else
              f"torch.matmul fp16 on {cores} host threads, a {rows}-row slab of the {size}^3 problem per step "
              f"(full problem ~{est_full:.1f} s/step)")
    line = {
        "impl": "reference", "metric": line_metric(world), "value": tflops, "unit": "TFLOPS",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16",
        "data": "synthetic",
        "config": line_config(world, os.environ.get("B200_DIST_TRANSPORT", "fused")),
        "cpu_baseline": {"value": tflops, "unit": "TFLOPS", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": tflops, "unit": "TFLOPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baselines():
    """torch.matmul / SDPA on the host cores, bounded samples (rank 0, N=1 only)."""
    import torch
    import torch.nn.functional as F
    cores = torch.get_num_threads()
    torch.manual_seed(0)
    a = torch.randn(S, S, dtype=torch.half)
    b = torch.randn(S, S, dtype=torch.half)
    torch.matmul(a[:512], b)
    t0 = time.perf_counter()
    torch.matmul(a, b)                       # the whole 8192^3 problem, once (about a second)
    dt = time.perf_counter() - t0
    gemm = {"value": 2.0 * S * S * S / dt / 1e12, "unit": "TFLOPS", "cores": cores, "kind": "reference",
            "sample": f"torch.matmul fp16 on host cores, the whole 8192^3 problem once ({dt:.1f} s)"}

    def sdpa_sample(B, H, N, D, max_reps, label):
        q, k, v = (torch.randn(B, H, N, D, dtype=torch.half) for _ in range(3))
        F.scaled_dot_product_attention(q[:, :1], k[:, :1], v[:, :1])
        reps, dt, t0 = 0, 0.0, time.perf_counter()
        while reps < max_reps and dt < 10.0:
            F.scaled_dot_product_attention(q, k, v)
            reps += 1
            dt = time.perf_counter() - t0
        return {"value": 4.0 * reps * B * H * N * N * D / dt / 1e12, "unit": "TFLOPS", "cores": cores, "kind": "reference",
                "sample": f"F.scaled_dot_product_attention fp16 on host cores, {reps} x (B{B} H{H} N{N} D{D}) of {label} ({dt:.1f} s)"}

    attn = sdpa_sample(1, 8, FA[2], FA[3], 16, "B4 H32")      # 16 x (B1 H8) = the full problem
    ffpa = sdpa_sample(1, 4, FF[2], FF[3], 8, "B2 H16")       # 8 x (B1 H4) = the full problem
    return gemm, attn, ffpa


def attention_row(torch, dev, world, rank, args, sync, shape, op, op_name, metric, kernel, peak_tf, peak_src, traffic_file,
                  host_op, want_e2e, dumps=None, dump_name=None):
    """One attention config: device-timed value, roofline, vendor SDPA, e2e through the host-buffer entry.
    With `dumps`, a row sample of the output of the last timed step goes to dumps[dump_name]."""
    import torch.distributed as dist
    import torch.nn.functional as F
    from leetcuda_b200 import _capi
    B, H, N, D = shape
    assert (B * H) % world == 0
    Bw, Hw = (B, H) if world == 1 else (1, B * H // world)      # (batch x head) units are independent
    torch.manual_seed(4321 + rank)
    nsets = 2 if 8 * Bw * Hw * N * D > 200e6 else 3              # rotate sets: > 126 MB L2 in flight
    sets = [[torch.randn(Bw, Hw, N, D, device=dev, dtype=torch.half) for _ in range(3)] for _ in range(nsets)]
    outs = [torch.empty(Bw, Hw, N, D, device=dev, dtype=torch.half) for _ in range(nsets)]

    def fstep(i):
        q, k, v = sets[i % nsets]
        op(q, k, v, outs[i % nsets], 2)

    settle()
    for i in range(args.warmup):
        fstep(i)
    sync()
    l1 = _capi.launch_count()
    with ClockSampler(dev.index) as row_clk:
        fms = cuda_time_ms(fstep, args.steps, sync)
    launches = _capi.launch_count() - l1
    if dumps is not None:
        dumps[dump_name] = sample_rows(outs[(args.steps - 1) % nsets], (1 << 20) // D, seed=D)   # 4 MB
    tf = torch.tensor([fms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tf, op=dist.ReduceOp.MAX)
    fms_step = tf.item() / args.steps
    fl = 4.0 * Bw * Hw * N * N * D * world
    fval = fl / (fms_step * 1e-3) / 1e12
    row = {
        "metric": metric, "value": fval, "unit": "TFLOPS", "ms_per_step": fms_step,
        "clocks": row_clk.summary(),
        "config": {"workload": f"attn_fwd_B{B}_H{H}_N{N}_D{D}_fp16", "op": op_name,
                   "sharding": "none" if world == 1 else f"(batch x head) split {world}-way, no collective",
                   "l2": f"{nsets} operand sets rotate ({8 * Bw * Hw * N * D / 1e6:.0f} MB each)"},
        "roofline": {"bound": "tensor", "achieved": fval / world, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": fval / world / peak_tf, "traffic": None, "peak_source": peak_src,
                     "kernel": kernel, "kernel_ms": fms_step, "algorithmic_flops": 4.0 * Bw * Hw * N * N * D,
                     "algorithmic_bytes": 8 * Bw * Hw * N * D},
    }
    prof = ROOT / "profiles" / traffic_file
    if prof.exists():
        try:
            row["roofline"]["traffic"] = json.loads(prof.read_text()).get("dram_bytes_per_launch")
        except Exception:
            pass
    if world == 1:
        q, k, v = sets[0]
        for _ in range(3):
            F.scaled_dot_product_attention(q, k, v)
        sms = cuda_time_ms(lambda i: F.scaled_dot_product_attention(*sets[i % nsets]), args.steps,
                           lambda: torch.cuda.synchronize()) / args.steps
        row["vendor"] = {"impl": "F.scaled_dot_product_attention (default backend)", "tflops": fl / (sms * 1e-3) / 1e12}
    if want_e2e and world == 1:
        # the C-ABI host-buffer entry (b200_fmha_fwd_f16_host): pinned q,k,v -> HBM, the kernel and the D2H of
        # o inside the call, pipelined over (batch x head) chunks; it returns when o is complete on the host
        hq, hk, hv = (torch.randn(B, H, N, D, dtype=torch.half).pin_memory() for _ in range(3))
        ho = torch.empty(B, H, N, D, dtype=torch.half).pin_memory()
        for _ in range(2):
            host_op(hq, hk, hv, ho)
        e_steps = max(3, min(args.steps, 10))
        e_ms = cuda_time_ms(lambda i: host_op(hq, hk, hv, ho), e_steps, lambda: torch.cuda.synchronize()) / e_steps
        row["e2e"] = {"value": fl / (e_ms * 1e-3) / 1e12, "unit": "TFLOPS", "h2d_bytes_per_step": 3 * B * H * N * D * 2,
                      "d2h_bytes_per_step": B * H * N * D * 2, "steps": e_steps,
                      "note": "b200_fmha_fwd_f16_host: pinned host q,k,v -> HBM, kernel, o -> pinned host inside the call, "
                              "pipelined over (batch x head) chunks (PCIe-bound)"}
        del hq, hk, hv, ho
    del sets, outs
    torch.cuda.empty_cache()
    return row, launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-secondary", action="store_true", help="skip the attention metrics and the next rows")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed row sample of what the last timed step of each GPU row computed to DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the GPU rows' outputs; --impl reference has none")

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if args.dump_outputs:
            raise SystemExit("--dump-outputs runs on one GPU")
        dist.init_process_group("nccl", device_id=dev)
    dumps = {} if args.dump_outputs else None

    from leetcuda_b200 import _capi, ffpa_attn, flash_attn, hgemm
    from leetcuda_b200 import dist as bdist

    peak_tf, peak_hbm, peak_src = measured_peaks()

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ------------------------------------------------------------------ HGEMM (primary)
    # N = 1: BASELINE configs[1], 8192^3.  N > 1: BASELINE configs[4], 16384^3 row-sharded over the
    # ranks (strong scaling): rank r owns rows [r*Mr, (r+1)*Mr) of A and C, B is replicated.
    if world == 1:
        Mr, Nn, Kk = S, S, S
    else:
        assert S16 % world == 0
        Mr, Nn, Kk = S16 // world, S16, S16
    torch.manual_seed(1234 + rank)
    NSETS = 3 if world == 1 else 2  # rotate operand sets (each >> 126 MB L2): no L2-resident re-reads
    As = [torch.randn(Mr, Kk, device=dev, dtype=torch.half) for _ in range(NSETS)]
    if world > 1:
        torch.manual_seed(99)  # B is replicated: same values on every rank
    Bs = [torch.randn(Kk, Nn, device=dev, dtype=torch.half) for _ in range(NSETS)]
    op = getattr(hgemm, OP)
    transport = os.environ.get("B200_DIST_TRANSPORT", "fused")
    sharded = bdist.RowShardedHgemm(Mr, Nn, Kk, world, rank, dev, transport=transport) if world > 1 else None
    Cs = [torch.empty(Mr, Nn, device=dev, dtype=torch.half) for _ in range(NSETS)] if world == 1 else None

    def step(i):
        j = i % NSETS
        if world == 1:
            op(As[j], Bs[j], Cs[j], 2, True, 2048)
        else:
            sharded(As[j], Bs[j])

    # N > 1, fused transport: the epilogue can push each finished box of C to every peer mapping (one TMA store per
    # peer) or once through the NVLS multicast mapping.  Which is faster depends on N (egress bytes: (N-1)x vs 1x the
    # shard); pick by a short untimed trial, all ranks agreeing on the max-over-ranks time.  B200_FUSED_EPILOGUE pins it.
    epilogue = os.environ.get("B200_FUSED_EPILOGUE", "")
    if world > 1 and transport == "fused" and not epilogue:
        trial = {}
        for mode in ("tma", "mc"):
            os.environ["B200_FUSED_EPILOGUE"] = mode
            try:
                for i in range(3):
                    step(i)
                sync()
                tms = torch.tensor([cuda_time_ms(step, 5, sync)], device=dev, dtype=torch.float64)
                dist.all_reduce(tms, op=dist.ReduceOp.MAX)
                trial[mode] = tms.item() / 5
            except Exception:
                trial[mode] = float("inf")
        epilogue = min(trial, key=trial.get)
        os.environ["B200_FUSED_EPILOGUE"] = epilogue
    elif world > 1 and transport == "fused":
        trial = {}

    for i in range(args.warmup):
        step(i)
    sync()
    l0 = _capi.launch_count()
    with ClockSampler(local) as clk:
        ms = cuda_time_ms(step, args.steps, sync)
    launches = _capi.launch_count() - l0
    if dumps is not None:   # before the roofline and cuBLAS legs below write into Cs again
        dumps["hgemm_c"] = sample_rows(Cs[(args.steps - 1) % NSETS], 1024, seed=0)   # 32 MB
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = t.item() / args.steps
    flops_rank = 2.0 * Mr * Nn * Kk
    flops_step = flops_rank * world
    value = flops_step / (ms_step * 1e-3) / 1e12

    # kernel-only duration for the roofline (compute kernel alone, this rank)
    def kern(i):
        j = i % NSETS
        if world == 1:
            op(As[j], Bs[j], Cs[j], 2, True, 2048)
        else:
            sharded.compute_only(As[j], Bs[j])
    k_ms = cuda_time_ms(kern, args.steps, lambda: torch.cuda.synchronize()) / args.steps
    tk = torch.tensor([k_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tk, op=dist.ReduceOp.MAX)
        k_ms = tk.item()
    ach = flops_rank / (k_ms * 1e-3) / 1e12
    roofline = {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": ach / peak_tf, "traffic": None, "peak_source": peak_src,
                "kernel": "hgemm_tcgen05_kernel<cta_group=2, NN>", "kernel_ms": k_ms,
                "algorithmic_flops": flops_rank, "algorithmic_bytes": 2 * (Mr * Kk + Kk * Nn + Mr * Nn)}
    if world > 1:
        gather = (world - 1) * Mr * Nn * 2
        roofline["fused_step"] = {
            "nvlink_bytes_in_per_rank": gather, "nvlink_peak_gbs": 770.0,
            "target_ms": max(flops_rank / (peak_tf * 1e12), gather / 770e9) * 1e3,
            "achieved_ms": ms_step, "compute_only_ms": k_ms,
            "epilogue": epilogue if transport == "fused" else None, "epilogue_trial_ms": trial if transport == "fused" else None,
            "note": "target = slower of (FLOPs / measured GEMM peak) and (bytes received over NVLink / 770 GB/s)"}
        # the stated baseline in the same run: GEMM into the rank's slice, then one ncclAllGather of C
        try:
            base = sharded if transport == "nccl" else bdist.RowShardedHgemm(Mr, Nn, Kk, world, rank, dev, transport="nccl")
            for i in range(3):
                base(As[i % NSETS], Bs[i % NSETS])
            sync()
            b_steps = max(3, min(args.steps, 10))
            b_ms = cuda_time_ms(lambda i: base(As[i % NSETS], Bs[i % NSETS]), b_steps, sync)
            tb = torch.tensor([b_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tb, op=dist.ReduceOp.MAX)
            roofline["fused_step"]["nccl_baseline_ms"] = tb.item() / b_steps
            roofline["fused_step"]["nccl_baseline_tflops"] = flops_step / (tb.item() / b_steps * 1e-3) / 1e12
            if base is not sharded:
                del base
        except Exception as e:
            roofline["fused_step"]["nccl_baseline_error"] = f"{type(e).__name__}: {e}"
    prof = ROOT / "profiles" / "hgemm_traffic.json"
    if prof.exists() and world == 1:
        try:
            roofline["traffic"] = json.loads(prof.read_text()).get("dram_bytes_per_launch")
        except Exception:
            pass

    # ------------------------------------------------------------------ attention (secondary) and FFPA large-D (config4)
    # (the three BASELINE single-GPU configs are measured back to back, before the long-running legs — host-buffer
    #  e2e, the 16384^3 strong-scaling point, the next rows — heat the chip; every row samples its own clocks)
    secondary = None
    config4 = None
    attn_d64 = None
    if not args.no_secondary:
        secondary, nl = attention_row(
            torch, dev, world, rank, args, sync, FA, flash_attn.flash_attn_mma_stages_split_q_shared_qkv,
            "flash_attn_mma_stages_split_q_shared_qkv", "FA-2 fp16 TFLOPS @B4H32N4096D128 (matmul FLOPs 4BHN^2D)",
            "attn_fwd_kernel<128> (two query tiles per CTA)", peak_tf, peak_src, "attn_traffic.json",
            flash_attn.fmha_host, True, dumps, "attn_o_d128")
        launches += nl
        try:
            config4, nl = attention_row(
                torch, dev, world, rank, args, sync, FF, ffpa_attn.ffpa_mma_acc_f32_L1,
                "ffpa_mma_acc_f32_L1", "FFPA fp16 TFLOPS @B2H16N2048D512 (matmul FLOPs 4BHN^2D)",
                "attn_pair_fwd_kernel (one query tile per CTA pair, cta_group::2)", peak_tf, peak_src,
                "attn_pair_traffic.json", flash_attn.fmha_host, True, dumps, "ffpa_o_d512")
            launches += nl
        except Exception as e:
            config4 = {"error": f"{type(e).__name__}: {e}"}
        # head dim 64 of the same op (the reference's default sweep covers D = 64, flash_attn_mma.py:497-502): its own roofline row
        try:
            attn_d64, nl = attention_row(
                torch, dev, world, rank, args, sync, (FA[0], FA[1], FA[2], 64), flash_attn.flash_attn_mma_stages_split_q_shared_qkv,
                "flash_attn_mma_stages_split_q_shared_qkv", "FA-2 fp16 TFLOPS @B4H32N4096D64 (matmul FLOPs 4BHN^2D)",
                "attn_fwd_kernel<64> (two query tiles per CTA, persistent grid)", peak_tf, peak_src, "attn_d64_traffic.json",
                flash_attn.fmha_host, False, dumps, "attn_o_d64")
            launches += nl
        except Exception as e:
            attn_d64 = {"error": f"{type(e).__name__}: {e}"}

    # ------------------------------------------------------------------ e2e (host buffers)
    ha = torch.randn(Mr, Kk, dtype=torch.half).pin_memory()
    hb = torch.randn(Kk, Nn, dtype=torch.half).pin_memory()
    hc = torch.empty(Mr, Nn, dtype=torch.half).pin_memory()
    da, db = As[0], Bs[0]

    def e2e_step(i):
        if world == 1:
            # the C-ABI host-buffer entry (b200_hgemm_f16_host): H2D of a and b, the GEMM and the D2H of
            # c all happen inside this call, pipelined over row panels; it returns when c is complete
            hgemm.hgemm_host(ha, hb, hc)
            return
        da.copy_(ha, non_blocking=True)
        db.copy_(hb, non_blocking=True)
        c_full = sharded(da, db)
        hc.copy_(c_full[rank * Mr:(rank + 1) * Mr], non_blocking=True)

    for i in range(2):
        e2e_step(i)
    e_steps = max(3, min(args.steps, 10 if world == 1 else 4))
    e_ms = cuda_time_ms(e2e_step, e_steps, sync)
    te = torch.tensor([e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = flops_step / (te.item() / e_steps * 1e-3) / 1e12
    e2e = {"value": e2e_val, "unit": "TFLOPS", "h2d_bytes_per_step": (Mr * Kk + Kk * Nn) * 2,
           "d2h_bytes_per_step": Mr * Nn * 2, "steps": e_steps,
           "note": ("b200_hgemm_f16_host: pinned host a,b -> HBM, GEMM, c -> pinned host inside the call, "
                    "pipelined over row and column panels (PCIe-bound)") if world == 1 else
                   "per rank: pinned host a,b -> HBM, op, this rank's c rows -> pinned host, every step (PCIe-bound)"}

    # ------------------------------------------------------------------ cuBLAS side by side
    cub = None
    if world == 1:
        for i in range(3):   # cuBLAS handle creation / heuristics stay outside the timed region
            torch.matmul(As[i % NSETS], Bs[i % NSETS], out=Cs[i % NSETS])
        cms = cuda_time_ms(lambda i: torch.matmul(As[i % NSETS], Bs[i % NSETS], out=Cs[i % NSETS]),
                           args.steps, lambda: torch.cuda.synchronize()) / args.steps
        cub = {"impl": "cuBLAS via torch.matmul (fp16, NN)", "tflops": flops_rank / (cms * 1e-3) / 1e12}
    del As, Bs, Cs, ha, hb, hc, sharded
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------ the N=1 point of the strong-scaling curve
    strong_n1 = None
    if world == 1 and not args.no_secondary:
        try:
            a16 = [torch.randn(S16, S16, device=dev, dtype=torch.half) for _ in range(2)]
            b16 = [torch.randn(S16, S16, device=dev, dtype=torch.half) for _ in range(2)]
            c16 = torch.empty(S16, S16, device=dev, dtype=torch.half)
            for i in range(3):
                op(a16[i % 2], b16[i % 2], c16, 2, True, 2048)
            n16 = max(3, min(args.steps, 10))
            m16 = cuda_time_ms(lambda i: op(a16[i % 2], b16[i % 2], c16, 2, True, 2048), n16,
                               lambda: torch.cuda.synchronize()) / n16
            strong_n1 = {"workload": "hgemm_nn_16384x16384x16384_fp16 on one GPU (the N=1 point of BASELINE configs[4])",
                         "ms_per_step": m16, "tflops": 2.0 * S16 ** 3 / (m16 * 1e-3) / 1e12, "steps": n16}
            del a16, b16, c16
            torch.cuda.empty_cache()
        except Exception as e:
            strong_n1 = {"error": f"{type(e).__name__}: {e}"}

    # ------------------------------------------------------------------ SURVEY §8f rows
    next_rows = None
    if world == 1 and not args.no_secondary:
        next_rows = []
        for fn in (row_sgemm_tf32, row_merge, row_rope_rmsnorm):
            try:
                got = fn(torch, dev, args, peak_tf, peak_hbm, peak_src)
                next_rows.extend(got if isinstance(got, list) else [got])
            except Exception as e:   # the headline line must survive a failure of the extra rows
                next_rows.append({"row": fn.__name__, "error": f"{type(e).__name__}: {e}"})
            torch.cuda.empty_cache()

    # ------------------------------------------------------------------ CPU baseline (rank 0, N=1)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu, cpu_a, cpu_f = cpu_baselines()
        if secondary is not None:
            secondary["cpu_baseline"] = cpu_a
        if isinstance(config4, dict) and "error" not in config4:
            config4["cpu_baseline"] = cpu_f

    if rank == 0:
        line = {
            "metric": line_metric(world), "value": value, "unit": "TFLOPS", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": line_config(world, transport),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": clk.summary(), "vendor": cub, "secondary": secondary, "config4": config4, "secondary_d64": attn_d64,
            "strong_scaling_n1": strong_n1, "next_rows": next_rows,
            "scaling_note": ("N=1 runs BASELINE configs[1] (8192^3); N>1 runs configs[4] (16384^3 split over the ranks, "
                             "total work fixed); strong_scaling_n1 on the N=1 line is the one-GPU 16384^3 figure"),
        }
        print(json.dumps(line), flush=True)
    if dumps is not None:
        import numpy as np
        out = Path(args.dump_outputs)
        out.mkdir(parents=True, exist_ok=True)
        for name, arr in dumps.items():
            np.save(out / f"{name}.npy", arr)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# SURVEY §8f rows (N = 1 only)
# ------------------------------------------------------------------------------------------------
def row_sgemm_tf32(torch, dev, args, peak_tf, peak_hbm, peak_src):
    """§8f-2: SGEMM through TF32 tensor cores."""
    from leetcuda_b200 import sgemm as SG
    Sg = 8192
    sa = [torch.randn(Sg, Sg, device=dev) for _ in range(2)]    # 2 sets x 3 x 256 MB > L2
    sb = [torch.randn(Sg, Sg, device=dev) for _ in range(2)]
    sc = [torch.empty(Sg, Sg, device=dev) for _ in range(2)]
    gfl = 2.0 * Sg ** 3
    for i in range(max(args.warmup, 3)):
        SG.sgemm_wmma_m16n16k8_mma4x2_warp2x4_stages(sa[i % 2], sb[i % 2], sc[i % 2], 2, False, 1)
    # the reference op: TF32 rounding of a and b in place + GEMM (3 launches of ours per step)
    op_ms = cuda_time_ms(lambda i: SG.sgemm_wmma_m16n16k8_mma4x2_warp2x4_stages(
        sa[i % 2], sb[i % 2], sc[i % 2], 2, False, 1), args.steps, lambda: torch.cuda.synchronize()) / args.steps
    # the GEMM kernel alone (operands already TF32-exact after the calls above)
    k_ms = cuda_time_ms(lambda i: SG.sgemm_tf32(sa[i % 2], sb[i % 2], sc[i % 2], round_inputs=False),
                        args.steps, lambda: torch.cuda.synchronize()) / args.steps
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    for _ in range(3):
        torch.matmul(sa[0], sb[0], out=sc[0])
    # vendor TF32: sustained (back to back) and burst (best single launch of 10, the way the bf16 burst peak was taken)
    v_ms = cuda_time_ms(lambda i: torch.matmul(sa[i % 2], sb[i % 2], out=sc[i % 2]), args.steps,
                        lambda: torch.cuda.synchronize()) / args.steps
    burst = min(cuda_time_ms(lambda i: torch.matmul(sa[0], sb[0], out=sc[0]), 1, lambda: torch.cuda.synchronize())
                for _ in range(10))
    torch.backends.cuda.matmul.allow_tf32 = prev
    ach = gfl / (k_ms * 1e-3) / 1e12
    tf32_nominal = 1125.0     # half the dense bf16 figure of B200_PROFILING.md (2250): a NOMINAL denominator
    return {
        "metric": "SGEMM TF32 TFLOPS @8192^3 (reference op: round a,b to TF32 in place + GEMM)",
        "value": gfl / (op_ms * 1e-3) / 1e12, "unit": "TFLOPS", "ms_per_step": op_ms,
        "config": {"workload": "sgemm_nn_8192x8192x8192_fp32_tf32", "op": "sgemm_wmma_m16n16k8_mma4x2_warp2x4_stages"},
        "roofline": {"bound": "tensor", "achieved": ach, "peak": tf32_nominal, "unit": "TFLOP/s",
                     "frac": ach / tf32_nominal, "traffic": None,
                     "peak_source": "NOMINAL dense TF32 (datasheet bf16 / 2; MEASURED_PEAKS.json has no TF32 entry) — "
                                    "see measured_vendor_burst for the in-run cuBLAS TF32 figure",
                     "measured_vendor_burst": gfl / (burst * 1e-3) / 1e12,
                     "frac_of_measured_vendor_burst": ach / (gfl / (burst * 1e-3) / 1e12),
                     "kernel": "hgemm_tcgen05_macro_kernel<NN, tf32> (512x256 per CTA pair)", "kernel_ms": k_ms,
                     "algorithmic_bytes": 3 * 4 * Sg * Sg},
        "vendor": {"impl": "cuBLAS TF32 via torch.matmul (allow_tf32), back to back", "tflops": gfl / (v_ms * 1e-3) / 1e12},
    }


def row_merge(torch, dev, args, peak_tf, peak_hbm, peak_src):
    """§8f-3: merge_attn_states, HBM-bound (3*D*2 + 12 bytes per token-head at fp16)."""
    from leetcuda_b200 import merge_attn_states as MA
    Tm, Hm, Dm = 131072, 16, 128          # 3 x 512 MB per set: far beyond L2
    mp = [torch.randn(Tm, Hm, Dm, device=dev, dtype=torch.half) for _ in range(2)]
    ms = [torch.randn(Tm, Hm, Dm, device=dev, dtype=torch.half) for _ in range(2)]
    mo = [torch.empty(Tm, Hm, Dm, device=dev, dtype=torch.half) for _ in range(2)]
    mpl = torch.randn(Hm, Tm, device=dev)
    msl = torch.randn(Hm, Tm, device=dev)
    mol = torch.empty(Hm, Tm, device=dev)
    for i in range(3):
        MA.merge_attn_states_cuda(mo[i % 2], mp[i % 2], mpl, ms[i % 2], msl, mol)
    m_ms = cuda_time_ms(lambda i: MA.merge_attn_states_cuda(mo[i % 2], mp[i % 2], mpl, ms[i % 2], msl, mol),
                        args.steps, lambda: torch.cuda.synchronize()) / args.steps
    m_bytes = Tm * Hm * (3 * Dm * 2 + 12)
    m_gbs = m_bytes / (m_ms * 1e-3) / 1e9
    row = {
        "metric": "merge_attn_states GB/s @T131072 H16 D128 fp16 (algorithmic bytes)", "value": m_gbs, "unit": "GB/s",
        "ms_per_step": m_ms,
        "config": {"workload": "merge_attn_states_T131072_H16_D128_fp16", "op": "merge_attn_states_cuda"},
        "roofline": {"bound": "hbm", "achieved": m_gbs, "peak": peak_hbm, "unit": "GB/s", "frac": m_gbs / peak_hbm,
                     "traffic": None, "peak_source": peak_src, "kernel": "merge_attn_states_kernel<half>",
                     "kernel_ms": m_ms, "algorithmic_bytes": m_bytes},
    }
    mprof = ROOT / "profiles" / "merge_traffic.json"
    if mprof.exists():
        try:
            row["roofline"]["traffic"] = json.loads(mprof.read_text()).get("dram_bytes_per_launch")
        except Exception:
            pass
    return row


def row_rope_rmsnorm(torch, dev, args, peak_tf, peak_hbm, peak_src):
    """§8f-4: the element-wise steps around attention (rope on q/k, rms-norm), HBM-bound."""
    from leetcuda_b200 import fused_ops as FO
    return FO.bench_rows(torch, dev, args.steps, peak_hbm, peak_src, cuda_time_ms)


if __name__ == "__main__":
    main()
