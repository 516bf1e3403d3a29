"""FP8 mode against bf16 and int8 codes: the config-2 denoise step of the video DiT and its seven GEMM shapes.

Steps: ltx_denoise_step at bench.py's config 2 -- 48 blocks, D = 4096, 768x512x25 video (N = 1536 tokens), S = 1024 text tokens,
seeded random-init weights (init_random_weights(1, ...)) -- in two forms: "plain" (no guidance: one B = 1 forward, the step
bench.py times) and "guided" (cfg scale 2 with a negative prompt: both passes as one batched B = 2 forward).  Three contexts hold
the same weights as bf16 (precision 16), FP8 (precision 8) and int8 codes (finalize_weights(8, 64)); after warm-up, --rounds
rounds time --steps steps of each mode and form in turn (CUDA events on the context's stream, and a host clock around a device
synchronise), then one profiled step per mode and form in a separate pass gives the per-class split (ltx_get_profile).

GEMMs: the seven Linears of a block at M = 1536 (one pass) and 3072 (the batched CFG pass), bf16 pair kernel (ltx_op_gemm)
against the FP8 pair kernel (ltx_op_gemm_fp8, quantiser not included), CUDA events over --reps launches after warm-up.  The
operands stay resident in the 126 MB L2 between launches where they fit (the D x D weights), as they do inside a step.

Prints the GPU name and power limit (nvidia-smi, same process) beside the numbers.

Usage (GPU box): python tools/fp8_bench.py [--layers 48] [--steps 3] [--rounds 3] [--warmup 2] [--reps 20] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ltx_video_swift_mlx_b200  # noqa: E402,F401
from ltx_video_swift_mlx_b200.context import LtxContext, LTXTransformerConfig  # noqa: E402

F, H, W, S, C, CAP, D = 4, 16, 24, 1024, 128, 3840, 4096
MODES = (("bf16", 16, 16), ("fp8", 8, 16), ("int8", 16, 8))   # name, precision, quant_bits
# name, N, K, epilogue mode of ltx_op_gemm (0 bf16, 1 GELU, 3 fp32 -- the gate * residual GEMMs write fp32)
GEMMS = (("attn1_qkv", 3 * D, D, 0), ("attn1_out", D, D, 3), ("attn2_q", D, D, 0), ("attn2_text_kv", D, D, 0),
         ("attn2_out", D, D, 3), ("ff_in", 4 * D, D, 1), ("ff_out", D, 4 * D, 3))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clk = (s.strip() for s in q.split(","))
    return dict(gpu=name, power_limit=power, max_sm_clock=clk)


def make_ctx(layers, precision, quant_bits):
    ctx = LtxContext(LTXTransformerConfig(num_layers=layers), 0)
    if precision != 16:
        ctx.set_precision(precision)
    ctx.init_random_weights(1, seed=101)
    ctx.finalize_weights(quant_bits=quant_bits, group_size=64)
    g = torch.Generator().manual_seed(1)
    noise = torch.randn(C, F, H, W, generator=g).numpy()

    def text():
        t = torch.randn(1, S, CAP, generator=g)
        return (t / t.pow(2).mean(-1, keepdim=True).sqrt()).bfloat16()
    ctx.denoise_begin(noise, (F, H, W), 0.7, text(), None, text(), None)
    return ctx


FORMS = (("plain", 1.0), ("guided", 2.0))   # cfg scale 1: the guidance pass is skipped


def step(ctx, n, cfg):
    for _ in range(n):
        ctx.denoise_step(0.7, 0.65, 0, cfg_scale=cfg)


def bench_steps(layers, steps, rounds, warmup):
    ctxs = {name: make_ctx(layers, p, q) for name, p, q in MODES}
    runs = [(m, f, cfg) for m in ctxs for f, cfg in FORMS]
    for m, _, cfg in runs:
        step(ctxs[m], warmup, cfg)
        ctxs[m].sync()
    dev = {(m, f): [] for m, f, _ in runs}
    host = {(m, f): [] for m, f, _ in runs}
    for _ in range(rounds):
        for m, f, cfg in runs:
            c = ctxs[m]
            st = torch.cuda.ExternalStream(c.stream)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c.sync()
            t0 = time.perf_counter()
            a.record(st)
            step(c, steps, cfg)
            b.record(st)
            c.sync()
            host[m, f].append((time.perf_counter() - t0) * 1e3 / steps)
            dev[m, f].append(a.elapsed_time(b) / steps)
    res = {m: {} for m in ctxs}
    for m, f, cfg in runs:   # profiled pass of its own: tracing slows the host
        c = ctxs[m]
        c.set_profiling(True)
        before = c.get_profile()
        step(c, 1, cfg)
        c.sync()
        after = c.get_profile()
        c.set_profiling(False)
        prof = {}
        for cls in after:
            n = after[cls]["launches"] - before[cls]["launches"]
            if n > 0:
                ms = after[cls]["ms"] - before[cls]["ms"]
                fl = after[cls]["flops"] - before[cls]["flops"]
                by = after[cls]["bytes"] - before[cls]["bytes"]
                prof[cls] = dict(ms=round(ms, 3), launches=n, tflops=round(fl / ms / 1e9, 1) if fl else 0.0,
                                 gbps=round(by / ms / 1e6, 1))
        res[m][f] = dict(ms_per_step=round(statistics.median(dev[m, f]), 2),
                         ms_per_step_host=round(statistics.median(host[m, f]), 2), rounds_ms=[round(x, 2) for x in dev[m, f]],
                         profile=prof)
    for c in ctxs.values():
        assert np.isfinite(c.denoise_get_latent()).all()
        c.close()
    return res


def bench_gemms(reps):
    ctx = LtxContext(LTXTransformerConfig(num_layers=1, num_attention_heads=1), 0)
    st = torch.cuda.ExternalStream(ctx.stream)
    g = torch.Generator(device="cuda").manual_seed(3)
    out = []
    for M in (1536, 3072):
        for name, N, K, mode in GEMMS:
            A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
            Wt = (torch.randn(N, K, device="cuda", generator=g) / K ** 0.5).bfloat16()
            bias = torch.zeros(N, device="cuda")
            Aq = torch.empty(M, K, device="cuda", dtype=torch.uint8)
            Wq = torch.empty(N, K, device="cuda", dtype=torch.uint8)
            sa, sw = torch.empty(M, device="cuda"), torch.empty(N, device="cuda")
            C_ = torch.empty(M, N, device="cuda", dtype=torch.float32 if mode == 3 else torch.bfloat16)
            torch.cuda.synchronize()
            ctx._check(ctx.lib.ltx_op_quantize_fp8(ctx.handle, A.data_ptr(), M, K, K, Aq.data_ptr(), sa.data_ptr()))
            ctx._check(ctx.lib.ltx_op_quantize_fp8(ctx.handle, Wt.data_ptr(), N, K, K, Wq.data_ptr(), sw.data_ptr()))
            runs = {
                "bf16": lambda: ctx.lib.ltx_op_gemm(ctx.handle, A.data_ptr(), Wt.data_ptr(), bias.data_ptr(), C_.data_ptr(),
                                                    M, N, K, mode, 0),
                "fp8": lambda: ctx.lib.ltx_op_gemm_fp8(ctx.handle, Aq.data_ptr(), sa.data_ptr(), Wq.data_ptr(), sw.data_ptr(),
                                                       bias.data_ptr(), C_.data_ptr(), M, N, K, mode, 0),
            }
            row = dict(gemm=name, M=M, N=N, K=K)
            for _ in range(2):   # alternate the two kernels, keep the better round of each
                for k, fn in runs.items():
                    for _ in range(3):
                        ctx._check(fn())
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(st)
                    for _ in range(reps):
                        fn()
                    b.record(st)
                    ctx.sync()
                    us = a.elapsed_time(b) * 1e3 / reps
                    if k + "_us" not in row or us < row[k + "_us"]:
                        row[k + "_us"] = round(us, 2)
            for k in runs:
                row[k + "_tflops"] = round(2.0 * M * N * K / (row[k + "_us"] * 1e-6) / 1e12, 1)
            row["speedup"] = round(row["bf16_us"] / row["fp8_us"], 3)
            out.append(row)
            print(json.dumps(row), flush=True)
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--layers", type=int, default=48)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "fp8_bench needs a GPU"
    info = gpu_info()
    print(json.dumps(info), flush=True)
    gemms = bench_gemms(args.reps)
    steps = bench_steps(args.layers, args.steps, args.rounds, args.warmup)
    print(json.dumps(steps), flush=True)
    res = dict(info, workload=dict(layers=args.layers, video="768x512x25", tokens=F * H * W, text_tokens=S, forms=dict(FORMS),
                                   steps_per_round=args.steps, rounds=args.rounds), steps=steps, gemms=gemms)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
