"""Audio + video CFG step of the LTX-2 dual model at full width: ltx_av_denoise_step with cfg 3 and rescale 0.7, the two
guidance passes as one batched B = 2 forward against two B = 1 forwards, alternated in one process.

Shape: 48 blocks, D = 4096, Da = 2048, video 768x512x25 (N = 1536 tokens), Ta = 26 audio tokens, S = 1024 text tokens,
random-init weights (init_random_weights(17, ...), as tools/ncu_av.py).  Runs bf16 weights, then int8 codes
(finalize_weights(8, 64)).  Per format: warm-up steps of both forms, then --rounds rounds of --steps timed steps of each
form (host clock around a device synchronise, and CUDA events on the context's stream), then one profiled step of each form
in a separate pass for the per-class split (ltx_get_profile).  Prints the GPU name and power limit beside the numbers.

Usage (GPU box): python tools/av_cfg_bench.py [--layers 48] [--steps 4] [--rounds 3] [--warmup 2] [--formats 16,8]"""
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

F, H, W, Ta, S, C, CAP = 4, 16, 24, 26, 1024, 128, 3840


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clk = (s.strip() for s in q.split(","))
    return dict(gpu=name, power_limit=power, max_sm_clock=clk)


def run_format(bits, layers, steps, rounds, warmup):
    ctx = LtxContext(LTXTransformerConfig(num_layers=layers), 0)
    ctx.init_random_weights(17, seed=101)
    ctx.finalize_weights(quant_bits=bits, group_size=64)
    g = torch.Generator().manual_seed(1)
    vn = torch.randn(C, F, H, W, generator=g).numpy()
    an = torch.randn(Ta, C, generator=g).numpy()

    def text():
        t = torch.randn(1, S, CAP, generator=g)
        return (t / t.pow(2).mean(-1, keepdim=True).sqrt()).bfloat16()
    ctx.av_denoise_begin(vn, an, (F, H, W), 0.7, text(), text(), None, text(), text(), None)
    st = torch.cuda.ExternalStream(ctx.stream)

    def step(batched, n):
        for _ in range(n):
            ctx.av_denoise_step(0.7, 0.65, 0, cfg_scale=3.0, rescale_phi=0.7, batched_cfg=batched)

    for batched in (True, False):
        step(batched, warmup)
    ctx.sync()
    host = {True: [], False: []}
    dev = {True: [], False: []}
    for _ in range(rounds):
        for batched in (True, False):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ctx.sync()
            t0 = time.perf_counter()
            a.record(st)
            step(batched, steps)
            b.record(st)
            ctx.sync()
            host[batched].append((time.perf_counter() - t0) * 1e3 / steps)
            dev[batched].append(a.elapsed_time(b) / steps)
    prof = {}
    for batched in (True, False):   # profiled pass of its own: tracing slows the host
        ctx.set_profiling(True)
        before = ctx.get_profile()
        step(batched, 1)
        ctx.sync()
        after = ctx.get_profile()
        ctx.set_profiling(False)
        prof["batched" if batched else "two_pass"] = {
            k: dict(ms=round(after[k]["ms"] - before[k]["ms"], 3), launches=after[k]["launches"] - before[k]["launches"])
            for k in after if after[k]["launches"] - before[k]["launches"] > 0}
    v, a_ = ctx.av_denoise_get_latents()
    assert np.isfinite(v).all() and np.isfinite(a_).all()
    ctx.close()
    res = dict(weights="bf16" if bits == 16 else f"int{bits}", layers=layers, steps_per_round=steps, rounds=rounds)
    for batched in (True, False):
        k = "batched" if batched else "two_pass"
        res[k + "_ms_per_step"] = round(statistics.median(dev[batched]), 2)
        res[k + "_ms_per_step_host"] = round(statistics.median(host[batched]), 2)
        res[k + "_rounds_ms"] = [round(x, 2) for x in dev[batched]]
    res["speedup"] = round(res["two_pass_ms_per_step"] / res["batched_ms_per_step"], 3)
    res["profile"] = prof
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--layers", type=int, default=48)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--formats", default="16,8")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "av_cfg_bench needs a GPU"
    info = gpu_info()
    print(json.dumps(info), flush=True)
    for bits in (int(b) for b in args.formats.split(",")):
        res = run_format(bits, args.layers, args.steps, args.rounds, args.warmup)
        res.update(info)
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
