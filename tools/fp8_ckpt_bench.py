"""FP8 mode from a bf16 checkpoint against FP8 mode from a scaled-FP8 (e4m3) checkpoint: load + finalize time, device memory,
and the config-2 denoise step.

Both arms hold the same model at the LTX-2 shape (48 blocks, D = 4096, caption 3840): seeded synthetic block Linears whose rows
each carry a power-of-two scale and one code of magnitude 448, so FP8 mode's per-row rule applied to the bf16 arm's decoded
values gives back exactly the e4m3 arm's codes and scales -- the two arms run the same kernels on the same operands, and the
final latents are compared bit for bit.  The bf16 arm loads the block Linears with ltx_load_tensor (bf16, converted at
finalize by dit_convert_fp8); the e4m3 arm with ltx_load_tensor_e4m3 (codes kept).  Every other tensor is the same bf16 / fp32
upload in both.  Host tensors sit in pinned memory; one host buffer per Linear shape serves all 48 blocks (the copy engine
reads it anew for every block, so the H2D cost is that of distinct data).

Per round, the arms run in turn, one context at a time: load (wall time to the last upload's return; device memory in use,
total - free from cudaMemGetInfo, polled after every load call, max kept), finalize (wall time, memory after), then the
config-2 plain step of bench.py (768x512x25 video -> N = 1536 tokens, S = 1024, cfg 1; --warmup steps, then --steps steps
timed with CUDA events on the context's stream), and memory after the context is closed.  Prints the GPU name and power
limit (nvidia-smi, same process) beside the numbers.

Usage (GPU box): python tools/fp8_ckpt_bench.py [--layers 48] [--rounds 2] [--steps 5] [--warmup 2] [--out FILE]"""
import argparse
import hashlib
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
BLOCK_LINEARS = (("attn1.to_q", D, D), ("attn1.to_k", D, D), ("attn1.to_v", D, D), ("attn1.to_out", D, D),
                 ("attn2.to_q", D, D), ("attn2.to_k", D, D), ("attn2.to_v", D, D), ("attn2.to_out", D, D),
                 ("ff.project_in.proj", 4 * D, D), ("ff.project_out", D, 4 * D))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clk = (s.strip() for s in q.split(","))
    return dict(gpu=name, power_limit=power, max_sm_clock=clk)


def used_gb():
    free, total = torch.cuda.mem_get_info(0)
    return (total - free) / 1e9


def coded_linear(n, k, g):
    """(e4m3 codes [n, k] as uint8, fp32 row scales [n], bf16 decoded values [n, k]), all pinned: w ~ N(0, 1/k) quantised by
    the per-row power-of-two rule, then the largest code of each row set to +-448."""
    w = torch.randn(n, k, generator=g) / k ** 0.5
    amax = w.abs().amax(1)
    s = torch.pow(2.0, torch.ceil(torch.log2(amax / 448.0)))
    q = (w / s[:, None]).clamp(-448.0, 448.0).to(torch.float8_e4m3fn).view(torch.uint8)
    rows = torch.arange(n)
    idx = w.abs().argmax(1)
    q[rows, idx] = (q[rows, idx] & 0x80) | 0x7E
    dec = (q.view(torch.float8_e4m3fn).float() * s[:, None]).bfloat16()
    return q.pin_memory(), s.float().pin_memory(), dec.pin_memory()


def other_tensors(layers, g):
    """every tensor outside the block Linears, under the names init_random_weights uses (same shapes and scales)"""
    t = {}

    def lin(name, n, k, scale=1.0):
        t[name + ".weight"] = (torch.randn(n, k, generator=g) * scale / k ** 0.5).bfloat16().pin_memory()
        t[name + ".bias"] = (torch.randn(n, generator=g) * 0.02).pin_memory()
    lin("patchify_proj", D, C)
    lin("adaln_single.emb.linear_1", D, 256)
    lin("adaln_single.emb.linear_2", D, D)
    lin("adaln_single.linear", 6 * D, D, 0.5)
    lin("caption_projection.linear_1", D, CAP)
    lin("caption_projection.linear_2", D, D)
    sst = (torch.randn(6, D, generator=g) * 0.1).pin_memory()
    norm = (1.0 + 0.1 * torch.randn(D, generator=g)).pin_memory()
    bias = (torch.randn(4 * D, generator=g) * 0.02).pin_memory()
    for i in range(layers):
        p = f"transformer_blocks.{i}."
        t[p + "scale_shift_table"] = sst
        for a in ("attn1", "attn2"):
            t[p + a + ".q_norm.weight"] = norm
            t[p + a + ".k_norm.weight"] = norm
        for name, n, _ in BLOCK_LINEARS:
            t[p + name + ".bias"] = bias[:n]
    t["scale_shift_table"] = (torch.randn(2, D, generator=g) * 0.1).pin_memory()
    lin("proj_out", C, D)
    return t


def run_arm(arm, layers, linears, others, steps, warmup, inputs):
    base = used_gb()
    peak = base
    t0 = time.perf_counter()
    ctx = LtxContext(LTXTransformerConfig(num_layers=layers), 0)
    ctx.set_precision(8)
    for k, v in others.items():
        ctx.load_tensor(k, v)
        peak = max(peak, used_gb())
    for i in range(layers):
        for name, n, k in BLOCK_LINEARS:
            q, s, dec = linears[n, k]
            key = f"transformer_blocks.{i}.{name}.weight"
            if arm == "e4m3":
                ctx.load_tensor_e4m3(key, q, s)
            else:
                ctx.load_tensor(key, dec)
            peak = max(peak, used_gb())
    ctx.sync()
    t1 = time.perf_counter()
    after_load = used_gb()
    ctx.finalize_weights()
    ctx.sync()
    t2 = time.perf_counter()
    after_finalize = used_gb()
    noise, pos, neg = inputs
    ctx.denoise_begin(noise, (F, H, W), 0.7, pos, None, neg, None)
    for _ in range(warmup):
        ctx.denoise_step(0.7, 0.65, 0, cfg_scale=1.0)
    ctx.sync()
    st = torch.cuda.ExternalStream(ctx.stream)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(steps):
        ctx.denoise_step(0.7, 0.65, 0, cfg_scale=1.0)
    b.record(st)
    ctx.sync()
    step_ms = a.elapsed_time(b) / steps
    after_steps = used_gb()
    lat = ctx.denoise_get_latent()
    assert np.isfinite(lat).all()
    ctx.close()
    torch.cuda.synchronize()
    return dict(load_s=round(t1 - t0, 3), finalize_s=round(t2 - t1, 3), load_finalize_s=round(t2 - t0, 3),
                mem_gb=dict(before=round(base, 2), peak_during_load=round(peak, 2), after_load=round(after_load, 2),
                            after_finalize=round(after_finalize, 2), after_steps=round(after_steps, 2),
                            after_close=round(used_gb(), 2)),
                step_ms=round(step_ms, 3), latent_sha1=hashlib.sha1(lat.tobytes()).hexdigest())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--layers", type=int, default=48)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    info = gpu_info()
    torch.cuda.init()
    g = torch.Generator().manual_seed(7)
    linears = {(n, k): coded_linear(n, k, g) for n, k in {(n, k) for _, n, k in BLOCK_LINEARS}}
    others = other_tensors(a.layers, g)
    noise = torch.randn(C, F, H, W, generator=g).numpy()

    def text():
        t = torch.randn(1, S, CAP, generator=g)
        return (t / t.pow(2).mean(-1, keepdim=True).sqrt()).bfloat16()
    inputs = (noise, text(), text())
    arms = ("bf16", "e4m3")
    rounds = {arm: [] for arm in arms}
    for _ in range(a.rounds):
        for arm in arms:
            rounds[arm].append(run_arm(arm, a.layers, linears, others, a.steps, a.warmup, inputs))
    summary = {}
    for arm in arms:
        rs = rounds[arm]
        summary[arm] = dict(load_finalize_s=statistics.median(r["load_finalize_s"] for r in rs),
                            load_s=statistics.median(r["load_s"] for r in rs),
                            finalize_s=statistics.median(r["finalize_s"] for r in rs),
                            step_ms=statistics.median(r["step_ms"] for r in rs),
                            peak_during_load_gb=max(r["mem_gb"]["peak_during_load"] for r in rs),
                            after_finalize_gb=max(r["mem_gb"]["after_finalize"] for r in rs))
    same = len({r["latent_sha1"] for arm in arms for r in rounds[arm]}) == 1
    res = dict(**info, layers=a.layers, D=D, steps=a.steps, warmup=a.warmup, tokens=F * H * W, text_tokens=S,
               latents_bit_identical_across_arms=same, summary=summary, rounds=rounds)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
