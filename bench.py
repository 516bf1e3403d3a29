#!/usr/bin/env python
"""bench.py -- DiT steps/s (+ VAE frames/s) of the LTX-2 denoise hot path on B200, the metric BASELINE.json names.

One "step" = one denoise step of the distilled LTX-2 video DiT at 768x512x25 frames (BASELINE config 2: N = 1536 video
tokens, S = 1024 text tokens, 48 blocks, D = 4096, bf16 weights, random-init on the device, synthetic inputs):
patchify -> 48-block forward -> unpatchify -> Euler update.  Step-invariant text projections are cached by the warm-up.

  value        steps/s of ONE video (latent resident in HBM, ltx_denoise_step), CUDA events on the library's stream.
               --gpus N > 1: the SAME video strong-scaled over N GPUs by Ulysses sequence parallelism (`scaling: "strong"`);
               N independent replicas (the trivial weak-scaling mode) are reported under extras.replicas
  e2e          steps/s through the host-buffer C ABI the Swift pipeline binds (ltx_dit_forward + ltx_guided_euler_step):
               pinned-host -> device copies of latent/timestep (+ text on a cache miss) and device -> host copies of the
               velocity and the new latent are inside the timed region
  parity       what the timed code computes, checked in the same process: a 2-block prefix of the model at the config-2
               shapes against the CPU oracle (rel-L2 <= 1e-2), the timed 48-block latent finite, the decoder on the real
               channel plan against the oracle (PSNR >= 40 dB); N > 1: the N-GPU latent / frames against this rank's own
               1-GPU run of the same inputs
  roofline     tensor-pipe roofline of the dominant kernel class (the tcgen05 GEMM): algorithmic FLOPs of the GEMM launches
               of one step / their summed device time (CUDA events around every launch, separate profiled pass)
  cpu_baseline the CPU oracle (a port of the reference's algorithm) on this box's host cores, bounded sample
  vae          secondary metric: frames/s of the video-VAE decode of the same clip (25 frames, 768x512)

`--impl reference` times the CPU port only (the Swift/MLX reference cannot be built in this image).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG2 = dict(width=768, height=512, frames=25, F=4, H=16, W=24, N=1536, S=1024)
D, L, HEADS, CAP, CIN = 4096, 48, 32, 3840, 128
WORKLOAD = ("LTX-2 distilled 13B-video DiT denoise step (BASELINE config 2): 768x512x25f -> N=1536 tokens, S=1024 text tokens, "
            "48 blocks, D=4096, 32 heads")


def dit_flops_per_step(N, S, cached_text=True):
    """SURVEY 8(d): per block 8ND^2 + 4N^2D + 4ND^2 (+ 4SD^2 text K/V when not cached) + 4NSD + 16ND^2."""
    blk = 8 * N * D * D + 4 * N * N * D + 4 * N * D * D + 4 * N * S * D + 16 * N * D * D
    if not cached_text:
        blk += 4 * S * D * D
    return L * blk + 2 * N * CIN * D * 2


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(tflops_sustained=j["bf16_tflops_sustained"], tflops_burst=j["bf16_tflops"], hbm_gbs=j["hbm_gbs"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(tflops_sustained=1400.0, tflops_burst=1590.0, hbm_gbs=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi during the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in self.rows)]
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(sm))


# ------------------------------------------------------------------------------------------------ CPU port arm
_CPU_CACHE = {}


def _cpu_port_inputs(O, cfg):
    """One transformer block's weights at the LTX-2 width plus the global (embedding / head) weights; the full-step timing
    re-uses the block for all 48 layers (same arithmetic, 1/48 of the 52 GB an fp32 copy of the model would need)."""
    g = torch.Generator().manual_seed(0)
    w = {}

    def lin(name, out_f, in_f):
        w[name + ".weight"] = torch.randn(out_f, in_f, generator=g) / math.sqrt(in_f)
        w[name + ".bias"] = torch.zeros(out_f)
    p = "transformer_blocks.0."
    w[p + "scale_shift_table"] = torch.randn(6, D, generator=g) * 0.1
    for a in ("attn1", "attn2"):
        for l in ("to_q", "to_k", "to_v", "to_out"):
            lin(p + f"{a}.{l}", D, D)
        w[p + f"{a}.q_norm.weight"] = torch.ones(D)
        w[p + f"{a}.k_norm.weight"] = torch.ones(D)
    lin(p + "ff.project_in.proj", 4 * D, D)
    lin(p + "ff.project_out", D, 4 * D)
    lin("patchify_proj", D, CIN)
    lin("adaln_single.emb.linear_1", D, 256)
    lin("adaln_single.emb.linear_2", D, D)
    lin("adaln_single.linear", 6 * D, D)
    lin("caption_projection.linear_1", D, CAP)
    lin("caption_projection.linear_2", D, D)
    w["scale_shift_table"] = torch.randn(2, D, generator=g) * 0.1
    lin("proj_out", CIN, D)
    x = torch.randn(1, CFG2["N"], D, generator=g)
    ctx = torch.randn(1, CFG2["S"], D, generator=g)
    ada = torch.randn(1, 1, 6, D, generator=g) * 0.1
    lat = torch.randn(1, CFG2["N"], CIN, generator=g)
    text = torch.randn(1, CFG2["S"], CAP, generator=g)
    rope = O.rope_table(cfg, CFG2["F"], CFG2["H"], CFG2["W"])
    return dict(w=w, x=x, ctx=ctx, ada=ada, rope=rope, lat=lat, text=text)


def cpu_port_step_seconds(sample_blocks=1, repeats=1):
    """Times the oracle (CPU port of the reference algorithm) on a bounded sample of the config-2 step: `sample_blocks`
    transformer blocks at the full shapes (N=1536, S=1024, D=4096, fp32), extrapolated to 48 blocks.
    Returns (seconds per full step, cores, description)."""
    from oracle import ltx_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = O.DiTConfig()
    if not _CPU_CACHE:
        _CPU_CACHE.update(_cpu_port_inputs(O, cfg))
    w, x, ctx, ada, rope = (_CPU_CACHE[k] for k in ("w", "x", "ctx", "ada", "rope"))
    best = float("inf")
    with torch.no_grad():
        for _ in range(repeats):
            t0 = time.perf_counter()
            y = x
            for _b in range(sample_blocks):
                y = O.block_forward(w, 0, y, ada, ctx, None, rope, cfg)
            best = min(best, (time.perf_counter() - t0) / sample_blocks)
    # text K/V are step-invariant in our arm (cached); the oracle recomputes them inside block_forward, which is what the
    # reference does every step as well (T/LTXAttention.swift:174-180), so the per-block time is used unchanged.
    return best * L, os.cpu_count() or 1, f"{sample_blocks} of {L} blocks at N=1536,S=1024,D=4096 fp32 (torch CPU), x{L}"


def cpu_port_full_step_seconds():
    """ONE true full step of the CPU port, not extrapolated: patchify projection, timestep MLPs, caption projection, RoPE
    table, all 48 block forwards (block 0's weights stand in for every layer), output head, Euler update.  ~26 s on 16 cores."""
    from oracle import ltx_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = O.DiTConfig()
    if not _CPU_CACHE:
        _CPU_CACHE.update(_cpu_port_inputs(O, cfg))
    base = _CPU_CACHE["w"]

    class Shared(dict):      # transformer_blocks.i.* -> transformer_blocks.0.*
        def __missing__(self, k):
            if k.startswith("transformer_blocks."):
                return base["transformer_blocks.0." + k.split(".", 2)[2]]
            raise KeyError(k)
    w = Shared(base)
    lat, text = _CPU_CACHE["lat"], _CPU_CACHE["text"]
    with torch.no_grad():
        t0 = time.perf_counter()
        v = O.dit_forward(w, cfg, lat, text, torch.tensor([0.7]), None, (CFG2["F"], CFG2["H"], CFG2["W"]))
        _ = lat + (0.5 - 0.7) * v
        return time.perf_counter() - t0


def run_reference(args, rank):
    if rank != 0:
        return
    times = []
    for i in range(args.warmup + args.steps):
        t, cores, desc = cpu_port_step_seconds(1, 1)
        if i >= args.warmup:
            times.append(t)
    sec = float(np.mean(times))
    full = None
    if not args.no_cpu_full_step:
        try:
            full = cpu_port_full_step_seconds()
        except Exception as e:   # report, do not hide
            full = f"failed: {e}"
    line = dict(metric="dit_steps_per_s", value=1.0 / sec, unit="steps/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=sec * 1e3, higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f32", data="synthetic",
                impl="reference", extrapolated=True,
                sample_ms_per_step=sec * 1e3 / L,
                config=dict(workload=WORKLOAD,
                            note="CPU port of the reference algorithm (oracle/); the Swift+MLX reference cannot be built here. Each "
                                 "timed step is ONE of the 48 blocks at the full shapes; value = 1 / (48 x that) -- extrapolated, so "
                                 "ms_per_step x steps exceeds the wall time of this run by design; full_step_s is one true 48-block step"),
                cpu_baseline=dict(value=1.0 / sec, unit="steps/s", cores=cores, kind="port", sample=desc, extrapolated=True,
                                  full_step_s=full, full_step_steps_per_s=(1.0 / full) if isinstance(full, float) else None),
                e2e=dict(value=1.0 / sec, unit="steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
def _unit_rms(t):
    return (t / t.pow(2).mean(-1, keepdim=True).sqrt()).bfloat16()


def _rel_l2(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy in float32, so that two builds run with the same arguments can be compared
    output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def parity_vs_oracle(local_rank):
    """The kernels the benchmark times, checked against the CPU oracle inside the benchmark process: (i) a 2-block prefix of
    the model at the config-2 shapes (N=1536, S=1024, D=4096 -- same tile fits, fused q|k|v, attention shapes as the timed
    48-block run), (ii) the decoder's real channel plan (base 1024, 5 blocks per stage) on a small latent."""
    from oracle import ltx_oracle as O   # checker only
    from ltx_video_swift_mlx_b200.context import LtxContext, LTXTransformerConfig
    out = {}
    torch.set_num_threads(os.cpu_count() or 1)
    F, H, W, N, S = CFG2["F"], CFG2["H"], CFG2["W"], CFG2["N"], CFG2["S"]
    ocfg = O.DiTConfig(num_layers=2)
    w = O.make_dit_weights(ocfg, 77)
    g = torch.Generator().manual_seed(78)
    lat = torch.randn(1, N, CIN, generator=g).bfloat16()
    text = _unit_rms(torch.randn(1, S, CAP, generator=g))
    sig = torch.tensor([0.725])
    t0 = time.perf_counter()
    with torch.no_grad():
        ref = O.dit_forward(w, ocfg, lat.float(), text.float(), sig, None, (F, H, W))
    t_oracle = time.perf_counter() - t0
    c = LtxContext(LTXTransformerConfig(num_layers=2), local_rank)
    c.load_weights(w)
    c.finalize_weights()
    got = c.dit_forward(lat, text, sig.numpy(), None, (F, H, W))
    c.close()
    err = _rel_l2(got, ref.numpy())
    out["dit_prefix_2_blocks_cfg2_shape"] = dict(rel_l2_vs_oracle=err, tol=1e-2, ok=bool(err <= 1e-2 and np.isfinite(got).all()),
                                                 oracle_cpu_s=t_oracle)
    del w
    vcfg = O.VAEConfig()
    vw = O.make_vae_weights(vcfg, 79)
    vw = {k: (O.bf16_round(v) if (k.endswith(".weight") and v.ndim >= 2) else v) for k, v in vw.items()}
    z = torch.randn(1, 128, 2, 4, 6, generator=g)
    with torch.no_grad():
        fref = O.decode_video(vw, vcfg, z)
    c = LtxContext(LTXTransformerConfig(num_layers=1, num_attention_heads=1), local_rank)
    c.load_weights(vw, prefix="vae.")
    c.finalize_weights()
    fr = c.vae_decode(z[0].numpy())
    c.close()
    p = float(O.psnr(torch.from_numpy(fr), fref))
    out["vae_full_channel_plan"] = dict(psnr_db_vs_oracle=p, bound_db=40.0, ok=bool(p >= 40.0), latent="2x4x6 (9 frames of 128x192)")
    return out


def run_ours(args, rank, world, local_rank):
    import ltx_video_swift_mlx_b200  # noqa: F401
    from ltx_video_swift_mlx_b200.context import LtxContext, LTXTransformerConfig, make_flags
    from ltx_video_swift_mlx_b200.scheduler import LTXScheduler
    from ltx_video_swift_mlx_b200 import dist as ltxdist

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    ctx = LtxContext(LTXTransformerConfig(), local_rank)
    ctx.init_random_weights(3, seed=1234)   # one model on every rank: sequence parallelism shards one video's tokens
    ctx.finalize_weights()
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local_rank))

    F, H, W, N, S = CFG2["F"], CFG2["H"], CFG2["W"], CFG2["N"], CFG2["S"]
    g = torch.Generator().manual_seed(1236)          # same video on every rank
    noise = torch.randn(1, CIN, F, H, W, generator=g)
    text = _unit_rms(torch.randn(1, S, CAP, generator=g))          # unit-RMS rows, mask all ones
    ntext = _unit_rms(torch.randn(1, S, CAP, generator=g))
    sigmas = LTXScheduler().set_timesteps(8, distilled=True, latent_token_count=N)
    pairs = [(sigmas[i], sigmas[i + 1]) for i in range(len(sigmas) - 1)]
    dev_sig = LTXScheduler().set_timesteps(40, distilled=False, latent_token_count=N)
    parity = {}

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if dist is None:
            return float(v)
        t = torch.tensor([v], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ok(flag):
        if dist is None:
            return bool(flag)
        t = torch.tensor([1 if flag else 0], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    def ev_time(c, strm, fn, reps, warm=0):
        for _ in range(warm):
            fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(strm)
        for i in range(reps):
            fn()
        b.record(strm)
        barrier()
        return max_over_ranks(a.elapsed_time(b) / reps)

    def full_denoise(c, guided=False, n_steps=None):
        """The whole schedule from the seeded noise; returns the final latent (host)."""
        if guided:
            c.denoise_begin(noise[0].numpy(), (F, H, W), dev_sig[0], text, None, ntext, None)
            for i in range(n_steps or 3):
                c.denoise_step(dev_sig[i], dev_sig[i + 1], i, cfg_scale=4.0, stg_scale=0.5, stg_blocks=(29,))
        else:
            c.denoise_begin(noise[0].numpy(), (F, H, W), sigmas[0], text, None)
            for i, (sg, sn) in enumerate(pairs[:n_steps] if n_steps else pairs):
                c.denoise_step(sg, sn, i)
        return c.denoise_get_latent()

    # ---------------- N > 1: the single-GPU answers this rank will hold the multi-GPU modes to (same inputs, same device)
    if world > 1:
        single_step1 = full_denoise(ctx, n_steps=1)
        single_plain = full_denoise(ctx)
        single_guided = full_denoise(ctx, guided=True)
        # replicas: N independent videos, one per GPU (weak scaling, no communication) -- reported as an extra
        ctx.denoise_begin(noise[0].numpy(), (F, H, W), sigmas[0], text, None)
        rep_no = [0]

        def rep_step():
            sg, sn = pairs[rep_no[0] % len(pairs)]
            ctx.denoise_step(sg, sn, rep_no[0] % len(pairs))
            rep_no[0] += 1
        t_rep = ev_time(ctx, stream, rep_step, max(4, min(args.steps, 8)), warm=3)
        ltxdist.init_context(ctx, sp_size=world, pass_groups=1)
        dist_step1 = full_denoise(ctx, n_steps=1)
        dist_plain = full_denoise(ctx)
        err1, err = _rel_l2(dist_step1, single_step1), _rel_l2(dist_plain, single_plain)
        # A rank's GEMMs sum K in a different order than the 1-GPU run once its row count takes the split-K weight-streaming
        # kernel (sp >= 4 here): the same arithmetic up to fp32 reassociation, which bf16 re-rounding turns into ~1e-4 per
        # forward and which compounds over the 8 steps.  One step is held to 1e-3, the whole schedule to 3e-3.
        parity["ulysses_vs_single_gpu"] = dict(one_step_rel_l2=err1, one_step_tol=1e-3, full_schedule_rel_l2=err, full_schedule_tol=3e-3,
                                               bit_identical=bool(np.array_equal(dist_plain, single_plain)),
                                               ok=all_ok(err1 <= 1e-3 and err <= 3e-3 and np.isfinite(dist_plain).all()), steps=len(pairs),
                                               peer_memory=bool(ctx.lib.ltx_dist_p2p_active(ctx.handle)))

    # ---------------- resident path (value): one video; Ulysses over all ranks when world > 1
    ctx.denoise_begin(noise[0].numpy(), (F, H, W), sigmas[0], text, None)
    step_no = [0]

    def resident_step():
        sg, sn = pairs[step_no[0] % len(pairs)]
        ctx.denoise_step(sg, sn, step_no[0] % len(pairs))
        step_no[0] += 1

    for _ in range(max(args.warmup, 3)):
        resident_step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    try:     # the sampler's nvidia-smi child must not outlive a failed run
        l0 = ctx.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            resident_step()
        e1.record(stream)
        barrier()
    finally:
        clocks = sampler.stop() if rank == 0 else None
    launches = (ctx.launch_count - l0) // args.steps
    ms_per_step = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    value = 1e3 / ms_per_step
    timed_latent = ctx.denoise_get_latent()
    parity["timed_latent_finite"] = all_ok(bool(np.isfinite(timed_latent).all() and np.abs(timed_latent).max() > 0))

    # ---------------- profiled pass: per-kernel-class device time of one step (not part of the timed value)
    ctx.set_profiling(True)
    ep0, ep1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ep0.record(stream)
    resident_step()
    ep1.record(stream)
    prof = ctx.get_profile()
    ctx.set_profiling(False)
    torch.cuda.synchronize()
    profiled_step_ms = ep0.elapsed_time(ep1)   # the same step run eagerly with an event pair around every kernel class scope

    # ---------------- e2e through the host-buffer ABI (the Swift seam), pinned host memory
    lat_host = torch.empty(1, N, CIN, dtype=torch.bfloat16).pin_memory()
    lat32 = (noise * sigmas[0]).contiguous().pin_memory()
    vel_lat = torch.empty_like(lat32).pin_memory()
    text_pin = text.pin_memory()
    ts = torch.zeros(1).pin_memory()
    from ltx_video_swift_mlx_b200 import latent_utils
    shape = latent_utils.VideoLatentShape(1, CIN, F, H, W)
    flags = make_flags(context_key=ctx.new_context_key())

    def host_step(i):
        sg, sn = pairs[i % len(pairs)]
        lat_host.copy_(torch.from_numpy(latent_utils.patchify(lat32.numpy())))     # host patchify + bf16 cast (:815)
        ts[0] = sg
        v = ctx.dit_forward(lat_host, text_pin, ts.numpy(), None, (F, H, W), flags)
        vel_lat.copy_(torch.from_numpy(latent_utils.unpatchify(v, shape)))
        ctx.guided_euler_step(lat32.numpy(), vel_lat.numpy(), sigma=sg, sigma_next=sn)

    for i in range(max(args.warmup, 3)):
        host_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        host_step(i)
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / args.steps)
    h2d = N * CIN * 2 + 4 + 2 * N * CIN * 4          # bf16 tokens + sigma ; latent + velocity for the Euler call
    d2h = N * CIN * 4 + N * CIN * 4                  # velocity ; updated latent
    parity["e2e_latent_finite"] = all_ok(bool(torch.isfinite(lat32).all()))

    extras = {}
    if world > 1:
        extras["replicas"] = dict(desc=f"{world} independent videos, one per GPU (weak scaling, no communication)",
                                  ms_per_step=t_rep, steps_per_s=world * 1e3 / t_rep)
        extras["ulysses"] = dict(desc=f"the headline: one video, sequence-parallel sp={world}", ms_per_step=ms_per_step,
                                 kernel_classes={k: v for k, v in prof.items() if v["launches"]})

    # ---------------- VAE decode (secondary metric), resident + host ABI; temporally sharded over the ranks when world > 1
    n_frames = 8 * (F - 1) + 1
    lat_dev = torch.randn(CIN, F, H, W, generator=torch.Generator().manual_seed(55)).cuda()
    frames_dev = torch.empty(n_frames, 32 * H, 32 * W, 3, device="cuda")
    torch.cuda.synchronize()
    vae_ms = ev_time(ctx, stream, lambda: ctx.vae_decode_dev(lat_dev.data_ptr(), (F, H, W), frames_dev.data_ptr()),
                     max(3, min(args.steps, 10)), warm=3)
    frames_sample = None
    if args.dump_outputs:
        # 2^20 of the 29.5 M frame values (118 MB in fp32) at fixed, seeded positions
        pick = np.sort(np.random.default_rng(0).choice(frames_dev.numel(), 1 << 20, replace=False))
        frames_sample = frames_dev.view(-1)[torch.from_numpy(pick).cuda()].cpu().numpy()
    ctx.set_profiling(True)
    ctx.vae_decode_dev(lat_dev.data_ptr(), (F, H, W), frames_dev.data_ptr())
    vprof = ctx.get_profile()
    ctx.set_profiling(False)
    torch.cuda.synchronize()
    frames_multi = frames_dev.cpu().numpy() if world > 1 else None
    lat_cpu = lat_dev.cpu().numpy()
    frames_host = ctx.pinned_empty((n_frames, 32 * H, 32 * W, 3))      # page-locked output buffer (ltx_host_alloc)
    ctx.vae_decode(lat_cpu, out=frames_host)
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        ctx.vae_decode(lat_cpu, out=frames_host)
    vae_e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / 3)
    parity["vae_frames_in_range"] = all_ok(bool(np.isfinite(frames_host).all() and frames_host.min() >= 0 and frames_host.max() <= 1
                                                and frames_host.std() > 0))

    def time_guided(c, strm, nsteps=3):
        """BASELINE config 3: dev schedule, CFG 4.0 + STG 0.5 at block 29 -> 3 forwards per step."""
        c.denoise_begin(noise[0].numpy(), (F, H, W), dev_sig[0], text, None, ntext, None)
        for i in range(2):
            c.denoise_step(dev_sig[i], dev_sig[i + 1], i, cfg_scale=4.0, stg_scale=0.5, stg_blocks=(29,))
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(strm)
        for i in range(2, 2 + nsteps):
            c.denoise_step(dev_sig[i], dev_sig[i + 1], i, cfg_scale=4.0, stg_scale=0.5, stg_blocks=(29,))
        b.record(strm)
        barrier()
        return max_over_ranks(a.elapsed_time(b) / nsteps)

    lat121 = torch.randn(CIN, 16, H, W, generator=torch.Generator().manual_seed(77))

    def time_vae121(c, strm, reps=2, fetch=False):
        """BASELINE config 4: 768x512x121 frames (latent 16x16x24)."""
        lat = lat121.cuda()
        out = torch.empty(121, 32 * H, 32 * W, 3, device="cuda")
        torch.cuda.synchronize()
        t = ev_time(c, strm, lambda: c.vae_decode_dev(lat.data_ptr(), (16, H, W), out.data_ptr()), reps, warm=1)
        fr = out.cpu().numpy() if fetch else None
        del lat, out
        return t, fr

    def cfg5_two_stage(sp):
        """BASELINE config 5 (generateVideoTwoStage, P/LTXPipeline.swift:2420-2709), int8 group-64 weights: stage 1 at
        768x512x257 (N = 12 672, 8 distilled steps) -> latent upscale 2x + AdaIN + re-noise on the device -> stage 2 at
        1536x1024x257 (N = 50 688, 3 refinement steps).  sp > 1: Ulysses over all ranks, the stage switch replicated."""
        from ltx_video_swift_mlx_b200.scheduler import STAGE_2_DISTILLED_SIGMA_VALUES as S2
        F5, H5, W5 = 33, 16, 24
        cq = LtxContext(LTXTransformerConfig(), local_rank)
        cq.init_random_weights(1 | 2 | 8, seed=99)   # DiT + VAE (latent statistics) + latent upscaler; same seed on every rank
        cq.finalize_weights(quant_bits=8)
        if sp > 1:
            ltxdist.init_context(cq, sp_size=sp, pass_groups=1)
        sq = torch.cuda.ExternalStream(cq.stream, device=torch.device("cuda", local_rank))
        g5 = torch.Generator().manual_seed(177)
        n1 = torch.randn(CIN, F5, H5, W5, generator=g5)
        n2 = torch.randn(CIN, F5, 2 * H5, 2 * W5, generator=g5)
        s1 = LTXScheduler().set_timesteps(8, distilled=True, latent_token_count=F5 * H5 * W5)
        res = {}

        def timed(fn):
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(sq)
            fn()
            b.record(sq)
            barrier()
            return max_over_ranks(a.elapsed_time(b))
        cq.denoise_begin(n1.numpy(), (F5, H5, W5), s1[0], text, None)
        cq.denoise_step(s1[0], s1[1], 0)       # untimed: builds the RoPE table, the text cache and the peer buffers
        t1 = timed(lambda: [cq.denoise_step(s1[i], s1[i + 1], i) for i in range(1, 8)]) / 7
        tu = timed(lambda: cq.denoise_upscale_stage(n2.numpy(), S2[0], 1.0))
        cq.denoise_step(S2[0], S2[1], 0)       # first stage-2 step builds the stage-2 RoPE table and buffers
        t2 = timed(lambda: [cq.denoise_step(S2[i], S2[i + 1], i) for i in range(1, 3)]) / 2
        cq.set_profiling(True)
        cq.denoise_step(S2[1], S2[2], 1)
        p5 = cq.get_profile()
        cq.set_profiling(False)
        lat = cq.denoise_get_latent()
        fl1, fl2 = dit_flops_per_step(F5 * H5 * W5, S), dit_flops_per_step(4 * F5 * H5 * W5, S)
        res.update(stage1_ms_per_step=t1, stage1_tokens=F5 * H5 * W5, stage1_tflops=fl1 / (t1 * 1e-3) / 1e12,
                   upscale_switch_ms=tu, stage2_ms_per_step=t2, stage2_tokens=4 * F5 * H5 * W5,
                   stage2_tflops=fl2 / (t2 * 1e-3) / 1e12, total_ms_8_plus_3_steps=8 * t1 + tu + 3 * t2,
                   final_latent_finite=all_ok(bool(np.isfinite(lat).all() and lat.std() > 0)),
                   peer_memory=bool(cq.lib.ltx_dist_p2p_active(cq.handle)) if sp > 1 else None,
                   stage2_kernel_classes={k: v for k, v in p5.items() if v["launches"]})
        if sp > 1:
            cq.dist_shutdown()
        cq.close()
        return res

    if world == 1:
        # qint8 weights (the reference's --transformer-quant qint8 path): same step on int8 group-64 weights
        try:
            cq = LtxContext(LTXTransformerConfig(), local_rank)
            cq.init_random_weights(1, seed=99)
            cq.finalize_weights(quant_bits=8)
            sq = torch.cuda.ExternalStream(cq.stream, device=torch.device("cuda", local_rank))
            cq.denoise_begin(noise[0].numpy(), (F, H, W), sigmas[0], text, None)
            qn = [0]

            def qstep():
                cq.denoise_step(pairs[qn[0] % len(pairs)][0], pairs[qn[0] % len(pairs)][1], qn[0] % len(pairs))
                qn[0] += 1
            tq = ev_time(cq, sq, qstep, 6, warm=3)
            cq.set_profiling(True)
            qstep()
            pq = cq.get_profile()
            cq.set_profiling(False)
            lq = cq.denoise_get_latent()
            extras["qint8"] = dict(desc="same step with int8 group-64 weights (dequant-fused tcgen05 GEMMs)", ms_per_step=tq,
                                   steps_per_s=1e3 / tq, latent_finite=bool(np.isfinite(lq).all()),
                                   kernel_classes={k: v for k, v in pq.items() if v["launches"]})
            cq.close()
            # the same quantised model with its dequantised values materialised once at load time (ltx_set_quant_storage)
            cm = LtxContext(LTXTransformerConfig(), local_rank)
            cm.set_quant_storage(True)
            cm.init_random_weights(1, seed=99)
            cm.finalize_weights(quant_bits=8)
            sm_ = torch.cuda.ExternalStream(cm.stream, device=torch.device("cuda", local_rank))
            cm.denoise_begin(noise[0].numpy(), (F, H, W), sigmas[0], text, None)
            mn = [0]

            def mstep():
                cm.denoise_step(pairs[mn[0] % len(pairs)][0], pairs[mn[0] % len(pairs)][1], mn[0] % len(pairs))
                mn[0] += 1
            tm = ev_time(cm, sm_, mstep, 6, warm=3)
            lm = cm.denoise_get_latent()
            extras["qint8_materialised"] = dict(desc="int8 group-64 quantised weights, dequantised values materialised as bf16 at load time "
                                                     "(ltx_set_quant_storage(1): same results as qint8, footprint of the bf16 model)",
                                                ms_per_step=tm, steps_per_s=1e3 / tm, latent_finite=bool(np.isfinite(lm).all()))
            cm.close()
        except Exception as e:   # report, do not hide
            extras["qint8"] = dict(error=str(e))
        # ---- the rows either side of the denoise loop (SURVEY 8f): dual audio/video model, VAE encoder, latent upscaler
        def ev1(fn, strm, reps=3, warm=1):
            for _ in range(warm):
                fn()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(strm)
            for _ in range(reps):
                fn()
            b.record(strm)
            torch.cuda.synchronize()
            return a.elapsed_time(b) / reps
        try:
            ca = LtxContext(LTXTransformerConfig(), local_rank)
            ca.init_random_weights(17, seed=101)          # video + audio / cross-modal tensors: the full LTX2Transformer
            ca.finalize_weights()
            sa = torch.cuda.ExternalStream(ca.stream, device=torch.device("cuda", local_rank))
            Ta = 26                                       # 25 frames at 24 fps = 1.04 s of audio at 25 latent frames / s
            vl = torch.randn(1, N, CIN, generator=g).bfloat16().cuda()
            al = torch.randn(1, Ta, CIN, generator=g).bfloat16().cuda()
            tx = text.cuda()
            sg2 = torch.tensor([0.7, 0.7], device="cuda")
            ov = torch.empty(1, N, CIN, device="cuda")
            oa = torch.empty(1, Ta, CIN, device="cuda")
            torch.cuda.synchronize()

            def av_step():
                ca._check(ca.lib.ltx_av_forward_dev(ca.handle, vl.data_ptr(), 1, al.data_ptr(), 1, tx.data_ptr(), tx.data_ptr(), 1,
                                                    sg2.data_ptr(), sg2.data_ptr() + 4, None, None, N, Ta, S, F, H, W, 77,
                                                    ov.data_ptr(), oa.data_ptr()))
            av_step()
            ta_ms = ev1(av_step, sa, reps=4)
            ca.set_profiling(True)
            av_step()
            pa = ca.get_profile()
            ca.set_profiling(False)
            extras["av_dual_forward"] = dict(
                desc=f"LTX2Transformer (dual audio/video, 48 blocks, D=4096 + Da=2048) forward, N={N} video + {Ta} audio tokens, S={S}",
                ms_per_forward=ta_ms, forwards_per_s=1e3 / ta_ms, outputs_finite=bool(torch.isfinite(ov).all() and torch.isfinite(oa).all()),
                kernel_classes={k: v for k, v in pa.items() if v["launches"]})
            ca.close()
            del vl, al, tx, ov, oa
        except Exception as e:
            extras["av_dual_forward"] = dict(error=str(e))
        try:
            ce = LtxContext(LTXTransformerConfig(), local_rank)
            ce.init_random_weights(2 | 4 | 8, seed=103)   # VAE decoder (latent statistics), encoder, upscaler
            ce.finalize_weights()
            se_ = torch.cuda.ExternalStream(ce.stream, device=torch.device("cuda", local_rank))
            px = (torch.rand(3, 1, 32 * H, 32 * W, generator=g) * 2 - 1).cuda()
            zl = torch.empty(CIN, 1, H, W, device="cuda")
            px25 = (torch.rand(3, 8 * (F - 1) + 1, 32 * H, 32 * W, generator=g) * 2 - 1).cuda()
            zl25 = torch.empty(CIN, F, H, W, device="cuda")
            lat1 = torch.randn(CIN, 33, H, W, generator=g).cuda()     # stage-1 latent of BASELINE config 5 (768x512x257)
            lat2 = torch.empty(CIN, 33, 2 * H, 2 * W, device="cuda")
            torch.cuda.synchronize()
            t_img = ev1(lambda: ce.vae_encode_dev(px.data_ptr(), (1, 32 * H, 32 * W), zl.data_ptr()), se_)
            t_clip = ev1(lambda: ce.vae_encode_dev(px25.data_ptr(), (8 * (F - 1) + 1, 32 * H, 32 * W), zl25.data_ptr()), se_)
            t_up = ev1(lambda: ce.upscale_latent_dev(lat1.data_ptr(), (33, H, W), lat2.data_ptr()), se_)
            ce.set_profiling(True)
            ce.upscale_latent_dev(lat1.data_ptr(), (33, H, W), lat2.data_ptr())
            pu = ce.get_profile()
            ce.set_profiling(False)
            extras["vae_encode"] = dict(desc="VideoEncoder + latent normalisation, 768x512", image_ms=t_img, clip_25f_ms=t_clip,
                                        clip_frames_per_s=(8 * (F - 1) + 1) * 1e3 / t_clip)
            extras["latent_upscale"] = dict(desc="upsampleLatents 33x16x24 -> 33x32x48 (stage switch of BASELINE config 5)",
                                            ms=t_up, kernel_classes={k: v for k, v in pu.items() if v["launches"]})
            ce.close()
            del px, zl, px25, zl25, lat1, lat2
        except Exception as e:
            extras["vae_encode"] = dict(error=str(e))
        tg = time_guided(ctx, stream)
        tv, _ = time_vae121(ctx, stream)
        extras["guided_cfg3"] = dict(desc="dev CFG 4.0 + STG 0.5 (3 forwards/step), 1 GPU", ms_per_step=tg, steps_per_s=1e3 / tg)
        extras["vae_121f"] = dict(desc="VAE decode 768x512x121f, 1 GPU", ms_per_decode=tv, frames_per_s=121e3 / tv)
        if not args.no_parity:
            try:
                parity.update(parity_vs_oracle(local_rank))
            except Exception as e:   # report, do not hide
                parity["oracle_check_error"] = str(e)
        if not args.no_cfg5:
            ctx.close()
            torch.cuda.empty_cache()
            try:
                extras["cfg5_two_stage"] = dict(desc="BASELINE config 5, int8 weights, 1 GPU: stage 1 N=12672 x 8 steps, device-resident "
                                                     "upscale + AdaIN + re-noise, stage 2 N=50688 x 3 steps", **cfg5_two_stage(1))
            except Exception as e:
                extras["cfg5_two_stage"] = dict(error=str(e))
    else:
        # sharded VAE on the same communicator: 25 frames (above, `vae`) and the 121-frame clip, both against this rank's 1-GPU decode
        tv, fr121 = time_vae121(ctx, stream, fetch=True)
        ctx.dist_shutdown()
        single = torch.empty(n_frames, 32 * H, 32 * W, 3, device="cuda")
        ctx.vae_decode_dev(lat_dev.data_ptr(), (F, H, W), single.data_ptr())
        torch.cuda.synchronize()
        s25 = single.cpu().numpy()
        _, s121 = time_vae121(ctx, stream, reps=1, fetch=True)
        d25, d121 = float(np.abs(frames_multi - s25).max()), float(np.abs(fr121 - s121).max())
        parity["vae_sharded_vs_single_gpu"] = dict(max_abs_diff_25f=d25, max_abs_diff_121f=d121,
                                                   bit_identical=bool(d25 == 0.0 and d121 == 0.0), tol=1e-4,
                                                   ok=all_ok(d25 <= 1e-4 and d121 <= 1e-4))
        del single, s25, s121, fr121
        extras["vae_121f_sharded"] = dict(desc=f"VAE decode 768x512x121f, {world} temporal shards + halo exchange",
                                          ms_per_decode=tv, frames_per_s=121e3 / tv)
        # pass-parallel guidance (BASELINE config 3): the conditional / unconditional / STG forwards on different GPU groups,
        # each group sequence-parallel over world / groups GPUs; best grouping reported, every grouping checked
        best = None
        for groups in (2, 3):
            if world % groups or HEADS % (world // groups):
                continue
            ltxdist.init_context(ctx, sp_size=world // groups, pass_groups=groups)
            out_g = full_denoise(ctx, guided=True)
            err = _rel_l2(out_g, single_guided)
            tg = time_guided(ctx, stream)
            ctx.dist_shutdown()
            rec = dict(groups=groups, sp=world // groups, ms_per_step=tg, steps_per_s=1e3 / tg, rel_l2_vs_single_gpu=err,
                       ok=all_ok(err <= 3e-3))
            extras.setdefault("guided_cfg3_groupings", []).append(rec)
            if best is None or tg < best["ms_per_step"]:
                best = rec
        ltxdist.init_context(ctx, sp_size=world, pass_groups=1)     # all passes sequentially, each over all GPUs
        out_g = full_denoise(ctx, guided=True)
        err = _rel_l2(out_g, single_guided)
        tg = time_guided(ctx, stream)
        ctx.dist_shutdown()
        rec = dict(groups=1, sp=world, ms_per_step=tg, steps_per_s=1e3 / tg, rel_l2_vs_single_gpu=err, ok=all_ok(err <= 3e-3))
        extras.setdefault("guided_cfg3_groupings", []).append(rec)
        if best is None or tg < best["ms_per_step"]:
            best = rec
        extras["guided_cfg3_pass_parallel"] = dict(desc="dev CFG 4.0 + STG 0.5 (BASELINE config 3), best grouping of passes x Ulysses", **best)
        parity["guided_pass_groups_vs_single_gpu"] = dict(ok=all(r["ok"] for r in extras["guided_cfg3_groupings"]), tol=3e-3, steps=3,
                                                          worst_rel_l2=max(r["rel_l2_vs_single_gpu"] for r in extras["guided_cfg3_groupings"]))
        if world >= 4 and not args.no_cfg5:
            ctx.close()
            torch.cuda.empty_cache()
            try:
                extras["cfg5_two_stage"] = dict(desc=f"BASELINE config 5, int8 weights, Ulysses sp={world}: stage 1 N=12672 x 8 steps, "
                                                     "upscale + AdaIN + re-noise, stage 2 N=50688 x 3 steps", **cfg5_two_stage(world))
            except Exception as e:   # report, do not hide
                extras["cfg5_two_stage"] = dict(error=str(e))

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        # the latent ltx_denoise_get_latent returns after the last timed step, and the frames of the last timed VAE decode
        dump_outputs(args.dump_outputs, dict(latent=timed_latent, vae_frames_sample=frames_sample))

    pk = peaks()
    # DRAM traffic of the dominant kernel: bytes of ONE FFN-in launch from the newest committed `ncu --set full` capture
    traffic, traffic_note = None, None
    try:
        import csv
        import glob
        cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r0*_gemm*ffn_in_ncu_raw.csv")))
        src = cands[-1]
        rows = list(csv.reader(open(src)))
        hdr, units, last = rows[0], rows[1], rows[-1]

        def _bytes(k):
            v, u = float(last[hdr.index(k)].replace(",", "")), units[hdr.index(k)]
            return v * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[u]
        traffic = _bytes("dram__bytes_read.sum") + _bytes("dram__bytes_write.sum")
        traffic_note = ("bytes of ONE FFN-in launch (M=1536,N=16384,K=4096; algorithmic 197.1e6), read from the committed capture "
                        f"profiles/{os.path.basename(src)} -- a citation of that capture's tree, not measured in this run")
    except Exception:
        pass
    gemm = prof["gemm"]
    achieved = gemm["flops"] / (gemm["ms"] * 1e-3) / 1e12 if gemm["ms"] > 0 else 0.0
    conv = vprof["conv3d"]
    cpu_sec, cores, desc = cpu_port_step_seconds(1, 1) if not args.no_cpu_baseline else (float("nan"), 0, "skipped")
    cpu_full = None
    if world == 1 and not args.no_cpu_baseline and not args.no_cpu_full_step:
        try:
            cpu_full = cpu_port_full_step_seconds()
        except Exception as e:
            cpu_full = f"failed: {e}"
    class_ms = sum(v["ms"] for v in prof.values())
    parity["all_ok"] = all((v if isinstance(v, bool) else v.get("ok", True)) for v in parity.values() if isinstance(v, (bool, dict)))
    line = dict(
        metric="dit_steps_per_s", value=value, unit="steps/s", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
        ms_per_step=ms_per_step, higher_is_better=True, scaling="strong", vs_baseline=None, dtype="bf16", data="synthetic",
        config=dict(workload=WORKLOAD, weights="bf16 random-init on the device, fp32 residual stream",
                    global_batch=1, l2="weights per step (26 GB) >> 126 MB L2; no flush needed",
                    parallelism=f"ulysses sp={world} (one video, tokens sharded, heads sharded inside self-attention)" if world > 1 else "single",
                    flops_per_step=dit_flops_per_step(N, S), step_tflops=dit_flops_per_step(N, S) / (ms_per_step * 1e-3) / 1e12),
        e2e=dict(value=1e3 / e2e_ms, unit="steps/s", ms_per_step=e2e_ms, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                 path="ltx_dit_forward + ltx_guided_euler_step with pinned host buffers (text cached by context_key)"),
        gpu_launches=int(launches),
        parity=parity,
        roofline=dict(bound="tensor", kernel="gemm_bf16_2cta / gemm_bf16_tcgen05 / gemm_swapab (all GEMM launches of one step)", achieved=achieved,
                      peak=pk["tflops_sustained"], unit="TFLOP/s", frac=achieved / pk["tflops_sustained"], traffic=traffic,
                      traffic_note=traffic_note,
                      peak_source=pk["source"] + ", sustained bf16", launches=gemm["launches"], ms=gemm["ms"]),
        kernel_classes={k: v for k, v in prof.items() if v["launches"]},
        step_minus_class_sum_ms=ms_per_step - class_ms,
        # the class times come from ONE eagerly launched step with an event pair around every scope: the GPU idles between the
        # scopes, draws less power and clocks higher than inside the back-to-back timed steps (see `clocks`: power-capped), so the
        # class sum can be SHORTER than the timed step; profiled_step_ms is that eager step's own device time, end to end
        profiled_step_ms=profiled_step_ms, profiled_step_minus_class_sum_ms=profiled_step_ms - class_ms,
        cpu_baseline=dict(value=1.0 / cpu_sec if cpu_sec == cpu_sec else None, unit="steps/s", cores=cores, kind="port", sample=desc,
                          extrapolated=True, full_step_s=cpu_full,
                          full_step_steps_per_s=(1.0 / cpu_full) if isinstance(cpu_full, float) else None),
        vae=dict(metric="vae_frames_per_s", value=n_frames / (vae_ms * 1e-3), unit="frames/s", ms_per_decode=vae_ms,
                 frames=n_frames, e2e_value=n_frames / (vae_e2e_ms * 1e-3), e2e_ms=vae_e2e_ms,
                 parallelism=f"{min(world, F)} temporal shards + per-conv halo exchange" if world > 1 else "single",
                 conv_tflops=conv["flops"] / (conv["ms"] * 1e-3) / 1e12 if conv["ms"] > 0 else None,
                 conv_frac_of_peak=(conv["flops"] / (conv["ms"] * 1e-3) / 1e12) / pk["tflops_sustained"] if conv["ms"] > 0 else None,
                 kernel_classes={k: v for k, v in vprof.items() if v["launches"]}),
        clocks=clocks,
        extras=extras,
    )
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def _positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {v}")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_positive_int, default=16, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what they computed to DIR/<name>.npy (float32): the denoised latent "
                         "and a seeded sample of the decoded frames")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cfg5", action="store_true", help="skip the two-stage 1536x1024x257 extra")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cpu-full-step", action="store_true", help="skip the one true 48-block CPU step (~26 s)")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-process oracle checks (N = 1)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours (the reference arm times one block of the CPU port and keeps no outputs)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
