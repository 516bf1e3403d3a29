"""VAE decode to fp32 frames against the decode straight to 8-bit frames (RGB8, I420) on one GPU.

The full decoder (LTX-2 channel plan, seeded random weights) at 768x512 with 25 and 121 frames (latents 4 / 16 x 16 x 24).
Per round the three output formats run in turn, in one process:
  resident     -- ltx_vae_decode_dev / ltx_vae_decode_u8_dev into device buffers: --iters decodes timed with CUDA events on
                  the context's stream, and with a host clock around the same decodes ending in a synchronise;
  host buffer  -- ltx_vae_decode / ltx_vae_decode_u8 from and into page-locked host buffers (ltx_host_alloc): latent upload,
                  decode, frame download and the synchronise, timed per call with events and with a host clock.
The median over --rounds is reported with the spread.  Each format is warmed up at each shape first.  The script also checks
that the RGB8 frames equal (uint8)(fp32 frames * 255) and the I420 frames equal ltx_frames_to_u8 of the fp32 frames, and
prints the GPU name and power limit (nvidia-smi, same process) beside the numbers.

Usage (GPU box): python tools/vae_u8_bench.py [--rounds 3] [--iters 3] [--out FILE]"""
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
from ltx_video_swift_mlx_b200 import _lib  # noqa: E402
from ltx_video_swift_mlx_b200.context import LtxContext, LTXTransformerConfig  # noqa: E402

H, W = 16, 24          # latent grid of 512 x 768
FORMATS = ("f32", "rgb8", "i420")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clk = (s.strip() for s in q.split(","))
    return dict(gpu=name, power_limit=power, max_sm_clock=clk)


def summary(xs):
    return dict(median=statistics.median(xs), min=min(xs), max=max(xs), n=len(xs))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    info = gpu_info()
    print(f"{info['gpu']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}", flush=True)
    ctx = LtxContext(LTXTransformerConfig(), 0)
    ctx.init_random_weights(2, seed=5)
    ctx.finalize_weights()
    stream = torch.cuda.ExternalStream(ctx.stream)
    codes = {"rgb8": _lib.LTX_FRAMES_RGB8, "i420": _lib.LTX_FRAMES_I420}
    result = dict(info, rounds=args.rounds, iters=args.iters, shapes={})
    for Fp in (4, 16):
        F, Ho, Wo = 8 * (Fp - 1) + 1, 32 * H, 32 * W
        lat = torch.randn(128, Fp, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(Fp)) * 0.5
        lat_host = ctx.pinned_empty((128, Fp, H, W))
        lat_host[...] = lat.cpu().numpy()
        dev = {"f32": torch.empty(F, Ho, Wo, 3, device="cuda")}
        host = {"f32": ctx.pinned_empty((F, Ho, Wo, 3))}
        for fmt, code in codes.items():
            dev[fmt] = torch.empty(ctx.lib.ltx_frames_u8_bytes(F, Ho, Wo, code), dtype=torch.uint8, device="cuda")
            host[fmt] = ctx.pinned_empty(ctx.frames_u8_shape(F, Ho, Wo, fmt), np.uint8)
        torch.cuda.synchronize()

        def resident(fmt):
            if fmt == "f32":
                ctx.vae_decode_dev(lat.data_ptr(), (Fp, H, W), dev[fmt].data_ptr())
            else:
                ctx.vae_decode_u8_dev(lat.data_ptr(), (Fp, H, W), dev[fmt].data_ptr(), fmt)

        def host_buffer(fmt):
            if fmt == "f32":
                ctx.vae_decode(lat_host, out=host[fmt])
            else:
                ctx.vae_decode_u8(lat_host, fmt, out=host[fmt])

        for fmt in FORMATS:   # warm-up (module loads, buffer growth)
            resident(fmt)
            host_buffer(fmt)
        ctx.sync()
        ref = dev["f32"].cpu().numpy()
        checks = dict(rgb8_equals_trunc_f32=bool(np.array_equal(dev["rgb8"].cpu().numpy().reshape(ref.shape),
                                                                (ref * np.float32(255)).astype(np.uint8))),
                      i420_equals_converter=bool(np.array_equal(dev["i420"].cpu().numpy().ravel(),
                                                                ctx.frames_to_u8(ref, "i420").ravel())),
                      host_equals_resident=all(np.array_equal(host[f].ravel().view(np.uint8), dev[f].cpu().numpy().ravel().view(np.uint8))
                                               for f in FORMATS))
        del ref
        rec = {f: dict(resident_event_ms=[], resident_host_ms=[], hostbuf_event_ms=[], hostbuf_host_ms=[]) for f in FORMATS}
        for _ in range(args.rounds):
            for fmt in FORMATS:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ctx.sync()
                t0 = time.perf_counter()
                a.record(stream)
                for _ in range(args.iters):
                    resident(fmt)
                b.record(stream)
                ctx.sync()
                t1 = time.perf_counter()
                rec[fmt]["resident_event_ms"].append(a.elapsed_time(b) / args.iters)
                rec[fmt]["resident_host_ms"].append((t1 - t0) * 1e3 / args.iters)
                ev, hc = [], []
                for _ in range(args.iters):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    t0 = time.perf_counter()
                    a.record(stream)
                    host_buffer(fmt)    # synchronises before it returns
                    b.record(stream)
                    t1 = time.perf_counter()
                    b.synchronize()
                    ev.append(a.elapsed_time(b))
                    hc.append((t1 - t0) * 1e3)
                rec[fmt]["hostbuf_event_ms"].append(statistics.median(ev))
                rec[fmt]["hostbuf_host_ms"].append(statistics.median(hc))
        out_bytes = {f: int(host[f].nbytes) for f in FORMATS}
        shape = dict(frames=F, height=Ho, width=Wo, output_bytes=out_bytes, checks=checks,
                     formats={f: {k: summary(v) for k, v in rec[f].items()} for f in FORMATS})
        result["shapes"][f"{Wo}x{Ho}x{F}"] = shape
        print(f"{Wo}x{Ho}x{F}: checks {checks}", flush=True)
        for f in FORMATS:
            s = shape["formats"][f]
            print(f"  {f:5s} {out_bytes[f] / 1e6:7.1f} MB  resident {s['resident_event_ms']['median']:7.2f} ms (events) "
                  f"{s['resident_host_ms']['median']:7.2f} ms (host)   host buffer {s['hostbuf_event_ms']['median']:7.2f} ms (events) "
                  f"{s['hostbuf_host_ms']['median']:7.2f} ms (host) [{s['hostbuf_host_ms']['min']:.2f}-{s['hostbuf_host_ms']['max']:.2f}]",
                  flush=True)
        del dev, host, lat_host
    ctx.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
