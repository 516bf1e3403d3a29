"""VAE decode timing (25-frame and 121-frame clips, 768x512) with the per-class profile; LTX_CONV_PAIR=0 runs one CTA per
voxel tile, LTX_CONV_SLAB=0 per-tap stages."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ltx_video_swift_mlx_b200  # noqa
from ltx_video_swift_mlx_b200.context import LtxContext, LTXTransformerConfig
ctx = LtxContext(LTXTransformerConfig(), 0)
ctx.init_random_weights(2, seed=5)
ctx.finalize_weights()
stream = torch.cuda.ExternalStream(ctx.stream)
for F in (4, 16):
    lat = torch.randn(128, F, 16, 24, device="cuda")
    out = torch.empty(8 * (F - 1) + 1, 512, 768, 3, device="cuda")
    torch.cuda.synchronize()
    for _ in range(2):
        ctx.vae_decode_dev(lat.data_ptr(), (F, 16, 24), out.data_ptr())
    ctx.sync()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(5):
        ctx.vae_decode_dev(lat.data_ptr(), (F, 16, 24), out.data_ptr())
    b.record(stream); ctx.sync(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 5
    ctx.set_profiling(True)
    ctx.vae_decode_dev(lat.data_ptr(), (F, 16, 24), out.data_ptr())
    p = ctx.get_profile()
    ctx.set_profiling(False)
    conv = p["conv3d"]
    print(f"{8*(F-1)+1:4d} frames: {ms:7.2f} ms  {(8*(F-1)+1)*1e3/ms:7.1f} frames/s   conv {conv['ms']:.2f} ms {conv['flops']/conv['ms']/1e9:.0f} TFLOP/s, "
          + ", ".join(f"{k} {v['ms']:.2f}" for k, v in p.items() if v['launches'] and k != 'conv3d'), flush=True)
