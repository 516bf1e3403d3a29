"""Micro-benchmark of the attention kernel on the DiT shapes.  R launches queued behind a 1 GB memset on the library's stream
(the host's issue latency is not in the number), CUDA events around the R.  ATT_SHAPES=a,b runs only those shapes;
LTX_ATT_PAIR=0 / 1 forces one CTA per query tile / CTA pairs."""
import os
import math, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ltx_video_swift_mlx_b200  # noqa
from ltx_video_swift_mlx_b200.context import LtxContext, LTXTransformerConfig
ctx = LtxContext(LTXTransformerConfig(num_layers=1, num_attention_heads=1), 0)
stream = torch.cuda.ExternalStream(ctx.stream)
big = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
for name, B, H, Nq, Nk, masked in [("self1536", 1, 32, 1536, 1536, False), ("cross1536", 1, 32, 1536, 1024, False), ("cross1536m", 1, 32, 1536, 1024, True),
                                   ("cfg_self", 2, 32, 1536, 1536, False), ("cfg_cross", 2, 32, 1536, 1024, False),
                                   ("sp8_self", 1, 4, 1536, 1536, False), ("sp8_cross", 1, 32, 192, 1024, False),
                                   ("self6144", 1, 32, 6144, 6144, False), ("self12672", 1, 32, 12672, 12672, False)]:
    if os.environ.get("ATT_SHAPES") and name not in os.environ["ATT_SHAPES"].split(","):
        continue
    D = H * 128
    R = 8 if Nq <= 6144 else 3
    q = torch.randn(B * Nq, D, device="cuda").bfloat16(); k = torch.randn(B * Nk, D, device="cuda").bfloat16()
    ldv = (Nk + 7) // 8 * 8
    vt = torch.randn(D, B * ldv, device="cuda").bfloat16(); o = torch.empty(B * Nq, D, device="cuda", dtype=torch.bfloat16)
    bias = torch.zeros(B, Nk, device="cuda") if masked else None
    def run():
        ctx._check(ctx.lib.ltx_op_attention(ctx.handle, q.data_ptr(), k.data_ptr(), vt.data_ptr(), ldv,
                                            bias.data_ptr() if masked else None, o.data_ptr(), B, H, Nq, Nk, 1 / math.sqrt(128)))
    run(); ctx.sync(); ts = []
    for _ in range(5):
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            big.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(R):
            run()
        e1.record(stream); ctx.sync(); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1) / R)
    t = sorted(ts)[len(ts) // 2]
    print(f"{name:10s}: {t*1e3:8.1f} us  {4*B*H*Nq*Nk*128/t/1e9:8.1f} TFLOP/s", flush=True)
