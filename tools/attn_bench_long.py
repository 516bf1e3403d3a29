import math, sys, os, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ltx_video_swift_mlx_b200  # noqa
from ltx_video_swift_mlx_b200.context import LtxContext, LTXTransformerConfig
ctx = LtxContext(LTXTransformerConfig(num_layers=1, num_attention_heads=1), 0)
stream = torch.cuda.ExternalStream(ctx.stream)
for H, N in [(8, 50688), (4, 50688), (32, 25344)]:
    D = H * 128
    q = torch.randn(N, D, device="cuda").bfloat16(); k = torch.randn(N, D, device="cuda").bfloat16()
    vt = torch.randn(D, N, device="cuda").bfloat16(); o = torch.empty(N, D, device="cuda", dtype=torch.bfloat16)
    run = lambda: ctx._check(ctx.lib.ltx_op_attention(ctx.handle, q.data_ptr(), k.data_ptr(), vt.data_ptr(), N, None, o.data_ptr(), 1, H, N, N, 1 / math.sqrt(128)))
    run(); ctx.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream); run(); run(); e1.record(stream); ctx.sync()
    t = e0.elapsed_time(e1) / 2
    print(f"H={H} N={N}: {t:8.2f} ms  {4*H*N*N*128/t/1e9:8.1f} TFLOP/s", flush=True)
