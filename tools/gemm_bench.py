"""Micro-benchmark of the tcgen05 GEMM on the DiT shapes (device time via CUDA events on the library stream)."""
import os
import math, os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ltx_video_swift_mlx_b200  # noqa
from ltx_video_swift_mlx_b200.context import LtxContext, LTXTransformerConfig

ctx = LtxContext(LTXTransformerConfig(num_layers=1, num_attention_heads=1), 0)
stream = torch.cuda.ExternalStream(ctx.stream)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
shapes = [("qk", 1536, 8192, 4096, 0), ("vT", 4096, 1536, 4096, 0), ("out", 1536, 4096, 4096, 2), ("ffn_in", 1536, 16384, 4096, 1),
          ("ffn_out", 1536, 4096, 16384, 2), ("proj_out", 1536, 128, 4096, 3), ("big", 8192, 8192, 8192, 0)]
def bench_q(name, M, N, K, bits, bn=0):
    A = torch.randn(M, K, device="cuda").bfloat16()
    Wt = (torch.randn(N, K, device="cuda") / math.sqrt(K)).bfloat16()
    q = torch.empty(N, K * bits // 8, device="cuda", dtype=torch.uint8); s = torch.empty(K // 64, N, device="cuda"); b = torch.empty(K // 64, N, device="cuda")
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16); bias = torch.zeros(N, device="cuda")
    torch.cuda.synchronize()
    ctx._check(ctx.lib.ltx_op_quantize(ctx.handle, Wt.data_ptr(), N, K, bits, q.data_ptr(), s.data_ptr(), b.data_ptr()))
    def run():
        ctx._check(ctx.lib.ltx_op_gemm_q(ctx.handle, A.data_ptr(), q.data_ptr(), s.data_ptr(), b.data_ptr(), bits, bias.data_ptr(), out.data_ptr(), M, N, K, 0, bn))
    for _ in range(3): run()
    ctx.sync(); ts = []
    for _ in range(10):
        flush.zero_(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); run(); e1.record(stream); ctx.sync(); ts.append(e0.elapsed_time(e1))
    t = sorted(ts)[len(ts) // 2]
    print(f"{name:9s} M={M} N={N} K={K} int{bits} bn={bn:5d}: {t*1e3:8.1f} us  {2*M*N*K/t/1e9:8.1f} TFLOP/s", flush=True)

for nm, M, N, K in ([("qk", 1536, 8192, 4096), ("out", 1536, 4096, 4096), ("ffn_in", 1536, 16384, 4096), ("ffn_out", 1536, 4096, 16384)] if '--quant' in sys.argv else []):
    for bits in (8, 4):
        # the dequant-fused kernel (ltx_op_gemm_q gives no bf16 panel, so M = 1536 stays on it): 0 = wave-fitted width, else forced
        for bn in (0, 256, 224, 192, 176, 128):
            bench_q(nm, M, N, K, bits, bn)

# M = 1536 shapes of the DiT block: the pair kernel at forced widths (1000 + width, 1000 = fitted); 0 = the library's own choice.  Timed like the small-M sweep below: R launches on R cold weight
# buffers queued behind a 2 GB memset, so the host's issue latency is not in the number.
shapes2 = [("qkv", 1536, 12288, 4096, 0), ("out", 1536, 4096, 4096, 2), ("q2", 1536, 4096, 4096, 0), ("ffn_in", 1536, 16384, 4096, 1),
           ("ffn_out", 1536, 4096, 16384, 2), ("cfg_qkv", 3072, 12288, 4096, 0), ("cfg_out", 3072, 4096, 4096, 2), ("big", 8192, 8192, 8192, 0)]
if '--bf16' in sys.argv:
    big = torch.empty(2 << 30, dtype=torch.uint8, device="cuda")
for name, M, N, K, mode in (shapes2 if '--bf16' in sys.argv else []):
    R = 4 if name == "big" else 8
    A = torch.randn(M, K, device="cuda").bfloat16()
    Bs = [(torch.randn(N, K, device="cuda") / math.sqrt(K)).bfloat16() for _ in range(R)]
    bias = torch.randn(max(M, N), device="cuda")
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    x = torch.zeros(M, N, device="cuda")
    g = torch.ones(N, device="cuda")
    for bn in [0, 1000, 1256, 1224, 1176, 1112]:
        def run(B):
            if mode == 2:
                ctx._check(ctx.lib.ltx_op_gemm_resid(ctx.handle, A.data_ptr(), B.data_ptr(), bias.data_ptr(), x.data_ptr(),
                                                     g.data_ptr(), g.data_ptr(), None, M, N, K, 0.5))
            else:
                ctx._check(ctx.lib.ltx_op_gemm(ctx.handle, A.data_ptr(), B.data_ptr(), bias.data_ptr(), out.data_ptr(), M, N, K, mode, bn))
        if mode == 2:
            if bn: os.environ["LTX_GEMM_FORCE_BN"] = str(bn)
            else: os.environ.pop("LTX_GEMM_FORCE_BN", None)
        run(Bs[0])
        ctx.sync()
        ts = []
        for _ in range(5):
            torch.cuda.synchronize()
            with torch.cuda.stream(stream):
                big.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for B in Bs:
                run(B)
            e1.record(stream); ctx.sync(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / R)
        t = sorted(ts)[len(ts) // 2]
        os.environ.pop("LTX_GEMM_FORCE_BN", None)
        print(f"{name:9s} M={M} N={N} K={K} mode={mode} bn={bn:5d}: {t*1e3:8.1f} us  {2*M*N*K/t/1e9:8.1f} TFLOP/s", flush=True)

# few activation rows (an Ulysses shard of the config-2 video: 192 rows at sp = 8, 384 at sp = 4): tile kernels (bn = 0) against
# the swap-AB weight-streaming kernel with (-2) / without (-3) split-K; GB/s = weight bytes / time.
# These kernels run 10-50 us, less than the host needs to issue one (ctypes + two tensor-map encodes + launch), so timing a
# single launch between two events measures the host.  Instead: a 2 GB memset is queued first on the library's stream (~0.6 ms:
# it flushes the L2 and lets the host run ahead), then R = 8 launches on R different weight buffers (each one cold), events
# around the 8.
small = [("qk", 8192, 4096, 0), ("v/q2", 4096, 4096, 0), ("out", 4096, 4096, 2), ("ffn_in", 16384, 4096, 1), ("ffn_out", 4096, 16384, 2)]
if '--small' in sys.argv:
    big = torch.empty(2 << 30, dtype=torch.uint8, device="cuda")
    R = 8
for M in ([192, 384, 96, 512, 768] if '--small' in sys.argv else []):
    for name, N, K, mode in small:
        A = torch.randn(M, K, device="cuda").bfloat16()
        Bs = [(torch.randn(N, K, device="cuda") / math.sqrt(K)).bfloat16() for _ in range(R)]
        bias = torch.randn(max(M, N), device="cuda")
        out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
        x = torch.zeros(M, N, device="cuda")
        g = torch.ones(N, device="cuda")
        for bn in ([0, -2, -3] if mode != 2 else [0, -2]):
            if bn != 0 and M > 512:
                continue
            def run(B):
                if mode == 2:   # gate * residual epilogue: ltx_op_gemm_resid attaches the workspace itself (swap-AB for 32 < M <= 512)
                    ctx._check(ctx.lib.ltx_op_gemm_resid(ctx.handle, A.data_ptr(), B.data_ptr(), bias.data_ptr(), x.data_ptr(),
                                                         g.data_ptr(), g.data_ptr(), None, M, N, K, 0.5))
                else:
                    ctx._check(ctx.lib.ltx_op_gemm(ctx.handle, A.data_ptr(), B.data_ptr(), bias.data_ptr(), out.data_ptr(), M, N, K, mode, bn))
            if mode == 2:
                if bn == 0: os.environ["LTX_GEMM_FORCE_BN"] = "1000"    # force the pair tile kernel (fitted width) for the comparison
                else: os.environ.pop("LTX_GEMM_FORCE_BN", None)
            run(Bs[0])
            ctx.sync()
            ts = []
            for _ in range(5):
                torch.cuda.synchronize()
                with torch.cuda.stream(stream):
                    big.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for B in Bs:
                    run(B)
                e1.record(stream); ctx.sync(); torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1) / R)
            t = sorted(ts)[len(ts) // 2]
            os.environ.pop("LTX_GEMM_FORCE_BN", None)
            print(f"{name:8s} M={M:4d} N={N:5d} K={K:5d} mode={mode} kernel={'tile' if bn == 0 else ('swapab+splitK' if bn == -2 else 'swapab')}: "
                  f"{t*1e3:8.1f} us  {2*M*N*K/t/1e9:7.1f} TFLOP/s  {N*K*2/t/1e6:7.1f} GB/s of weights", flush=True)
