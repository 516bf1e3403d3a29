"""Out-of-bounds net for the kernels with ragged edges (compute-sanitizer is closed on the GPU pool, so this is the memcheck we
have): every output buffer carries NaN guard rows / columns that must still be NaN after the call, every input is surrounded
by NaN that must never reach a valid output, and the valid region must match the reference.  Covers the attention kernel
(ragged query / key counts, batch boundaries), the row kernels (row counts that do not fill a CTA), the implicit-GEMM
convolution (ragged spatial tiles, narrow Cout) and the column-blocked / partially column-blocked GEMM epilogues that the
sequence-parallel path stores into peer memory with."""
import math

import pytest
import torch

from helpers import O, product, rel_l2

pytestmark = pytest.mark.gpu
NAN = float("nan")


@pytest.fixture(scope="module")
def ctx():
    c = product().LtxContext(product().LTXTransformerConfig(num_layers=1, num_attention_heads=1), 0)
    yield c
    c.close()


@pytest.mark.parametrize("B,H,HD,Nq,Nk", [(1, 2, 128, 1, 1), (1, 2, 128, 129, 65), (2, 2, 128, 100, 100), (3, 1, 128, 257, 63),
                                          (2, 4, 64, 70, 130), (1, 1, 128, 127, 1537)])
def test_attention_guards(ctx, B, H, HD, Nq, Nk):
    D = H * HD
    g = torch.Generator(device="cuda").manual_seed(B + H + Nq + Nk)
    pad = 3
    # q / k buffers: valid rows followed by NaN rows (a tile that ran past B*N rows would pull them in)
    q = torch.full((B * Nq + pad, D), NAN, device="cuda", dtype=torch.bfloat16)
    k = torch.full((B * Nk + pad, D), NAN, device="cuda", dtype=torch.bfloat16)
    q[:B * Nq] = torch.randn(B * Nq, D, device="cuda", generator=g).bfloat16()
    k[:B * Nk] = torch.randn(B * Nk, D, device="cuda", generator=g).bfloat16()
    v = torch.randn(B * Nk, D, device="cuda", generator=g).bfloat16()
    ldv = (Nk + 7) // 8 * 8 + 8
    vt = torch.full((D, B * ldv), NAN, device="cuda", dtype=torch.bfloat16)            # NaN between the batches' columns
    for b in range(B):
        vt[:, b * ldv: b * ldv + Nk] = v[b * Nk:(b + 1) * Nk].t()
    o = torch.full((B * Nq + pad, D), NAN, device="cuda", dtype=torch.bfloat16)
    scale = 1 / math.sqrt(HD)
    torch.cuda.synchronize()
    if HD == 128:
        ctx._check(ctx.lib.ltx_op_attention(ctx.handle, q.data_ptr(), k.data_ptr(), vt.data_ptr(), ldv, None, o.data_ptr(), B, H, Nq, Nk, scale))
    else:
        ctx._check(ctx.lib.ltx_op_attention_hd(ctx.handle, q.data_ptr(), k.data_ptr(), vt.data_ptr(), ldv, None, o.data_ptr(), B, H, HD, Nq, Nk, scale))
    ctx.sync()
    assert torch.isnan(o[B * Nq:].float()).all(), "rows past B*Nq were written"
    assert torch.isfinite(o[:B * Nq].float()).all(), "padding (NaN) reached a valid output"
    qh = q[:B * Nq].float().view(B, Nq, H, HD).permute(0, 2, 1, 3)
    kh = k[:B * Nk].float().view(B, Nk, H, HD).permute(0, 2, 1, 3)
    vh = v.float().view(B, Nk, H, HD).permute(0, 2, 1, 3)
    ref = (torch.softmax(qh @ kh.transpose(-1, -2) * scale, -1) @ vh).permute(0, 2, 1, 3).reshape(B * Nq, D)
    assert rel_l2(o[:B * Nq].float(), ref) <= 1e-2


@pytest.mark.parametrize("M,D", [(1, 4096), (3, 4096), (5, 4096), (193, 4096), (7, 512), (2, 256)])
def test_row_kernels_guards(ctx, M, D):
    """rmsnorm_mod and qknorm_rope with row counts below / not a multiple of the CTA count (persistent streaming CTAs at
    D = 4096, one row per CTA otherwise): nothing is written behind the M rows and every row is written."""
    g = torch.Generator(device="cuda").manual_seed(M + D)
    pad = 5
    x = torch.full((M + pad, D), NAN, device="cuda")
    x[:M] = torch.randn(M, D, device="cuda", generator=g)
    ts, tc, as_, ac = [torch.randn(D, device="cuda", generator=g) * 0.3 for _ in range(4)]
    out = torch.full((M + pad, D), NAN, device="cuda", dtype=torch.bfloat16)
    torch.cuda.synchronize()
    ctx._check(ctx.lib.ltx_op_rmsnorm_mod(ctx.handle, x.data_ptr(), out.data_ptr(), M, D, ts.data_ptr(), tc.data_ptr(),
                                          as_.data_ptr(), ac.data_ptr(), 1e-6, 0))
    ctx.sync()
    assert torch.isnan(out[M:].float()).all() and torch.isfinite(out[:M].float()).all()
    ref = O.rms_norm(x[:M], None, 1e-6) * (1 + tc + ac) + ts + as_
    assert rel_l2(out[:M].float(), ref) <= 4e-3
    # q/k norm + RoPE in place: the rows behind M must stay NaN
    heads = D // 128
    y = torch.full((M + pad, D), NAN, device="cuda", dtype=torch.bfloat16)
    y0 = torch.randn(M, D, device="cuda", generator=g).bfloat16()
    y[:M] = y0
    w = 1 + 0.1 * torch.randn(D, device="cuda", generator=g)
    cos = torch.rand(M, D // 2, device="cuda", generator=g)
    sin = torch.sqrt(1 - cos * cos)
    torch.cuda.synchronize()
    ctx._check(ctx.lib.ltx_op_qknorm_rope(ctx.handle, y.data_ptr(), M, D, w.data_ptr(), cos.data_ptr(), sin.data_ptr(), M, 1e-6))
    ctx.sync()
    assert torch.isnan(y[M:].float()).all() and torch.isfinite(y[:M].float()).all()
    n = O.rms_norm(y0.float(), w, 1e-6).view(M, heads, 2, 64)                  # split RoPE: (x1, x2) = the two halves of a head
    c3, s3 = cos.view(M, heads, 64), sin.view(M, heads, 64)
    ref = torch.stack([n[:, :, 0] * c3 - n[:, :, 1] * s3, n[:, :, 1] * c3 + n[:, :, 0] * s3], 2).reshape(M, D)
    assert rel_l2(y[:M].float(), ref) <= 4e-3


def test_row_kernels_refuse_misaligned_rows(ctx):
    """At D = 4096 the rows (and the RoPE tables) reach the kernels by bulk copies, which need 16-byte aligned sources: a
    pointer off that alignment is refused with code 2, and nothing is written."""
    from ltx_video_swift_mlx_b200._lib import LtxError
    M, D = 3, 4096
    x = torch.randn(M * D + 4, device="cuda")
    tb = torch.zeros(4, D, device="cuda")
    out = torch.full((M, D), NAN, device="cuda", dtype=torch.bfloat16)
    torch.cuda.synchronize()
    with pytest.raises(LtxError) as e:
        ctx._check(ctx.lib.ltx_op_rmsnorm_mod(ctx.handle, x.data_ptr() + 4, out.data_ptr(), M, D, tb[0].data_ptr(), tb[1].data_ptr(),
                                              tb[2].data_ptr(), tb[3].data_ptr(), 1e-6, 0))
    assert e.value.code == 2
    y = torch.randn(M * D + 8, device="cuda").bfloat16()
    y0 = y.clone()
    w = torch.ones(D, device="cuda")
    tabs = torch.rand(2, M * D // 2 + 4, device="cuda")
    for yp, cp in ((y.data_ptr() + 2, tabs[0].data_ptr()), (y.data_ptr(), tabs[0].data_ptr() + 4)):
        with pytest.raises(LtxError) as e:
            ctx._check(ctx.lib.ltx_op_qknorm_rope(ctx.handle, yp, M, D, w.data_ptr(), cp, tabs[1].data_ptr(), M, 1e-6))
        assert e.value.code == 2
    ctx.sync()
    assert torch.isnan(out.float()).all() and torch.equal(y, y0)


@pytest.mark.parametrize("T,H,W,Cin,Cout", [(1, 3, 5, 64, 48), (2, 7, 9, 64, 64), (3, 5, 130, 128, 128), (1, 17, 3, 128, 256)])
def test_conv3d_guards(ctx, T, H, W, Cin, Cout):
    """Spatial extents that do not fill the 128-voxel tiles, Cout below / at the tile width: nothing lands behind the output
    volume and every voxel is written."""
    g = torch.Generator().manual_seed(T * H * W + Cin + Cout)
    x = torch.randn(1, Cin, T, H, W, generator=g)
    w = O.bf16_round(torch.randn(Cout, Cin, 3, 3, 3, generator=g) / math.sqrt(27 * Cin))
    b = torch.randn(Cout, generator=g) * 0.1
    ref = O.conv3d_full(O.bf16_round(x), w, b, causal=False)[0].permute(1, 2, 3, 0)
    x_cl = x[0].permute(1, 2, 3, 0).contiguous().cuda()
    w_dev = w.permute(2, 3, 4, 0, 1).reshape(27, Cout, Cin).contiguous().cuda().bfloat16()
    b_dev = b.cuda()
    n = T * H * W * Cout
    buf = torch.full((n + 4096,), NAN, device="cuda")
    torch.cuda.synchronize()
    ctx._check(ctx.lib.ltx_op_conv3d(ctx.handle, x_cl.data_ptr(), w_dev.data_ptr(), b_dev.data_ptr(), buf.data_ptr(), T, H, W, Cin, Cout, 0))
    ctx.sync()
    assert torch.isnan(buf[n:]).all(), "the convolution wrote behind its output volume"
    out = buf[:n].view(T, H, W, Cout)
    assert torch.isfinite(out).all()
    assert rel_l2(out, ref) <= 1e-4


@pytest.mark.parametrize("M,bn", [(192, -2), (192, 0), (1536, 0), (100, -2), (700, 0)])
def test_gemm_column_blocked_epilogue_guards(ctx, M, bn):
    """The Ulysses send layout: columns >= col_from leave in blocks of `cb` columns, block j to its own base (a peer's buffer in
    the real path), the columns before col_from stay row-major -- q | k | v as one projection.  Each destination carries a
    guard row; nothing else may be touched."""
    N, K, cb, col_from = 768, 256, 128, 512
    g = torch.Generator(device="cuda").manual_seed(M + bn)
    A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    Wt = (torch.randn(N, K, device="cuda", generator=g) / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, device="cuda", generator=g)
    plain = torch.full((M + 1, col_from), NAN, device="cuda", dtype=torch.bfloat16)
    nblk = (N - col_from) // cb
    blocks = torch.full((nblk, M + 1, cb), NAN, device="cuda", dtype=torch.bfloat16)
    torch.cuda.synchronize()
    ctx._check(ctx.lib.ltx_op_gemm_blocked(ctx.handle, A.data_ptr(), Wt.data_ptr(), bias.data_ptr(), plain.data_ptr(), blocks.data_ptr(),
                                           M, N, K, col_from, cb, (M + 1) * cb, bn))
    ctx.sync()
    ref = A.float() @ Wt.float().t() + bias
    assert torch.isnan(plain[M].float()).all() and torch.isnan(blocks[:, M].float()).all()
    assert rel_l2(plain[:M].float(), ref[:, :col_from]) <= 4e-3
    for j in range(nblk):
        assert rel_l2(blocks[j, :M].float(), ref[:, col_from + j * cb: col_from + (j + 1) * cb]) <= 4e-3
