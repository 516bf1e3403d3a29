"""FP8 mode (ltx_set_precision(ctx, 8)): the e4m3 row quantiser equals its CPU restatement bit for bit, the FP8 pair GEMM
equals the float64 product of its decoded operands within a bound set from the first B200 run, the FP8 DiT matches the oracle
restatement of FP8 mode, and the mode keeps the bit-for-bit identities of the bf16 mode."""
import math

import numpy as np
import pytest
import torch

from fp8_ref import decode, fp8_blocks, quantize_rows
from helpers import O, product, rel_l2, small_dit_config

pytestmark = pytest.mark.gpu
LTX_ERR_UNSUPPORTED = 5

# Bounds set from the first B200 run (NVIDIA B200, 1000 W power limit); the measured value is beside each.
GEMM_BOUND = 1e-6        # |C - ref| / sum_k |a_k b_k| over all elements, fp32 outputs; measured 2.1e-7 (K up to 16384): the
                         # kind::f8f6f4 accumulator behaves as fp32 here, not as the ~14-bit accumulator reported for Hopper
FWD_ORACLE_TOL = 2e-2    # velocity rel-L2 against the FP8 restatement of the oracle; measured 1.2e-2 (D = 256), 5.7e-3 (D = 4096)
FWD_DRIFT_TOL = 5e-2     # velocity rel-L2 against the bf16 forward (the format's own drift); measured 2.2e-2 / 1.3e-2
LOOP_TOL = 3e-2          # 4-step guided loop against the oracle loop in FP8 mode; measured 1.75e-2 (plain and image-to-video)
MEASURED = {}


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k, v in sorted(MEASURED.items()):
        print(f"fp8 measured {k}: {v:.3e}")


@pytest.fixture(scope="module")
def ctx():
    c = product().LtxContext(product().LTXTransformerConfig(num_layers=1, num_attention_heads=1), 0)
    yield c
    c.close()


def _note(key, v):
    MEASURED[key] = max(MEASURED.get(key, 0.0), float(v))


def _rows(M, K, seed):
    """bf16 rows with the edge cases of the format: 448, 449, amax 1e-3, a zero row, a 1e4-times-median outlier, tiny values."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(M, K, generator=g) * torch.pow(2.0, torch.randint(-8, 8, (M, 1), generator=g).float())
    x[0] = x[0] / x[0].abs().max() * 448.0
    x[0, 5] = 448.0
    x[1, 3] = 449.0
    x[2] = x[2] / x[2].abs().max() * 1e-3
    x[3] = 0.0
    x[4, 7] = 1e4 * float(x[4].abs().median())
    x[5] = x[5] * 1e-30
    return x.bfloat16()


@pytest.mark.parametrize("M,K,pitch", [(40, 256, 0), (24, 4096, 0), (9, 16384, 0), (37, 272, 48)])
def test_quantize_rows_matches_restatement(ctx, M, K, pitch):
    x = _rows(M, K, M + K)
    ld = K + pitch
    buf = torch.full((M, ld), 3e38, dtype=torch.bfloat16)   # the pitch padding must not be read
    buf[:, :K] = x
    buf = buf.cuda()
    codes = torch.full((M, K), 0xAA, dtype=torch.uint8, device="cuda")
    scales = torch.full((M,), float("nan"), device="cuda")
    torch.cuda.synchronize()
    ctx._check(ctx.lib.ltx_op_quantize_fp8(ctx.handle, buf.data_ptr(), M, K, ld, codes.data_ptr(), scales.data_ptr()))
    ctx.sync()
    q, s = quantize_rows(x)
    assert torch.equal(scales.cpu().double(), s)
    assert torch.equal(codes.cpu(), q)
    assert float(s[3]) == 1.0 and int(q[3].abs().sum()) == 0


def _operands(M, N, K, seed):
    g = torch.Generator().manual_seed(seed)
    a = (torch.randn(M, K, generator=g) * torch.pow(2.0, torch.randint(-4, 4, (M, 1), generator=g).float())).bfloat16()
    w = (torch.randn(N, K, generator=g) / math.sqrt(K)).bfloat16()
    qa, sa = quantize_rows(a)
    qw, sw = quantize_rows(w)
    bias = torch.randn(N, generator=g) * 0.1
    da, dw = decode(qa, sa), decode(qw, sw)
    ref = da @ dw.t() + bias.double()
    denom = da.abs() @ dw.abs().t()
    dev = [t.cuda() for t in (qa, sa.float(), qw, sw.float(), bias)]
    return dev, ref, denom


def _gelu(x):
    return 0.5 * x * (1 + torch.tanh(math.sqrt(2 / math.pi) * (x + 0.044715 * x ** 3)))


@pytest.mark.parametrize("M,N,K,mode,bn", [
    (1, 264, 272, 3, 0), (33, 520, 4112, 3, 64), (300, 264, 1040, 3, 176), (1536, 4096, 4096, 3, 0),
    (1536, 1000, 4112, 3, 256), (1536, 4096, 16384, 3, 0), (3072, 4096, 4096, 3, 0),
    (300, 520, 272, 0, 128), (1, 256, 4096, 0, 0), (1536, 12288, 4096, 0, 256), (33, 264, 1040, 1, 96),
    (1536, 16384, 4096, 1, 0), (1536, 520, 4112, 4, 208), (300, 1000, 272, 4, 80),
])
def test_gemm_fp8_against_decoded_product(ctx, M, N, K, mode, bn):
    (qa, sa, qw, sw, bias), ref, denom = _operands(M, N, K, M * 7 + N + K + mode)
    dt = torch.float32 if mode == 3 else torch.bfloat16
    out = torch.full((M + 2, N), float("nan"), device="cuda", dtype=dt)    # guard rows either side
    torch.cuda.synchronize()
    ctx._check(ctx.lib.ltx_op_gemm_fp8(ctx.handle, qa.data_ptr(), sa.data_ptr(), qw.data_ptr(), sw.data_ptr(), bias.data_ptr(),
                                       out[1].data_ptr(), M, N, K, mode, bn))
    ctx.sync()
    o = out.double().cpu()
    assert torch.isnan(o[0]).all() and torch.isnan(o[M + 1]).all()
    o = o[1:M + 1]
    assert torch.isfinite(o).all()
    if mode == 3:
        err = float(((o - ref).abs() / denom).max())
        _note("gemm_err_over_sum_abs", err)
        assert err <= GEMM_BOUND, err
        return
    act = {0: lambda t: t, 1: _gelu, 4: lambda t: t * torch.sigmoid(t)}[mode]
    want = act(ref)
    # the product bound (activations are 1.13-Lipschitz at most), half a bf16 ulp, and the approximate tanh / exp of the epilogue
    tol = 1.2 * GEMM_BOUND * denom + 2.0 ** -8 * want.abs() + (1e-3 * ref.abs() if mode != 0 else 0.0)
    assert bool(((o - want).abs() <= tol).all()), float(((o - want).abs() - tol).max())


@pytest.mark.parametrize("M", [300, 1536])
def test_gemm_fp8_vt_split_and_gate_residual_restate_the_plain_product(ctx, M):
    D = 256
    N, K = 3 * D, 1040
    (qa, sa, qw, sw, bias), _, _ = _operands(M, N, K, M + 11)
    args = (qa.data_ptr(), sa.data_ptr(), qw.data_ptr(), sw.data_ptr(), bias.data_ptr())
    plain = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    plain32 = torch.empty(M, N, device="cuda")
    ldt = (M + 7) // 8 * 8
    qk = torch.full((M, 2 * D), float("nan"), device="cuda", dtype=torch.bfloat16)
    vt = torch.full((D, ldt), float("nan"), device="cuda", dtype=torch.bfloat16)
    g = torch.Generator(device="cuda").manual_seed(M)
    x0 = torch.randn(M, N, device="cuda", generator=g)
    ga, gb = torch.randn(N, device="cuda", generator=g), torch.randn(N, device="cuda", generator=g)
    x = x0.clone()
    shadow = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    torch.cuda.synchronize()
    ctx._check(ctx.lib.ltx_op_gemm_fp8(ctx.handle, *args, plain.data_ptr(), M, N, K, 0, 256))
    ctx._check(ctx.lib.ltx_op_gemm_fp8(ctx.handle, *args, plain32.data_ptr(), M, N, K, 3, 256))
    ctx._check(ctx.lib.ltx_op_gemm_fp8_ex(ctx.handle, *args, qk.data_ptr(), vt.data_ptr(), 2 * D, ldt, None, None, None, None,
                                          M, N, K, 256))
    ctx._check(ctx.lib.ltx_op_gemm_fp8_ex(ctx.handle, *args, None, None, 0, 0, x.data_ptr(), ga.data_ptr(), gb.data_ptr(),
                                          shadow.data_ptr(), M, N, K, 0))
    ctx.sync()
    assert torch.equal(qk, plain[:, :2 * D])
    assert torch.equal(vt[:, :M], plain[:, 2 * D:].t())
    want = x0 + plain32 * (ga + gb)
    assert torch.allclose(x, want, rtol=1e-6, atol=1e-6)
    assert torch.equal(shadow, x.bfloat16())


def _ctx(pcfg, w, precision):
    c = product().LtxContext(pcfg, 0)
    if precision != 16:
        c.set_precision(precision)
    c.load_weights(w)
    c.finalize_weights()
    return c


def _inputs(ocfg, N, S, seed, B=1):
    g = torch.Generator().manual_seed(seed)
    lat = torch.randn(B, N, ocfg.in_channels, generator=g).bfloat16()
    cx = torch.randn(B, S, ocfg.caption_channels, generator=g)
    return lat, (cx / cx.pow(2).mean(-1, keepdim=True).sqrt()).bfloat16()


@pytest.mark.parametrize("layers,heads,fhw,S", [(2, 2, (2, 4, 6), 40), (1, 32, (6, 16, 16), 1024)])
def test_fp8_forward_against_oracle_and_bf16(layers, heads, fhw, S):
    ocfg, pcfg = small_dit_config(layers, heads)
    w = O.make_dit_weights(ocfg, 40 + layers)
    N = fhw[0] * fhw[1] * fhw[2]
    lat, cx = _inputs(ocfg, N, S, 7)
    sig = torch.tensor([0.6])
    c8 = _ctx(pcfg, w, 8)
    out8 = c8.dit_forward(lat, cx, sig.numpy(), None, fhw)
    c8.close()
    c16 = _ctx(pcfg, w, 16)
    out16 = c16.dit_forward(lat, cx, sig.numpy(), None, fhw)
    c16.close()
    assert np.isfinite(out8).all()
    with fp8_blocks():
        ref8 = O.dit_forward(w, ocfg, lat.float(), cx.float(), sig, None, fhw)
    e_or, e_drift = rel_l2(out8, ref8), rel_l2(out8, out16)
    _note(f"forward_vs_fp8_oracle_D{heads * 128}", e_or)
    _note(f"forward_drift_vs_bf16_D{heads * 128}", e_drift)
    assert e_or <= FWD_ORACLE_TOL, e_or
    assert 1e-5 < e_drift <= FWD_DRIFT_TOL, e_drift


def test_fp8_mode_bit_identities():
    ocfg, pcfg = small_dit_config(3, 2)
    w = O.make_dit_weights(ocfg, 51)
    c = _ctx(pcfg, w, 8)
    fhw, S = (3, 4, 8), 40
    g = torch.Generator().manual_seed(52)
    noise = torch.randn(1, 128, *fhw, generator=g)
    _, cx = _inputs(ocfg, 96, S, 53)
    _, ncx = _inputs(ocfg, 96, S, 54)
    sigmas = O.set_timesteps(4, False, 96)

    def loop(**kw):
        c.denoise_begin(noise[0].numpy(), fhw, sigmas[0], cx, None, ncx, None)
        for i in range(len(sigmas) - 1):
            c.denoise_step(sigmas[i], sigmas[i + 1], i, cfg_scale=3.0, rescale_phi=0.5, **kw)
        return c.denoise_get_latent()

    c.set_graphs(False)
    sep = loop(batched_cfg=False)
    bat = loop(batched_cfg=True)
    np.testing.assert_array_equal(bat, sep)                       # batched CFG = two B = 1 passes
    stg_share = loop(stg_scale=0.4, stg_blocks=(1,), share_stg_prefix=True)
    stg_full = loop(stg_scale=0.4, stg_blocks=(1,), share_stg_prefix=False)
    np.testing.assert_array_equal(stg_share, stg_full)            # STG prefix sharing changes nothing
    c.set_graphs(True)
    graphed = loop(batched_cfg=True)
    captures, replays = c.graph_stats()
    assert captures >= 1 and replays >= 1, (captures, replays)
    np.testing.assert_array_equal(graphed, bat)                   # captured-graph replay = eager
    c.close()


@pytest.mark.parametrize("i2v", [False, True])
def test_fp8_guided_loop_against_oracle(i2v):
    ocfg, pcfg = small_dit_config(2, 2)
    w = O.make_dit_weights(ocfg, 61)
    c = _ctx(pcfg, w, 8)
    fhw, S = (3, 4, 6), 40
    g = torch.Generator().manual_seed(62)
    noise = torch.randn(1, 128, *fhw, generator=g)
    _, cx = _inputs(ocfg, 72, S, 63)
    _, ncx = _inputs(ocfg, 72, S, 64)
    sigmas = O.set_timesteps(4, False, 72)
    kw = dict(neg_context=ncx.float(), cfg_scale=3.0, phi=0.5)
    if i2v:
        init = noise * sigmas[0]
        init[:, :, 0] = torch.randn(128, 4, 6, generator=g) * 0.5
        with fp8_blocks():
            ref = O.denoise_loop(w, ocfg, noise, cx.float(), None, sigmas, frame0_conditioned=True, init_latent=init, **kw)
        c.denoise_begin((init[0] / sigmas[0]).numpy(), fhw, sigmas[0], cx, None, ncx, None)
    else:
        with fp8_blocks():
            ref = O.denoise_loop(w, ocfg, noise, cx.float(), None, sigmas, **kw)
        c.denoise_begin(noise[0].numpy(), fhw, sigmas[0], cx, None, ncx, None)
    for i in range(len(sigmas) - 1):
        c.denoise_step(sigmas[i], sigmas[i + 1], i, cfg_scale=3.0, rescale_phi=0.5, i2v_frame0_conditioned=i2v)
    out = c.denoise_get_latent()
    c.close()
    err = rel_l2(out, ref[0])
    _note(f"loop_vs_fp8_oracle_i2v{int(i2v)}", err)
    assert err <= LOOP_TOL, err


def _code(fn):
    with pytest.raises(product().LtxError) as e:
        fn()
    return e.value.code


def test_fp8_mode_refusals():
    ocfg, pcfg = small_dit_config(1, 2)
    w = O.make_dit_weights(ocfg, 71)
    c = product().LtxContext(pcfg, 0)
    c.set_precision(8)
    c.load_weights(w)
    assert _code(lambda: c.finalize_weights(quant_bits=8)) == LTX_ERR_UNSUPPORTED
    assert _code(lambda: c.finalize_weights(quant_bits=4)) == LTX_ERR_UNSUPPORTED
    c.finalize_weights()                                   # the refused calls left the weights as they were
    assert _code(lambda: c.set_precision(16)) != 0
    lat, cx = _inputs(ocfg, 48, 40, 72)
    fhw = (2, 4, 6)
    v = c.dit_forward(lat, cx, np.array([0.5], dtype=np.float32), None, fhw)
    assert np.isfinite(v).all()
    # the dual audio/video model: refused before anything is read or written
    out_v = np.full((1, 48, 128), 7.0, dtype=np.float32)
    out_a = np.full((1, 11, 128), 7.0, dtype=np.float32)
    al = np.zeros((1, 11, 128), dtype=np.float32)
    lv = lat.float().numpy()
    cxf = cx.float().numpy()
    P = lambda a: a.ctypes.data   # noqa: E731
    sig = np.array([0.5], dtype=np.float32)
    lib, h = c.lib, c.handle
    assert lib.ltx_av_forward(h, P(lv), 0, P(al), 0, P(cxf), P(cxf), 0, 0.5, 0.5, None, None, 48, 11, 40, *fhw, 0, P(out_v),
                              P(out_a)) == LTX_ERR_UNSUPPORTED
    assert lib.ltx_av_forward_batch(h, P(lv), 0, P(al), 0, P(cxf), P(cxf), 0, P(sig), 0, P(sig), None, None, 1, 48, 11, 40, *fhw, 0,
                                    P(out_v), P(out_a)) == LTX_ERR_UNSUPPORTED
    noise = np.zeros((128, *fhw), dtype=np.float32)
    anoise = np.zeros((11, 128), dtype=np.float32)
    assert lib.ltx_av_denoise_begin(h, P(noise), P(anoise), *fhw, 11, 1.0, P(cxf), P(cxf), 0, None, None, None, None,
                                    40) == LTX_ERR_UNSUPPORTED
    assert (out_v == 7.0).all() and (out_a == 7.0).all()
    c.close()
    # ltx_set_precision(8) after the DiT weights are loaded
    c = product().LtxContext(pcfg, 0)
    c.load_weights(w)
    assert _code(lambda: c.set_precision(8)) == LTX_ERR_UNSUPPORTED
    c.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_fp8_mode_refuses_sequence_parallel_forward():
    import threading
    ocfg, pcfg = small_dit_config(1, 2)
    w = O.make_dit_weights(ocfg, 81)
    ctxs = [product().LtxContext(pcfg, d) for d in (0, 1)]
    for cc in ctxs:
        cc.set_precision(8)
        cc.load_weights(w)
        cc.finalize_weights()
    product().LtxContext.dist_init_local(ctxs, sp_size=2, pass_groups=1)
    lat, cx = _inputs(ocfg, 48, 40, 82)
    res = {}

    def work(i):
        try:
            ctxs[i].dit_forward(lat, cx, np.array([0.5], dtype=np.float32), None, (2, 4, 6))
            res[i] = 0
        except product().LtxError as e:
            res[i] = e.code

    ts = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=300)
    assert res == {0: LTX_ERR_UNSUPPORTED, 1: LTX_ERR_UNSUPPORTED}
    ts = [threading.Thread(target=cc.dist_shutdown) for cc in ctxs]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=120)
    for cc in ctxs:
        cc.close()
