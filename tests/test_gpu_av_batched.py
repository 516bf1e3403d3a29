"""The dual audio / video transformer on a batch of two items (ltx_av_forward_batch) and the audio + video loop's batched
guidance pass: oracle parity at B = 2, each item bit-identical to its B = 1 call (the audio stream's 2 x Ta rows on the 64-row
form of the weight-streaming GEMM, per-item modulation rows in the row kernels), the batched loop equal to the two-pass loop,
and the refusals."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import O, product, rel_l2

pytestmark = pytest.mark.gpu
TOL = 1e-2   # the bound of the B = 1 oracle parity test


def _setup(layers, heads, aheads, seed, caption=192, quant_bits=16):
    ctxmod = product()
    ocfg = O.DiTConfig(num_layers=layers, num_heads=heads, head_dim=128, caption_channels=caption)
    av = O.AVConfig(audio_heads=aheads)
    pcfg = ctxmod.LTXTransformerConfig(num_layers=layers, num_attention_heads=heads, caption_channels=caption,
                                       audio_num_attention_heads=aheads)
    w = O.make_av_weights(ocfg, av, seed)
    ctx = ctxmod.LtxContext(pcfg, 0)
    ctx.load_weights(w)
    ctx.finalize_weights(quant_bits=quant_bits)
    return ocfg, av, w, ctx


def _text(g, B, S, caption):
    t = torch.randn(B, S, caption, generator=g)
    return (t / t.pow(2).mean(-1, keepdim=True).sqrt()).bfloat16()


def _batch(fhw, Ta, S, caption, seed, masked=(0, 0)):
    """Two items with different latents, prompts and masks (masked[b] leading key positions of item b are off)."""
    g = torch.Generator().manual_seed(seed)
    N = fhw[0] * fhw[1] * fhw[2]
    vl = torch.randn(2, N, 128, generator=g).bfloat16()
    al = torch.randn(2, Ta, 128, generator=g).bfloat16()
    vc, ac = _text(g, 2, S, caption), _text(g, 2, S, caption)
    mask = None
    if any(masked):
        mask = torch.ones(2, S, dtype=torch.int32)
        for b, m in enumerate(masked):
            mask[b, :m] = 0
    return vl, al, vc, ac, mask


def _item(t, b):
    return None if t is None else t[b:b + 1]


def _check_items_bit_identical(ctx, vl, al, vc, ac, vs, as_, mask, fhw):
    """The B = 2 call, then each item alone at B = 1: equal bit for bit."""
    ov, oa = ctx.av_forward(vl, al, vc, ac, vs, as_, fhw, mask, mask)
    assert ov.shape[0] == 2 and oa.shape[0] == 2
    assert np.isfinite(ov).all() and np.isfinite(oa).all()
    for b in range(2):
        vsb = vs[b:b + 1] if vs.ndim == 2 else float(vs[b])
        iv, ia = ctx.av_forward(_item(vl, b), _item(al, b), _item(vc, b), _item(ac, b), vsb, float(as_[b]), fhw,
                                _item(mask, b), _item(mask, b))
        assert np.isfinite(iv).all() and np.isfinite(ia).all()
        assert np.array_equal(ov[b:b + 1], iv), (b, np.abs(ov[b:b + 1] - iv).max())
        assert np.array_equal(oa[b:b + 1], ia), (b, np.abs(oa[b:b + 1] - ia).max())
    return ov, oa


@pytest.mark.parametrize("layers,heads,aheads,fhw,Ta,S,masked,per_token", [
    (2, 2, 2, (2, 4, 6), 11, 40, (5, 0), False),
    (2, 2, 4, (3, 4, 4), 26, 24, (3, 7), False),      # 52 audio rows: the 64-row weight-streaming form
    (2, 2, 2, (3, 4, 6), 11, 40, (0, 0), True),       # video sigmas [2, N]
    (2, 2, 4, (2, 4, 6), 26, 40, (4, 4), True),
])
def test_av_batch_matches_oracle(layers, heads, aheads, fhw, Ta, S, masked, per_token):
    ocfg, av, w, ctx = _setup(layers, heads, aheads, seed=layers * 100 + heads * 10 + aheads + 7)
    vl, al, vc, ac, mask = _batch(fhw, Ta, S, 192, 31, masked)
    N = fhw[0] * fhw[1] * fhw[2]
    if per_token:
        vs = torch.stack([torch.linspace(0.3, 0.8, N), torch.linspace(0.9, 0.4, N)])
        vs[:, :fhw[1] * fhw[2]] = 0.0
    else:
        vs = torch.tensor([0.7, 0.35])
    as_ = torch.tensor([0.55, 0.9])
    rv, ra = O.av_dit_forward(w, ocfg, av, vl.float(), al.float(), vc.float(), ac.float(), vs, as_, mask, mask, fhw, Ta)
    ov, oa = ctx.av_forward(vl, al, vc, ac, vs.numpy(), as_.numpy(), fhw, mask, mask)
    assert np.isfinite(ov).all() and np.isfinite(oa).all()
    for b in range(2):
        assert rel_l2(ov[b], rv[b]) <= TOL, (b, rel_l2(ov[b], rv[b]))
        assert rel_l2(oa[b], ra[b]) <= TOL, (b, rel_l2(oa[b], ra[b]))
    # the two items really differ (different prompts and sigmas), and a cached text K / V call gives the same numbers
    assert rel_l2(ov[0], ov[1]) > 1e-2
    ov2, oa2 = ctx.av_forward(vl, al, vc, ac, vs.numpy(), as_.numpy(), fhw, mask, mask, context_key=11)
    ov3, oa3 = ctx.av_forward(vl, al, vc, ac, vs.numpy(), as_.numpy(), fhw, mask, mask, context_key=11)
    assert np.array_equal(ov2, ov) and np.array_equal(oa2, oa) and np.array_equal(ov3, ov) and np.array_equal(oa3, oa)
    ctx.close()


@pytest.mark.parametrize("fhw,Ta,S,masked,per_token", [
    ((2, 4, 6), 11, 40, (0, 0), False),     # N = 48, Ta = 11: both audio items on the 32-row form, video on the tile kernel
    ((2, 4, 6), 26, 40, (0, 0), False),     # 52 audio rows: the 64-row form (V^T with per-item column blocks, per-item gates)
    ((3, 4, 6), 17, 24, (0, 0), False),     # 34 audio rows
    ((2, 4, 6), 32, 24, (6, 0), False),     # 64 audio rows, mask on one prompt only
    ((3, 4, 8), 26, 40, (6, 9), False),     # 96 -> 192 video rows: one-CTA tiles at B = 1, CTA pairs at B = 2; both masked
    ((2, 4, 6), 26, 40, (0, 0), True),      # per-token sigmas
])
def test_av_batch_items_bit_identical_to_single_calls(fhw, Ta, S, masked, per_token):
    ocfg, av, w, ctx = _setup(2, 2, 2, seed=41)
    vl, al, vc, ac, mask = _batch(fhw, Ta, S, 192, 17, masked)
    N = fhw[0] * fhw[1] * fhw[2]
    if per_token:
        vs = np.stack([np.linspace(0.2, 0.9, N), np.linspace(0.8, 0.3, N)]).astype(np.float32)
        vs[:, :fhw[1] * fhw[2]] = 0.0
    else:
        vs = np.array([0.8, 0.45], dtype=np.float32)
    _check_items_bit_identical(ctx, vl, al, vc, ac, vs, np.array([0.6, 0.25], dtype=np.float32), mask, fhw)
    ctx.close()


def test_av_batch_int8_items_bit_identical():
    """int8 codes through the dequant-fused GEMM (N = 48 -> 96 video rows stay below the 257-row panel switch)."""
    _, _, _, ctx = _setup(2, 2, 2, seed=43, quant_bits=8)
    fhw, Ta, S = (2, 4, 6), 26, 40
    vl, al, vc, ac, mask = _batch(fhw, Ta, S, 192, 19, (3, 0))
    _check_items_bit_identical(ctx, vl, al, vc, ac, np.array([0.7, 0.4], dtype=np.float32),
                               np.array([0.7, 0.3], dtype=np.float32), mask, fhw)
    ctx.close()


def test_av_batch_full_width_block_bit_identical():
    """One block at the LTX-2 widths (D = 4096, Da = 2048) and the flagship shape (N = 1536, Ta = 26, S = 1024): the
    D-specialised row kernels, the pair GEMMs at 3072 rows and the 64-row weight-streaming form at 52 rows."""
    ctxmod = product()
    ctx = ctxmod.LtxContext(ctxmod.LTXTransformerConfig(num_layers=1), 0)
    ctx.init_random_weights(17, seed=3)
    ctx.finalize_weights()
    fhw, Ta, S = (4, 16, 24), 26, 1024
    vl, al, vc, ac, mask = _batch(fhw, Ta, S, 3840, 23, (100, 0))
    ov, oa = _check_items_bit_identical(ctx, vl, al, vc, ac, np.array([0.9, 0.5], dtype=np.float32),
                                        np.array([0.9, 0.5], dtype=np.float32), mask, fhw)
    assert ov.std() > 0.05 and oa.std() > 0.05
    ctx.close()


def _loop_inputs(seed, fhw, Ta, S, i2v):
    g = torch.Generator().manual_seed(seed)
    vn, an = torch.randn(1, 128, *fhw, generator=g), torch.randn(1, Ta, 128, generator=g)
    img = torch.randn(1, 128, 1, fhw[1], fhw[2], generator=g) if i2v else None
    vc, ac, nvc, nac = (_text(g, 1, S, 192) for _ in range(4))
    mask = torch.ones(1, S, dtype=torch.int32)
    mask[:, :3] = 0
    nmask = torch.ones(1, S, dtype=torch.int32)
    nmask[:, :7] = 0
    return vn, an, img, vc, ac, nvc, nac, mask, nmask


@pytest.mark.parametrize("i2v", [False, True])
def test_av_batched_cfg_loop_equals_two_pass_loop_and_oracle(i2v):
    """A 4-step CFG + rescale loop with masked prompts: the batched guidance forward gives the two-pass loop's latents bit for
    bit, stays within the multi-step bound of the oracle loop, and really ran (fewer GEMM launches per step)."""
    from ltx_video_swift_mlx_b200.pipeline import denoise_av_resident
    ocfg, av, w, ctx = _setup(2, 2, 2, seed=81)
    fhw, Ta, S = (3, 4, 6), 26, 40
    vn, an, img, vc, ac, nvc, nac, mask, nmask = _loop_inputs(9, fhw, Ta, S, i2v)
    sig = O.set_timesteps(8, True, 72)[3:8]
    kw = dict(cfg_scale=3.0, guidance_rescale=0.7, image_latent=None if img is None else img.numpy())
    launches = {}
    out = {}
    for batched in (True, False):
        ctx.set_profiling(True)
        before = ctx.get_profile()["gemm"]["launches"]
        out[batched] = denoise_av_resident(ctx, vn.numpy(), an.numpy(), vc, ac, mask, sig, nvc, nac, nmask, batched_cfg=batched, **kw)
        launches[batched] = ctx.get_profile()["gemm"]["launches"] - before
        ctx.set_profiling(False)
    (bv, ba), (sv, sa) = out[True], out[False]
    assert np.isfinite(bv).all() and np.isfinite(ba).all()
    assert np.array_equal(bv, sv) and np.array_equal(ba, sa)
    assert 0 < launches[True] < launches[False], launches
    rv, ra = O.av_denoise_loop(w, ocfg, av, vn, an, vc.float(), ac.float(), mask, sig, nvc.float(), nac.float(), nmask,
                               cfg_scale=3.0, phi=0.7, image_latent=img)
    assert rel_l2(bv, rv) <= 2e-2 and rel_l2(ba, ra) <= 2e-2, (rel_l2(bv, rv), rel_l2(ba, ra))
    ctx.close()


def test_av_batch_refusals_write_nothing():
    from ltx_video_swift_mlx_b200._lib import LTX_BF16, LtxError
    _, _, _, ctx = _setup(1, 2, 2, seed=3)
    fhw, Ta, S = (2, 4, 6), 11, 24
    N = 48
    g = torch.Generator().manual_seed(1)
    vl3, al3 = torch.randn(3, N, 128, generator=g).bfloat16(), torch.randn(3, Ta, 128, generator=g).bfloat16()
    vc3, ac3 = _text(g, 3, S, 192), _text(g, 3, S, 192)
    with pytest.raises(LtxError) as e:                                   # B = 3: unsupported
        ctx.av_forward(vl3, al3, vc3, ac3, np.full(3, 0.5, np.float32), np.full(3, 0.5, np.float32), fhw)
    assert e.value.code == 5
    with pytest.raises(LtxError) as e:                                   # audio batch of 1 against a video batch of 2
        ctx.av_forward(vl3[:2], al3[:1], vc3[:2], ac3[:2], np.full(2, 0.5, np.float32), np.full(2, 0.5, np.float32), fhw)
    assert e.value.code == 2
    with pytest.raises(LtxError) as e:                                   # three sigmas for two items
        ctx.av_forward(vl3[:2], al3[:2], vc3[:2], ac3[:2], np.full(3, 0.5, np.float32), np.full(2, 0.5, np.float32), fhw)
    assert e.value.code == 2
    # the C entry points directly, outputs NaN-prefilled: a refusal leaves them untouched
    vl, al, vc, ac = (t[:2].contiguous() for t in (vl3, al3, vc3, ac3))
    sig3 = np.full(3, 0.5, np.float32)
    ov = np.full((3, N, 128), np.nan, np.float32)
    oa = np.full((3, Ta, 128), np.nan, np.float32)
    p = lambda t: C.c_void_p(t.data_ptr() if isinstance(t, torch.Tensor) else t.ctypes.data)   # noqa: E731
    for B, null_audio in ((3, False), (2, True), (0, False)):
        rc = ctx.lib.ltx_av_forward_batch(ctx.handle, p(vl3 if B == 3 else vl), LTX_BF16, None if null_audio else p(al3 if B == 3 else al),
                                          LTX_BF16, p(vc3 if B == 3 else vc), p(ac3 if B == 3 else ac), LTX_BF16, p(sig3), 0,
                                          p(sig3), None, None, B, N, Ta, S, *fhw, 0, p(ov), p(oa))
        assert rc == (5 if B == 3 else 2), (B, null_audio, rc)
        assert np.isnan(ov).all() and np.isnan(oa).all()
    # bad shape (N != F*H*W) on the device entry point
    dv = torch.full((2, N, 128), float("nan"), device="cuda")
    da = torch.full((2, Ta, 128), float("nan"), device="cuda")
    dsig = torch.full((2,), 0.5, device="cuda")
    dvl, dal, dvc, dac = vl.cuda(), al.cuda(), vc.cuda(), ac.cuda()
    rc = ctx.lib.ltx_av_forward_batch_dev(ctx.handle, p(dvl), LTX_BF16, p(dal), LTX_BF16, p(dvc), p(dac), LTX_BF16, p(dsig), 0,
                                          p(dsig), None, None, 2, N + 1, Ta, S, *fhw, 0, p(dv), p(da))
    torch.cuda.synchronize()
    assert rc == 2
    assert torch.isnan(dv).all() and torch.isnan(da).all()
    ctx.close()


def _gelu_tanh(x):
    return 0.5 * x * (1.0 + torch.tanh(0.7978845608028654 * (x + 0.044715 * x ** 3)))


@pytest.mark.parametrize("M", [33, 52, 64])
@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4, "vt"])
def test_skinny_gemm_64_row_form_matches_fp64(M, mode):
    """The 64-row form of the weight-streaming GEMM (two items of <= 32 rows) against a float64 product of bf16-exact operands,
    for every epilogue it serves: bf16 / GELU / SiLU / fp32 outputs, the gate * residual update with one gate row per item,
    and the V^T store with a padded column block per item.  Rows 0..31 also equal the 32-row form's, bit for bit."""
    N, K = 96, 512
    g = torch.Generator(device="cuda").manual_seed(M * 7 + (5 if mode == "vt" else mode))
    A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    Wt = (torch.randn(N, K, device="cuda", generator=g) / K ** 0.5).bfloat16()
    bias = torch.randn(N, device="cuda", generator=g)
    ref = A.double() @ Wt.double().t() + bias.double()
    _, _, _, ctx = _setup(1, 2, 2, seed=1)
    lib, h = ctx.lib, ctx.handle
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())   # noqa: E731
    if mode == 2:
        rpg = M if M % 2 else M // 2
        ga = torch.randn(M // rpg, N, device="cuda", generator=g)
        gb = torch.randn(N, device="cuda", generator=g)
        x0 = torch.randn(M, N, device="cuda", generator=g)
        x = x0.clone()
        ctx._check(lib.ltx_op_gemm_skinny(h, p(A), p(Wt), p(bias), None, p(x), p(ga), p(gb), rpg, M, N, K, 2, 2, 0))
        ctx.sync()
        gate = (ga.double().repeat_interleave(rpg, 0) + gb.double())
        want = x0.double() + ref * gate
        assert torch.isfinite(x).all()
        assert (x.double() - want).norm() / want.norm() <= 1e-5
        ctx.close()
        return
    if mode == "vt":
        if M % 2:
            ctx.close()
            pytest.skip("the per-item V^T store splits M into two equal items")
        rows, ld = M // 2, (M // 2 + 7) // 8 * 8 + 8
        out = torch.full((N, 2 * ld), float("nan"), device="cuda", dtype=torch.bfloat16)
        ctx._check(lib.ltx_op_gemm_skinny(h, p(A), p(Wt), p(bias), p(out), None, None, None, 0, M, N, K, 0, 2, ld))
        ctx.sync()
        for i in range(2):
            got = out[:, i * ld:i * ld + rows].double().t()
            assert torch.isfinite(got).all()
            assert (got - ref[i * rows:(i + 1) * rows]).norm() / ref[i * rows:(i + 1) * rows].norm() <= 4e-3
            assert torch.isnan(out[:, i * ld + rows:(i + 1) * ld].float()).all()    # the padding is never written
        ctx.close()
        return
    dt = torch.float32 if mode == 3 else torch.bfloat16
    out = torch.full((M + 1, N), float("nan"), device="cuda", dtype=dt)
    ctx._check(lib.ltx_op_gemm_skinny(h, p(A), p(Wt), p(bias), p(out), None, None, None, 0, M, N, K, mode, 2, 0))
    ctx.sync()
    want = ref
    if mode == 1:
        want = _gelu_tanh(ref)
    if mode == 4:
        want = ref * torch.sigmoid(ref)
    got = out[:M].double()
    assert torch.isfinite(got).all() and torch.isnan(out[M].float()).all()
    assert (got - want).norm() / want.norm() <= (1e-5 if mode == 3 else 4e-3)
    # rows of the first item on the 32-row form: the same bits
    one = torch.full((32, N), float("nan"), device="cuda", dtype=dt)
    ctx._check(lib.ltx_op_gemm_skinny(h, p(A[:32].contiguous()), p(Wt), p(bias), p(one), None, None, None, 0, 32, N, K, mode, 1, 0))
    ctx.sync()
    assert torch.equal(one, out[:32])
    ctx.close()
