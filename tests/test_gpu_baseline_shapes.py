"""Parity at the BASELINE.json shapes themselves (the small-shape suites never reach the tile-width fit, the fused q|k|v
projection, the 3-way tap split or the 256-wide conv tiles that the benchmarked configurations take):

  * config 2: the LTX-2 width (D = 4096, 32 heads, caption 3840) at N = 1536 video tokens (4x16x24) and S = 1024 text tokens,
    a 4-block prefix of the 48-block model against the oracle (C/LTXConfig.swift:122-139, T/LTXTransformer.swift:235-486);
    the same prefix with int8 group-64 weights (P/LTXPipeline.swift:323-333) against the bf16 model;
  * config 4's decoder: the real channel plan (base 1024, 5 res blocks per stage, V/VideoDecoder.swift:331-355) on the
    config-2 latent 4x16x24 (25 frames of 512x768) against the oracle, PSNR >= 50 dB (57.8 dB measured on a B200 at 1000 W).
The oracle needs a few seconds of CPU per case at these sizes."""
import numpy as np
import pytest
import torch

from helpers import O, product, rel_l2

pytestmark = pytest.mark.gpu

FHW, N, S = (4, 16, 24), 1536, 1024
LAYERS = 4


@pytest.fixture(scope="module")
def cfg2():
    ocfg = O.DiTConfig(num_layers=LAYERS)                       # every other field is the LTX-2 default
    assert ocfg.inner_dim == 4096 and ocfg.num_heads == 32 and ocfg.caption_channels == 3840
    w = O.make_dit_weights(ocfg, 2024)
    g = torch.Generator().manual_seed(1236)
    lat = torch.randn(1, N, ocfg.in_channels, generator=g).bfloat16()
    text = torch.randn(1, S, ocfg.caption_channels, generator=g)
    text = (text / text.pow(2).mean(-1, keepdim=True).sqrt()).bfloat16()
    sig = torch.tensor([0.725])
    with torch.no_grad():
        ref = O.dit_forward(w, ocfg, lat.float(), text.float(), sig, None, FHW)
    return dict(ocfg=ocfg, w=w, lat=lat, text=text, sig=sig, ref=ref)


def _ctx(cfg2, quant_bits=16):
    ctxmod = product()
    ctx = ctxmod.LtxContext(ctxmod.LTXTransformerConfig(num_layers=LAYERS), 0)
    ctx.load_weights(cfg2["w"])
    ctx.finalize_weights(quant_bits=quant_bits)
    return ctx


def test_cfg2_shape_forward_matches_oracle(cfg2):
    ctx = _ctx(cfg2)
    out = ctx.dit_forward(cfg2["lat"], cfg2["text"], cfg2["sig"].numpy(), None, FHW)
    assert out.shape == (1, N, 128) and np.isfinite(out).all()
    err = rel_l2(out, cfg2["ref"])
    assert err <= 1e-2, err
    # the resident step (patchify -> forward -> unpatchify -> Euler) at the same shape: one Euler step from the same tokens
    lat_cfhw = cfg2["lat"].float()[0].t().reshape(128, *FHW).contiguous()          # tokens [N, C] -> latent [C, F, H, W]
    ctx.denoise_begin(lat_cfhw.numpy(), FHW, 1.0, cfg2["text"], None)
    ctx.denoise_step(float(cfg2["sig"][0]), 0.4, 0)
    got = ctx.denoise_get_latent()
    v = cfg2["ref"][0].t().reshape(128, *FHW)
    want = lat_cfhw + (0.4 - float(cfg2["sig"][0])) * v
    assert rel_l2(got, want) <= 1e-2
    ctx.close()


def test_cfg2_shape_masked_text_and_two_prompts(cfg2):
    """The additive-mask path at S = 1024, and two prompts back to back on one context: the second must not see the first
    one's projected text (same padded S, same cache key -- the host entry point fingerprints its buffers)."""
    ctxmod = product()
    ctx = _ctx(cfg2)
    mask = torch.ones(1, S, dtype=torch.int32)
    mask[:, :300] = 0
    with torch.no_grad():
        ref_m = O.dit_forward(cfg2["w"], cfg2["ocfg"], cfg2["lat"].float(), cfg2["text"].float(), cfg2["sig"], mask, FHW)
    fl = ctxmod.make_flags(context_key=7)
    out_m = ctx.dit_forward(cfg2["lat"], cfg2["text"], cfg2["sig"].numpy(), mask, FHW, fl)
    assert rel_l2(out_m, ref_m) <= 1e-2
    out_u = ctx.dit_forward(cfg2["lat"], cfg2["text"], cfg2["sig"].numpy(), None, FHW, fl)      # same key, other mask
    assert rel_l2(out_u, cfg2["ref"]) <= 1e-2
    g = torch.Generator().manual_seed(99)
    text2 = torch.randn(1, S, 3840, generator=g)
    text2 = (text2 / text2.pow(2).mean(-1, keepdim=True).sqrt()).bfloat16()
    out_2 = ctx.dit_forward(cfg2["lat"], text2, cfg2["sig"].numpy(), None, FHW, fl)             # same key, other prompt
    fresh = _ctx(cfg2)
    want_2 = fresh.dit_forward(cfg2["lat"], text2, cfg2["sig"].numpy(), None, FHW)
    np.testing.assert_array_equal(out_2, want_2)
    assert rel_l2(out_2, out_u) > 1e-2                                                            # the prompt matters
    fresh.close()
    ctx.close()


@pytest.mark.parametrize("bits,tol", [(8, 3e-2), (4, 0.35)])
def test_cfg2_shape_quantised_weights(cfg2, bits, tol):
    """int8 / int4 group-64 weights at M = 1536 (the large-M dequant path): drift against the oracle on the bf16 weights, and
    the two quantised runs of the same input are bit-identical (no data race in the conversion pipeline)."""
    ctx = _ctx(cfg2, quant_bits=bits)
    a = ctx.dit_forward(cfg2["lat"], cfg2["text"], cfg2["sig"].numpy(), None, FHW)
    b = ctx.dit_forward(cfg2["lat"], cfg2["text"], cfg2["sig"].numpy(), None, FHW)
    assert np.isfinite(a).all()
    np.testing.assert_array_equal(a, b)
    err = rel_l2(a, cfg2["ref"])
    assert 1e-5 < err <= tol, err
    ctx.close()


def test_full_vae_plan_at_cfg2_latent():
    ctxmod = product()
    ocfg = O.VAEConfig()                                           # base 1024, 5 blocks per stage
    assert ocfg.base_channels == 1024 and ocfg.blocks_per_stage == 5
    w = O.make_vae_weights(ocfg, 404)
    w = {k: (O.bf16_round(v) if (k.endswith(".weight") and v.ndim >= 2) else v) for k, v in w.items()}
    ctx = ctxmod.LtxContext(ctxmod.LTXTransformerConfig(num_layers=1, num_attention_heads=1), 0)
    ctx.load_weights(w, prefix="vae.")
    ctx.finalize_weights()
    z = torch.randn(1, 128, *FHW, generator=torch.Generator().manual_seed(405))
    with torch.no_grad():
        ref = O.decode_video(w, ocfg, z)
    out = ctx.vae_decode(z[0].numpy())
    assert out.shape == tuple(ref.shape) == (25, 512, 768, 3)
    assert np.isfinite(out).all() and out.min() >= 0 and out.max() <= 1
    p = O.psnr(torch.from_numpy(out), ref)
    assert p >= 50.0, p
    ctx.close()
