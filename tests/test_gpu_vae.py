"""Video-VAE decode parity against the CPU oracle: PSNR >= 50 dB on [0,1] frames (bf16 activations into the convs; every case
measured 58.4-61.4 dB on a B200 at 1000 W)."""
import numpy as np
import pytest
import torch

from helpers import O, make_ctx_with_vae, small_vae_config

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("base,blocks,fhw", [(512, 1, (2, 3, 4)), (512, 2, (3, 4, 6)), (1024, 1, (1, 2, 3))])
def test_vae_decode_matches_oracle(base, blocks, fhw):
    ocfg, pcfg = small_vae_config(base, blocks)
    ctx, w = make_ctx_with_vae(ocfg, pcfg, seed=base + blocks)
    g = torch.Generator().manual_seed(31)
    z = torch.randn(1, 128, *fhw, generator=g)
    ref = O.decode_video(w, ocfg, z)
    out = ctx.vae_decode(z[0].numpy())
    assert out.shape == tuple(ref.shape) == (8 * (fhw[0] - 1) + 1, 32 * fhw[1], 32 * fhw[2], 3)
    assert np.isfinite(out).all() and out.min() >= 0 and out.max() <= 1
    p = O.psnr(torch.from_numpy(out), ref)
    assert p >= 50.0, p
    ctx.close()


def test_vae_decode_timestep_conditioned():
    """decodeVideo(timestep: 0.05) -- noise injection + time-embedded scale/shift tables (V/VideoDecoder.swift:368-375,
    100-114, 419-436); the noise is passed in as data (SURVEY H7)."""
    ocfg, pcfg = small_vae_config(512, 1)
    ctx, w = make_ctx_with_vae(ocfg, pcfg, seed=41)
    g = torch.Generator().manual_seed(43)
    z = torch.randn(1, 128, 2, 3, 4, generator=g)
    nz = torch.randn(1, 128, 2, 3, 4, generator=g)
    ref = O.decode_video(w, ocfg, z, timestep=0.05, decode_noise=nz)
    out = ctx.vae_decode(z[0].numpy(), timestep=0.05, decode_noise=nz[0].numpy())
    assert O.psnr(torch.from_numpy(out), ref) >= 50.0
    plain = ctx.vae_decode(z[0].numpy())
    assert O.psnr(torch.from_numpy(plain), ref) < 35.0      # the conditioning really changes the frames
    ctx.close()


def test_vae_decode_causal():
    """causal: true -- two leading frame copies instead of one leading + one trailing (V/VideoConvolution.swift:281-294); covers the
    fused conv1 -> conv2 hand-over and the halo fill with the causal frame offset."""
    ocfg, pcfg = small_vae_config(512, 2)
    ocfg.causal = True
    ctx, w = make_ctx_with_vae(ocfg, pcfg, seed=51)
    z = torch.randn(1, 128, 3, 3, 4, generator=torch.Generator().manual_seed(53))
    ref = O.decode_video(w, ocfg, z)
    out = ctx.vae_decode(z[0].numpy(), causal=True)
    assert O.psnr(torch.from_numpy(out), ref) >= 50.0
    noncausal = ctx.vae_decode(z[0].numpy(), causal=False)
    assert O.psnr(torch.from_numpy(noncausal), ref) < 35.0
    ctx.close()


@pytest.mark.parametrize("frames,tile,overlap,timed", [(5, 3, 1, False), (6, 4, 2, False), (4, 2, 1, True), (5, 2, 0, False)])
def test_vae_decode_temporal_tiling(frames, tile, overlap, timed):
    """decodeVideo's tiled branch (decodeWithTemporalTiling, V/VideoDecoder.swift:517-602): overlapping chunks decoded
    independently, 8 * overlap frames cross-faded, clip after the blend.  Checked (i) against the oracle restatement (PSNR) and
    (ii) tightly against the same blend done on the host from the library's own per-chunk decodes.  (4, 2, 1) has three 9-frame chunks (8 of each cross-faded) and the
    timestep-conditioned tables; (5, 2, 0) is pure concatenation ending in a one-frame chunk."""
    from ltx_video_swift_mlx_b200.vae import VideoDecoder, decode_video
    ocfg, pcfg = small_vae_config(512, 1)
    ctx, w = make_ctx_with_vae(ocfg, pcfg, seed=61)
    g = torch.Generator().manual_seed(63)
    z = torch.randn(1, 128, frames, 2, 3, generator=g)
    nz = torch.randn(1, 128, frames, 2, 3, generator=g) if timed else None
    ts = 0.05 if timed else None
    ref = O.decode_video(w, ocfg, z, timestep=ts, decode_noise=nz, temporal_tile_size=tile, temporal_tile_overlap=overlap)
    out = decode_video(z.numpy(), VideoDecoder(ctx), timestep=ts, temporal_tile_size=tile, temporal_tile_overlap=overlap,
                       decode_noise=None if nz is None else nz.numpy())
    assert out.shape == tuple(ref.shape), (out.shape, ref.shape)
    assert out.shape[0] == ctx.lib.ltx_vae_tiled_frames(frames, tile, overlap)
    assert np.isfinite(out).all() and out.min() >= 0 and out.max() <= 1
    assert O.psnr(torch.from_numpy(out), ref) >= 50.0
    # (ii) the same chunk schedule on the host; interior frames of a chunk (never clipped away) must agree to fp32 rounding
    stride, po = tile - overlap, 8 * overlap
    chunks, start = [], 0
    while True:
        end = min(start + tile, frames)
        chunks.append(ctx.vae_decode(z[0, :, start:end].numpy(), timestep=ts,
                                     decode_noise=None if nz is None else nz[0, :, start:end].numpy()))
        if end >= frames:
            break
        start += stride
    def unclipped(a):
        return (a > 1e-3) & (a < 1 - 1e-3)
    res, ok = chunks[0], unclipped(chunks[0])
    for nxt in chunks[1:]:
        if 0 < po < res.shape[0] and po < nxt.shape[0]:
            wts = (np.arange(po, dtype=np.float32) / np.float32(po)).reshape(po, 1, 1, 1)
            res = np.concatenate([res[:-po], res[-po:] * (1 - wts) + nxt[:po] * wts, nxt[po:]], axis=0)
            ok = np.concatenate([ok[:-po], ok[-po:] & unclipped(nxt[:po]), unclipped(nxt[po:])], axis=0)
        else:
            res = np.concatenate([res, nxt], axis=0)
            ok = np.concatenate([ok, unclipped(nxt)], axis=0)
    # the library blends before the clip, the host copy after it: they agree wherever no source value sat on a rail
    assert ok.mean() > 0.3
    assert np.abs(out - res)[ok].max() <= 2e-5
    # a latent no longer than one tile takes the single pass
    one = decode_video(z[:, :, :tile].numpy(), VideoDecoder(ctx), timestep=ts, temporal_tile_size=tile,
                       decode_noise=None if nz is None else nz[:, :, :tile].numpy())
    assert np.array_equal(one, chunks[0])
    ctx.close()


def test_vae_tiled_arguments():
    from ltx_video_swift_mlx_b200._lib import LtxError
    ocfg, pcfg = small_vae_config(512, 1)
    ctx, _ = make_ctx_with_vae(ocfg, pcfg, seed=61)
    assert ctx.lib.ltx_vae_tiled_frames(16, 8, 1) == 57 + 57 + 9 - 16      # chunks [0,8) [7,15) [14,16): 57, 57, 9 frames
    assert ctx.lib.ltx_vae_tiled_frames(16, 0, 1) == 121 and ctx.lib.ltx_vae_tiled_frames(4, 8, 1) == 25
    assert ctx.lib.ltx_vae_tiled_frames(16, 4, 4) == -1
    with pytest.raises(LtxError) as e:
        ctx.vae_decode_tiled(np.zeros((128, 6, 2, 3), dtype=np.float32), 3, 3)
    assert e.value.code == 2
    ctx.close()


def test_vae_decode_conv_forms_agree(monkeypatch):
    """The three main-loop forms of the convolution on the full-width channel plan: CTA pairs add the taps up in the order of the
    one-CTA form (bit-identical frames); slab stages use another order (same frames to 2e-3 on [0, 1])."""
    ocfg, pcfg = small_vae_config(1024, 1)
    ctx, w = make_ctx_with_vae(ocfg, pcfg, seed=61)
    z = torch.randn(128, 3, 4, 6, generator=torch.Generator().manual_seed(67)).numpy()
    frames = {}
    for name, pair, slab in (("single", "0", "0"), ("pair", "1", "0"), ("pair+slab", "1", "1")):
        monkeypatch.setenv("LTX_CONV_PAIR", pair)
        monkeypatch.setenv("LTX_CONV_SLAB", slab)
        frames[name] = ctx.vae_decode(z)
    ctx.close()
    assert np.array_equal(frames["single"], frames["pair"])
    assert float(np.abs(frames["pair+slab"] - frames["pair"]).max()) <= 2e-3
    assert not np.array_equal(frames["pair+slab"], frames["pair"])      # the slab form really ran
