"""8-bit frames from the VAE decode (include/ltxcuda.h: ltx_vae_decode_u8*, ltx_vae_decode_tiled_u8*, ltx_frames_to_u8*).

RGB8 written by conv_out's epilogue must equal (np.float32(frames) * np.float32(255)).astype(np.uint8) of the fp32 decode of the
same latent, bit for bit; I420 must equal the converter applied to the fp32 frames (and the numpy float32 restatement) bit for
bit, and lie within one code of the float64 restatement."""
import ctypes as C
import threading

import numpy as np
import pytest
import torch

from frames_u8_ref import i420, i420_f64
from helpers import O, make_ctx_with_vae, product, small_vae_config

pytestmark = pytest.mark.gpu

ctxmod = product()
from ltx_video_swift_mlx_b200 import _lib  # noqa: E402
from ltx_video_swift_mlx_b200.vae import VideoDecoder, decode_video, decode_video_u8  # noqa: E402

RGB8, I420 = _lib.LTX_FRAMES_RGB8, _lib.LTX_FRAMES_I420


def trunc255(frames):
    return (np.float32(frames) * np.float32(255)).astype(np.uint8)


def check_i420(ctx, frames, got, what):
    conv = ctx.frames_to_u8(frames, "i420")
    assert np.array_equal(got, conv), what
    assert np.array_equal(got, i420(frames)), what
    d = np.abs(got.astype(int) - i420_f64(frames).astype(int))
    print(f"{what}: I420 codes off the float64 restatement: {int((d > 0).sum())} of {d.size} (max {int(d.max())})")
    assert d.max() <= 1, what


@pytest.fixture(scope="module")
def small():
    ocfg, pcfg = small_vae_config(512, 2)
    ctx, _ = make_ctx_with_vae(ocfg, pcfg, seed=71)
    yield ctx
    ctx.close()


@pytest.mark.parametrize("fhw,timed,causal", [((2, 3, 4), False, False), ((3, 2, 3), True, False), ((3, 3, 4), False, True),
                                              ((1, 2, 2), False, False)])
def test_fused_u8_decode_matches_fp32_decode(small, fhw, timed, causal):
    g = torch.Generator().manual_seed(sum(fhw) + 10 * timed + 100 * causal)
    z = torch.randn(128, *fhw, generator=g).numpy()
    nz = torch.randn(128, *fhw, generator=g).numpy() if timed else None
    ts = 0.05 if timed else None
    ref = small.vae_decode(z, timestep=ts, decode_noise=nz, causal=causal)
    assert 0.05 < float((ref > 0).mean()) and float((ref < 1).mean()) > 0.05     # frames inside the clip range, not saturated
    rgb = small.vae_decode_u8(z, "rgb8", timestep=ts, decode_noise=nz, causal=causal)
    assert rgb.shape == ref.shape and np.array_equal(rgb, trunc255(ref))
    assert np.array_equal(small.frames_to_u8(ref, "rgb8"), rgb)
    yuv = small.vae_decode_u8(z, "i420", timestep=ts, decode_noise=nz, causal=causal)
    assert yuv.shape == (ref.shape[0], ref.shape[1] * 3 // 2, ref.shape[2])
    check_i420(small, ref, yuv, f"fhw={fhw} timed={timed} causal={causal}")


def test_u8_dev_entry_points_match_host(small):
    z = torch.randn(128, 2, 3, 4, generator=torch.Generator().manual_seed(3))
    lat = z.cuda()
    F, H, W = 9, 96, 128
    f32 = torch.empty(F, H, W, 3, device="cuda")
    small.vae_decode_dev(lat.data_ptr(), (2, 3, 4), f32.data_ptr())
    for fmt in ("rgb8", "i420"):
        code = RGB8 if fmt == "rgb8" else I420
        n = small.lib.ltx_frames_u8_bytes(F, H, W, code)
        a, b = torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda")
        small.vae_decode_u8_dev(lat.data_ptr(), (2, 3, 4), a.data_ptr(), fmt)
        small.frames_to_u8_dev(f32.data_ptr(), (F, H, W), b.data_ptr(), fmt)
        small.sync()
        host = small.vae_decode_u8(z.numpy(), fmt)
        assert np.array_equal(a.cpu().numpy(), host.ravel()) and np.array_equal(b.cpu().numpy(), host.ravel()), fmt


@pytest.mark.parametrize("frames,tile,overlap,timed", [(5, 3, 1, False), (4, 2, 1, True), (5, 2, 0, False), (2, 4, 1, False)])
def test_tiled_u8_decode_equals_converter_of_tiled_fp32(frames, tile, overlap, timed):
    ocfg, pcfg = small_vae_config(512, 1)
    ctx, _ = make_ctx_with_vae(ocfg, pcfg, seed=61)
    g = torch.Generator().manual_seed(67)
    z = torch.randn(1, 128, frames, 2, 3, generator=g).numpy()
    nz = torch.randn(1, 128, frames, 2, 3, generator=g).numpy() if timed else None
    ts = 0.05 if timed else None
    dec = VideoDecoder(ctx)
    ref = decode_video(z, dec, timestep=ts, temporal_tile_size=tile, temporal_tile_overlap=overlap, decode_noise=nz)
    for fmt in ("rgb8", "i420"):
        got = decode_video_u8(z, dec, fmt, timestep=ts, temporal_tile_size=tile, temporal_tile_overlap=overlap, decode_noise=nz)
        assert np.array_equal(got, ctx.frames_to_u8(ref, fmt)), fmt
    assert np.array_equal(decode_video_u8(z, dec, "rgb8", timestep=ts, temporal_tile_size=tile, temporal_tile_overlap=overlap,
                                          decode_noise=nz), trunc255(ref))
    ctx.close()


def test_flagship_shape_768x512x25():
    """The full decoder (random weights) at 768 x 512 x 25 frames: the fused stores against the fp32 decode."""
    ctx = ctxmod.LtxContext(ctxmod.LTXTransformerConfig(), 0)
    ctx.init_random_weights(2, seed=5)
    ctx.finalize_weights()
    lat = torch.randn(128, 4, 16, 24, device="cuda", generator=torch.Generator(device="cuda").manual_seed(9)) * 0.5
    F, H, W = 25, 512, 768
    f32 = torch.empty(F, H, W, 3, device="cuda")
    ctx.vae_decode_dev(lat.data_ptr(), (4, 16, 24), f32.data_ptr())
    outs = {}
    for fmt, code in (("rgb8", RGB8), ("i420", I420)):
        buf = torch.empty(ctx.lib.ltx_frames_u8_bytes(F, H, W, code), dtype=torch.uint8, device="cuda")
        ctx.vae_decode_u8_dev(lat.data_ptr(), (4, 16, 24), buf.data_ptr(), fmt)
        ctx.sync()
        outs[fmt] = buf.cpu().numpy().reshape(ctx.frames_u8_shape(F, H, W, fmt))
    ref = f32.cpu().numpy()
    print(f"768x512x25: {float(((ref > 0) & (ref < 1)).mean()):.3f} of the samples inside (0, 1)")
    assert np.array_equal(outs["rgb8"], trunc255(ref))
    check_i420(ctx, ref, outs["i420"], "768x512x25")
    ctx.close()


def test_refusals_write_nothing(small):
    lib, h = small.lib, small.handle
    z = np.ascontiguousarray(torch.randn(128, 2, 2, 3, generator=torch.Generator().manual_seed(1)).numpy())
    zp = z.ctypes.data_as(C.c_void_p)
    n = lib.ltx_frames_u8_bytes(9, 64, 96, RGB8)
    host = np.full(n, 0xA5, dtype=np.uint8)
    hp = host.ctypes.data_as(C.c_void_p)
    dev = torch.full((n,), 0xA5, dtype=torch.uint8, device="cuda")
    lat = torch.from_numpy(z).cuda()
    frames = np.random.default_rng(0).random((9, 64, 96, 3), dtype=np.float32)
    fdev = torch.from_numpy(frames).cuda()
    got = C.c_int(-7)
    for fmt in (0, 3, -1):
        assert lib.ltx_vae_decode_u8(h, zp, 2, 2, 3, -1.0, None, 0, fmt, hp) == 2
        assert lib.ltx_vae_decode_u8_dev(h, lat.data_ptr(), 2, 2, 3, -1.0, None, 0, fmt, dev.data_ptr()) == 2
        assert lib.ltx_vae_decode_tiled_u8(h, zp, 2, 2, 3, -1.0, None, 0, 1, 0, fmt, hp, C.byref(got)) == 2
        assert lib.ltx_vae_decode_tiled_u8_dev(h, lat.data_ptr(), 2, 2, 3, -1.0, None, 0, 1, 0, fmt, dev.data_ptr(), C.byref(got)) == 2
        assert lib.ltx_frames_to_u8(h, frames.ctypes.data_as(C.c_void_p), 9, 64, 96, fmt, hp) == 2
        assert lib.ltx_frames_to_u8_dev(h, fdev.data_ptr(), 9, 64, 96, fmt, dev.data_ptr()) == 2
    for fmt in (RGB8, I420):
        assert lib.ltx_vae_decode_u8(h, zp, 2, 2, 3, -1.0, None, 0, fmt, None) == 2
        assert lib.ltx_vae_decode_u8_dev(h, lat.data_ptr(), 2, 2, 3, -1.0, None, 0, fmt, None) == 2
        assert lib.ltx_vae_decode_tiled_u8(h, zp, 2, 2, 3, -1.0, None, 0, 1, 0, fmt, None, C.byref(got)) == 2
        assert lib.ltx_vae_decode_tiled_u8_dev(h, lat.data_ptr(), 2, 2, 3, -1.0, None, 0, 1, 0, fmt, None, C.byref(got)) == 2
        assert lib.ltx_frames_to_u8(h, frames.ctypes.data_as(C.c_void_p), 9, 64, 96, fmt, None) == 2
        assert lib.ltx_frames_to_u8_dev(h, fdev.data_ptr(), 9, 64, 96, fmt, None) == 2
    # I420 of an odd width, and a misaligned device output for the fused store
    assert lib.ltx_frames_to_u8(h, frames.ctypes.data_as(C.c_void_p), 9, 64, 95, I420, hp) == 2
    assert lib.ltx_frames_to_u8_dev(h, fdev.data_ptr(), 9, 64, 95, I420, dev.data_ptr()) == 2
    assert lib.ltx_vae_decode_u8_dev(h, lat.data_ptr(), 2, 2, 3, -1.0, None, 0, RGB8, dev.data_ptr() + 1) == 2
    small.sync()
    assert (host == 0xA5).all() and bool((dev == 0xA5).all()) and got.value == -7


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_u8_decode_matches_single_gpu():
    """ltx_dist_init_local: two contexts in one process decode temporal slabs and gather the 8-bit planes; same bytes as one GPU."""
    ocfg, pcfg = small_vae_config(512, 1)
    w = O.make_vae_weights(ocfg, 8)
    w = {k: (O.bf16_round(v) if (k.endswith(".weight") and v.ndim >= 2) else v) for k, v in w.items()}
    z = torch.randn(128, 5, 3, 4, generator=torch.Generator().manual_seed(5)).numpy()

    def make(dev):
        c = ctxmod.LtxContext(pcfg, dev)
        c.load_weights(w, prefix="vae.")
        c.finalize_weights()
        return c

    def work(c, out, key):
        try:
            out[key] = {fmt: c.vae_decode_u8(z, fmt) for fmt in ("rgb8", "i420")}
        except Exception as e:   # surfaced by the assertions below
            out[key] = e

    single = make(0)
    ref = {}
    work(single, ref, "single")
    single.close()
    assert not isinstance(ref["single"], Exception), ref["single"]
    ctxs = [make(0), make(1)]
    ctxmod.LtxContext.dist_init_local(ctxs, sp_size=1, pass_groups=2)
    res = {}
    threads = [threading.Thread(target=work, args=(c, res, i)) for i, c in enumerate(ctxs)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout=600)
    for i in range(2):
        assert not isinstance(res.get(i), Exception), res.get(i)
        for fmt in ("rgb8", "i420"):
            assert np.array_equal(res[i][fmt], ref["single"][fmt]), (i, fmt)

    def shut(c):
        c.dist_shutdown()
    ts = [threading.Thread(target=shut, args=(c,)) for c in ctxs]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=120)
    for c in ctxs:
        c.close()
