"""The 8-bit frame formats (include/ltxcuda.h: LTX_FRAMES_RGB8, LTX_FRAMES_I420) on the GPU-less host: the numpy restatement
the GPU tests compare against, held to hand-computed anchors, and the host-only ltx_frames_u8_bytes."""
import numpy as np
import pytest

from frames_u8_ref import i420, i420_f64, rgb8
from helpers import product

product()
from ltx_video_swift_mlx_b200 import _lib  # noqa: E402
from ltx_video_swift_mlx_b200.context import LtxContext  # noqa: E402

f32 = np.float32


def solid(rgb, H=2, W=2):
    return np.broadcast_to(np.asarray(rgb, dtype=f32), (1, H, W, 3)).copy()


def yuv_of(rgb):
    out = i420(solid(rgb))[0]
    return int(out[0, 0]), int(out[2, 0]), int(out[2, 1])     # Y of pixel (0, 0), then U and V (one byte each at 2 x 2)


@pytest.mark.parametrize("rgb,expect", [
    ((1, 1, 1), (235, 128, 128)),      # white: the top of the luma range, no chroma
    ((0, 0, 0), (16, 128, 128)),       # black
    ((1, 0, 0), (63, 102, 240)),       # BT.709 limited-range primaries (ITU-R BT.709-6 with 8-bit quantisation)
    ((0, 1, 0), (173, 42, 26)),
    ((0, 0, 1), (32, 240, 118)),
    ((0.5, 0.5, 0.5), (126, 128, 128)),  # 16 + 109.5 = 125.5: ties go to even
])
def test_i420_anchors(rgb, expect):
    assert yuv_of(rgb) == expect
    assert tuple(int(x) for x in i420_f64(solid(rgb))[0][[0, 2, 2], [0, 0, 1]]) == expect


def test_i420_layout_and_chroma_mean():
    """Per frame Y [H][W] | U [H/2][W/2] | V [H/2][W/2]; the chroma of a cell comes from its mean colour."""
    fr = np.zeros((2, 4, 6, 3), dtype=f32)
    fr[1, 0, 0] = (1, 0, 0)           # one red pixel in the first cell of frame 1
    out = i420(fr)
    assert out.shape == (2, 6, 6) and out.dtype == np.uint8
    flat = out.reshape(2, -1)
    y, u, v = flat[:, :24].reshape(2, 4, 6), flat[:, 24:30].reshape(2, 2, 3), flat[:, 30:].reshape(2, 2, 3)
    assert (flat[0] == np.r_[np.full(24, 16), np.full(12, 128)]).all()
    assert y[1, 0, 0] == 63 and (y[1].ravel()[1:] == 16).all()
    # mean colour (0.25, 0, 0): Y'_m = 0.05315, Cb = 128 - 6.416 -> 122, Cr = 128 + 28.0 -> 156
    assert (u[1, 0, 0], v[1, 0, 0]) == (122, 156)
    assert (u[1].ravel()[1:] == 128).all() and (v[1].ravel()[1:] == 128).all()


def test_rgb8_truncates_v_times_255():
    v = np.array([0, 1, 0.5, 1 / 255, 254.5 / 255, -0.25, 1.5, np.nextafter(f32(1), f32(0))], dtype=f32)
    assert rgb8(v).tolist() == [0, 255, 127, int(f32(1 / 255) * f32(255)), 254, 0, 255, 254]
    # at every code boundary: the first fp32 value whose product reaches k gives k, the one below it k - 1
    for k in range(1, 256):
        x = f32(k) / f32(255)
        while f32(x * f32(255)) < k:
            x = np.nextafter(x, f32(2))
        while f32(np.nextafter(x, f32(0)) * f32(255)) >= k:
            x = np.nextafter(x, f32(0))
        assert rgb8(np.array([x, np.nextafter(x, f32(0))], dtype=f32)).tolist() == [k, k - 1], k


def test_i420_fp32_within_one_code_of_float64():
    fr = np.random.default_rng(0).random((3, 16, 24, 3), dtype=f32)
    d = np.abs(i420(fr).astype(int) - i420_f64(fr).astype(int))
    assert d.max() <= 1


def test_frames_u8_bytes():
    lib = _lib.load()
    assert lib.ltx_frames_u8_bytes(25, 512, 768, _lib.LTX_FRAMES_RGB8) == 25 * 512 * 768 * 3
    assert lib.ltx_frames_u8_bytes(25, 512, 768, _lib.LTX_FRAMES_I420) == 25 * 512 * 768 * 3 // 2
    assert lib.ltx_frames_u8_bytes(121, 512, 768, _lib.LTX_FRAMES_RGB8) == 142_737_408       # 571 MB as fp32
    assert lib.ltx_frames_u8_bytes(1, 3, 5, _lib.LTX_FRAMES_RGB8) == 45
    for bad in ((1, 3, 4, _lib.LTX_FRAMES_I420), (1, 4, 5, _lib.LTX_FRAMES_I420), (1, 4, 4, 0), (1, 4, 4, 3), (0, 4, 4, 1),
                (1, -2, 4, 1), (1, 4, 0, 2)):
        assert lib.ltx_frames_u8_bytes(*bad) == 0, bad
    assert LtxContext.frames_u8_shape(9, 64, 96, "rgb8") == (9, 64, 96, 3)
    assert LtxContext.frames_u8_shape(9, 64, 96, "i420") == (9, 96, 96)
    assert int(np.prod(LtxContext.frames_u8_shape(9, 64, 96, "i420"))) == lib.ltx_frames_u8_bytes(9, 64, 96, _lib.LTX_FRAMES_I420)
