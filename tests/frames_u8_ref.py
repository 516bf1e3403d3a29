"""numpy restatements of the 8-bit frame formats of include/ltxcuda.h (LTX_FRAMES_RGB8, LTX_FRAMES_I420).

`rgb8` and `i420` repeat the library's fp32 arithmetic (csrc/frames_u8.cuh) step by step: every operation is one float32
operation rounded to nearest, so they agree with the device bit for bit.  `i420_f64` is the same definition evaluated in
float64, the yardstick the fp32 codes are held to within one code."""
import numpy as np

f32 = np.float32
KR, KG, KB = f32(0.2126), f32(0.7152), f32(0.0722)


def rgb8(frames):
    """[F, H, W, 3] float -> uint8 (uint8)(clip01(v) * 255.0f): one fp32 multiply, then truncation."""
    v = np.clip(np.asarray(frames, dtype=f32), f32(0), f32(1))
    return (v * f32(255)).astype(np.uint8)


def _luma(r, g, b):
    return (KR * r + KG * g) + KB * b


def _code(x):
    return np.clip(np.rint(x), 0, 255).astype(np.uint8)


def _planes(frames, dtype):
    v = np.clip(np.asarray(frames, dtype=f32), f32(0), f32(1)).astype(dtype)
    F, H, W, _ = v.shape
    assert H % 2 == 0 and W % 2 == 0, "I420 needs even H and W"
    cells = v.reshape(F, H // 2, 2, W // 2, 2, 3)
    p = [cells[:, :, 0, :, 0], cells[:, :, 0, :, 1], cells[:, :, 1, :, 0], cells[:, :, 1, :, 1]]   # pixel i = 2 * row + col
    return v, p


def _pack(y, cb, cr):
    F, H, W = y.shape
    return np.concatenate([y.reshape(F, -1), cb.reshape(F, -1), cr.reshape(F, -1)], axis=1).reshape(F, H * 3 // 2, W)


def i420(frames):
    """[F, H, W, 3] float -> [F, 3H/2, W] uint8 (Y | U | V planes per frame), BT.709 limited range in float32."""
    v, p = _planes(frames, f32)
    y = _code(f32(16) + f32(219) * _luma(v[..., 0], v[..., 1], v[..., 2]))
    m = (((p[0] + p[1]) + p[2]) + p[3]) * f32(0.25)
    ym = _luma(m[..., 0], m[..., 1], m[..., 2])
    cb = _code(f32(128) + (f32(224) * (m[..., 2] - ym)) / f32(1.8556))
    cr = _code(f32(128) + (f32(224) * (m[..., 0] - ym)) / f32(1.5748))
    return _pack(y, cb, cr)


def i420_f64(frames):
    """The same definition in float64 (means of the cell's four pixels, Cb / Cr from the mean colour)."""
    v, p = _planes(frames, np.float64)
    kr, kg, kb = 0.2126, 0.7152, 0.0722
    y = _code(16 + 219 * (kr * v[..., 0] + kg * v[..., 1] + kb * v[..., 2]))
    m = (p[0] + p[1] + p[2] + p[3]) / 4
    ym = kr * m[..., 0] + kg * m[..., 1] + kb * m[..., 2]
    cb = _code(128 + 224 * (m[..., 2] - ym) / 1.8556)
    cr = _code(128 + 224 * (m[..., 0] - ym) / 1.5748)
    return _pack(y, cb, cr)
