"""CPU restatement of FP8 mode (ltx_set_precision(ctx, 8)) for the tests: the per-row e4m3 format, and the oracle forward with
every Linear inside the transformer blocks run on e4m3 operands.

Format (one definition for weight rows = output channels and activation rows = tokens):
  s = 2^ceil(log2(amax / 448)) (a power of two; 1 for a zero row),  q = e4m3_rn_satfinite(x / s),  x ~= q * s.
x / s and q * s are exact, so the restatement is bit for bit.  e4m3 is torch.float8_e4m3fn; values are clamped to +-448 before
the cast because torch turns an overflow into NaN (the library's conversion saturates)."""
import contextlib

import torch

from helpers import O

E4M3_MAX = 448.0


def row_scales(x: torch.Tensor) -> torch.Tensor:
    """The least power of two s with amax <= 448 * s per row (float64 [M]); amax = f * 2^e, f in [0.5, 1), 448 = 0.875 * 2^9."""
    amax = x.to(torch.float64).abs().amax(-1)
    f, e = torch.frexp(amax)
    e = torch.where(f <= 0.875, e - 9, e - 8)
    s = torch.ldexp(torch.ones_like(amax), e)
    return torch.where(amax > 0, s, torch.ones_like(s))


def quantize_rows(x: torch.Tensor):
    """x [M, K] -> (e4m3 codes as uint8 [M, K], scales float64 [M])."""
    x64 = x.to(torch.float64)
    s = row_scales(x64)
    y = (x64 / s[:, None]).clamp(-E4M3_MAX, E4M3_MAX)
    return y.to(torch.float8_e4m3fn).view(torch.uint8), s


def decode(codes: torch.Tensor, scales: torch.Tensor) -> torch.Tensor:
    return codes.view(torch.float8_e4m3fn).to(torch.float64) * scales.to(torch.float64)[:, None]


def fake_quant(x: torch.Tensor) -> torch.Tensor:
    """The float64 values FP8 mode feeds the tensor cores for the rows of x (any leading shape)."""
    x2 = x.reshape(-1, x.shape[-1])
    return decode(*quantize_rows(x2)).reshape(x.shape)


_plain_linear = O.linear


def _linear(x, w, name):
    if not name.startswith("transformer_blocks."):
        return _plain_linear(x, w, name)
    y = fake_quant(x) @ fake_quant(w[name + ".weight"]).t()
    return y.to(x.dtype) + w[name + ".bias"].to(x.dtype)


@contextlib.contextmanager
def fp8_blocks():
    """Inside: the oracle's block Linears (attn1 / attn2 q, k, v, to_out, FFN in / out) quantise their input rows and weight
    rows as FP8 mode does and multiply in float64; everything else is the plain oracle."""
    O.linear = _linear
    try:
        yield
    finally:
        O.linear = _plain_linear
