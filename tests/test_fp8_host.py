"""FP8 mode on the CPU: known answers of the e4m3 row format, and the FP8 restatement of the oracle forward really acts."""
import math

import torch

from fp8_ref import decode, fp8_blocks, quantize_rows, row_scales
from helpers import O


def test_448_is_the_largest_finite_code():
    q, s = quantize_rows(torch.tensor([[448.0, -448.0, 1.0]]))
    assert float(s[0]) == 1.0
    assert q[0].tolist() == [0x7E, 0xFE, 0x38]


def test_power_of_two_scale_rule():
    for amax, want in [(448.0, 1.0), (449.0, 2.0), (1e-3, 2.0 ** -18), (896.0, 2.0), (897.0, 4.0), (224.0, 0.5)]:
        s = float(row_scales(torch.tensor([[amax, -amax / 3]]))[0])
        assert s == want, (amax, s)
        assert s == 2.0 ** math.ceil(math.log2(amax / 448.0))
        assert amax / s <= 448.0 < 2 * amax / s


def test_subnormal_codes():
    # with s = 1 the e4m3 subnormals are k * 2^-9, k = 1..7; half of the smallest rounds to even (zero), 1.5 of it up
    x = torch.tensor([[448.0, 2.0 ** -9, 3 * 2.0 ** -9, 7 * 2.0 ** -9, 2.0 ** -10, 1.5 * 2.0 ** -9, -2.0 ** -9]])
    q, s = quantize_rows(x)
    assert float(s[0]) == 1.0
    assert q[0].tolist() == [0x7E, 0x01, 0x03, 0x07, 0x00, 0x02, 0x81]
    assert decode(q, s)[0, 1:4].tolist() == [2.0 ** -9, 3 * 2.0 ** -9, 7 * 2.0 ** -9]


def test_zero_row():
    q, s = quantize_rows(torch.zeros(2, 32))
    assert s.tolist() == [1.0, 1.0]
    assert int(q.abs().sum()) == 0


def test_outlier_row():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 256, generator=g).bfloat16().float()
    med = float(x.abs().median())
    x[0, 17] = 1e4 * med
    q, s = quantize_rows(x)
    assert float(s[0]) == 2.0 ** math.ceil(math.log2(float(x.abs().max()) / 448.0))
    d = decode(q, s)
    assert abs(float(d[0, 17]) / float(x[0, 17]) - 1) <= 2.0 ** -4            # 3 mantissa bits
    # the rest of the row moves down the format (s = 16 here): half a step of 3 mantissa bits, or of the subnormal spacing
    assert torch.isfinite(d).all()
    err = (d - x.double()).abs()
    assert bool((err <= torch.maximum(2.0 ** -4 * x.double().abs(), torch.full_like(err, 2.0 ** -10 * float(s[0])))).all())
    assert int((q[0] & 0x78).eq(0).sum()) > 0                                   # some subnormal / zero codes among them


def test_codes_round_to_nearest_even_and_saturate():
    x = torch.tensor([[1.0, 1.0625, 1.1875, 440.0, 464.0 - 1e-6, -300.0]])
    q, s = quantize_rows(x)
    d = decode(q, s)[0].tolist()
    assert float(s[0]) == 2.0                   # amax 464 > 448
    # x / s = 0.5, 0.53125, 0.59375 (steps of 1/16 there: the last two are ties, to even), 220, 232-, -150 (steps of 16)
    assert d == [1.0, 1.0, 1.25, 448.0, 448.0, -288.0]


def test_fp8_oracle_forward_differs_from_plain():
    ocfg = O.DiTConfig(num_layers=1, num_heads=2, head_dim=128, caption_channels=192)
    w = O.make_dit_weights(ocfg, 3)
    g = torch.Generator().manual_seed(1)
    fhw = (1, 2, 4)
    lat = torch.randn(1, 8, 128, generator=g)
    cx = torch.randn(1, 6, 192, generator=g)
    sig = torch.tensor([0.5])
    plain = O.dit_forward(w, ocfg, lat, cx, sig, None, fhw)
    with fp8_blocks():
        fp8 = O.dit_forward(w, ocfg, lat, cx, sig, None, fhw)
    again = O.dit_forward(w, ocfg, lat, cx, sig, None, fhw)
    assert O.rel_l2(fp8, plain) > 1e-4
    assert torch.equal(again, plain)     # the switch is scoped
