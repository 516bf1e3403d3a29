"""The VAE convolution piece by piece against float64 restatements: the padding prologue (vae_prep_kernel: every mode, pad bit
and channel bin), the halo fill of the fused res-block groups, and every epilogue of the implicit-GEMM conv (residual, in
place, tap split, the 9-tap per-frame conv, depth-to-space, unpatchify, the fused hand-overs to the next conv) under all three
main-loop forms.  Then the bit-identities the multi-GPU decode rests on: CTA pairs vs one CTA per tile, mode 4 vs mode 0, and a
temporal shard vs the whole clip (slab stages, tap split, and a tile width that the short shard narrows).

Operands are bf16-exact.  Bounds:
  * fp32 outputs: |got - ref| <= 5e-5 * (|W| * |x| + |bias| + |resid|) per element (|W| * |x|: the float64 conv of the absolute
    values) and rel-L2 <= 2e-5;
  * bf16 outputs: within one bf16 ulp of the float64 value, plus 2^-16 of the pre-activation's terms (fp32 rounding of a sum
    that cancels to ~0 is more than an ulp of the result); >= 99.9 % bit-equal to the correctly rounded value (copies: 100 %).
Every output buffer is NaN-prefilled and carries a NaN guard tail."""
import ctypes as C
import math

import pytest
import torch

from helpers import O, product

pytestmark = pytest.mark.gpu
NAN = float("nan")
CAUSAL, ZERO_HW, ZERO_T = 1, 2, 4
GUARD = 4096
FP32_TOL, FP32_REL_L2 = 5e-5, 2e-5


@pytest.fixture(scope="module")
def ctx():
    c = product().LtxContext(product().LTXTransformerConfig(num_layers=1, num_attention_heads=1), 0)
    yield c
    c.close()


@pytest.fixture(params=["single", "pair", "pair+slab"])
def conv_form(request, monkeypatch):
    """LTX_CONV_PAIR / LTX_CONV_SLAB (read by the launcher on every call): one CTA per voxel tile; CTA pairs wherever Cin comes
    in 128-channel stages; pairs with slab stages for tiles up to 128 columns (the default)."""
    set_form(monkeypatch, request.param)
    return request.param


def set_form(monkeypatch, form):
    monkeypatch.setenv("LTX_CONV_PAIR", "0" if form == "single" else "1")
    monkeypatch.setenv("LTX_CONV_SLAB", "1" if form == "pair+slab" else "0")


def plan(T, H, W, Cin, Cout, mode=0, ntaps=27):
    """What the launcher decides on this device (the plan reads LTX_CONV_PAIR / LTX_CONV_SLAB as the launcher does)."""
    out = (C.c_int32 * 7)()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    from ltx_video_swift_mlx_b200 import _lib
    assert _lib.load().ltx_conv3d_plan(T, H, W, Cin, Cout, mode, ntaps, sms, out) == 0
    p = dict(zip(("bn", "pair", "slab", "bt", "bh", "bw", "ksplit"), list(out)))
    p["tiles"] = -(-T // p["bt"]) * -(-H // p["bh"]) * -(-W // p["bw"])
    return p


def check_form(p, form, Cin, Cout):
    """The plan takes the form the fixture asked for."""
    pairs = form != "single" and Cin % 128 == 0
    assert p["pair"] == int(pairs), (form, p)
    assert p["slab"] == int(pairs and form == "pair+slab" and Cout < 256), (form, p)


def ptr(t):
    return None if t is None else t.data_ptr()


def nan_buf(shape, dtype=torch.float32, head=0):
    """NaN buffer: `head` elements, the tensor, GUARD elements; returns (buffer, view)."""
    n = math.prod(shape)
    buf = torch.full((head + n + GUARD,), NAN, device="cuda", dtype=dtype)
    return buf, buf[head:head + n].view(shape)


def assert_guard(buf, n, head=0):
    assert torch.isnan(buf[head + n:].float()).all(), "written behind the output"
    if head:
        assert torch.isnan(buf[:head].float()).all(), "written before the output"


def silu(v):
    return v * torch.sigmoid(v)


def bf16_ulp(r):
    _, e = torch.frexp(r.abs())
    return torch.where(r == 0, torch.zeros_like(r), torch.ldexp(torch.ones_like(r), e - 8))


def check_bf16(got, ref, slack=0.0, min_equal=0.999, what=""):
    """got (bf16) against ref (float64): within one ulp of ref + slack everywhere, >= min_equal bit-equal to ref rounded to
    nearest even (computed in float64: a float32 detour would round twice)."""
    g, ulp = got.double(), bf16_ulp(ref)
    assert torch.isfinite(g).all(), what
    err = (g - ref).abs()
    lim = ulp + slack
    worst = (err / lim.clamp_min(1e-300)).max().item()
    assert (err <= lim).all(), f"{what}: {int((err > lim).sum())} elements off by more than one bf16 ulp (worst {worst:.2f} ulp)"
    rounded = torch.where(ulp > 0, torch.round(ref / ulp.clamp_min(1e-300)) * ulp, ref)
    eq = (g == rounded).double().mean().item()
    assert eq >= min_equal, f"{what}: only {eq:.5f} bit-equal"
    print(f"[measured] {what}: worst {worst:.3f} of the bound, bit-equal {eq:.6f}")
    return eq


def check_fp32(got, ref, den, what=""):
    assert torch.isfinite(got).all(), what
    e = ((got.double() - ref).abs() / den).max().item()
    rl2 = ((got.double() - ref).norm() / ref.norm()).item()
    print(f"[measured] {what}: per-element {e:.3e}, rel-L2 {rl2:.3e}")
    assert e <= FP32_TOL, f"{what}: per-element error {e:.3e}"
    assert rl2 <= FP32_REL_L2, f"{what}: rel-L2 {rl2:.3e}"


# ---------------------------------------------------------------------------------------------------- float64 restatements
def pad_ref(x, pad):
    """fp32 [T,H,W,C] -> float64 [T+2,H+2,W+2,C] padded as the decoder / encoder / upscaler pad, plus the mask of the voxels
    that the zero padding owns."""
    T, H, W, Cc = x.shape
    xc = x.double().permute(3, 0, 1, 2)                                            # [C,T,H,W]
    one = torch.ones(1, T, H, W, device=x.device, dtype=torch.float64)
    if pad & ZERO_HW:
        xc, m = torch.nn.functional.pad(xc, (1, 1, 1, 1)), torch.nn.functional.pad(one, (1, 1, 1, 1))
    else:
        xc, m = torch.nn.functional.pad(xc, (1, 1, 1, 1), mode="reflect"), torch.nn.functional.pad(one, (1, 1, 1, 1), value=1.0)
    if pad & ZERO_T:
        z = torch.zeros_like(xc[:, :1])
        xc, m = torch.cat([z, xc, z], 1), torch.cat([z[:1], m, z[:1]], 1)
    elif pad & CAUSAL:
        xc, m = torch.cat([xc[:, :1], xc[:, :1], xc], 1), torch.cat([m[:, :1], m[:, :1], m], 1)
    else:
        xc, m = torch.cat([xc[:, :1], xc, xc[:, -1:]], 1), torch.cat([m[:, :1], m, m[:, -1:]], 1)
    return xc.permute(1, 2, 3, 0), m[0] == 0


def act_ref(v, mode, a, b):
    """The prologue's activation on float64 [..., C]; returns (value, slack) -- slack = 2^-16 of the pre-activation's terms."""
    if mode == 0:
        return v, torch.zeros_like(v)
    if mode == 2:
        sc = 1 + (a.double() if a is not None else 0.0)
        sh = b.double() if b is not None else torch.zeros_like(v[..., 0:1])
        u = v / torch.sqrt(v.pow(2).mean(-1, keepdim=True) + 1e-8) * sc
    else:
        sh = b.double()
        u = v * a.double()
    pre, slack = u + sh, (u.abs() + sh.abs()) * 2.0 ** -16
    return (pre if mode == 1 else silu(pre)), slack


def conv_ref(xp, w, T, H, W):
    """float64 cross-correlation of a padded channels-last volume: (conv, conv of the absolute values), [T,H,W,Cout] each.  27 taps,
    or 9 (the dt = 1 taps: weight i is tap 9 + i)."""
    ntaps, Cout, Cin = w.shape
    X, Wd = xp.double(), w.double()
    acc = torch.zeros(T * H * W, Cout, device=xp.device, dtype=torch.float64)
    acc_abs = torch.zeros_like(acc)
    for i in range(ntaps):
        tap = i if ntaps == 27 else 9 + i
        dt, dh, dw = tap // 9, (tap // 3) % 3, tap % 3
        xs = X[dt:dt + T, dh:dh + H, dw:dw + W].reshape(-1, Cin)
        acc += xs @ Wd[i].t()
        acc_abs += xs.abs() @ Wd[i].abs().t()
    return acc.view(T, H, W, Cout), acc_abs.view(T, H, W, Cout)


def handover_ref(y, scale, shift):
    """float64 prologue mode 2 of the next conv on [T,H,W,C] (tables nullable)."""
    return act_ref(y.double(), 2, scale, shift)


def to_ncthw(v):
    return v.permute(3, 0, 1, 2).unsqueeze(0)


def from_ncthw(v):
    return v[0].permute(1, 2, 3, 0)


def d2s_ref(conv, resid, Cin, t_shift):
    """depth-to-space (2,2,2) of the conv + the 4x tiled depth-to-space of the conv input (V/VideoDecoder.swift:214-251); the
    first output frame is dropped unless t_shift."""
    Cout = conv.shape[-1]
    r = O.depth_to_space(to_ncthw(resid), Cin // 8)
    v = O.depth_to_space(to_ncthw(conv), Cout // 8) + torch.cat([r, r, r, r], 1)
    return from_ncthw(v if t_shift else v[:, :, 1:])


def unpatchify_ref(v):
    return from_ncthw(O.vae_unpatchify(to_ncthw(v), 4))


def conv_inputs(T, H, W, Cin, Cout, ntaps=27, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    xp = torch.randn(T + 2, H + 2, W + 2, Cin, device="cuda", generator=g).bfloat16()
    w = (torch.randn(ntaps, Cout, Cin, device="cuda", generator=g) / math.sqrt(ntaps * Cin)).bfloat16()
    b = (torch.randn(Cout, device="cuda", generator=g) * 0.1).bfloat16().float()
    return xp, w, b, g


# ---------------------------------------------------------------------------------------------------- entry points
def run_prep(ctx, x, mode, a, b, pad):
    T, H, W, Cc = x.shape
    buf, out = nan_buf((T + 2, H + 2, W + 2, Cc), torch.bfloat16)
    torch.cuda.synchronize()
    ctx._check(ctx.lib.ltx_op_vae_prep(ctx.handle, x.data_ptr(), buf.data_ptr(), T, H, W, Cc, mode, ptr(a), ptr(b), pad))
    ctx.sync()
    assert_guard(buf, out.numel())
    return out


def run_conv(ctx, xp, w, b, T, H, W, mode=0, resid=None, inplace=False, t_shift=0, no_clip=0, scale=None, shift=None,
             next_tshift=1):
    """ltx_op_conv3d_epi into fresh NaN buffers; checks the guards (and, for the hand-over, that only the interior of next_pad
    was written).  Returns (out, next_pad interior)."""
    ntaps, Cout, Cin = w.shape
    out = npad = buf = nbuf = None
    head = 0
    if mode in (0, 4):
        buf, out = nan_buf((T, H, W, Cout))
        if inplace:
            out.copy_(resid)
            resid = out
    elif mode == 1:
        head = 4 * H * W * (Cout // 8)      # one output frame in front: the frame that t_shift = 0 drops must stay unwritten
        buf, out = nan_buf((2 * T - 1 + t_shift, 2 * H, 2 * W, Cout // 8), head=head)
    elif mode == 2:
        buf, out = nan_buf((T, 4 * H, 4 * W, 3))
    if mode in (3, 4):
        nbuf, npad = nan_buf((T + 2, H + 2, W + 2, Cout), torch.bfloat16)
    torch.cuda.synchronize()
    ctx._check(ctx.lib.ltx_op_conv3d_epi(ctx.handle, xp.data_ptr(), w.data_ptr(), b.data_ptr(), T, H, W, Cin, Cout, ntaps, mode,
                                         ptr(out), ptr(resid), t_shift, no_clip, ptr(npad), ptr(scale), ptr(shift), next_tshift))
    ctx.sync()
    if buf is not None:
        assert_guard(buf, out.numel(), head)
        assert torch.isfinite(out).all(), "an output element was not written"
    interior = None
    if npad is not None:
        assert_guard(nbuf, npad.numel())
        inner = torch.zeros(npad.shape[:3], dtype=torch.bool, device="cuda")
        inner[next_tshift:next_tshift + T, 1:H + 1, 1:W + 1] = True
        assert torch.isnan(npad[~inner].float()).all(), "the hand-over wrote a padding voxel"
        interior = npad[next_tshift:next_tshift + T, 1:H + 1, 1:W + 1]
        assert torch.isfinite(interior.float()).all(), "an interior voxel of next_pad was not written"
    return out, interior


# ---------------------------------------------------------------------------------------------------- a. prologue
PREP_CHANNELS = [48, 64, 128, 192, 256, 384, 512, 1024, 2048]      # every VPL bin (1, 2, 4, 8, 16), C not a multiple of 128
PREP_MODES = [(0, False), (1, True), (2, True), (2, False), (3, True)]
PREP_PADS = [0, CAUSAL, ZERO_HW | CAUSAL, ZERO_HW | ZERO_T]
PREP_VOLS = [(1, 2, 2), (3, 7, 9), (5, 16, 24), (2, 2, 5)]
PREP_CASES = [(Cc, mode, tables, PREP_PADS[(i + j) % 4], PREP_VOLS[(i + 2 * j) % 4])
              for i, Cc in enumerate(PREP_CHANNELS) for j, (mode, tables) in enumerate(PREP_MODES)]


@pytest.mark.parametrize("Cc,mode,tables,pad,vol", PREP_CASES)
def test_prep(ctx, Cc, mode, tables, pad, vol):
    T, H, W = vol
    g = torch.Generator(device="cuda").manual_seed(Cc * 31 + mode * 7 + pad + T * H * W)
    x = (torch.randn(T, H, W, Cc, device="cuda", generator=g) * 1.5).bfloat16().float()
    a = b = None
    if tables:
        a = (torch.randn(Cc, device="cuda", generator=g) * (0.3 if mode == 2 else 1.0)).bfloat16().float()
        b = (torch.randn(Cc, device="cuda", generator=g) * 0.5).bfloat16().float()
    got = run_prep(ctx, x, mode, a, b, pad)
    padded, zero = pad_ref(x, pad)
    ref, slack = act_ref(padded, mode, a, b)
    ref = torch.where(zero[..., None], torch.zeros_like(ref), ref)       # zero padding is written after the activation
    assert (got[zero] == 0).all()
    if mode == 0:
        assert torch.equal(got.double(), ref)
    else:
        check_bf16(got, ref, slack, what=f"prologue mode {mode}{'' if tables or mode != 2 else ' (no tables)'} C={Cc}")


# ---------------------------------------------------------------------------------------------------- b. halo fill
HALO_CASES = [(pad, Cc, T, hw) for pad in (0, CAUSAL, CAUSAL | ZERO_HW, ZERO_HW | ZERO_T) for Cc in (64, 128, 256, 1024)
              for T, hw in zip((1, 2, 5), ((2, 9), (7, 2), (2, 2)) if Cc != 1024 else ((2, 9), (7, 2), (6, 10)))]


@pytest.mark.parametrize("pad,Cc,T,hw", HALO_CASES)
def test_halo_fill(ctx, pad, Cc, T, hw):
    H, W = hw
    g = torch.Generator(device="cuda").manual_seed(pad * 1000 + Cc + T * 7 + H)
    x = torch.randn(T, H, W, Cc, device="cuda", generator=g).bfloat16()
    ts = 1 if pad & ZERO_T else (2 if pad & CAUSAL else 1)
    buf, vol = nan_buf((T + 2, H + 2, W + 2, Cc), torch.bfloat16)
    vol[ts:ts + T, 1:H + 1, 1:W + 1] = x
    torch.cuda.synchronize()
    ctx._check(ctx.lib.ltx_op_vae_halo_fill(ctx.handle, buf.data_ptr(), T, H, W, Cc, pad))
    ctx.sync()
    assert_guard(buf, vol.numel())
    ref, zero = pad_ref(x.float(), pad)
    ref[zero] = 0
    assert torch.equal(vol, ref.bfloat16())


@pytest.mark.parametrize("pad,Cc,vol", [(0, 128, (3, 7, 9)), (CAUSAL, 256, (2, 16, 24)), (CAUSAL | ZERO_HW, 128, (1, 2, 5)),
                                        (ZERO_HW | ZERO_T, 256, (4, 5, 2))])
def test_halo_fill_completes_the_prologue(ctx, pad, Cc, vol):
    """What vae_resgroup_fused relies on: the halo fill of the interior of prep(x) is prep(x), bit for bit."""
    T, H, W = vol
    g = torch.Generator(device="cuda").manual_seed(Cc + pad)
    x = torch.randn(T, H, W, Cc, device="cuda", generator=g)
    a, b = torch.randn(Cc, device="cuda", generator=g) * 0.3, torch.randn(Cc, device="cuda", generator=g) * 0.3
    full = run_prep(ctx, x, 2, a, b, pad)
    ts = 1 if pad & ZERO_T else (2 if pad & CAUSAL else 1)
    buf, vol = nan_buf(full.shape, torch.bfloat16)
    vol[ts:ts + T, 1:H + 1, 1:W + 1] = full[ts:ts + T, 1:H + 1, 1:W + 1]
    torch.cuda.synchronize()
    ctx._check(ctx.lib.ltx_op_vae_halo_fill(ctx.handle, buf.data_ptr(), T, H, W, Cc, pad))
    ctx.sync()
    assert_guard(buf, vol.numel())
    assert torch.equal(vol, full)


# ---------------------------------------------------------------------------------------------------- c. epilogues
# (T, H, W, Cin, Cout, what the default plan must show)
MODE0_CASES = [
    (5, 8, 8, 128, 128, "odd"),          # odd number of voxel tiles: the pair's second tile lies past the volume
    (3, 6, 10, 128, 48, "narrow"),       # Cout = 48: a 64-wide tile, partly empty
    (2, 16, 24, 512, 512, "ksplit"),     # tile-starved: taps split by dt + the reduction pass (bias, residual)
    (9, 32, 48, 256, 256, "bn256"),
    (2, 5, 7, 64, 128, "single"),        # Cin = 64: one CTA per tile in every form
]


def expect(p, tag):
    if tag == "odd":
        assert p["tiles"] % 2 == 1
    elif tag == "ksplit":
        assert p["ksplit"] == 3
    elif tag == "bn256":
        assert p["bn"] == 256 and p["ksplit"] == 1
    elif tag == "narrow":
        assert p["bn"] == 64
    elif tag == "slab":
        assert p["slab"] == 1
    if tag != "ksplit":
        assert p["ksplit"] == 1


@pytest.mark.parametrize("T,H,W,Cin,Cout,tag", MODE0_CASES)
@pytest.mark.parametrize("inplace", [False, True])
def test_mode0_residual(ctx, conv_form, T, H, W, Cin, Cout, tag, inplace):
    p = plan(T, H, W, Cin, Cout, 0)
    check_form(p, conv_form, Cin, Cout)
    expect(p, tag)
    xp, w, b, g = conv_inputs(T, H, W, Cin, Cout, seed=T * H * W + Cin + Cout)
    resid = torch.randn(T, H, W, Cout, device="cuda", generator=g)
    out, _ = run_conv(ctx, xp, w, b, T, H, W, 0, resid, inplace)
    conv, cabs = conv_ref(xp, w, T, H, W)
    check_fp32(out, conv + b.double() + resid.double(), cabs + b.double().abs() + resid.double().abs(),
               f"mode 0 + residual{' in place' if inplace else ''} {T}x{H}x{W} {Cin}->{Cout} {conv_form}")


@pytest.mark.parametrize("T,H,W,Cin,Cout,tag", [(3, 16, 24, 128, 128, "slab"), (5, 32, 48, 128, 512, "bn256")])
def test_nine_taps(ctx, conv_form, T, H, W, Cin, Cout, tag):
    """The upscaler's per-frame 3x3 conv: weights [9][Cout][Cin], only the dt = 1 taps."""
    p = plan(T, H, W, Cin, Cout, 0, 9)
    check_form(p, conv_form, Cin, Cout)
    if conv_form == "pair+slab" or tag != "slab":
        expect(p, tag)
    xp, w, b, _ = conv_inputs(T, H, W, Cin, Cout, ntaps=9, seed=9 * T + Cout)
    out, _ = run_conv(ctx, xp, w, b, T, H, W, 0)
    conv, cabs = conv_ref(xp, w, T, H, W)
    check_fp32(out, conv + b.double(), cabs + b.double().abs(), f"9 taps {T}x{H}x{W} {Cin}->{Cout} {conv_form}")


@pytest.mark.parametrize("T,H,W,Cin", [(1, 8, 8, 128), (3, 6, 10, 256), (2, 4, 6, 512)])
@pytest.mark.parametrize("t_shift", [0, 1])
def test_mode1_depth_to_space(ctx, conv_form, T, H, W, Cin, t_shift):
    Cout = 4 * Cin
    check_form(plan(T, H, W, Cin, Cout, 1), conv_form, Cin, Cout)
    xp, w, b, g = conv_inputs(T, H, W, Cin, Cout, seed=T + Cin + t_shift)
    x = torch.randn(T, H, W, Cin, device="cuda", generator=g)                  # the conv's unpadded input: the residual
    out, _ = run_conv(ctx, xp, w, b, T, H, W, 1, x, t_shift=t_shift)
    conv, cabs = conv_ref(xp, w, T, H, W)
    ref = d2s_ref(conv + b.double(), x.double(), Cin, t_shift)
    den = d2s_ref(cabs + b.double().abs(), x.double().abs(), Cin, t_shift)
    check_fp32(out, ref, den, f"mode 1 {T}x{H}x{W} {Cin}->{Cout} t_shift {t_shift} {conv_form}")


@pytest.mark.parametrize("T,H,W,Cin", [(2, 5, 7, 64), (3, 8, 12, 128)])
@pytest.mark.parametrize("no_clip", [0, 1])
def test_mode2_unpatchify(ctx, conv_form, T, H, W, Cin, no_clip):
    Cout = 48
    check_form(plan(T, H, W, Cin, Cout, 2), conv_form, Cin, Cout)
    xp, w, b, g = conv_inputs(T, H, W, Cin, Cout, seed=T + Cin)
    b = (torch.randn(Cout, device="cuda", generator=g) * 2.5).bfloat16().float()   # both rails of the clip are reached
    out, _ = run_conv(ctx, xp, w, b, T, H, W, 2, no_clip=no_clip)
    conv, cabs = conv_ref(xp, w, T, H, W)
    ref = (unpatchify_ref(conv + b.double()) + 1) * 0.5
    den = (unpatchify_ref(cabs + b.double().abs()) + 1) * 0.5
    assert (ref < 0).float().mean() > 0.05 and (ref > 1).float().mean() > 0.05
    if not no_clip:
        ref = ref.clamp(0, 1)
        assert out.min() >= 0 and out.max() <= 1
    check_fp32(out, ref, den, f"mode 2 {T}x{H}x{W} {Cin}->48 no_clip {no_clip} {conv_form}")


@pytest.mark.parametrize("T,H,W,Cout", [(5, 8, 8, 128), (2, 8, 12, 256)])
@pytest.mark.parametrize("next_tshift", [1, 2])
@pytest.mark.parametrize("tables", [True, False])
def test_modes3_4_handover(ctx, conv_form, T, H, W, Cout, next_tshift, tables):
    """conv1 -> conv2 (mode 3) and conv2 -> next conv1 (mode 4, in place on the residual stream, as vae_resgroup_fused runs
    them): the bf16 interior of next_pad against the float64 prologue of the conv's own fp32 values, and mode 4's fp32 output
    bit-equal to mode 0's."""
    Cin = Cout
    for mode in (3, 4):
        check_form(plan(T, H, W, Cin, Cout, mode), conv_form, Cin, Cout)
    xp, w, b, g = conv_inputs(T, H, W, Cin, Cout, seed=T * Cout + next_tshift)
    resid = torch.randn(T, H, W, Cout, device="cuda", generator=g)
    sc = sh = None
    if tables:
        sc, sh = torch.randn(Cout, device="cuda", generator=g) * 0.3, torch.randn(Cout, device="cuda", generator=g) * 0.3
    tag = f"{T}x{H}x{W} {Cout} next_tshift {next_tshift}{'' if tables else ' no tables'} {conv_form}"
    conv, cabs = conv_ref(xp, w, T, H, W)

    y0, _ = run_conv(ctx, xp, w, b, T, H, W, 0)
    check_fp32(y0, conv + b.double(), cabs + b.double().abs(), f"mode 0 {tag}")
    _, np3 = run_conv(ctx, xp, w, b, T, H, W, 3, scale=sc, shift=sh, next_tshift=next_tshift)
    check_bf16(np3, *handover_ref(y0, sc, sh), what=f"mode 3 next_pad {tag}")
    check_bf16(np3, handover_ref(conv + b.double(), sc, sh)[0], slack=math.inf, min_equal=0.99, what=f"mode 3 vs float64 chain {tag}")
    # mode 3 and the prologue kernel on mode 0's output: two implementations of one formula (other sum-of-squares order)
    prep = run_prep(ctx, y0, 2, sc, sh, CAUSAL if next_tshift == 2 else 0)[next_tshift:next_tshift + T, 1:H + 1, 1:W + 1]
    check_bf16(prep, *handover_ref(y0, sc, sh), what=f"prologue on mode 0 output {tag}")

    y0r, _ = run_conv(ctx, xp, w, b, T, H, W, 0, resid)
    y4, np4 = run_conv(ctx, xp, w, b, T, H, W, 4, resid, inplace=True, scale=sc, shift=sh, next_tshift=next_tshift)
    check_fp32(y4, conv + b.double() + resid.double(), cabs + b.double().abs() + resid.double().abs(), f"mode 4 out {tag}")
    assert torch.equal(y4, y0r), "mode 4's fp32 output differs from mode 0's"
    check_bf16(np4, *handover_ref(y4, sc, sh), what=f"mode 4 next_pad {tag}")
    check_bf16(np4, handover_ref(conv + b.double() + resid.double(), sc, sh)[0], slack=math.inf, min_equal=0.99,
               what=f"mode 4 vs float64 chain {tag}")


# ---------------------------------------------------------------------------------------------------- d. invariants
# (T, H, W, Cin, Cout, ntaps, mode)
FORM_CASES = [(5, 8, 8, 128, 128, 27, 0), (2, 16, 24, 512, 512, 27, 0), (3, 16, 24, 128, 128, 9, 0), (3, 6, 10, 256, 1024, 27, 1),
              (3, 8, 12, 128, 48, 27, 2), (5, 8, 8, 128, 128, 27, 3), (2, 8, 12, 256, 256, 27, 4), (5, 8, 8, 128, 128, 27, 4)]


@pytest.mark.parametrize("T,H,W,Cin,Cout,ntaps,mode", FORM_CASES)
def test_forms_agree(ctx, monkeypatch, T, H, W, Cin, Cout, ntaps, mode):
    """CTA pairs add the taps up in the order of one CTA per tile: bit-identical in every epilogue.  Slab stages use another
    order: within the fp32 bound of each other, and not identical (the slab form really ran)."""
    xp, w, b, g = conv_inputs(T, H, W, Cin, Cout, ntaps, seed=T + Cout + mode)
    resid = torch.randn(T, H, W, Cin if mode == 1 else Cout, device="cuda", generator=g) if mode in (0, 1, 4) else None
    sc, sh = torch.randn(Cout, device="cuda", generator=g) * 0.3, torch.randn(Cout, device="cuda", generator=g) * 0.3
    res, plans = {}, {}
    for form in ("single", "pair", "pair+slab"):
        set_form(monkeypatch, form)
        plans[form] = plan(T, H, W, Cin, Cout, mode, ntaps)
        check_form(plans[form], form, Cin, Cout)
        res[form] = run_conv(ctx, xp, w, b, T, H, W, mode, resid, inplace=mode == 4, t_shift=1 if mode == 1 else 0,
                             scale=sc, shift=sh, next_tshift=2)
    assert plans["pair"]["pair"] == 1
    for i in range(2):
        if res["single"][i] is not None:
            assert torch.equal(res["single"][i], res["pair"][i]), f"pair vs single CTA, output {i}"
    if plans["pair+slab"]["slab"]:
        outs = [res[f][0] if res[f][0] is not None else res[f][1] for f in ("pair", "pair+slab")]
        assert not torch.equal(*outs), "slab stages should sum in another order"
        if res["pair"][0] is not None:
            conv, cabs = conv_ref(xp, w, T, H, W)
            den = cabs + b.double().abs() + (resid.double().abs() if mode in (0, 4) else 0)
            if mode == 2:
                den = (unpatchify_ref(den) + 1) * 0.5
            assert ((outs[1].double() - outs[0].double()).abs() <= 2 * FP32_TOL * den).all()
        else:
            conv, _ = conv_ref(xp, w, T, H, W)
            check_bf16(outs[1], handover_ref(conv + b.double(), sc, sh)[0], slack=math.inf, min_equal=0.99, what="mode 3 slab")
    else:
        for i in range(2):
            if res["pair"][i] is not None:
                assert torch.equal(res["pair"][i], res["pair+slab"][i])


# (name, T, H, W, Cin, Cout, modes, shard [f0, f1))
SHARD_CASES = [("slab", 6, 16, 24, 128, 128, (0, 4), (2, 5)),
               ("ksplit", 4, 16, 24, 512, 512, (0,), (1, 3)),
               ("bn 256 -> 128", 8, 32, 48, 256, 512, (0,), (3, 5)),
               ("bn 256 -> 128, d2s", 8, 32, 48, 128, 512, (1,), (3, 5))]


@pytest.mark.parametrize("name,T,H,W,Cin,Cout,modes,shard", SHARD_CASES, ids=[c[0] for c in SHARD_CASES])
def test_temporal_shard_is_bit_identical(ctx, conv_form, name, T, H, W, Cin, Cout, modes, shard):
    """A rank of the multi-GPU decode convolves padded frames [f0, f1 + 2) of the clip's padded volume (its halo frames come
    from the neighbours): its output must be frames [f0, f1) of the whole clip's, bit for bit -- also where the launcher
    narrows the tile width for the short shard.  Depth-to-space on a shard keeps its first frame (t_shift = 1): frames
    [2 f0 - 1, 2 f1 - 1) of the whole clip."""
    f0, f1 = shard
    Ts = f1 - f0
    xp, w, b, g = conv_inputs(T, H, W, Cin, Cout, seed=T * H + Cout)
    xs = xp[f0:f1 + 2].contiguous()
    for mode in modes:
        pw, ps = plan(T, H, W, Cin, Cout, mode), plan(Ts, H, W, Cin, Cout, mode)
        check_form(pw, conv_form, Cin, Cout)
        assert {k: pw[k] for k in ("pair", "slab", "ksplit")} == {k: ps[k] for k in ("pair", "slab", "ksplit")}
        print(f"[plan] {name} mode {mode} {conv_form}: whole clip {pw}, shard {ps}")
        if name == "ksplit":
            assert pw["ksplit"] == 3
        if name.startswith("bn"):
            assert (pw["bn"], ps["bn"]) == (256, 128), (pw, ps)
        if name == "slab" and conv_form == "pair+slab":
            assert pw["slab"] == 1
        if mode == 1:
            x = torch.randn(T, H, W, Cin, device="cuda", generator=g)
            whole, _ = run_conv(ctx, xp, w, b, T, H, W, 1, x, t_shift=0)
            part, _ = run_conv(ctx, xs, w, b, Ts, H, W, 1, x[f0:f1].contiguous(), t_shift=1)
            assert torch.equal(part, whole[2 * f0 - 1:2 * f1 - 1])
            continue
        resid = torch.randn(T, H, W, Cout, device="cuda", generator=g)
        sc, sh = torch.randn(Cout, device="cuda", generator=g) * 0.3, torch.randn(Cout, device="cuda", generator=g) * 0.3
        kw = dict(inplace=True, scale=sc, shift=sh, next_tshift=2) if mode == 4 else {}
        whole, wpad = run_conv(ctx, xp, w, b, T, H, W, mode, resid, **kw)
        part, ppad = run_conv(ctx, xs, w, b, Ts, H, W, mode, resid[f0:f1].contiguous(), **kw)
        assert torch.equal(part, whole[f0:f1])
        if mode == 4:
            assert torch.equal(ppad, wpad[f0:f1])


# ---------------------------------------------------------------------------------------------------- argument checks
def test_bad_arguments_are_refused(ctx):
    """Now that the prologue, the halo fill and every epilogue are reachable from outside, the launchers refuse what their
    kernels cannot do (code 2, before anything is launched), and the context stays usable."""
    from ltx_video_swift_mlx_b200._lib import LtxError
    T, H, W, Cin = 2, 8, 8, 128
    xp, w, b, g = conv_inputs(T, H, W, Cin, 512)
    out = torch.zeros(2 * T * 4 * H * 4 * W * 64, device="cuda")          # big enough for every layout below
    resid = torch.zeros(T * H * W * 512, device="cuda")
    npad = torch.zeros((T + 2) * (H + 2) * (W + 2) * 256, device="cuda", dtype=torch.bfloat16)
    tab = torch.zeros(512, device="cuda")

    def conv(Cout, mode, o=out, r=resid, t_shift=0, np_=npad, sc=None, sh=None, nts=1):
        return ctx.lib.ltx_op_conv3d_epi(ctx.handle, xp.data_ptr(), w.data_ptr(), b.data_ptr(), T, H, W, Cin, Cout, 27, mode,
                                         ptr(o), ptr(r), t_shift, 0, ptr(np_), ptr(sc), ptr(sh), nts)
    refused = {
        "unpatchify with Cout != 48": lambda: conv(64, 2),
        "unpatchify with Cout = 96": lambda: conv(96, 2),
        "t_shift 2": lambda: conv(512, 1, t_shift=2),
        "t_shift -1": lambda: conv(512, 1, t_shift=-1),
        "next_tshift 0": lambda: conv(128, 3, nts=0),
        "next_tshift 3": lambda: conv(128, 4, nts=3),
        "mode 0 without out": lambda: conv(128, 0, o=None),
        "mode 1 without out": lambda: conv(512, 1, o=None),
        "mode 1 without resid": lambda: conv(512, 1, r=None),
        "mode 2 without out": lambda: conv(48, 2, o=None),
        "mode 3 without next_pad": lambda: conv(128, 3, np_=None),
        "mode 4 without next_pad": lambda: conv(128, 4, np_=None),
        "mode 4 without resid": lambda: conv(128, 4, r=None),
        "mode 3 with only next_scale": lambda: conv(128, 3, sc=tab),
        "mode 3 at Cout 192 (a 128-wide tile)": lambda: conv(192, 3),
        "mode 5": lambda: conv(128, 5),
        "prologue mode 4": lambda: ctx.lib.ltx_op_vae_prep(ctx.handle, resid.data_ptr(), npad.data_ptr(), T, H, W, 64, 4, None, None, 0),
        "prologue mode 1 without tables": lambda: ctx.lib.ltx_op_vae_prep(ctx.handle, resid.data_ptr(), npad.data_ptr(), T, H, W, 64, 1,
                                                                           None, None, 0),
        "prologue mode 2 with only a": lambda: ctx.lib.ltx_op_vae_prep(ctx.handle, resid.data_ptr(), npad.data_ptr(), T, H, W, 64, 2,
                                                                        tab.data_ptr(), None, 0),
        "prologue pad 8": lambda: ctx.lib.ltx_op_vae_prep(ctx.handle, resid.data_ptr(), npad.data_ptr(), T, H, W, 64, 0, None, None, 8),
        "halo fill pad 8": lambda: ctx.lib.ltx_op_vae_halo_fill(ctx.handle, npad.data_ptr(), T, H, W, 64, 8),
    }
    torch.cuda.synchronize()
    for what, call in refused.items():
        with pytest.raises(LtxError) as e:
            ctx._check(call())
        assert e.value.code == 2, what
    ctx._check(conv(512, 0))
    ctx.sync()
