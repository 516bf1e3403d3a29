"""Scaled-FP8 transformer checkpoints (an F8_E4M3 "X.weight" with "X.weight_scale" beside it): ltx_load_safetensors and
ltx_load_tensor_e4m3 decode them bit for bit as the decoded values would load in bf16 / int8 / fp32 modes, FP8 mode keeps the
file's codes and scales, and every malformed file is refused without leaving a tensor behind."""
import contextlib
import ctypes as C
import json
import math
import os
import struct

import numpy as np
import pytest
import torch

from fp8_ref import fake_quant
from helpers import O, product, rel_l2, small_dit_config

pytestmark = pytest.mark.gpu
LTX_ERR_INVALID_ARGUMENT, LTX_ERR_WEIGHTS = 2, 4
# FP8 mode's bounds (tests/test_gpu_fp8.py); measured on an NVIDIA B200 at a 1000 W power limit beside each
FWD_ORACLE_TOL = 2e-2    # forward against the oracle on the file's decoded weights; measured 1.14e-2
LOOP_TOL = 3e-2          # 4-step guided loop, same oracle; measured 1.78e-2
MEASURED = {}


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k, v in sorted(MEASURED.items()):
        print(f"fp8 checkpoint measured {k}: {v:.3e}")


# ---------------------------------------------------------------------------------------------------------- file writer
_DTYPES = {torch.float32: "F32", torch.bfloat16: "BF16", torch.float16: "F16", torch.float8_e4m3fn: "F8_E4M3",
           torch.float8_e5m2: "F8_E5M2"}


def write_safetensors(path, tensors, dtypes=None):
    """tensors: name -> torch tensor (F32 / BF16 / F16 / F8_E4M3 / F8_E5M2 from its dtype); dtypes overrides the header's dtype
    string of a name (for malformed files)."""
    header, blobs, off = {}, [], 0
    for k, v in tensors.items():
        v = v.contiguous()
        raw = v.reshape(-1).view(torch.uint8).numpy().tobytes() if v.numel() else b""
        header[k] = {"dtype": (dtypes or {}).get(k, _DTYPES[v.dtype]), "shape": list(v.shape),
                     "data_offsets": [off, off + len(raw)]}
        blobs.append(raw)
        off += len(raw)
    hj = json.dumps(header).encode()
    hj += b" " * ((8 - len(hj) % 8) % 8)
    with open(path, "wb") as f:
        f.write(struct.pack("<Q", len(hj)))
        f.write(hj)
        for b in blobs:
            f.write(b)


# ---------------------------------------------------------------------------------------------------------- checkpoints
def encode(w, scale):
    """e4m3 codes of w / scale (scale [1] or [N]); values beyond +-448 saturate."""
    s = scale.reshape(-1, 1).double() if scale.numel() > 1 else scale.double().reshape(1, 1)
    return (w.double() / s).clamp(-448.0, 448.0).to(torch.float8_e4m3fn)


def decode_bf16(codes, scale):
    s = scale.float().reshape(-1, 1) if scale.numel() > 1 else scale.float().reshape(1, 1)
    return (codes.float() * s).bfloat16()


def decode_f32(codes, scale):
    s = scale.float().reshape(-1, 1) if scale.numel() > 1 else scale.float().reshape(1, 1)
    return codes.float() * s


def decode_f64(codes, scale):
    """What FP8 mode multiplies by: the code times the fp32 scale."""
    s = scale.float().double().reshape(-1, 1) if scale.numel() > 1 else scale.float().double().reshape(1, 1)
    return codes.double() * s


# which Linears arrive as codes, and how they are scaled: "t" one scale per tensor, "c" one per output channel
BLOCK_PLAN = {"attn1.to_q": "t", "attn1.to_k": "c", "attn1.to_out": "c", "attn2.to_q": "t", "attn2.to_k": "c",
              "attn2.to_v": "t", "ff.project_in.proj": "c", "ff.project_out": "t"}          # attn1.to_v, attn2.to_out: bf16
OUTER_PLAN = {"patchify_proj": "c", "caption_projection.linear_2": "t", "adaln_single.linear": "c", "proj_out": "t"}


def _scale(w, kind, pow2, g):
    amax = w.double().abs().amax(1)
    if kind == "t":
        if pow2:
            return torch.tensor([2.0 ** math.ceil(math.log2(float(amax.max()) / 448.0))])
        return torch.tensor([0.0137])   # a non-power of two
    if pow2:
        return torch.pow(2.0, torch.ceil(torch.log2(amax / 448.0))).float()
    return (amax / 448.0 * (1.0 + 0.5 * torch.rand(w.shape[0], generator=g, dtype=torch.float64))).float()


def build_checkpoint(w, layers, plans, pow2=False, seed=0, scale_dtype=torch.float32):
    """-> (file tensors, {post-mapping weight key: (codes, fp32 scale)}).  pow2: power-of-two scales and a code of magnitude
    448 in every row, so that FP8 mode's per-row rule applied to the decoded values gives back the same codes and scales."""
    g = torch.Generator().manual_seed(seed)
    names = [p for p in plans[1]] + [f"transformer_blocks.{i}.{p}" for i in range(layers) for p in plans[0]]
    kinds = {**plans[1], **{f"transformer_blocks.{i}.{p}": k for i in range(layers) for p, k in plans[0].items()}}
    file, coded = {}, {}
    for k, v in w.items():
        file[k] = v.bfloat16() if v.ndim >= 2 else v.float()
    for n in names:
        wt = w[n + ".weight"]
        s = _scale(wt, kinds[n], pow2, g).to(scale_dtype).float()
        q = encode(wt, s)
        if pow2:   # the largest code of every row becomes +-448
            qb = q.view(torch.uint8).clone()
            idx = q.float().abs().argmax(1)
            rows = torch.arange(q.shape[0])
            qb[rows, idx] = (qb[rows, idx] & 0x80) | 0x7E
            q = qb.view(torch.float8_e4m3fn)
        file[n + ".weight"] = q
        file[n + ".weight_scale"] = s.to(scale_dtype).reshape([] if kinds[n] == "t" else [-1])
        file[n + ".input_scale"] = torch.tensor(1.0)
        coded[n + ".weight"] = (q.view(torch.uint8), s)
    return file, coded


def decoded_weights(w, coded, how):
    out = dict(w)
    for k, (q, s) in coded.items():
        out[k] = how(q.view(torch.float8_e4m3fn), s)
    return out


# ---------------------------------------------------------------------------------------------------------- contexts
def _ctx(pcfg, precision=16):
    c = product().LtxContext(pcfg, 0)
    if precision != 16:
        c.set_precision(precision)
    return c


def _from_file(pcfg, path, precision=16, which=1, quant_bits=16, materialise=False, finalize=True):
    c = _ctx(pcfg, precision)
    n = c.load_safetensors(path, which)
    if materialise:
        c.set_quant_storage(True)
    if finalize:
        c.finalize_weights(quant_bits)
    return c, n


def _from_dict(pcfg, w, precision=16, quant_bits=16, materialise=False, finalize=True):
    c = _ctx(pcfg, precision)
    c.load_weights(w)
    if materialise:
        c.set_quant_storage(True)
    if finalize:
        c.finalize_weights(quant_bits)
    return c


def _inputs(ocfg, N, S, seed, B=1):
    g = torch.Generator().manual_seed(seed)
    lat = torch.randn(B, N, ocfg.in_channels, generator=g).bfloat16()
    cx = torch.randn(B, S, ocfg.caption_channels, generator=g)
    return lat, (cx / cx.pow(2).mean(-1, keepdim=True).sqrt()).bfloat16()


FHW, S = (2, 4, 6), 40


def _forward(c, ocfg, B=1, seed=7):
    lat, cx = _inputs(ocfg, FHW[0] * FHW[1] * FHW[2], S, seed, B)
    sig = np.array([0.6, 0.35][:B], dtype=np.float32)
    return c.dit_forward(lat, cx, sig, None, FHW)


def _wf32(w):
    return {k: v.float() for k, v in w.items()}


@pytest.fixture(scope="module")
def setup(tmp_path_factory):
    ocfg, pcfg = small_dit_config(2, 2)
    w = O.make_dit_weights(ocfg, 101)
    d = tmp_path_factory.mktemp("fp8ckpt")
    file, coded = build_checkpoint(w, 2, (BLOCK_PLAN, OUTER_PLAN), seed=3)
    path = os.path.join(d, "scaled_fp8.safetensors")
    write_safetensors(path, file)
    file2, coded2 = build_checkpoint(w, 2, (BLOCK_PLAN, OUTER_PLAN), pow2=True, seed=4, scale_dtype=torch.bfloat16)
    path2 = os.path.join(d, "scaled_fp8_pow2.safetensors")
    write_safetensors(path2, file2)
    return dict(ocfg=ocfg, pcfg=pcfg, w=w, path=path, coded=coded, path2=path2, coded2=coded2, dir=d,
                n_tensors=len(w))


# ---------------------------------------------------------------------------------------------------------- 1, 2: decode
@pytest.mark.parametrize("quant_bits,materialise", [(16, False), (8, False), (8, True)])
def test_bf16_mode_equals_decoded_bf16_load(setup, quant_bits, materialise):
    s = setup
    a, n = _from_file(s["pcfg"], s["path"], quant_bits=quant_bits, materialise=materialise)
    assert n == s["n_tensors"]
    b = _from_dict(s["pcfg"], (decoded_weights(s["w"], s["coded"], decode_bf16)), quant_bits=quant_bits,
                   materialise=materialise)
    va, vb = _forward(a, s["ocfg"]), _forward(b, s["ocfg"])
    assert np.isfinite(va).all()
    np.testing.assert_array_equal(va, vb)
    a.close(); b.close()


def test_fp32_mode_equals_decoded_fp32_load(setup):
    s = setup
    a, _ = _from_file(s["pcfg"], s["path"], precision=32)
    b = _from_dict(s["pcfg"], _wf32(decoded_weights(s["w"], s["coded"], decode_f32)), precision=32)
    np.testing.assert_array_equal(_forward(a, s["ocfg"]), _forward(b, s["ocfg"]))
    a.close(); b.close()


def test_load_tensor_e4m3_equals_the_file(setup):
    """The C ABI entry point (per-tensor and per-channel scales, float8 or uint8 codes) loads what the file loader loads."""
    s = setup
    a, _ = _from_file(s["pcfg"], s["path"])
    b = _ctx(s["pcfg"])
    b.load_weights({k: v for k, v in (s["w"]).items() if k not in s["coded"]})
    for i, (k, (q, sc)) in enumerate(s["coded"].items()):
        b.load_tensor_e4m3(k, q.view(torch.float8_e4m3fn) if i % 2 else q.numpy(), sc if sc.numel() > 1 else float(sc))
    b.finalize_weights()
    np.testing.assert_array_equal(_forward(a, s["ocfg"]), _forward(b, s["ocfg"]))
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------------------- 3: FP8 keeps codes
def _loop(c, ocfg, graphs):
    fhw = (3, 4, 4)
    g = torch.Generator().manual_seed(52)
    noise = torch.randn(1, 128, *fhw, generator=g)
    _, cx = _inputs(ocfg, 48, S, 53)
    _, ncx = _inputs(ocfg, 48, S, 54)
    sigmas = O.set_timesteps(4, False, 48)
    c.set_graphs(graphs)
    c.denoise_begin(noise[0].numpy(), fhw, sigmas[0], cx, None, ncx, None)
    for i in range(len(sigmas) - 1):
        c.denoise_step(sigmas[i], sigmas[i + 1], i, cfg_scale=3.0, rescale_phi=0.5, batched_cfg=True)
    return c.denoise_get_latent()


def test_fp8_mode_keeps_file_codes_bit_for_bit(setup):
    s = setup
    dec = decoded_weights(s["w"], s["coded2"], decode_bf16)
    # the decode is exact in bf16 here: the twin's weights hold exactly code * scale
    for k, (q, sc) in s["coded2"].items():
        assert torch.equal(dec[k].double(), decode_f64(q.view(torch.float8_e4m3fn), sc)), k
    bf_path = os.path.join(s["dir"], "decoded_bf16.safetensors")
    write_safetensors(bf_path, {k: (v.bfloat16() if v.ndim >= 2 else v.float()) for k, v in dec.items()})
    a, n = _from_file(s["pcfg"], s["path2"], precision=8)
    b, nb = _from_file(s["pcfg"], bf_path, precision=8)
    assert n == nb == s["n_tensors"]
    for B in (1, 2):
        va, vb = _forward(a, s["ocfg"], B), _forward(b, s["ocfg"], B)
        assert np.isfinite(va).all()
        np.testing.assert_array_equal(va, vb)
    la, lb = _loop(a, s["ocfg"], True), _loop(b, s["ocfg"], True)
    captures, replays = a.graph_stats()
    assert captures >= 1 and replays >= 1, (captures, replays)
    np.testing.assert_array_equal(la, lb)
    np.testing.assert_array_equal(la, _loop(a, s["ocfg"], False))
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------------------- 4: FP8 vs oracle
@contextlib.contextmanager
def fp8_file_blocks(coded):
    """Inside: the oracle's block Linears multiply fake-quantised activation rows (FP8 mode's per-row rule) by the file's
    decoded weights in float64 where the file holds codes, and by fake-quantised weight rows where it holds bf16."""
    plain = O.linear
    exact = {k: decode_f64(q.view(torch.float8_e4m3fn), sc) for k, (q, sc) in coded.items()}

    def linear(x, w, name):
        if not name.startswith("transformer_blocks."):
            return plain(x, w, name)
        wk = name + ".weight"
        wt = exact[wk] if wk in exact else fake_quant(w[wk])
        return (fake_quant(x) @ wt.t()).to(x.dtype) + w[name + ".bias"].to(x.dtype)
    O.linear = linear
    try:
        yield
    finally:
        O.linear = plain


def test_fp8_mode_arbitrary_scales_against_oracle(setup):
    s = setup
    ocfg = s["ocfg"]
    c, _ = _from_file(s["pcfg"], s["path"], precision=8)
    # non-block Linears are decoded to bf16 storage: the oracle gets those values
    w_or = decoded_weights(s["w"], {k: v for k, v in s["coded"].items() if not k.startswith("transformer_blocks.")},
                           lambda q, sc: decode_bf16(q, sc).float())
    lat, cx = _inputs(ocfg, 48, S, 7)
    out = c.dit_forward(lat, cx, np.array([0.6], dtype=np.float32), None, FHW)
    with fp8_file_blocks(s["coded"]):
        ref = O.dit_forward(w_or, ocfg, lat.float(), cx.float(), torch.tensor([0.6]), None, FHW)
    err = rel_l2(out, ref)
    MEASURED["forward_vs_oracle"] = err
    assert err <= FWD_ORACLE_TOL, err
    fhw = (3, 4, 6)
    g = torch.Generator().manual_seed(62)
    noise = torch.randn(1, 128, *fhw, generator=g)
    _, pcx = _inputs(ocfg, 72, S, 63)
    _, ncx = _inputs(ocfg, 72, S, 64)
    sigmas = O.set_timesteps(4, False, 72)
    with fp8_file_blocks(s["coded"]):
        ref = O.denoise_loop(w_or, ocfg, noise, pcx.float(), None, sigmas, neg_context=ncx.float(), cfg_scale=3.0, phi=0.5)
    c.denoise_begin(noise[0].numpy(), fhw, sigmas[0], pcx, None, ncx, None)
    for i in range(len(sigmas) - 1):
        c.denoise_step(sigmas[i], sigmas[i + 1], i, cfg_scale=3.0, rescale_phi=0.5)
    err = rel_l2(c.denoise_get_latent(), ref[0])
    MEASURED["loop_vs_oracle"] = err
    assert err <= LOOP_TOL, err
    c.close()


# ---------------------------------------------------------------------------------------------------------- 5: dual model
def test_dual_model_decodes_to_bf16(setup, tmp_path):
    ocfg = O.DiTConfig(num_layers=1, num_heads=2, head_dim=128, caption_channels=192)
    av = O.AVConfig(audio_heads=2)
    pcfg = product().LTXTransformerConfig(num_layers=1, num_attention_heads=2, caption_channels=192, audio_num_attention_heads=2)
    w = O.make_av_weights(ocfg, av, 9)
    block = {**BLOCK_PLAN, "audio_attn1.to_q": "c", "audio_attn1.to_v": "t", "audio_attn2.to_out": "c",
             "audio_ff.project_in.proj": "t", "audio_to_video_attn.to_k": "c", "audio_to_video_attn.to_out": "t",
             "video_to_audio_attn.to_q": "t", "video_to_audio_attn.to_v": "c"}
    outer = {**OUTER_PLAN, "audio_patchify_proj": "c", "audio_caption_projection.linear_1": "t"}
    file, coded = build_checkpoint(w, 1, (block, outer), seed=5)
    path = os.path.join(tmp_path, "av_fp8.safetensors")
    write_safetensors(path, file)
    a, n = _from_file(pcfg, path, which=5)
    assert n == len(w)
    b = _from_dict(pcfg, (decoded_weights(w, coded, decode_bf16)))
    g = torch.Generator().manual_seed(3)
    fhw, Ta = (2, 4, 6), 11
    vl, al = torch.randn(1, 48, 128, generator=g).bfloat16(), torch.randn(1, Ta, 128, generator=g).bfloat16()
    vc, ac = torch.randn(1, S, 192, generator=g).bfloat16(), torch.randn(1, S, 192, generator=g).bfloat16()
    oa = a.av_forward(vl, al, vc, ac, 0.6, 0.4, fhw)
    ob = b.av_forward(vl, al, vc, ac, 0.6, 0.4, fhw)
    assert np.isfinite(oa[0]).all() and np.isfinite(oa[1]).all()
    np.testing.assert_array_equal(oa[0], ob[0])
    np.testing.assert_array_equal(oa[1], ob[1])
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------------------- 6: LoRA
def test_lora_on_codes_equals_lora_on_decoded_twin(setup):
    s = setup
    g = torch.Generator().manual_seed(11)
    D = s["ocfg"].inner_dim
    loras = {"transformer_blocks.0.attn2.to_q.weight": (D, D), "transformer_blocks.1.ff.project_in.proj.weight": (4 * D, D),
             "transformer_blocks.1.attn1.to_k.weight": (D, D)}
    facs = {k: ((torch.randn(8, i, generator=g) * 0.05).bfloat16(), (torch.randn(o, 8, generator=g) * 0.05).bfloat16())
            for k, (o, i) in loras.items()}
    # power-of-two scales: the Linears that stay codes match their twins' conversion bit for bit (test above)
    a, _ = _from_file(s["pcfg"], s["path2"], precision=8, finalize=False)
    b = _from_dict(s["pcfg"], decoded_weights(s["w"], s["coded2"], decode_bf16), precision=8, finalize=False)
    for c in (a, b):
        for k, (dn, up) in facs.items():
            c.fuse_lora(k, dn, up, 0.75)
        c.finalize_weights()
    va, vb = _forward(a, s["ocfg"]), _forward(b, s["ocfg"])
    assert np.isfinite(va).all()
    np.testing.assert_array_equal(va, vb)
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------------------- 7: refusals
PROBE = "aaa_probe.weight"   # sorts first: uploaded before anything the refusal is about


def _code(fn):
    with pytest.raises(product().LtxError) as e:
        fn()
    return e.value.code


def _absent(c, key):
    """fuse_lora names a tensor that is not loaded -> LTX_ERR_WEIGHTS before anything else happens"""
    dn, up = torch.zeros(8, 16), torch.zeros(16, 8)
    return _code(lambda: c.fuse_lora(key, dn, up, 1.0)) == LTX_ERR_WEIGHTS


def _bad_files(s):
    file, _ = build_checkpoint(s["w"], 2, (BLOCK_PLAN, OUTER_PLAN), seed=3)
    file[PROBE] = torch.randn(16, 16).bfloat16()
    wk = "transformer_blocks.1.attn2.to_k.weight"          # per-channel
    tk = "transformer_blocks.0.ff.project_out.weight"      # per-tensor
    N = file[wk].shape[0]
    cases = {}

    def case(name, edit, dtypes=None, which=1):
        f = dict(file)
        edit(f)
        cases[name] = (f, dtypes, which)
    case("no_scale", lambda f: f.pop(wk + "_scale"))
    case("scale_shape_n2", lambda f: f.__setitem__(wk + "_scale", torch.ones(N, 2)))
    case("scale_shape_2", lambda f: f.__setitem__(tk + "_scale", torch.ones(2)))
    case("scale_dtype_f16", lambda f: f.__setitem__(wk + "_scale", torch.ones(N, dtype=torch.float16)))
    case("scale_zero", lambda f: f.__setitem__(tk + "_scale", torch.tensor(0.0)))
    case("scale_negative", lambda f: f.__setitem__(wk + "_scale", -torch.ones(N)))
    case("scale_inf", lambda f: f.__setitem__(tk + "_scale", torch.tensor(float("inf"))))
    case("scale_nan", lambda f: f.__setitem__(wk + "_scale", torch.full((N,), float("nan")).bfloat16()))
    case("e5m2", lambda f: f.__setitem__("transformer_blocks.0.attn1.to_v.weight",
                                         f["transformer_blocks.0.attn1.to_v.weight"].float().to(torch.float8_e5m2)))

    def coded_other(key, shape):
        def edit(f):
            f[key] = torch.ones(shape).to(torch.float8_e4m3fn)
            f[key + "_scale"] = torch.tensor(1.0)
        return edit
    case("e4m3_bias", coded_other("transformer_blocks.0.attn1.to_q.bias", (256,)))
    case("e4m3_norm", coded_other("transformer_blocks.0.attn1.q_norm.weight", (256,)))
    case("e4m3_table", coded_other("transformer_blocks.0.scale_shift_table", (6, 256)))

    def nan_code(code):
        def edit(f):
            q = f[wk].view(torch.uint8).clone()
            q[3, 5] = code
            f[wk] = q.view(torch.float8_e4m3fn)
        return edit
    case("nan_7f", nan_code(0x7F))
    case("nan_ff", nan_code(0xFF))
    # a VAE file with an e4m3 conv kernel
    vae = {"decoder.conv_in.conv.weight": torch.ones(8, 8, 3, 3, 3).to(torch.float8_e4m3fn),
           "decoder.conv_in.conv.weight_scale": torch.tensor(1.0), "decoder.aaa.weight": torch.randn(4, 4)}
    cases["vae_e4m3"] = (vae, None, 2)
    vae2 = {"decoder.time_embedder.linear_1.weight": torch.ones(8, 8).to(torch.float8_e4m3fn),
            "decoder.time_embedder.linear_1.weight_scale": torch.tensor(1.0)}
    cases["vae_e4m3_linear"] = (vae2, None, 2)
    return cases


@pytest.mark.parametrize("precision", [16, 8])
def test_refusals_leave_nothing_behind(setup, precision):
    s = setup
    ref_ctx, _ = _from_file(s["pcfg"], s["path"], precision=precision)
    ref = _forward(ref_ctx, s["ocfg"])
    ref_ctx.close()
    c = _ctx(s["pcfg"], precision)
    for name, (f, dtypes, which) in _bad_files(s).items():
        p = os.path.join(s["dir"], f"bad_{name}_{precision}.safetensors")
        write_safetensors(p, f, dtypes)
        assert _code(lambda: c.load_safetensors(p, which)) == LTX_ERR_WEIGHTS, name
        assert _absent(c, PROBE) and _absent(c, "vae.aaa.weight"), name
    # the C ABI: n_scales other than 1 or N, and a NaN code
    q = torch.zeros(16, 32, dtype=torch.uint8)
    shape = (C.c_int64 * 2)(16, 32)
    for n_scales in (0, 2, 15, 17):
        sc = np.ones(max(n_scales, 1), dtype=np.float32)
        rc = c.lib.ltx_load_tensor_e4m3(c.handle, b"transformer_blocks.0.attn1.to_q.weight", q.numpy().ctypes.data,
                                        sc.ctypes.data, n_scales, shape, 2)
        assert rc == LTX_ERR_INVALID_ARGUMENT, n_scales
    assert _code(lambda: c.load_tensor_e4m3("transformer_blocks.0.attn1.to_q.weight", q, [1.0, -1.0] + [1.0] * 14)) == LTX_ERR_WEIGHTS
    assert _code(lambda: c.load_tensor_e4m3("vae.up_blocks_0.time_embedder.linear_1.weight", q, 1.0)) == LTX_ERR_WEIGHTS
    assert _code(lambda: c.load_tensor_e4m3("transformer_blocks.0.attn1.to_q.bias", q, 1.0)) == LTX_ERR_WEIGHTS
    qn = q.clone()
    qn[7, 9] = 0xFF
    assert _code(lambda: c.load_tensor_e4m3("transformer_blocks.0.attn1.to_q.weight", qn, 1.0)) == LTX_ERR_WEIGHTS
    assert _absent(c, "transformer_blocks.0.attn1.to_q.weight")
    # a good file still loads in full and computes what a fresh context computes
    assert c.load_safetensors(s["path"], 1) == s["n_tensors"]
    c.finalize_weights()
    np.testing.assert_array_equal(_forward(c, s["ocfg"]), ref)
    c.close()
