"""LtxContext: owner of one libltxcuda context (one GPU).  Thin, typed wrapper over the C ABI; all arithmetic happens
inside libltxcuda.so."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import (LTX_BF16, LTX_F16, LTX_F32, LTX_FRAMES_I420, LTX_FRAMES_RGB8, LtxConfig, LtxDitFlags, LtxError,
                   LtxStepParams)


@dataclass
class LTXTransformerConfig:
    """Mirror of LTXTransformerConfig (Configuration/LTXConfig.swift:83-156) + the VAE channel plan."""
    num_layers: int = 48
    num_attention_heads: int = 32
    attention_head_dim: int = 128
    in_channels: int = 128
    out_channels: int = 128
    caption_channels: int = 3840
    ffn_mult: int = 4
    rope_theta: float = 10000.0
    max_pos: Tuple[int, int, int] = (20, 2048, 2048)
    timestep_scale_multiplier: float = 1000.0
    norm_eps: float = 1e-6
    vae_latent_channels: int = 128
    vae_base_channels: int = 1024
    vae_blocks_per_stage: int = 5
    vae_patch_size: int = 4
    vae_encoder_base_channels: int = 128     # VideoEncoder channel plan (random init only)
    upscaler_mid_channels: int = 1024        # SpatialUpscaler(midChannels:) (random init only)
    upscaler_blocks: int = 4
    audio_num_attention_heads: int = 32      # audio stream of LTX2Transformer (Configuration/LTXConfig.swift:134-173)
    audio_attention_head_dim: int = 64
    audio_in_channels: int = 128
    audio_max_pos: int = 20

    @property
    def inner_dim(self) -> int:
        return self.num_attention_heads * self.attention_head_dim

    def to_c(self) -> LtxConfig:
        c = LtxConfig()
        c.num_layers, c.num_heads, c.head_dim = self.num_layers, self.num_attention_heads, self.attention_head_dim
        c.in_channels, c.out_channels, c.caption_channels = self.in_channels, self.out_channels, self.caption_channels
        c.ffn_mult, c.rope_theta = self.ffn_mult, self.rope_theta
        for i in range(3):
            c.max_pos[i] = self.max_pos[i]
        c.timestep_scale_multiplier, c.norm_eps = self.timestep_scale_multiplier, self.norm_eps
        c.vae_latent_channels, c.vae_base_channels = self.vae_latent_channels, self.vae_base_channels
        c.vae_blocks_per_stage, c.vae_patch_size = self.vae_blocks_per_stage, self.vae_patch_size
        c.vae_encoder_base_channels, c.upscaler_mid_channels = self.vae_encoder_base_channels, self.upscaler_mid_channels
        c.upscaler_blocks = self.upscaler_blocks
        c.audio_num_heads, c.audio_head_dim = self.audio_num_attention_heads, self.audio_attention_head_dim
        c.audio_in_channels, c.audio_max_pos = self.audio_in_channels, self.audio_max_pos
        return c


def _host(a, dtype=None) -> np.ndarray:
    """Contiguous host ndarray from a numpy array or a CPU torch tensor (bf16 tensors are viewed as uint16)."""
    if hasattr(a, "detach"):
        import torch
        t = a.detach().cpu().contiguous()
        if t.dtype == torch.bfloat16:
            return t.view(torch.uint16).numpy()
        a = t.numpy()
    a = np.ascontiguousarray(a)
    if dtype is not None and a.dtype != dtype:
        a = np.ascontiguousarray(a.astype(dtype))
    return a


def _dtype_code(a) -> int:
    if hasattr(a, "detach"):
        import torch
        return {torch.float32: LTX_F32, torch.bfloat16: LTX_BF16, torch.float16: LTX_F16}[a.dtype]
    return {np.dtype(np.float32): LTX_F32, np.dtype(np.float16): LTX_F16, np.dtype(np.uint16): LTX_BF16}[np.asarray(a).dtype]


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _frames_format(format) -> int:
    """Frame format code from "rgb8" / "i420" or an ltx_frames_format code (other codes go to the library, which refuses them)."""
    if isinstance(format, str):
        return {"rgb8": LTX_FRAMES_RGB8, "i420": LTX_FRAMES_I420}[format.lower()]
    return int(format)


def make_flags(stg_blocks: Sequence[int] = (), skip_self_attn: bool = False, skip_ff: bool = False,
               cas_blocks: Sequence[int] = (), cross_attn_scale: float = 1.0, context_key: int = 0) -> LtxDitFlags:
    f = LtxDitFlags()
    f.n_stg_blocks = len(stg_blocks)
    for i, b in enumerate(stg_blocks):
        f.stg_blocks[i] = int(b)
    f.skip_self_attn, f.skip_ff = int(skip_self_attn), int(skip_ff)
    f.n_cas_blocks = len(cas_blocks)
    for i, b in enumerate(cas_blocks):
        f.cas_blocks[i] = int(b)
    f.cross_attn_scale = float(cross_attn_scale)
    f.context_key = int(context_key)
    return f


def map_weight_key(which: int, file_key: str) -> Optional[str]:
    """mapTransformerKey (which=1) / mapVAEWeights (which=2) for one checkpoint key; None = skipped by the loader."""
    buf = C.create_string_buffer(512)
    rc = _lib.load().ltx_map_weight_key(int(which), file_key.encode(), buf, 512)
    if rc != 0:
        raise LtxError(rc, "ltx_map_weight_key failed")
    s = buf.value.decode()
    return s or None


class LtxContext:
    def __init__(self, config: Optional[LTXTransformerConfig] = None, device: int = 0):
        self.lib = _lib.load()
        self.config = config or LTXTransformerConfig()
        self.device = device
        h = C.c_void_p()
        cfg = self.config.to_c()
        rc = self.lib.ltx_ctx_create(C.byref(cfg), device, C.byref(h))
        if rc != 0:
            raise LtxError(rc, self.lib.ltx_last_error(None).decode())
        self.handle = h

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc: int):
        if rc != 0:
            raise LtxError(rc, self.lib.ltx_last_error(self.handle).decode())

    def close(self):
        if getattr(self, "handle", None):
            self.lib.ltx_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        self._check(self.lib.ltx_sync(self.handle))

    @property
    def launch_count(self) -> int:
        return int(self.lib.ltx_launch_count(self.handle))

    @property
    def stream(self) -> int:
        p = C.c_void_p()
        self._check(self.lib.ltx_get_stream(self.handle, C.byref(p)))
        return p.value or 0

    def set_graphs(self, enabled: bool):
        """Captured-step replay (CUDA graphs) on / off; off also drops what was captured."""
        self._check(self.lib.ltx_set_graphs(self.handle, int(enabled)))

    def graph_stats(self) -> Tuple[int, int]:
        """(captures, replays) so far."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        self._check(self.lib.ltx_graph_stats(self.handle, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def set_profiling(self, enabled: bool):
        self._check(self.lib.ltx_set_profiling(self.handle, int(enabled)))

    PROFILE_CLASSES = ("gemm", "attention", "rows", "conv3d", "vae_prologue", "other", "comm")

    def get_profile(self) -> Dict[str, dict]:
        n = 8
        ms, fl, by = (C.c_double * n)(), (C.c_double * n)(), (C.c_double * n)()
        cnt = (C.c_uint64 * n)()
        self._check(self.lib.ltx_get_profile(self.handle, ms, fl, by, cnt, n))
        return {name: dict(ms=ms[i], flops=fl[i], bytes=by[i], launches=int(cnt[i]))
                for i, name in enumerate(self.PROFILE_CLASSES)}

    # ------------------------------------------------------------------ multi-GPU
    @staticmethod
    def dist_unique_id() -> bytes:
        lib = _lib.load()
        buf = C.create_string_buffer(128)
        rc = lib.ltx_dist_get_unique_id(buf)
        if rc != 0:
            raise LtxError(rc, lib.ltx_last_error(None).decode())
        return buf.raw

    def dist_init(self, unique_id: bytes, rank: int, world_size: int, sp_size: int = 1, pass_groups: int = 1):
        assert len(unique_id) == 128
        self._check(self.lib.ltx_dist_init(self.handle, unique_id, rank, world_size, sp_size, pass_groups))

    @staticmethod
    def dist_init_local(contexts: Sequence["LtxContext"], sp_size: int = 1, pass_groups: Optional[int] = None):
        """All ranks in this process: contexts[i] (one per device) becomes rank i.  Collective calls must then be issued
        concurrently, one host thread per context (ctypes releases the GIL while a call runs)."""
        n = len(contexts)
        if pass_groups is None:
            pass_groups = n // sp_size
        arr = (C.c_void_p * n)(*[c.handle for c in contexts])
        contexts[0]._check(contexts[0].lib.ltx_dist_init_local(arr, n, int(sp_size), int(pass_groups)))

    def dist_shutdown(self):
        self._check(self.lib.ltx_dist_shutdown(self.handle))

    # ------------------------------------------------------------------ weights
    def load_tensor(self, key: str, value):
        code = _dtype_code(value)
        a = _host(value)
        shape = (C.c_int64 * max(1, a.ndim))(*a.shape)
        self._check(self.lib.ltx_load_tensor(self.handle, key.encode(), _ptr(a), code, shape, a.ndim))

    def load_tensor_e4m3(self, key: str, codes, scale):
        """A transformer Linear weight [N, K] of a scaled-FP8 checkpoint: codes as a torch.float8_e4m3fn tensor or uint8 codes
        (numpy or torch), scale one value (per tensor) or N values (per output channel); w = e4m3(code) * scale.  Decoded to the
        mode's storage, or kept as codes for the block Linears in FP8 mode (ltx_load_tensor_e4m3)."""
        if hasattr(codes, "detach"):
            import torch
            t = codes.detach().cpu().contiguous()
            if t.dtype == torch.float8_e4m3fn:
                t = t.view(torch.uint8)
            codes = t.numpy()
        q = np.ascontiguousarray(codes)
        if q.dtype != np.uint8 or q.ndim != 2:
            raise LtxError(2, "load_tensor_e4m3: codes must be a 2-D float8_e4m3fn or uint8 tensor")
        s = np.ascontiguousarray(np.asarray(scale.detach().cpu().float() if hasattr(scale, "detach") else scale,
                                            dtype=np.float32).reshape(-1))
        shape = (C.c_int64 * 2)(*q.shape)
        self._check(self.lib.ltx_load_tensor_e4m3(self.handle, key.encode(), _ptr(q), _ptr(s), s.size, shape, 2))

    def load_weights(self, weights: Dict[str, object], prefix: str = ""):
        for k, v in weights.items():
            self.load_tensor(prefix + k, v)

    def load_safetensors(self, path: str, which: int) -> int:
        """LTXWeightLoader.loadTransformerWeights (which=1) / loadVAEWeights (2) / loadVAEEncoderWeights (3) /
        loadSpatialUpscaler (4): reads the checkpoint, maps the keys and uploads the tensors.  Returns the number taken."""
        n = C.c_int(0)
        self._check(self.lib.ltx_load_safetensors(self.handle, str(path).encode(), int(which), C.byref(n)))
        return n.value

    def fuse_lora(self, key: str, down, up, scale: float = 1.0):
        """LoRAAdapter.fuseWeights for one layer: W[key] += scale * up @ down (down [r, in], up [out, r]); before finalize_weights."""
        code = _dtype_code(down)
        assert _dtype_code(up) == code
        d, u = _host(down), _host(up)
        assert d.ndim == 2 and u.ndim == 2 and d.shape[0] == u.shape[1]
        self._check(self.lib.ltx_fuse_lora(self.handle, key.encode(), _ptr(d), _ptr(u), code, int(d.shape[0]), float(scale)))

    def set_precision(self, bits: int):
        """16 = bf16 mode (default), 32 = fp32 mode (fp32 DiT weights, split-bf16 tensor-core GEMMs), 8 = FP8 mode (the block
        Linears run as e4m3 x e4m3 GEMMs with per-row power-of-two scales; no quantised weights, sequence parallelism or dual
        audio/video model); before loading weights."""
        self._check(self.lib.ltx_set_precision(self.handle, int(bits)))

    def set_quant_storage(self, materialise: bool):
        """False (default): quantised weights stay as codes; True: their dequantised bf16 values replace the weights at
        finalize time (same results, bf16 speed and footprint).  Before finalize_weights(quant_bits=8 | 4)."""
        self._check(self.lib.ltx_set_quant_storage(self.handle, int(materialise)))

    def init_random_weights(self, which: int = 3, seed: int = 0):
        self._check(self.lib.ltx_init_random_weights(self.handle, which, seed))

    def finalize_weights(self, quant_bits: int = 16, group_size: int = 64):
        self._check(self.lib.ltx_finalize_weights(self.handle, quant_bits, group_size))

    # ------------------------------------------------------------------ DiT
    def dit_forward(self, latent, context, timesteps, mask, fhw: Tuple[int, int, int],
                    flags: Optional[LtxDitFlags] = None) -> np.ndarray:
        """Host-buffer call (the Swift seam): latent [B,N,C], context [B,S,Cc], timesteps [B], mask [B,S]|None."""
        lc, cc = _dtype_code(latent), _dtype_code(context)
        lat, ctx = _host(latent), _host(context)
        ts = _host(timesteps, np.float32)
        per_token = 1 if ts.ndim == 2 else 0
        mk = None if mask is None else _host(mask, np.int32)
        B, N = lat.shape[0], lat.shape[1]
        S = ctx.shape[1]
        out = np.empty((B, N, self.config.out_channels), dtype=np.float32)
        F, H, W = fhw
        self._check(self.lib.ltx_dit_forward(self.handle, _ptr(lat), lc, _ptr(ctx), cc, _ptr(ts), per_token, _ptr(mk), B, N, S, F, H, W,
                                             C.byref(flags) if flags is not None else None, _ptr(out)))
        return out

    def dit_forward_dev(self, latent_ptr: int, latent_dtype: int, context_ptr: int, context_dtype: int, ts_ptr: int,
                        mask_ptr: Optional[int], B: int, N: int, S: int, fhw, flags: Optional[LtxDitFlags], out_ptr: int):
        F, H, W = fhw
        self._check(self.lib.ltx_dit_forward_dev(self.handle, latent_ptr, latent_dtype, context_ptr, context_dtype, ts_ptr, 0,
                                                 mask_ptr, B, N, S, F, H, W,
                                                 C.byref(flags) if flags is not None else None, out_ptr))

    def av_forward(self, video_latent, audio_latent, video_context, audio_context, video_sigma, audio_sigma,
                   fhw: Tuple[int, int, int], video_mask=None, audio_mask=None, context_key: int = 0):
        """LTX2Transformer.callAsFunction: video_latent [B,N,C], audio_latent [B,Ta,Ca], contexts [B,S,Cc], B = 1 or 2 ->
        (video velocity [B,N,C], audio velocity [B,Ta,Ca]) fp32.  video_sigma: a float, or an array [B] / [1,N] / [N] / [B,N]
        (per-token sigmas: videoTimesteps of the image-to-video mode); audio_sigma: a float or [B]; masks [B,S] or None.
        Mismatched batch tensors raise LtxError code 2; B > 2 code 5 (the library's refusal)."""
        vc, ac, cc = _dtype_code(video_latent), _dtype_code(audio_latent), _dtype_code(video_context)
        assert _dtype_code(audio_context) == cc, "both contexts must have the same dtype"
        vl, al, vx, axx = _host(video_latent), _host(audio_latent), _host(video_context), _host(audio_context)
        B, N, Ta, S = vl.shape[0], vl.shape[1], al.shape[1], vx.shape[1]
        vm = None if video_mask is None else _host(video_mask, np.int32)
        am = None if audio_mask is None else _host(audio_mask, np.int32)
        F, H, W = fhw
        if B != 1:
            vs = _host(np.asarray(video_sigma, dtype=np.float32).reshape(-1), np.float32)
            as_ = _host(np.asarray(audio_sigma, dtype=np.float32).reshape(-1), np.float32)
            per_token = vs.size == B * N and vs.size != B
            ok = (al.shape[0] == B and vx.shape[0] == B and _host(audio_context).shape[:2] == (B, S) and as_.size == B
                  and (vs.size == B or per_token)
                  and all(m is None or m.size == B * S for m in (vm, am)))
            if not ok:
                raise LtxError(2, "dual forward: batch tensors must all have B items ([B,N,C], [B,Ta,Ca], [B,S,Cc], "
                                  "sigmas [B] / [B,N], masks [B,S])")
            ov = np.full((B, N, self.config.out_channels), np.nan, dtype=np.float32)
            oa = np.full((B, Ta, self.config.audio_in_channels), np.nan, dtype=np.float32)
            self._check(self.lib.ltx_av_forward_batch(self.handle, _ptr(vl), vc, _ptr(al), ac, _ptr(vx), _ptr(axx), cc, _ptr(vs),
                                                      int(per_token), _ptr(as_), _ptr(vm), _ptr(am), B, N, Ta, S, F, H, W,
                                                      int(context_key), _ptr(ov), _ptr(oa)))
            return ov, oa
        assert al.shape[0] == 1, "video and audio latents must have the same batch"
        ov = np.empty((1, N, self.config.out_channels), dtype=np.float32)
        oa = np.empty((1, Ta, self.config.audio_in_channels), dtype=np.float32)
        audio_sigma = float(np.asarray(audio_sigma).reshape(-1)[0])
        if not np.isscalar(video_sigma) and np.asarray(video_sigma).size > 1:
            vs = np.ascontiguousarray(_host(video_sigma, np.float32).reshape(-1))
            assert vs.size == N, "per-token video sigmas must have N entries"
            self._check(self.lib.ltx_av_forward_tokens(self.handle, _ptr(vl), vc, _ptr(al), ac, _ptr(vx), _ptr(axx), cc, _ptr(vs),
                                                       float(audio_sigma), _ptr(vm), _ptr(am), N, Ta, S, F, H, W,
                                                       int(context_key), _ptr(ov), _ptr(oa)))
            return ov, oa
        video_sigma = float(np.asarray(video_sigma).reshape(-1)[0])
        self._check(self.lib.ltx_av_forward(self.handle, _ptr(vl), vc, _ptr(al), ac, _ptr(vx), _ptr(axx), cc, float(video_sigma),
                                            float(audio_sigma), _ptr(vm), _ptr(am), N, Ta, S, F, H, W, int(context_key),
                                            _ptr(ov), _ptr(oa)))
        return ov, oa

    def clear_caches(self):
        """clearRoPECache + the text-projection caches of both streams (video and, in the dual model, audio)."""
        self._check(self.lib.ltx_dit_clear_caches(self.handle))

    def new_context_key(self) -> int:
        """A context_key no earlier call on this context has used: the host-seam loops take one per prompt per generation, so a
        second generation never finds the first one's projected text under its key."""
        self._key_serial = getattr(self, "_key_serial", 0) + 1
        return 0x6000000000000000 + self._key_serial

    # ------------------------------------------------------------------ guidance + Euler
    def guided_euler_step(self, latent: np.ndarray, v_cond, v_uncond=None, v_stg=None, v_prev=None, use_prev: bool = False,
                          cfg_scale: float = 1.0, rescale_phi: float = 0.0, stg_scale: float = 0.0, ge_gamma: float = 0.0,
                          sigma: float = 1.0, sigma_next: float = 0.0) -> np.ndarray:
        """In place on `latent` (fp32 host array); `v_prev` (if given) is updated with the velocity used."""
        assert latent.dtype == np.float32 and latent.flags["C_CONTIGUOUS"]
        vc = _host(v_cond, np.float32)
        vu = None if v_uncond is None else _host(v_uncond, np.float32)
        vs = None if v_stg is None else _host(v_stg, np.float32)
        if v_prev is not None:
            assert v_prev.dtype == np.float32 and v_prev.flags["C_CONTIGUOUS"]
        self._check(self.lib.ltx_guided_euler_step(self.handle, _ptr(latent), _ptr(vc), _ptr(vu), _ptr(vs), _ptr(v_prev),
                                                   int(use_prev), latent.size, cfg_scale, rescale_phi, stg_scale, ge_gamma,
                                                   sigma, sigma_next))
        return latent

    # ------------------------------------------------------------------ resident denoise session
    def denoise_begin(self, noise, fhw, sigma0: float, context, mask=None, neg_context=None, neg_mask=None):
        nz = _host(noise, np.float32)
        cc = _dtype_code(context)
        ctx = _host(context)
        S = ctx.shape[-2]
        mk = None if mask is None else _host(mask, np.int32)
        nctx = None if neg_context is None else _host(neg_context)
        nmk = None if neg_mask is None else _host(neg_mask, np.int32)
        F, H, W = fhw
        self._check(self.lib.ltx_denoise_begin(self.handle, _ptr(nz), F, H, W, sigma0, _ptr(ctx), cc, _ptr(mk), _ptr(nctx),
                                               _ptr(nmk), S))
        self._session_shape = (self.config.in_channels, F, H, W)

    def denoise_begin_from_latent(self, latent, noise, noise_scale: float, fhw, context, mask=None, neg_context=None,
                                  neg_mask=None, frame0_latent=None):
        """Stage-2 start point (P/LTXPipeline.swift:2636-2657): latent = noise_scale * noise + (1 - noise_scale) * latent."""
        lt, nz = _host(latent, np.float32), _host(noise, np.float32)
        f0 = None if frame0_latent is None else _host(frame0_latent, np.float32)
        cc = _dtype_code(context)
        ctx = _host(context)
        S = ctx.shape[-2]
        mk = None if mask is None else _host(mask, np.int32)
        nctx = None if neg_context is None else _host(neg_context)
        nmk = None if neg_mask is None else _host(neg_mask, np.int32)
        F, H, W = fhw
        self._check(self.lib.ltx_denoise_begin_from_latent(self.handle, _ptr(lt), _ptr(nz), float(noise_scale), _ptr(f0), F, H, W,
                                                           _ptr(ctx), cc, _ptr(mk), _ptr(nctx), _ptr(nmk), S))
        self._session_shape = (self.config.in_channels, F, H, W)

    def denoise_upscale_stage(self, noise, noise_scale: float, adain_factor: float = 1.0):
        """Device-resident stage switch of generateVideoTwoStage (:2594-2647): upscale 2x, AdaIN against stage 1, re-noise."""
        Cc, F, H, W = self._session_shape
        nz = _host(noise, np.float32)
        assert nz.size == Cc * F * 4 * H * W, "noise must have the stage-2 shape [C, F, 2H, 2W]"
        self._check(self.lib.ltx_denoise_upscale_stage(self.handle, _ptr(nz), float(noise_scale), float(adain_factor)))
        self._session_shape = (Cc, F, 2 * H, 2 * W)

    def denoise_set_frame0(self, frame0_latent):
        f0 = _host(frame0_latent, np.float32)
        Cc, F, H, W = self._session_shape
        assert f0.size == Cc * H * W
        self._check(self.lib.ltx_denoise_set_frame0(self.handle, _ptr(f0)))

    def denoise_step(self, sigma: float, sigma_next: float, step_index: int, cfg_scale: float = 1.0, rescale_phi: float = 0.0,
                     stg_scale: float = 0.0, stg_blocks: Sequence[int] = (), ge_gamma: float = 0.0,
                     share_stg_prefix: bool = True, i2v_frame0_conditioned: bool = False, batched_cfg: bool = True):
        p = LtxStepParams()
        p.i2v_frame0_conditioned = int(i2v_frame0_conditioned)
        p.disable_stg_prefix_sharing = 0 if share_stg_prefix else 1
        p.disable_batched_cfg = 0 if batched_cfg else 1
        p.sigma, p.sigma_next, p.cfg_scale, p.rescale_phi = sigma, sigma_next, cfg_scale, rescale_phi
        p.stg_scale, p.ge_gamma, p.step_index = stg_scale, ge_gamma, step_index
        p.n_stg_blocks = len(stg_blocks)
        for i, b in enumerate(stg_blocks):
            p.stg_blocks[i] = int(b)
        self._check(self.lib.ltx_denoise_step(self.handle, C.byref(p)))

    # ------------------------------------------------------------------ resident audio + video denoise session
    def av_denoise_begin(self, video_noise, audio_noise, fhw, sigma0: float, video_context, audio_context, mask=None,
                         neg_video_context=None, neg_audio_context=None, neg_mask=None):
        """video_noise [C,F,H,W], audio_noise [Ta,Ca] fp32 (generateVideoWithAudio, Pipeline/LTXPipeline.swift:1255-1259)."""
        vn, an = _host(video_noise, np.float32), _host(audio_noise, np.float32)
        cc = _dtype_code(video_context)
        assert _dtype_code(audio_context) == cc, "both contexts must have the same dtype"
        vx, ax = _host(video_context), _host(audio_context)
        S = vx.shape[-2]
        mk = None if mask is None else _host(mask, np.int32)
        nvx = None if neg_video_context is None else _host(neg_video_context)
        nax = None if neg_audio_context is None else _host(neg_audio_context)
        nmk = None if neg_mask is None else _host(neg_mask, np.int32)
        F, H, W = fhw
        Ta = an.shape[-2]
        self._check(self.lib.ltx_av_denoise_begin(self.handle, _ptr(vn), _ptr(an), F, H, W, Ta, sigma0, _ptr(vx), _ptr(ax), cc,
                                                  _ptr(mk), _ptr(nvx), _ptr(nax), _ptr(nmk), S))
        self._session_shape = (self.config.in_channels, F, H, W)
        self._av_session_audio_shape = (Ta, self.config.audio_in_channels)

    def av_denoise_step(self, sigma: float, sigma_next: float, step_index: int = 0, cfg_scale: float = 1.0,
                        rescale_phi: float = 0.0, i2v_frame0_conditioned: bool = False, batched_cfg: bool = True):
        """batched_cfg: with CFG on one GPU, run the conditional and unconditional passes as one B = 2 forward (same values)."""
        p = LtxStepParams()
        p.i2v_frame0_conditioned = int(i2v_frame0_conditioned)
        p.disable_batched_cfg = 0 if batched_cfg else 1
        p.sigma, p.sigma_next, p.cfg_scale, p.rescale_phi, p.step_index = sigma, sigma_next, cfg_scale, rescale_phi, step_index
        self._check(self.lib.ltx_av_denoise_step(self.handle, C.byref(p)))

    def av_denoise_get_latents(self):
        ov = np.empty(self._session_shape, dtype=np.float32)
        oa = np.empty(self._av_session_audio_shape, dtype=np.float32)
        self._check(self.lib.ltx_av_denoise_get_latents(self.handle, _ptr(ov), _ptr(oa)))
        return ov, oa

    def denoise_get_latent(self) -> np.ndarray:
        out = np.empty(self._session_shape, dtype=np.float32)
        self._check(self.lib.ltx_denoise_get_latent(self.handle, _ptr(out)))
        return out

    def denoise_latent_dev(self) -> int:
        p = C.c_void_p()
        self._check(self.lib.ltx_denoise_latent_dev(self.handle, C.byref(p)))
        return p.value

    # ------------------------------------------------------------------ VAE
    def pinned_empty(self, shape, dtype=np.float32) -> np.ndarray:
        """ndarray over page-locked host memory (ltx_host_alloc), for buffers handed to the host-pointer entry points; the
        memory is released when the array (and every view of it) is garbage-collected."""
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        rc = self.lib.ltx_host_alloc(C.byref(p), max(n, 1))
        if rc != 0:
            raise LtxError(rc, "ltx_host_alloc failed")
        lib = self.lib

        class _Owner:
            def __init__(self, addr):
                self.addr = addr

            def __del__(self):
                lib.ltx_host_free(C.c_void_p(self.addr))
        buf = (C.c_char * max(n, 1)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
        self._pinned = getattr(self, "_pinned", [])
        owner = _Owner(p.value)
        # keep the owner alive as long as the base buffer object is: numpy holds `buf`, `buf` holds the owner
        buf._owner = owner
        return arr

    def vae_decode(self, latent, timestep: Optional[float] = None, decode_noise=None, causal: bool = False,
                   out: Optional[np.ndarray] = None) -> np.ndarray:
        lat = _host(latent, np.float32)
        if lat.ndim == 5:
            lat = lat[0]
        Cc, Fp, Hp, Wp = lat.shape
        lat = np.ascontiguousarray(lat)
        nz = None if decode_noise is None else _host(decode_noise, np.float32)
        shape = (8 * (Fp - 1) + 1, 32 * Hp, 32 * Wp, 3)
        if out is None:
            out = np.empty(shape, dtype=np.float32)
        assert out.shape == shape and out.dtype == np.float32 and out.flags["C_CONTIGUOUS"]
        self._check(self.lib.ltx_vae_decode(self.handle, _ptr(lat), Fp, Hp, Wp, -1.0 if timestep is None else float(timestep),
                                            _ptr(nz), int(causal), _ptr(out)))
        return out

    def vae_decode_tiled(self, latent, tile_size: int, tile_overlap: int = 1, timestep: Optional[float] = None,
                         decode_noise=None, causal: bool = False) -> np.ndarray:
        """decodeVideo's temporally tiled branch (decodeWithTemporalTiling, Models/VAE/VideoDecoder.swift:517-602)."""
        lat = _host(latent, np.float32)
        if lat.ndim == 5:
            lat = lat[0]
        Cc, Fp, Hp, Wp = lat.shape
        lat = np.ascontiguousarray(lat)
        nz = None if decode_noise is None else np.ascontiguousarray(_host(decode_noise, np.float32).reshape(lat.shape))
        nf = self.lib.ltx_vae_tiled_frames(Fp, int(tile_size), int(tile_overlap))
        if nf <= 0:
            raise LtxError(2, "temporal tile overlap must be in [0, tile size)")
        out = np.empty((nf, 32 * Hp, 32 * Wp, 3), dtype=np.float32)
        got = C.c_int(0)
        self._check(self.lib.ltx_vae_decode_tiled(self.handle, _ptr(lat), Fp, Hp, Wp, -1.0 if timestep is None else float(timestep),
                                                  _ptr(nz), int(causal), int(tile_size), int(tile_overlap), _ptr(out),
                                                  C.byref(got)))
        assert got.value == nf
        return out

    def vae_decode_dev(self, latent_ptr: int, fhw, out_ptr: int, causal: bool = False):
        Fp, Hp, Wp = fhw
        self._check(self.lib.ltx_vae_decode_dev(self.handle, latent_ptr, Fp, Hp, Wp, -1.0, None, int(causal), out_ptr))

    # ------------------------------------------------------------------ 8-bit frames (decodeVideo -> tensorToImages)
    @staticmethod
    def frames_u8_shape(F: int, H: int, W: int, format) -> Tuple[int, ...]:
        """Array shape of 8-bit frames: RGB8 (F, H, W, 3); I420 (F, 3H/2, W) -- each frame's Y, U and V planes one after
        another, the usual two-dimensional view of I420."""
        return (F, H, W, 3) if _frames_format(format) == LTX_FRAMES_RGB8 else (F, H * 3 // 2, W)

    def vae_decode_u8(self, latent, format="rgb8", timestep: Optional[float] = None, decode_noise=None, causal: bool = False,
                      out: Optional[np.ndarray] = None) -> np.ndarray:
        """vae_decode straight to 8-bit frames, written by conv_out's epilogue; format "rgb8" or "i420" (ltxcuda.h)."""
        fmt = _frames_format(format)
        lat = _host(latent, np.float32)
        if lat.ndim == 5:
            lat = lat[0]
        Cc, Fp, Hp, Wp = lat.shape
        lat = np.ascontiguousarray(lat)
        nz = None if decode_noise is None else _host(decode_noise, np.float32)
        shape = self.frames_u8_shape(8 * (Fp - 1) + 1, 32 * Hp, 32 * Wp, fmt)
        if out is None:
            out = np.empty(shape, dtype=np.uint8)
        assert out.shape == shape and out.dtype == np.uint8 and out.flags["C_CONTIGUOUS"]
        self._check(self.lib.ltx_vae_decode_u8(self.handle, _ptr(lat), Fp, Hp, Wp, -1.0 if timestep is None else float(timestep),
                                               _ptr(nz), int(causal), fmt, _ptr(out)))
        return out

    def vae_decode_tiled_u8(self, latent, tile_size: int, tile_overlap: int = 1, format="rgb8",
                            timestep: Optional[float] = None, decode_noise=None, causal: bool = False) -> np.ndarray:
        """vae_decode_tiled, then the 8-bit conversion of the blended and clipped frames."""
        fmt = _frames_format(format)
        lat = _host(latent, np.float32)
        if lat.ndim == 5:
            lat = lat[0]
        Cc, Fp, Hp, Wp = lat.shape
        lat = np.ascontiguousarray(lat)
        nz = None if decode_noise is None else np.ascontiguousarray(_host(decode_noise, np.float32).reshape(lat.shape))
        nf = self.lib.ltx_vae_tiled_frames(Fp, int(tile_size), int(tile_overlap))
        if nf <= 0:
            raise LtxError(2, "temporal tile overlap must be in [0, tile size)")
        out = np.empty(self.frames_u8_shape(nf, 32 * Hp, 32 * Wp, fmt), dtype=np.uint8)
        got = C.c_int(0)
        self._check(self.lib.ltx_vae_decode_tiled_u8(self.handle, _ptr(lat), Fp, Hp, Wp,
                                                     -1.0 if timestep is None else float(timestep), _ptr(nz), int(causal),
                                                     int(tile_size), int(tile_overlap), fmt, _ptr(out), C.byref(got)))
        assert got.value == nf
        return out

    def vae_decode_u8_dev(self, latent_ptr: int, fhw, out_ptr: int, format="rgb8", causal: bool = False,
                          timestep: Optional[float] = None, noise_ptr: Optional[int] = None):
        """Device pointers; out_ptr holds ltx_frames_u8_bytes(8(F'-1)+1, 32H', 32W', format) bytes, 4-byte aligned."""
        Fp, Hp, Wp = fhw
        self._check(self.lib.ltx_vae_decode_u8_dev(self.handle, latent_ptr, Fp, Hp, Wp, -1.0 if timestep is None else float(timestep),
                                                   noise_ptr, int(causal), _frames_format(format), out_ptr))

    def frames_to_u8(self, frames, format="rgb8") -> np.ndarray:
        """fp32 frames [F, H, W, 3] (clipped to [0, 1]) -> 8-bit frames, the arithmetic of the fused decode."""
        fmt = _frames_format(format)
        fr = _host(frames, np.float32)
        F, H, W, _ = fr.shape
        out = np.empty(self.frames_u8_shape(F, H, W, fmt), dtype=np.uint8)
        self._check(self.lib.ltx_frames_to_u8(self.handle, _ptr(fr), F, H, W, fmt, _ptr(out)))
        return out

    def frames_to_u8_dev(self, frames_ptr: int, fhw, out_ptr: int, format="rgb8"):
        F, H, W = fhw
        self._check(self.lib.ltx_frames_to_u8_dev(self.handle, frames_ptr, F, H, W, _frames_format(format), out_ptr))

    # ------------------------------------------------------------------ VAE encoder / latent upscaler / AdaIN
    def vae_encode(self, pixels, normalize: bool = True) -> np.ndarray:
        """pixels [3,T,H,W] (or [1,3,T,H,W]) fp32 -> latent [128, ceil(T/8), H/32, W/32] (VideoEncoder + encodeImage stats)."""
        px = _host(pixels, np.float32)
        if px.ndim == 5:
            px = np.ascontiguousarray(px[0])
        _, T, H, W = px.shape
        out = np.empty((self.config.vae_latent_channels, (T + 7) // 8, H // 32, W // 32), dtype=np.float32)
        self._check(self.lib.ltx_vae_encode(self.handle, _ptr(px), T, H, W, int(normalize), _ptr(out)))
        return out

    def vae_encode_dev(self, pixels_ptr: int, thw, out_ptr: int, normalize: bool = True):
        T, H, W = thw
        self._check(self.lib.ltx_vae_encode_dev(self.handle, pixels_ptr, T, H, W, int(normalize), out_ptr))

    def upscale_latent(self, latent) -> np.ndarray:
        """upsampleLatents: [128,F,H,W] (normalised) -> [128,F,2H,2W]."""
        lat = _host(latent, np.float32)
        if lat.ndim == 5:
            lat = np.ascontiguousarray(lat[0])
        Cc, F, H, W = lat.shape
        out = np.empty((Cc, F, 2 * H, 2 * W), dtype=np.float32)
        self._check(self.lib.ltx_upscale_latent(self.handle, _ptr(lat), F, H, W, _ptr(out)))
        return out

    def upscale_latent_dev(self, latent_ptr: int, fhw, out_ptr: int):
        F, H, W = fhw
        self._check(self.lib.ltx_upscale_latent_dev(self.handle, latent_ptr, F, H, W, out_ptr))

    def adain_filter(self, latent, reference, factor: float = 1.0) -> np.ndarray:
        """adainFilterLatent: latent [C,...] takes the per-channel mean/std of reference [C,...]; returns a new array."""
        lat = np.array(_host(latent, np.float32), copy=True)
        ref = _host(reference, np.float32)
        Cc = lat.shape[0]
        self._check(self.lib.ltx_adain_filter(self.handle, _ptr(lat), lat.size // Cc, _ptr(ref), ref.size // Cc, Cc, float(factor)))
        return lat
