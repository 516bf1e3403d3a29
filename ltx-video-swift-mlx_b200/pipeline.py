"""The generateVideo step loop (Pipeline/LTXPipeline.swift:793-956) over libltxcuda, in two forms:

* `denoise_host_seam`  -- call-for-call what the Swift pipeline does at the three seams of SURVEY 8b: host latent ->
  LTXTransformer(...) 1-3x per step -> guided Euler, all through host buffers (H2D/D2H every call).  This is the `e2e`
  path of bench.py.
* `denoise_resident`   -- the device-resident fast path (ltx_denoise_begin / ltx_denoise_step): latent, text caches and
  GE state stay in HBM; one D2H at the end."""
from __future__ import annotations

from typing import List, Optional, Sequence

import numpy as np

from .context import LtxContext
from .latent_utils import VideoLatentShape, patchify, unpatchify
from .transformer import LTXTransformer


def denoise_host_seam(ctx: LtxContext, noise: np.ndarray, context, mask, sigmas: Sequence[float], neg_context=None,
                      neg_mask=None, cfg_scale: float = 1.0, guidance_rescale: float = 0.0, stg_scale: float = 0.0,
                      stg_blocks: Sequence[int] = (29,), ge_gamma: float = 0.0, cache_text: bool = True) -> np.ndarray:
    """noise [1,C,F,H,W] fp32 host.  Returns the final latent [1,C,F,H,W]."""
    _, C, F, H, W = noise.shape
    shape = VideoLatentShape(1, C, F, H, W)
    tr = LTXTransformer(ctx)
    latent = np.ascontiguousarray(noise.astype(np.float32) * np.float32(sigmas[0]))      # :793
    v_prev = np.zeros_like(latent)
    use_cfg = cfg_scale > 1.0 and neg_context is not None
    # one fresh cache key per prompt per generation: the projected text is step-invariant inside this loop only
    key_pos = ctx.new_context_key() if cache_text else 0
    key_neg = ctx.new_context_key() if cache_text else 0
    for step in range(len(sigmas) - 1):
        sg, sn = float(sigmas[step]), float(sigmas[step + 1])
        tok = patchify(latent)                                                            # :815 (cast to bf16 on device)
        ts = np.array([sg], dtype=np.float32)
        vc = unpatchify(tr(tok, context, ts, mask, shape.fhw, context_key=key_pos), shape)
        vu = vs = None
        if use_cfg:                                                                       # :829-848
            vu = unpatchify(tr(tok, neg_context, ts, neg_mask, shape.fhw, context_key=key_neg), shape)
        if stg_scale > 0:                                                                 # :897-921
            tr.set_stg_skip_flags(True, False, stg_blocks)
            vs = unpatchify(tr(tok, context, ts, mask, shape.fhw, context_key=key_pos), shape)
            tr.clear_stg_skip_flags()
        ctx.guided_euler_step(latent, vc, vu, vs, v_prev, use_prev=step > 0, cfg_scale=cfg_scale,
                              rescale_phi=guidance_rescale, stg_scale=stg_scale, ge_gamma=ge_gamma, sigma=sg, sigma_next=sn)
    return latent


def denoise_resident(ctx: LtxContext, noise: np.ndarray, context, mask, sigmas: Sequence[float], neg_context=None,
                     neg_mask=None, cfg_scale: float = 1.0, guidance_rescale: float = 0.0, stg_scale: float = 0.0,
                     stg_blocks: Sequence[int] = (29,), ge_gamma: float = 0.0, fetch: bool = True) -> Optional[np.ndarray]:
    _, C, F, H, W = noise.shape
    ctx.denoise_begin(noise[0], (F, H, W), float(sigmas[0]), context, mask, neg_context, neg_mask)
    for step in range(len(sigmas) - 1):
        ctx.denoise_step(float(sigmas[step]), float(sigmas[step + 1]), step, cfg_scale, guidance_rescale, stg_scale,
                         tuple(stg_blocks) if stg_scale > 0 else (), ge_gamma)
    return ctx.denoise_get_latent()[None] if fetch else None


def generate_two_stage_resident(ctx: LtxContext, noise1: np.ndarray, noise2: np.ndarray, context, mask, sigmas1: Sequence[float],
                                sigmas2: Sequence[float], adain_factor: float = 1.0, image_latent_half=None,
                                image_latent_full=None) -> np.ndarray:
    """generateVideoTwoStage (Pipeline/LTXPipeline.swift:2420-2720), denoising + latent glue only, device-resident:
    stage 1 at half resolution (distilled schedule) -> upscale 2x + AdaIN + re-noise with sigmas2[0] (:2594-2647) ->
    stage 2 refinement.  noise1 [1,C,F,H,W], noise2 [1,C,F,2H,2W].  The optional image latents condition frame 0 (I2V)."""
    _, C, F, H, W = noise1.shape
    i2v = image_latent_half is not None
    ctx.denoise_begin(noise1[0], (F, H, W), float(sigmas1[0]), context, mask)
    if i2v:
        ctx.denoise_set_frame0(image_latent_half)
    for i in range(len(sigmas1) - 1):
        ctx.denoise_step(float(sigmas1[i]), float(sigmas1[i + 1]), i, i2v_frame0_conditioned=i2v)
    ctx.denoise_upscale_stage(noise2[0], float(sigmas2[0]), adain_factor)
    if i2v:
        ctx.denoise_set_frame0(image_latent_full)
    for i in range(len(sigmas2) - 1):
        ctx.denoise_step(float(sigmas2[i]), float(sigmas2[i + 1]), i, i2v_frame0_conditioned=i2v)
    return ctx.denoise_get_latent()[None]


def denoise_av_host_seam(ctx: LtxContext, video_noise: np.ndarray, audio_noise: np.ndarray, video_context, audio_context, mask,
                         sigmas: Sequence[float], neg_video_context=None, neg_audio_context=None, neg_mask=None,
                         cfg_scale: float = 1.0, guidance_rescale: float = 0.0, cache_text: bool = True,
                         image_latent: Optional[np.ndarray] = None, inject_noise: Optional[Sequence[np.ndarray]] = None,
                         image_cond_noise_scale: float = 0.0):
    """The audio + video denoise loop of generateVideoWithAudio (Pipeline/LTXPipeline.swift:1277-1404) at the Swift seams: one
    LTX2Transformer call per step (two with CFG), CFG / rescale / scheduler.step on the video latent through
    ltx_guided_euler_step, CFG + plain Euler on the packed audio latent.  video_noise [1,C,F,H,W], audio_noise [1,Ta,Ca] fp32.
    image_latent [1,C,1,H,W] selects the image-to-video branch (:1262-1298, 1381-1391): frame 0 holds the image latent
    (optionally re-noised per step with the caller's draws, inject_noise[step] * scale * sigma^2), the video timesteps are per
    token (0 on frame 0), and the Euler update leaves frame 0 untouched.  Returns (video latent, audio latent)."""
    _, C, F, H, W = video_noise.shape
    shape = VideoLatentShape(1, C, F, H, W)
    v_lat = np.ascontiguousarray(video_noise.astype(np.float32) * np.float32(sigmas[0]))       # :1255-1259
    a_lat = np.ascontiguousarray(audio_noise.astype(np.float32) * np.float32(sigmas[0]))
    cond_mask = None
    if image_latent is not None:
        v_lat[:, :, 0:1] = np.asarray(image_latent, dtype=np.float32)
        cond_mask = np.zeros((1, F * H * W), dtype=np.float32)
        cond_mask[:, :H * W] = 1.0
    use_cfg = cfg_scale > 1.0 and neg_video_context is not None
    key_pos = ctx.new_context_key() if cache_text else 0
    key_neg = ctx.new_context_key() if cache_text else 0
    for step in range(len(sigmas) - 1):
        sg, sn = float(sigmas[step]), float(sigmas[step + 1])
        if image_latent is not None and image_cond_noise_scale > 0 and sg > 0 and inject_noise is not None:
            v_lat[:, :, 0:1] = (np.asarray(image_latent, dtype=np.float32) + np.float32(image_cond_noise_scale)
                                * np.asarray(inject_noise[step], dtype=np.float32) * np.float32(sg * sg))
        tok = patchify(v_lat)
        vsg = sg if cond_mask is None else np.float32(sg) * (1.0 - cond_mask)                  # :1294-1298
        pv, pa = ctx.av_forward(tok, a_lat, video_context, audio_context, vsg, sg, shape.fhw, mask, mask,
                                context_key=key_pos)
        vc, vu = unpatchify(pv, shape), None
        va = pa
        if use_cfg:                                                                            # :1310-1362
            nv, na = ctx.av_forward(tok, a_lat, neg_video_context, neg_audio_context, vsg, sg, shape.fhw, neg_mask, neg_mask,
                                    context_key=key_neg)
            vu = unpatchify(nv, shape)
            va = pa + np.float32(cfg_scale - 1.0) * (pa - na)                                  # applyCFG on the audio velocity
        frame0 = v_lat[:, :, 0:1].copy() if image_latent is not None else None
        ctx.guided_euler_step(v_lat, vc, vu, None, None, cfg_scale=cfg_scale if use_cfg else 1.0,
                              rescale_phi=guidance_rescale if use_cfg else 0.0, sigma=sg, sigma_next=sn)
        if frame0 is not None:                    # :1381-1391: the element-wise Euler update is discarded on frame 0
            v_lat[:, :, 0:1] = frame0
        a_lat = a_lat + np.float32(sn - sg) * va                                               # :1402
    return v_lat, a_lat


def denoise_av_resident(ctx: LtxContext, video_noise: np.ndarray, audio_noise: np.ndarray, video_context, audio_context, mask,
                        sigmas: Sequence[float], neg_video_context=None, neg_audio_context=None, neg_mask=None,
                        cfg_scale: float = 1.0, guidance_rescale: float = 0.0, image_latent: Optional[np.ndarray] = None,
                        inject_noise: Optional[Sequence[np.ndarray]] = None, image_cond_noise_scale: float = 0.0,
                        batched_cfg: bool = True):
    """The same loop on the device-resident session (ltx_av_denoise_begin / _step): latents, text caches and velocities stay
    in HBM, the only per-step host traffic is the optional re-noised conditioning frame.  batched_cfg: run the two guidance
    passes as one B = 2 forward (same values).  Returns (video latent [1,C,F,H,W], audio latent [1,Ta,Ca])."""
    _, C, F, H, W = video_noise.shape
    ctx.av_denoise_begin(video_noise[0], audio_noise[0], (F, H, W), float(sigmas[0]), video_context, audio_context, mask,
                         neg_video_context, neg_audio_context, neg_mask)
    i2v = image_latent is not None
    if i2v:
        ctx.denoise_set_frame0(np.asarray(image_latent, dtype=np.float32))
    for step in range(len(sigmas) - 1):
        sg, sn = float(sigmas[step]), float(sigmas[step + 1])
        if i2v and image_cond_noise_scale > 0 and sg > 0 and inject_noise is not None:
            ctx.denoise_set_frame0(np.asarray(image_latent, dtype=np.float32) + np.float32(image_cond_noise_scale)
                                   * np.asarray(inject_noise[step], dtype=np.float32) * np.float32(sg * sg))
        ctx.av_denoise_step(sg, sn, step, cfg_scale, guidance_rescale, i2v_frame0_conditioned=i2v, batched_cfg=batched_cfg)
    v, a = ctx.av_denoise_get_latents()
    return v[None], a[None]
