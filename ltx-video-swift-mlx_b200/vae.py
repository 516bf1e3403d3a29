"""decodeVideo -- host mirror of Models/VAE/VideoDecoder.swift:466-508 over libltxcuda."""
from __future__ import annotations

from typing import Optional

import numpy as np

from .context import LtxContext


class VideoDecoder:
    """Handle on the decoder weights held by an LtxContext (VideoDecoder(), causal: false by default, :320)."""

    def __init__(self, ctx: LtxContext, causal: bool = False):
        self.ctx = ctx
        self.causal = causal
        self.timestep_conditioning = False


def decode_video(latent, decoder: VideoDecoder, timestep: Optional[float] = None, temporal_tile_size: int = 0,
                 temporal_tile_overlap: int = 1, decode_noise=None) -> np.ndarray:
    """latent [1,128,F',H',W'] or [128,F',H',W'] fp32 -> frames [F,H,W,3] fp32 in [0,1].
    temporal_tile_size > 0 with more latent frames than one tile takes the reference's overlap-blend tiling (:482-494,
    517-602; off by default there: vaeTemporalTileSize 0, Configuration/MemoryOptimizationConfig.swift:78-84) -- an
    approximation kept for drop-in behaviour; on B200 the exact single pass (or the exact multi-GPU temporal sharding) fits."""
    lat = np.asarray(latent, dtype=np.float32)
    frames_lat = lat.shape[-3]
    if temporal_tile_size > 0 and frames_lat > temporal_tile_size:
        return decoder.ctx.vae_decode_tiled(lat, temporal_tile_size, temporal_tile_overlap, timestep, decode_noise, decoder.causal)
    return decoder.ctx.vae_decode(lat, timestep, decode_noise, decoder.causal)


def decode_video_u8(latent, decoder: VideoDecoder, format="rgb8", timestep: Optional[float] = None, temporal_tile_size: int = 0,
                    temporal_tile_overlap: int = 1, decode_noise=None) -> np.ndarray:
    """decode_video followed by tensorToImages (U/VideoExporter.swift:543-580) in one call: 8-bit frames, "rgb8" [F,H,W,3]
    or "i420" [F,3H/2,W] (BT.709 limited range), as include/ltxcuda.h defines them.  Only the 8-bit frames cross PCIe."""
    lat = np.asarray(latent, dtype=np.float32)
    frames_lat = lat.shape[-3]
    if temporal_tile_size > 0 and frames_lat > temporal_tile_size:
        return decoder.ctx.vae_decode_tiled_u8(lat, temporal_tile_size, temporal_tile_overlap, format, timestep, decode_noise,
                                               decoder.causal)
    return decoder.ctx.vae_decode_u8(lat, format, timestep, decode_noise, decoder.causal)


class VideoEncoder:
    """Handle on the encoder weights held by an LtxContext (VideoEncoder(causal: true), Models/VAE/VideoEncoder.swift:211)."""

    def __init__(self, ctx: LtxContext):
        self.ctx = ctx

    def __call__(self, pixels) -> np.ndarray:
        """VideoEncoder.callAsFunction (:270-312): [1,3,T,H,W] -> latent mean [1,128,T',H/32,W/32] (not normalised)."""
        return self.ctx.vae_encode(pixels, normalize=False)[None]


def encode_image(pixels, encoder: VideoEncoder) -> np.ndarray:
    """encodeImage (Pipeline/LTXPipeline.swift:1902-1932) after the image has been loaded and resized: encode and
    normalise with the decoder's per-channel statistics.  pixels [1,3,1,H,W] in [-1,1] -> [1,128,1,H/32,W/32]."""
    return encoder.ctx.vae_encode(pixels, normalize=True)[None]
