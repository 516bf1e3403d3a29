"""ctypes binding of libltxcuda.so (include/ltxcuda.h).  There is no fallback: if the shared library is missing or
cannot be loaded, importing the product path raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libltxcuda.so")

LTX_F32, LTX_BF16, LTX_F16 = 0, 1, 2
LTX_MAX_FLAG_BLOCKS = 64
LTX_FRAMES_RGB8, LTX_FRAMES_I420 = 1, 2     # ltx_frames_format


class LtxConfig(C.Structure):
    _fields_ = [
        ("num_layers", C.c_int32), ("num_heads", C.c_int32), ("head_dim", C.c_int32), ("in_channels", C.c_int32),
        ("out_channels", C.c_int32), ("caption_channels", C.c_int32), ("ffn_mult", C.c_int32), ("rope_theta", C.c_float),
        ("max_pos", C.c_int32 * 3), ("timestep_scale_multiplier", C.c_float), ("norm_eps", C.c_float),
        ("vae_latent_channels", C.c_int32), ("vae_base_channels", C.c_int32), ("vae_blocks_per_stage", C.c_int32),
        ("vae_patch_size", C.c_int32), ("vae_encoder_base_channels", C.c_int32), ("upscaler_mid_channels", C.c_int32),
        ("upscaler_blocks", C.c_int32), ("audio_num_heads", C.c_int32), ("audio_head_dim", C.c_int32),
        ("audio_in_channels", C.c_int32), ("audio_max_pos", C.c_int32),
    ]


class LtxDitFlags(C.Structure):
    _fields_ = [
        ("n_stg_blocks", C.c_int32), ("stg_blocks", C.c_int32 * LTX_MAX_FLAG_BLOCKS), ("skip_self_attn", C.c_int32),
        ("skip_ff", C.c_int32), ("n_cas_blocks", C.c_int32), ("cas_blocks", C.c_int32 * LTX_MAX_FLAG_BLOCKS),
        ("cross_attn_scale", C.c_float), ("context_key", C.c_uint64),
    ]


class LtxStepParams(C.Structure):
    _fields_ = [
        ("sigma", C.c_float), ("sigma_next", C.c_float), ("cfg_scale", C.c_float), ("rescale_phi", C.c_float),
        ("stg_scale", C.c_float), ("ge_gamma", C.c_float), ("n_stg_blocks", C.c_int32),
        ("stg_blocks", C.c_int32 * LTX_MAX_FLAG_BLOCKS), ("step_index", C.c_int32),
        ("i2v_frame0_conditioned", C.c_int32), ("disable_stg_prefix_sharing", C.c_int32), ("disable_batched_cfg", C.c_int32),
    ]


# name -> (restype, argtypes); must list every symbol declared in include/ltxcuda.h (tests/test_abi.py checks it)
_P, _I, _F, _U64, _SZ, _I64 = C.c_void_p, C.c_int, C.c_float, C.c_uint64, C.c_size_t, C.c_int64
SIGNATURES = {
    "ltx_config_default": (None, [C.POINTER(LtxConfig)]),
    "ltx_version": (C.c_char_p, []),
    "ltx_ctx_create": (_I, [C.POINTER(LtxConfig), _I, C.POINTER(_P)]),
    "ltx_ctx_destroy": (_I, [_P]),
    "ltx_last_error": (C.c_char_p, [_P]),
    "ltx_sync": (_I, [_P]),
    "ltx_load_tensor": (_I, [_P, C.c_char_p, _P, _I, C.POINTER(_I64), _I]),
    "ltx_load_tensor_e4m3": (_I, [_P, C.c_char_p, _P, _P, _I64, C.POINTER(_I64), _I]),
    "ltx_load_safetensors": (_I, [_P, C.c_char_p, _I, C.POINTER(_I)]),
    "ltx_map_weight_key": (_I, [_I, C.c_char_p, C.c_char_p, _SZ]),
    "ltx_fuse_lora": (_I, [_P, C.c_char_p, _P, _P, _I, _I, _F]),
    "ltx_set_precision": (_I, [_P, _I]),
    "ltx_set_quant_storage": (_I, [_P, _I]),
    "ltx_init_random_weights": (_I, [_P, _I, _U64]),
    "ltx_finalize_weights": (_I, [_P, _I, _I]),
    "ltx_dit_forward": (_I, [_P, _P, _I, _P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _I, C.POINTER(LtxDitFlags), _P]),
    "ltx_dit_forward_dev": (_I, [_P, _P, _I, _P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _I, C.POINTER(LtxDitFlags), _P]),
    "ltx_av_forward": (_I, [_P, _P, _I, _P, _I, _P, _P, _I, _F, _F, _P, _P, _I, _I, _I, _I, _I, _I, _U64, _P, _P]),
    "ltx_av_forward_dev": (_I, [_P, _P, _I, _P, _I, _P, _P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _U64, _P, _P]),
    "ltx_av_forward_tokens": (_I, [_P, _P, _I, _P, _I, _P, _P, _I, _P, _F, _P, _P, _I, _I, _I, _I, _I, _I, _U64, _P, _P]),
    "ltx_av_forward_tokens_dev": (_I, [_P, _P, _I, _P, _I, _P, _P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _U64, _P, _P]),
    "ltx_av_forward_batch": (_I, [_P, _P, _I, _P, _I, _P, _P, _I, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _U64, _P, _P]),
    "ltx_av_forward_batch_dev": (_I, [_P, _P, _I, _P, _I, _P, _P, _I, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _U64, _P, _P]),
    "ltx_dit_clear_caches": (_I, [_P]),
    "ltx_guided_euler_step": (_I, [_P, _P, _P, _P, _P, _P, _I, _SZ, _F, _F, _F, _F, _F, _F]),
    "ltx_guided_euler_step_dev": (_I, [_P, _P, _P, _P, _P, _P, _I, _SZ, _F, _F, _F, _F, _F, _F]),
    "ltx_denoise_begin": (_I, [_P, _P, _I, _I, _I, _F, _P, _I, _P, _P, _P, _I]),
    "ltx_denoise_step": (_I, [_P, C.POINTER(LtxStepParams)]),
    "ltx_denoise_get_latent": (_I, [_P, _P]),
    "ltx_denoise_latent_dev": (_I, [_P, C.POINTER(_P)]),
    "ltx_av_denoise_begin": (_I, [_P, _P, _P, _I, _I, _I, _I, _F, _P, _P, _I, _P, _P, _P, _P, _I]),
    "ltx_av_denoise_step": (_I, [_P, C.POINTER(LtxStepParams)]),
    "ltx_av_denoise_get_latents": (_I, [_P, _P, _P]),
    "ltx_vae_decode": (_I, [_P, _P, _I, _I, _I, _F, _P, _I, _P]),
    "ltx_vae_decode_dev": (_I, [_P, _P, _I, _I, _I, _F, _P, _I, _P]),
    "ltx_vae_tiled_frames": (_I, [_I, _I, _I]),
    "ltx_vae_decode_tiled": (_I, [_P, _P, _I, _I, _I, _F, _P, _I, _I, _I, _P, _P]),
    "ltx_vae_decode_tiled_dev": (_I, [_P, _P, _I, _I, _I, _F, _P, _I, _I, _I, _P, _P]),
    "ltx_frames_u8_bytes": (_SZ, [_I, _I, _I, _I]),
    "ltx_vae_decode_u8": (_I, [_P, _P, _I, _I, _I, _F, _P, _I, _I, _P]),
    "ltx_vae_decode_u8_dev": (_I, [_P, _P, _I, _I, _I, _F, _P, _I, _I, _P]),
    "ltx_vae_decode_tiled_u8": (_I, [_P, _P, _I, _I, _I, _F, _P, _I, _I, _I, _I, _P, _P]),
    "ltx_vae_decode_tiled_u8_dev": (_I, [_P, _P, _I, _I, _I, _F, _P, _I, _I, _I, _I, _P, _P]),
    "ltx_frames_to_u8": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "ltx_frames_to_u8_dev": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "ltx_vae_encode": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "ltx_vae_encode_dev": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "ltx_upscale_latent": (_I, [_P, _P, _I, _I, _I, _P]),
    "ltx_upscale_latent_dev": (_I, [_P, _P, _I, _I, _I, _P]),
    "ltx_adain_filter": (_I, [_P, _P, _SZ, _P, _SZ, _I, _F]),
    "ltx_adain_filter_dev": (_I, [_P, _P, _SZ, _P, _SZ, _I, _F]),
    "ltx_denoise_begin_from_latent": (_I, [_P, _P, _P, _F, _P, _I, _I, _I, _P, _I, _P, _P, _P, _I]),
    "ltx_denoise_upscale_stage": (_I, [_P, _P, _F, _F]),
    "ltx_denoise_set_frame0": (_I, [_P, _P]),
    "ltx_dist_get_unique_id": (_I, [_P]),
    "ltx_dist_init": (_I, [_P, _P, _I, _I, _I, _I]),
    "ltx_dist_init_local": (_I, [_P, _I, _I, _I]),
    "ltx_dist_shutdown": (_I, [_P]),
    "ltx_dist_p2p_active": (_I, [_P]),
    "ltx_dist_info": (_I, [_P, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "ltx_host_alloc": (_I, [C.POINTER(_P), _SZ]),
    "ltx_host_free": (_I, [_P]),
    "ltx_launch_count": (_U64, [_P]),
    "ltx_get_stream": (_I, [_P, C.POINTER(_P)]),
    "ltx_set_profiling": (_I, [_P, _I]),
    "ltx_set_graphs": (_I, [_P, _I]),
    "ltx_graph_stats": (_I, [_P, _P, _P]),
    "ltx_get_profile": (_I, [_P, _P, _P, _P, _P, _I]),
    "ltx_op_gemm": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I]),
    "ltx_op_gemm_blocked": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, C.c_int64, _I]),
    "ltx_op_gemm_resid": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _F]),
    "ltx_op_gemm_skinny": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, C.c_int64]),
    "ltx_op_quantize": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "ltx_op_dequantize": (_I, [_P, _P, _P, _P, _I, _I, _I, _P]),
    "ltx_op_gemm_q": (_I, [_P, _P, _P, _P, _P, _I, _P, _P, _I, _I, _I, _I, _I]),
    "ltx_op_quantize_fp8": (_I, [_P, _P, _I, _I, _I64, _P, _P]),
    "ltx_op_gemm_fp8": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I]),
    "ltx_op_gemm_fp8_ex": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I64, _P, _P, _P, _P, _I, _I, _I, _I]),
    "ltx_op_attention": (_I, [_P, _P, _P, _P, _I64, _P, _P, _I, _I, _I, _I, _F]),
    "ltx_op_attention_hd": (_I, [_P, _P, _P, _P, _I64, _P, _P, _I, _I, _I, _I, _I, _F]),
    "ltx_op_attention_blocks": (_I, [_P, _P, _P, _P, _I64, _I, _I, _I, _F, C.POINTER(_P), _I, _I]),
    "ltx_op_rmsnorm_mod": (_I, [_P, _P, _P, _I, _I, _P, _P, _P, _P, _F, _I]),
    "ltx_op_qknorm_rope": (_I, [_P, _P, _I, _I, _P, _P, _P, _I, _F]),
    "ltx_op_conv3d": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I]),
    "ltx_conv3d_plan": (_I, [_I, _I, _I, _I, _I, _I, _I, _I, C.POINTER(C.c_int32)]),
    "ltx_op_vae_prep": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _I]),
    "ltx_op_vae_halo_fill": (_I, [_P, _P, _I, _I, _I, _I, _I]),
    "ltx_op_conv3d_epi": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _I, _I, _P, _P, _P, _I]),
}

_lib = None


def load() -> C.CDLL:
    """Loads libltxcuda.so (built in-tree by csrc/build.sh / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `bash ltx-video-swift-mlx_b200/csrc/build.sh` "
            "(there is no CPU / PyTorch fallback for the product path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class LtxError(RuntimeError):
    """Mirrors LTXError (LTXVideo.swift:66-107): code 1 invalidConfiguration, 2/3 generationFailed, 4 weightLoadingFailed."""

    def __init__(self, code: int, message: str):
        super().__init__(f"[ltxcuda error {code}] {message}")
        self.code = code
