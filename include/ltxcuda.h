/* ltxcuda.h -- C ABI of libltxcuda.so: the B200 (sm_100a) implementation of the LTX-2 denoise hot path.
 *
 * The reference (VincentGourbin/ltx-video-swift-mlx) has no plugin/FFI interface: every model is a Swift Module
 * calling MLX directly.  This header is the drop-in boundary at the three narrowest Swift call sites (SURVEY 8b);
 * each entry point cites the Swift symbol it replaces (paths relative to Sources/LTXVideo/).  A SwiftPM C target
 * (`CLTXCuda`, see INTEGRATION.md) exposes it to the unchanged `LTXPipeline`.
 *
 * Conventions
 *   - plain pointers and sizes only; the caller owns every host buffer, the library owns device memory and weights;
 *   - every function returns 0 on success, non-zero on failure (LTX_ERR_*); `ltx_last_error` gives the message
 *     (maps to LTXError.generationFailed / .weightLoadingFailed / .invalidConfiguration, LTXVideo.swift:66-107);
 *   - no CPU fallback: without an sm_100a device `ltx_ctx_create` fails;
 *   - a context is thread-compatible (calls are serialised by `actor LTXPipeline`, Pipeline/LTXPipeline.swift:117);
 *   - `*_dev` variants take device pointers, enqueue on the context stream and do not synchronise.
 */
#ifndef LTXCUDA_H_
#define LTXCUDA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define LTX_OK 0
#define LTX_ERR_INVALID_CONFIGURATION 1 /* LTXError.invalidConfiguration */
#define LTX_ERR_INVALID_ARGUMENT 2      /* LTXError.generationFailed (bad shapes / pointers) */
#define LTX_ERR_CUDA 3                  /* LTXError.generationFailed (device error) */
#define LTX_ERR_WEIGHTS 4               /* LTXError.weightLoadingFailed */
#define LTX_ERR_UNSUPPORTED 5

typedef enum { LTX_F32 = 0, LTX_BF16 = 1, LTX_F16 = 2 } ltx_dtype;

typedef struct ltx_ctx ltx_ctx;

/* Mirrors LTXTransformerConfig (Configuration/LTXConfig.swift:83-156) plus the VAE channel plan
 * (Models/VAE/VideoDecoder.swift:331-355).  Zero-initialise and call ltx_config_default for the LTX-2 values. */
typedef struct {
  int32_t num_layers;        /* 48 */
  int32_t num_heads;         /* 32 */
  int32_t head_dim;          /* 128 (only value supported by the attention kernel) */
  int32_t in_channels;       /* 128 */
  int32_t out_channels;      /* 128 */
  int32_t caption_channels;  /* 3840 */
  int32_t ffn_mult;          /* 4 */
  float rope_theta;          /* 10000 */
  int32_t max_pos[3];        /* {20, 2048, 2048} */
  float timestep_scale_multiplier; /* 1000 */
  float norm_eps;            /* 1e-6 */
  int32_t vae_latent_channels;   /* 128 */
  int32_t vae_base_channels;     /* 1024 */
  int32_t vae_blocks_per_stage;  /* 5 */
  int32_t vae_patch_size;        /* 4 */
  /* used by ltx_init_random_weights only (loaded checkpoints carry their own shapes):
   * VideoEncoder channel plan base (Models/VAE/VideoEncoder.swift:229-262) and SpatialUpscaler(midChannels:numBlocksPerStage:)
   * (Models/Upscaler/SpatialUpscaler.swift:181-185) */
  int32_t vae_encoder_base_channels; /* 128 */
  int32_t upscaler_mid_channels;     /* 1024 */
  int32_t upscaler_blocks;           /* 4 */
  /* audio stream of the dual audio/video transformer (Configuration/LTXConfig.swift:134-173) */
  int32_t audio_num_heads;           /* 32 */
  int32_t audio_head_dim;            /* 64 */
  int32_t audio_in_channels;         /* 128 (= audio_out_channels) */
  int32_t audio_max_pos;             /* 20 */
} ltx_config;

void ltx_config_default(ltx_config* cfg);
const char* ltx_version(void);

/* LTXPipeline.init / loadModels (Pipeline/LTXPipeline.swift:189,217): one context per GPU. */
int ltx_ctx_create(const ltx_config* cfg, int device, ltx_ctx** out);
int ltx_ctx_destroy(ltx_ctx* ctx);
const char* ltx_last_error(const ltx_ctx* ctx);
int ltx_sync(ltx_ctx* ctx);

/* Weight ingestion: replaces LTXWeightLoader.applyTransformerWeights / applyVAEWeights
 * (Utils/ModelDownloader.swift:972-1064).  `key` is the post-mapping name (mapTransformerKey :756-803,
 * mapVAEWeights :808-899), e.g. "transformer_blocks.3.attn1.to_q.weight", "vae.up_blocks_0.res_blocks.0.conv1.conv.weight"
 * (VAE keys carry the prefix "vae.").  Matrices / conv kernels are stored as bf16 (the loader's fp32->bf16 cast,
 * :1005-1012), vectors and tables as fp32. */
int ltx_load_tensor(ltx_ctx* ctx, const char* key, const void* host_data, ltx_dtype dtype, const int64_t* shape, int ndim);
/* Reads a .safetensors checkpoint and loads the tensors of the hot path under their post-mapping names -- the counterpart of
 * LTXWeightLoader.loadTransformerWeights / loadVAEWeights (Utils/ModelDownloader.swift:605-659) with the key mapping of
 * mapTransformerKey (:756-803) and mapVAEWeights (:808-899).  which: 1 = video transformer (unified checkpoint: only the
 * "model.diffusion_model." tensors; audio / cross-modal / connector tensors are skipped as with includeAudio:false),
 * 2 = VAE decoder (stand-alone VAE file or the "vae." tensors of a unified checkpoint; encoder tensors are skipped),
 * 3 = VAE encoder (the "encoder." tensors of the same files, mapVAEEncoderWeights :1224-1280, names prefixed "vae_encoder."),
 * 4 = latent upscaler file (loadSpatialUpscaler, Models/Upscaler/SpatialUpscaler.swift:262-300, names prefixed "upscaler.";
 * conv kernels are taken in the checkpoint's (O, I, kD, kH, kW) layout),
 * 5 = dual audio/video transformer (loadTransformerWeights(includeAudio: true), :605-639: the audio_*, av_ca_* and
 * cross-modal tensors are kept under their own names).  ltx_map_weight_key also accepts which = 6: a LoRA layer key ->
 * the model weight it patches (LoRAKeyMapper.loraKeyToModelKey, LoRA/LoRALoader.swift:209-243).
 * F32 / BF16 / F16 tensors are accepted, and for which = 1 and 5 also scaled-FP8 Linears (the layout of ltx_load_tensor_e4m3,
 * assumed from the ".weight_scale" / ".input_scale" side keys the reference's loader filters): "X.weight" in F8_E4M3
 * (e4m3fn) [N, K] with "X.weight_scale" in F32 / BF16 of shape [] / [1] / [N] / [N, 1]; "X.input_scale" is ignored (FP8 mode
 * quantises activations per token row at run time).  Mixed files are fine.  Refused with LTX_ERR_WEIGHTS: F8_E4M3 without a
 * valid scale (or with a scale that is not finite and > 0), F8_E5M2, F8_E4M3 on anything but a 2-D transformer ".weight"
 * (and in the VAE / encoder / upscaler files), NaN codes.  The whole header is validated before anything is uploaded; the NaN
 * check runs during the upload, and a refused file leaves none of its tensors in the context.  n_loaded (nullable) receives
 * the number of tensors taken.  Follow with ltx_finalize_weights.  ltx_map_weight_key exposes the name mapping alone (no
 * context, no GPU): it writes the mapped name, or an empty string for a tensor the loader skips, into out[cap]. */
int ltx_load_safetensors(ltx_ctx* ctx, const char* path, int which, int* n_loaded);
/* The code-carrying twin of ltx_load_tensor, for callers that parse scaled-FP8 checkpoints themselves: the transformer Linear
 * weight `key` (post-mapping name, ending in ".weight") of shape[ndim = 2] = [N, K] given as e4m3 (e4m3fn) codes[N * K] and
 * fp32 scales[n_scales], n_scales = 1 (one scale per tensor) or N (one per output channel): w[n][k] = e4m3(code) * scale.
 * bf16 and int8 / int4 modes store the decoded bf16 values (the rounding an fp32 file of w gets), fp32 mode the fp32 products.
 * FP8 mode keeps the codes of the Linears inside the transformer blocks as they are, with their scales as the GEMM's row
 * scales (no second rounding, half the bytes of bf16); the other Linears are decoded to bf16.  (The dual audio/video model
 * has no FP8 mode; ltx_load_safetensors with which = 5 decodes its tensors in every mode.)  n_scales other than 1 or N, ndim != 2 or null pointers:
 * LTX_ERR_INVALID_ARGUMENT; a key outside the transformer, a scale that is not finite and > 0, or a NaN code (0x7F / 0xFF,
 * checked on the device; the tensor is then not loaded): LTX_ERR_WEIGHTS. */
int ltx_load_tensor_e4m3(ltx_ctx* ctx, const char* key, const uint8_t* codes, const float* scales, int64_t n_scales,
                         const int64_t* shape, int ndim);
int ltx_map_weight_key(int which, const char* file_key, char* out, size_t cap);
/* LoRA fuse at load time -- LoRAAdapter.fuseWeights (LoRA/LoRAAdapter.swift:64-166) with the delta of LoRAWeights.getDelta
 * (LoRA/LoRALoader.swift:162-178): W[out, in] += scale * up[out, rank] @ down[rank, in] on the loaded tensor `key` (post-mapping
 * name; ltx_map_weight_key(6, loraLayerKey) is LoRAKeyMapper.loraKeyToModelKey :209-243).  Call after loading the base weights
 * and BEFORE ltx_finalize_weights: quantisation then sees the merged weight (the reference dequantises, merges, requantises).
 * rank must be a multiple of 8; scale = user scale * alpha / rank as computed by the reference's loader.  A weight held as
 * e4m3 codes (FP8 mode, loaded from a scaled-FP8 checkpoint) is decoded to bf16 first and the delta added there; finalize then
 * converts it by FP8 mode's per-row rule: "merge, then quantise", as for int8. */
int ltx_fuse_lora(ltx_ctx* ctx, const char* key, const void* down, const void* up, ltx_dtype dtype, int rank, float scale);
/* Precision of the DiT path.  16 (default): the reference's "bf16" mode -- bf16 weights and tensor-core operands, fp32
 * accumulation / residual stream / norms / softmax; velocity within rel-L2 1e-2 of the fp32 graph.  32: fp32 mode -- DiT
 * matrices stay fp32, activations fp32, every Linear runs as a split-bf16 (3-term) tensor-core product that is exact to
 * fp32 rounding, attention in fp32; velocity within rel-L2 1e-4 (the mode BASELINE config 0, "random-init fp32", is checked
 * in); single GPU, no quantisation.  8: FP8 mode -- at ltx_finalize_weights every Linear inside the transformer blocks
 * (attn1 q|k|v and to_out, attn2 q, text k / v and to_out, FFN in / out) becomes e4m3 codes with one power-of-two scale per output channel (s = 2^ceil(log2(amax /
 * 448)), q = e4m3_rn_satfinite(w / s); the bf16 copies are freed, about half the DiT's weight bytes), and each of those GEMMs
 * quantises its activation rows by the same rule and runs e4m3 x e4m3 -> fp32 on the tensor cores (tcgen05 kind::f8f6f4),
 * scaled back per row and column before the bias.  Those Linears that arrive as e4m3 codes (a scaled-FP8 checkpoint through
 * ltx_load_safetensors or ltx_load_tensor_e4m3) keep the file's codes and take the file's scale (per tensor, broadcast, or
 * per output channel) as their row scale instead: nothing is rounded twice and no bf16 copy of them is ever made.
 * Patchify, caption projection, timestep MLPs / AdaLN and proj_out stay bf16 (decoded when they arrive as codes).
 * FP8 mode refuses quant_bits != 16, sequence parallelism (pass groups are fine) and the dual audio/video model
 * (LTX_ERR_UNSUPPORTED).  Must be called before the DiT weights are loaded (8 after that: LTX_ERR_UNSUPPORTED); the VAE is
 * unaffected in every mode. */
int ltx_set_precision(ltx_ctx* ctx, int bits);
/* Where quantised weights live (takes effect at the next ltx_finalize_weights with quant_bits 8 / 4).  0 (default): as codes --
 * 13 GB (int8) / 6.5 GB (int4) for the video DiT; every GEMM dequantises on the fly (fused kernel for M <= 256, a per-GEMM bf16
 * panel above).  1: materialised -- every Linear is quantised exactly as in mode 0 and its dequantised values (s * q + beta,
 * rounded to bf16: the operand values the fused kernels feed the tensor cores) replace the bf16 weight once, at load time; the
 * codes are dropped.  Same results bit for bit as mode 0 at the speed and footprint of the bf16 model: the reference quantises to
 * fit 32 GB of unified memory (Pipeline/LTXPipeline.swift:323-333), which a 180 GB B200 does not need. */
int ltx_set_quant_storage(ltx_ctx* ctx, int materialise);
/* Random-init weights of the configured architecture, generated on the device (no checkpoints in this environment).
 * which: bit mask, 1 = DiT, 2 = VAE decoder, 4 = VAE encoder, 8 = latent upscaler, 16 = the audio / cross-modal tensors of the
 * dual audio/video transformer (use 17 for the whole LTX2Transformer). */
int ltx_init_random_weights(ltx_ctx* ctx, int which, uint64_t seed);
/* Packs the loaded tensors into kernel layouts.  quant_bits: 16 = bf16; 8 / 4 replace every GEMM weight of the DiT by
 * per-64-group affine codes (w ~= s*q + beta) consumed by the dequant-fused GEMM -- the counterpart of
 * quantize(model:groupSize:64,bits:) (Pipeline/LTXPipeline.swift:323-333).  The exact MLX rounding rule is not in the
 * reference tree; ours is plain min/max affine with bf16 scales (DESIGN.md).  Each component (DiT, VAE decoder, VAE encoder,
 * upscaler) is packed once: the call may be repeated after loading a further component (loadVAEEncoder on demand,
 * Pipeline/LTXPipeline.swift:1870-1884). */
int ltx_finalize_weights(ltx_ctx* ctx, int quant_bits, int group_size);

/* Per-forward runtime flags: setSTGSkipFlags / clearSTGSkipFlags / setCrossAttentionScale
 * (Models/Transformer/LTXTransformer.swift:497-526). */
#define LTX_MAX_FLAG_BLOCKS 64
typedef struct {
  int32_t n_stg_blocks;                      /* blocks whose skip flags are set (empty = normal pass) */
  int32_t stg_blocks[LTX_MAX_FLAG_BLOCKS];
  int32_t skip_self_attn;                    /* applied to stg_blocks */
  int32_t skip_ff;
  int32_t n_cas_blocks;                      /* blocks with a cross-attention scale != 1 */
  int32_t cas_blocks[LTX_MAX_FLAG_BLOCKS];
  float cross_attn_scale;
  uint64_t context_key;  /* 0: recompute caption projection + text K/V; else cache them under this key (step-invariant) */
} ltx_dit_flags;

/* LTXTransformer.callAsFunction(latent:context:timesteps:contextMask:latentShape:)
 * (Models/Transformer/LTXTransformer.swift:235-486).
 *   latent   [B, N, in_channels]   (N = F*H*W, token order F-major then H then W, Pipeline/LatentUtils.swift:29-31)
 *   context  [B, S, caption_channels]
 *   timesteps[B] sigma in [0,1], or [B,N] per token when ts_per_token != 0 (image-conditioned denoise())
 *   mask     [B, S] int32, 1 = attend, NULL = all ones
 *   out      [B, N, out_channels] fp32 velocity
 * Host-pointer variant copies in/out and synchronises. */
int ltx_dit_forward(ltx_ctx* ctx, const void* latent, ltx_dtype latent_dtype, const void* context, ltx_dtype context_dtype,
                    const float* timesteps, int ts_per_token, const int32_t* mask, int B, int N, int S, int F, int H,
                    int W, const ltx_dit_flags* flags, float* out_velocity);
int ltx_dit_forward_dev(ltx_ctx* ctx, const void* latent, ltx_dtype latent_dtype, const void* context,
                        ltx_dtype context_dtype, const float* timesteps, int ts_per_token, const int32_t* mask, int B, int N,
                        int S, int F, int H, int W, const ltx_dit_flags* flags, float* out_velocity);
/* LTX2Transformer.callAsFunction(videoLatent:audioLatent:videoContext:audioContext:videoTimesteps:audioTimesteps:
 * videoContextMask:audioContextMask:videoLatentShape:audioNumFrames:) (Models/Transformer/LTX2Transformer.swift:240-392): the dual
 * audio/video ("19 B") model -- per block video and audio self-attention, text cross-attention on both streams, audio->video
 * and video->audio cross-modal attention, both feed-forwards (Models/Transformer/LTX2TransformerBlock.swift:174-297).
 *   video_latent [1, N, in_channels], audio_latent [1, Ta, audio_in_channels] (bf16 or fp32), contexts [1, S, caption_channels],
 *   one sigma per stream, masks [1, S] int32 or NULL; out_video [1, N, out_channels], out_audio [1, Ta, audio_in_channels] fp32.
 * context_key != 0 caches the text K / V of both streams.  Weights: bf16, or int8 / int4 after ltx_finalize_weights(ctx, 8 | 4, 64)
 * (quantize(model: ltx2, groupSize: 64, bits:), Pipeline/LTXPipeline.swift:491).  One GPU; B = 1 here, B = 2 through
 * ltx_av_forward_batch. */
int ltx_av_forward(ltx_ctx* ctx, const void* video_latent, ltx_dtype video_dtype, const void* audio_latent, ltx_dtype audio_dtype,
                   const void* video_context, const void* audio_context, ltx_dtype context_dtype, float video_sigma,
                   float audio_sigma, const int32_t* video_mask, const int32_t* audio_mask, int N, int Ta, int S, int F, int H,
                   int W, uint64_t context_key, float* out_video, float* out_audio);
int ltx_av_forward_dev(ltx_ctx* ctx, const void* video_latent, ltx_dtype video_dtype, const void* audio_latent,
                       ltx_dtype audio_dtype, const void* video_context, const void* audio_context, ltx_dtype context_dtype,
                       const float* video_sigma, const float* audio_sigma, const int32_t* video_mask, const int32_t* audio_mask,
                       int N, int Ta, int S, int F, int H, int W, uint64_t context_key, float* out_video, float* out_audio);
/* The same call with videoTimesteps of shape [1, N] -- one sigma per video token: the image-to-video branch of
 * generateVideoWithAudio feeds sigma * (1 - conditioningMask) (Pipeline/LTXPipeline.swift:1293-1298), and the main video
 * AdaLN-single, both cross-modal video embedders and the output head's embedded timestep are then evaluated per token
 * (Models/Transformer/LTX2Transformer.swift:273-298, 370-377).  video_sigmas [N] fp32; the audio stream keeps one sigma. */
int ltx_av_forward_tokens(ltx_ctx* ctx, const void* video_latent, ltx_dtype video_dtype, const void* audio_latent,
                          ltx_dtype audio_dtype, const void* video_context, const void* audio_context, ltx_dtype context_dtype,
                          const float* video_sigmas, float audio_sigma, const int32_t* video_mask, const int32_t* audio_mask, int N,
                          int Ta, int S, int F, int H, int W, uint64_t context_key, float* out_video, float* out_audio);
int ltx_av_forward_tokens_dev(ltx_ctx* ctx, const void* video_latent, ltx_dtype video_dtype, const void* audio_latent,
                              ltx_dtype audio_dtype, const void* video_context, const void* audio_context, ltx_dtype context_dtype,
                              const float* video_sigmas, const float* audio_sigma, const int32_t* video_mask,
                              const int32_t* audio_mask, int N, int Ta, int S, int F, int H, int W, uint64_t context_key,
                              float* out_video, float* out_audio);
/* LTX2Transformer.callAsFunction (Models/Transformer/LTX2Transformer.swift:240-392) on a batch, with the conventions of
 * ltx_dit_forward: B items (1 or 2, e.g. the conditional and unconditional passes of a CFG step) in one forward.
 *   video_latent [B, N, in_channels], audio_latent [B, Ta, audio_in_channels] (bf16 or fp32), contexts [B, S, caption_channels];
 *   video_sigmas [B], or [B, N] when video_ts_per_token != 0; audio_sigmas [B]; masks [B, S] int32 or NULL;
 *   out_video [B, N, out_channels], out_audio [B, Ta, audio_in_channels] fp32.
 * Each item attends within itself only, and its outputs equal those of the B = 1 call on that item alone, bit for bit.
 * B > 2, and B = 2 on a sequence-parallel (Ulysses) context, return LTX_ERR_UNSUPPORTED; bad sizes or NULL tensors
 * LTX_ERR_INVALID_ARGUMENT.  Refused calls write nothing.  Host-pointer variant copies in/out and synchronises. */
int ltx_av_forward_batch(ltx_ctx* ctx, const void* video_latent, ltx_dtype video_dtype, const void* audio_latent,
                         ltx_dtype audio_dtype, const void* video_context, const void* audio_context, ltx_dtype context_dtype,
                         const float* video_sigmas, int video_ts_per_token, const float* audio_sigmas, const int32_t* video_mask,
                         const int32_t* audio_mask, int B, int N, int Ta, int S, int F, int H, int W, uint64_t context_key,
                         float* out_video, float* out_audio);
int ltx_av_forward_batch_dev(ltx_ctx* ctx, const void* video_latent, ltx_dtype video_dtype, const void* audio_latent,
                             ltx_dtype audio_dtype, const void* video_context, const void* audio_context, ltx_dtype context_dtype,
                             const float* video_sigmas, int video_ts_per_token, const float* audio_sigmas,
                             const int32_t* video_mask, const int32_t* audio_mask, int B, int N, int Ta, int S, int F, int H, int W,
                             uint64_t context_key, float* out_video, float* out_audio);
/* LTXTransformer.clearRoPECache (:202) + drops the cached text K/V. */
int ltx_dit_clear_caches(ltx_ctx* ctx);

/* applyCFG + applyGuidanceRescale (Pipeline/LatentUtils.swift:131-183), STG / GE lines (Pipeline/LTXPipeline.swift:920-927)
 * and LTXScheduler.step(latent:velocity:sigma:sigmaNext:) (Scheduler/LTXScheduler.swift:305-327), fused, fp32.
 *   latent in/out [n]; v_uncond / v_stg / v_prev may be NULL; v_prev is read (if use_prev) and then overwritten with
 *   the velocity actually used (the GE momentum state). */
int ltx_guided_euler_step(ltx_ctx* ctx, float* latent, const float* v_cond, const float* v_uncond, const float* v_stg,
                          float* v_prev, int use_prev, size_t n, float cfg_scale, float rescale_phi, float stg_scale,
                          float ge_gamma, float sigma, float sigma_next);
int ltx_guided_euler_step_dev(ltx_ctx* ctx, float* latent, const float* v_cond, const float* v_uncond, const float* v_stg,
                              float* v_prev, int use_prev, size_t n, float cfg_scale, float rescale_phi, float stg_scale,
                              float ge_gamma, float sigma, float sigma_next);

/* Device-resident fast path for the generateVideo step loop (Pipeline/LTXPipeline.swift:793-956): the latent, both
 * text contexts and the GE state stay in HBM between steps. */
typedef struct {
  float sigma, sigma_next;
  float cfg_scale;      /* <= 1: no unconditional pass */
  float rescale_phi;
  float stg_scale;      /* <= 0: no perturbed pass */
  float ge_gamma;
  int32_t n_stg_blocks;
  int32_t stg_blocks[LTX_MAX_FLAG_BLOCKS];
  int32_t step_index;   /* GE applies for step_index > 0 */
  int32_t i2v_frame0_conditioned; /* image-to-video loop (denoise(), Pipeline/LTXPipeline.swift:2237-2252, 2344-2357): the
                                     first latent frame is a clean conditioning frame -> its tokens get timestep 0
                                     (per-token timesteps sigma * (1 - mask)) and the Euler update skips it */
  int32_t disable_stg_prefix_sharing; /* 0 (default): the STG pass reuses the conditional pass's blocks before the first
                                         perturbed block (identical inputs -> identical values); 1: recompute them */
  int32_t disable_batched_cfg;        /* 0 (default): on one GPU the conditional and unconditional passes run as ONE B = 2
                                         forward, as denoise() batches them (Pipeline/LTXPipeline.swift:2234-2269) -- in both
                                         ltx_denoise_step and ltx_av_denoise_step; 1: as two B = 1 forwards, the way
                                         generateVideo / generateVideoWithAudio issue them (:829-848, :1300-1362).  Same values
                                         per pass.  LTX_BATCHED_CFG=0 in the environment also selects two forwards. */
} ltx_step_params;
/* noise [in_channels, F, H, W] fp32 host; latent = noise * sigma0 (:793).  neg_context may be NULL. */
int ltx_denoise_begin(ltx_ctx* ctx, const float* noise, int F, int H, int W, float sigma0, const void* context,
                      ltx_dtype context_dtype, const int32_t* mask, const void* neg_context, const int32_t* neg_mask, int S);
int ltx_denoise_step(ltx_ctx* ctx, const ltx_step_params* p);
/* copies the current latent [in_channels, F, H, W] fp32 to the host (synchronises). */
int ltx_denoise_get_latent(ltx_ctx* ctx, float* latent_out);
/* device pointer of the resident latent (for chaining into ltx_vae_decode_dev). */
int ltx_denoise_latent_dev(ltx_ctx* ctx, float** latent_dev);

/* The step loop of generateVideoWithAudio (Pipeline/LTXPipeline.swift:1255-1404), device resident: both latents, the text K / V
 * of both streams and the velocities stay in HBM; one call per step.
 *   begin : video_noise [in_channels, F, H, W], audio_noise [Ta, audio_in_channels] (the packed audio latent) fp32 host; both
 *           are scaled by sigma0 (:1255-1259); contexts [S, caption_channels]; one mask serves both streams (textMask); the
 *           negative contexts (a pair, or both NULL) enable CFG.
 *   step  : per pass one LTX2Transformer forward (two with CFG, :1300-1362; on one GPU without Ulysses both passes run as
 *           one B = 2 forward, item 0 conditional, unless disable_batched_cfg or LTX_BATCHED_CFG=0 -- same values per pass);
 *           video = applyCFG (+ rescale) + scheduler.step,
 *           audio = applyCFG + latent += (sigma_next - sigma) * velocity (:1402).  Reads sigma, sigma_next, cfg_scale,
 *           rescale_phi and i2v_frame0_conditioned of ltx_step_params (per-token video timesteps sigma * (1 - mask) and an
 *           untouched frame 0, :1293-1298, 1381-1391; set the frame with ltx_denoise_set_frame0); STG / GE are not part of
 *           this loop (LTX_ERR_UNSUPPORTED).
 *   get   : either output may be NULL.  ltx_denoise_latent_dev / ltx_denoise_set_frame0 act on the video latent. */
int ltx_av_denoise_begin(ltx_ctx* ctx, const float* video_noise, const float* audio_noise, int F, int H, int W, int Ta,
                         float sigma0, const void* video_context, const void* audio_context, ltx_dtype context_dtype,
                         const int32_t* mask, const void* neg_video_context, const void* neg_audio_context,
                         const int32_t* neg_mask, int S);
int ltx_av_denoise_step(ltx_ctx* ctx, const ltx_step_params* p);
int ltx_av_denoise_get_latents(ltx_ctx* ctx, float* video_latent_out, float* audio_latent_out);

/* decodeVideo(latent:decoder:timestep:temporalTileSize:temporalTileOverlap:) untiled
 * (Models/VAE/VideoDecoder.swift:466-508 -> VideoDecoder.callAsFunction :358-449).
 *   latent [128, F', H', W'] fp32 ; timestep < 0 = none ; decode_noise (same shape) required when timestep >= 0;
 *   out_frames [8(F'-1)+1, 32H', 32W', 3] fp32 in [0,1]. */
int ltx_vae_decode(ltx_ctx* ctx, const float* latent, int Fp, int Hp, int Wp, float timestep, const float* decode_noise,
                   int causal, float* out_frames);
int ltx_vae_decode_dev(ltx_ctx* ctx, const float* latent, int Fp, int Hp, int Wp, float timestep,
                       const float* decode_noise, int causal, float* out_frames);
/* decodeVideo with temporalTileSize > 0 and more latent frames than one tile (Models/VAE/VideoDecoder.swift:482-494 ->
 * decodeWithTemporalTiling :517-602): chunks of tile_size latent frames at stride tile_size - tile_overlap are decoded
 * independently, the 8 * tile_overlap frames they share are cross-faded linearly (weight j / (8 overlap) on the later chunk),
 * and the result is normalised and clipped.  This is the reference's memory-saving approximation (Fp <= tile_size, or
 * tile_size <= 0, is the exact single pass); its frame count follows the chunk arithmetic -- ltx_vae_tiled_frames gives it
 * (-1 for an invalid tile / overlap pair) so that the caller can size out_frames [frames, 32H', 32W', 3].  With
 * timestep >= 0 each chunk mixes in its own slice of decode_noise. */
int ltx_vae_tiled_frames(int Fp, int tile_size, int tile_overlap);
int ltx_vae_decode_tiled(ltx_ctx* ctx, const float* latent, int Fp, int Hp, int Wp, float timestep, const float* decode_noise,
                         int causal, int tile_size, int tile_overlap, float* out_frames, int* out_num_frames);
int ltx_vae_decode_tiled_dev(ltx_ctx* ctx, const float* latent, int Fp, int Hp, int Wp, float timestep,
                             const float* decode_noise, int causal, int tile_size, int tile_overlap, float* out_frames,
                             int* out_num_frames);

/* 8-bit frames.  The value v of a sample is what the fp32 entry points return: clip01((x + 1) / 2).
 *   LTX_FRAMES_RGB8: [F, H, W, 3] uint8, q = (uint8_t)(v * 255.0f) -- one fp32 multiply, then truncation.  This is
 *                    tensorToImages (U/VideoExporter.swift:543-580: clip, x 255, to uint8) as SURVEY section 2 row 21
 *                    describes it, with MLX's float -> uint8 cast; the rounding rule is taken from that description.
 *   LTX_FRAMES_I420: planar 4:2:0, BT.709, limited range; per frame Y [H][W] | U [H/2][W/2] | V [H/2][W/2], frames one
 *                    after another.  Y = rint(16 + 219 Y'), Y' = 0.2126 R + 0.7152 G + 0.0722 B per pixel;
 *                    Cb = rint(128 + 224 (B_m - Y'_m) / 1.8556), Cr = rint(128 + 224 (R_m - Y'_m) / 1.5748), where m is
 *                    the mean colour of the 2x2 cell (((p00 + p01) + p10) + p11) * 0.25 per component and Y'_m its luma.
 *                    fp32 arithmetic, round to nearest, ties to even. */
typedef enum { LTX_FRAMES_RGB8 = 1, LTX_FRAMES_I420 = 2 } ltx_frames_format;
/* Bytes of F frames of H x W pixels in `format`; 0 for a bad format, a non-positive size, or odd H / W in I420.  Host only. */
size_t ltx_frames_u8_bytes(int F, int H, int W, int format);
/* decodeVideo -> tensorToImages (U/VideoExporter.swift:543-580) as one call: the arguments of ltx_vae_decode /
 * ltx_vae_decode_tiled, and `out` holds ltx_frames_u8_bytes(frames, 32H', 32W', format) bytes.  The untiled decode writes
 * the 8-bit frames from conv_out's epilogue (no fp32 frame buffer; a temporally sharded decode gathers the 8-bit planes);
 * the tiled one converts after its blend and clip.  Same bytes as ltx_frames_to_u8 of the fp32 decode.  A bad format or
 * out == NULL returns LTX_ERR_INVALID_ARGUMENT before anything is written.  _dev: device pointers, `out` 4-byte aligned. */
int ltx_vae_decode_u8(ltx_ctx* ctx, const float* latent, int Fp, int Hp, int Wp, float timestep, const float* decode_noise,
                      int causal, int format, uint8_t* out);
int ltx_vae_decode_u8_dev(ltx_ctx* ctx, const float* latent, int Fp, int Hp, int Wp, float timestep,
                          const float* decode_noise, int causal, int format, uint8_t* out);
int ltx_vae_decode_tiled_u8(ltx_ctx* ctx, const float* latent, int Fp, int Hp, int Wp, float timestep,
                            const float* decode_noise, int causal, int tile_size, int tile_overlap, int format, uint8_t* out,
                            int* out_num_frames);
int ltx_vae_decode_tiled_u8_dev(ltx_ctx* ctx, const float* latent, int Fp, int Hp, int Wp, float timestep,
                                const float* decode_noise, int causal, int tile_size, int tile_overlap, int format,
                                uint8_t* out, int* out_num_frames);
/* tensorToImages (U/VideoExporter.swift:543-580) for frames already decoded: fp32 [F, H, W, 3] (clipped to [0, 1] first)
 * -> `format`, the same arithmetic as the fused decode.  Refusals as above; I420 needs even H and W. */
int ltx_frames_to_u8(ltx_ctx* ctx, const float* frames, int F, int H, int W, int format, uint8_t* out);
int ltx_frames_to_u8_dev(ltx_ctx* ctx, const float* frames, int F, int H, int W, int format, uint8_t* out);

/* VideoEncoder.callAsFunction (Models/VAE/VideoEncoder.swift:270-312), the encoder half of encodeImage
 * (Pipeline/LTXPipeline.swift:1902-1932): pixels [3, T, H, W] fp32 (the reference feeds [-1, 1]), H and W multiples of 32
 * -> latent mean [128, ceil(T/8), H/32, W/32] fp32 (T = 8k+1 frames -> k+1 latent frames; an image is T = 1).
 * normalize != 0 applies (latent - mean_of_means) / std_of_means with the decoder's statistics, as encodeImage does
 * (:1920-1926).  Weights: "vae_encoder.*" tensors (ltx_load_safetensors which = 3 or ltx_load_tensor). */
int ltx_vae_encode(ltx_ctx* ctx, const float* pixels, int T, int H, int W, int normalize, float* latent_out);
int ltx_vae_encode_dev(ltx_ctx* ctx, const float* pixels, int T, int H, int W, int normalize, float* latent_out);

/* upsampleLatents(_:upscaler:latentMean:latentStd:) (Models/Upscaler/SpatialUpscaler.swift:360-383; inlined at
 * Pipeline/LTXPipeline.swift:1694-1708, 2594-2619): latent [128, F, H, W] fp32 (normalised) -> denormalise ->
 * SpatialUpscaler (:215-258) -> renormalise -> [128, F, 2H, 2W].  Weights: "upscaler.*" tensors. */
int ltx_upscale_latent(ltx_ctx* ctx, const float* latent, int F, int H, int W, float* out);
int ltx_upscale_latent_dev(ltx_ctx* ctx, const float* latent, int F, int H, int W, float* out);

/* adainFilterLatent(_:reference:factor:) (Pipeline/LatentUtils.swift:201-227): per-channel statistics over (F, H, W) of
 * latent [channels, n_per_channel] are replaced by those of reference [channels, n_ref_per_channel]; in place. */
int ltx_adain_filter(ltx_ctx* ctx, float* latent, size_t n_per_channel, const float* reference, size_t n_ref_per_channel,
                     int channels, float factor);
int ltx_adain_filter_dev(ltx_ctx* ctx, float* latent, size_t n_per_channel, const float* reference, size_t n_ref_per_channel,
                         int channels, float factor);

/* Starts a resident denoise session from an existing latent instead of pure noise -- stage 2 of generateVideoTwoStage
 * (Pipeline/LTXPipeline.swift:2636-2647): latent = noise_scale * noise + (1 - noise_scale) * latent.  latent and noise are
 * [in_channels, F, H, W] fp32 host buffers; frame0_latent (nullable, [in_channels, 1, H, W]) overwrites the first latent
 * frame afterwards (the full-resolution image latent of I2V stage 2, :2650-2657).  Text arguments as ltx_denoise_begin. */
int ltx_denoise_begin_from_latent(ltx_ctx* ctx, const float* latent, const float* noise, float noise_scale,
                                  const float* frame0_latent, int F, int H, int W, const void* context, ltx_dtype context_dtype,
                                  const int32_t* mask, const void* neg_context, const int32_t* neg_mask, int S);
/* Device-resident glue between the two stages (generateVideoTwoStage :2594-2647) without a host round trip: takes the
 * current session latent [C, F, H, W] as the stage-1 output, upscales it 2x (ltx_upscale_latent), applies AdaIN against
 * the stage-1 latent (factor adain_factor), mixes in noise [C, F, 2H, 2W] (host, fp32) with noise_scale and makes the
 * result the session latent at (F, 2H, 2W); the text contexts of the session are kept. */
int ltx_denoise_upscale_stage(ltx_ctx* ctx, const float* noise, float noise_scale, float adain_factor);
/* latent[:, 0, :, :] = frame0_latent (host, [in_channels, 1, H, W] fp32): the clean conditioning frame of the
 * image-to-video loops (Pipeline/LTXPipeline.swift:1132-1160, 2650-2657); combine with ltx_step_params.i2v_frame0_conditioned. */
int ltx_denoise_set_frame0(ltx_ctx* ctx, const float* frame0_latent);

/* ---- multi-GPU: one process and one context per GPU of an NVLink/NVSwitch box; NCCL communicators are owned by the context.
 * The reference has no multi-device code (SURVEY 2a); correctness contract: N-GPU result == 1-GPU result.
 *   world_size = pass_groups * sp_size, rank = group * sp_size + sp_rank.
 *   sp_size     : Ulysses sequence parallelism of ltx_dit_forward* / ltx_denoise_step (tokens sharded over the sp ranks for
 *                 row-wise ops, heads sharded inside self-attention, NCCL all-to-all in between); must divide num_heads and N.
 *                 Every rank passes the full inputs and receives the full velocity.
 *   pass_groups : ltx_denoise_step runs pass p (conditional, unconditional, STG) on group p % pass_groups and broadcasts
 *                 the velocities; the guided Euler update is replicated.
 *   ltx_vae_decode* shards the latent frames in contiguous temporal slabs over all ranks, exchanging one boundary frame
 *   per convolution with each neighbour (exact, unlike the reference's overlap-blend tiling); every rank gets all frames.
 * ltx_dist_get_unique_id fills a 128-byte NCCL id on one rank; the caller ships it to the others (torch.distributed, MPI, ...). */
int ltx_dist_get_unique_id(void* id_out_128);
int ltx_dist_init(ltx_ctx* ctx, const void* unique_id_128, int rank, int world_size, int sp_size, int pass_groups);
int ltx_dist_info(const ltx_ctx* ctx, int* rank, int* world_size, int* sp_size, int* pass_groups);
/* 1 when the Ulysses exchange of this context runs over peer memory: every sp rank's receive buffer is mapped into its
 * peers (CUDA IPC over NVLink / NVSwitch), the V-projection GEMM epilogue, the q/k norm+RoPE kernel and the attention
 * epilogue store their head / token blocks straight into the destination rank's buffer, and a release/acquire flag barrier
 * replaces the NCCL all-to-all.  Established lazily by the first sequence-parallel forward; 0 = NCCL all-to-all (mapping
 * unavailable or LTX_P2P=0). */
int ltx_dist_p2p_active(const ltx_ctx* ctx);
/* The same wiring for contexts that all live in ONE process (one per device; contexts[i] becomes rank i): the shape a Swift
 * host needs, whose pipeline is a single actor in a single process (Pipeline/LTXPipeline.swift:117) and has no launcher.
 * Afterwards the collective entry points must be called concurrently, one host thread per context.  Peer memory between
 * same-process ranks is plain peer access (no IPC handles). */
int ltx_dist_init_local(ltx_ctx** contexts, int n, int sp_size, int pass_groups);
/* Destroys the communicators (collective); the context can be re-initialised with a different layout afterwards. */
int ltx_dist_shutdown(ltx_ctx* ctx);

/* Page-locked host memory for the caller's input / output buffers (frames, latents): the host-pointer entry points copy
 * with cudaMemcpyAsync, which only reaches PCIe speed (and only overlaps) from pinned memory -- a pageable 118 MB frame
 * buffer costs ~24 ms per 25-frame decode, a pinned one ~2 ms.  The Swift adapter wraps the pointer in an MLXArray / Data
 * without copying. */
int ltx_host_alloc(void** ptr, size_t bytes);
int ltx_host_free(void* ptr);

/* Number of kernels launched by this context so far (bench.py reports the per-step delta as gpu_launches). */
uint64_t ltx_launch_count(const ltx_ctx* ctx);
/* The CUDA stream (cudaStream_t) every kernel of this context is enqueued on -- for CUDA-event timing by the caller. */
int ltx_get_stream(ltx_ctx* ctx, void** stream);
/* Per-kernel-class device timing (the B200 counterpart of GenerationTimings / --profile, LTXVideo.swift:255-297):
 * when enabled, every launch is bracketed by CUDA events on the context stream.  ltx_get_profile synchronises, sums
 * elapsed ms / algorithmic flops / algorithmic bytes / launch counts per class and clears the records.
 * Classes: 0 GEMM, 1 attention, 2 norm/RoPE rows, 3 conv3d, 4 VAE prologue, 5 other; n_classes must be >= 8. */
int ltx_set_profiling(ltx_ctx* ctx, int enabled);
/* Captured steps.  In the steady state of a denoise loop (text projections cached, RoPE table built) ltx_denoise_step and
 * ltx_dit_forward issue a fixed sequence of ~600 launches on fixed buffers; the library runs the sequence eagerly once per
 * (shape, flags, buffers), captures it into a CUDA graph on the second occurrence and replays the graph afterwards -- the
 * B200 counterpart of MLX's lazy graph + eval() (Pipeline/LTXPipeline.swift:950-952).  Same results bit for bit.
 * ltx_set_graphs(ctx, 0) turns it off (and drops the captured graphs); ltx_graph_stats reports captures / replays so far. */
int ltx_set_graphs(ltx_ctx* ctx, int enabled);
int ltx_graph_stats(const ltx_ctx* ctx, uint64_t* captures, uint64_t* replays);
int ltx_get_profile(ltx_ctx* ctx, double* ms, double* flops, double* bytes, uint64_t* counts, int n_classes);

/* ---- diagnostic single-kernel entry points (device pointers; used by the parity tests and the profiler) ---- */
/* C[M,N] = A[M,K] B[N,K]^T (+bias[N]) ; mode: 0 bf16 out, 1 gelu bf16 out, 3 fp32 out, 4 silu bf16 out; force_bn: 0 auto, a tile
 * width, -1 = the weight-streaming kernel for M <= 32 (error if the shape is not eligible), -2 / -3 = the few-row (M <= 512)
 * swap-AB weight-streaming kernel with / without its split-K workspace. */
int ltx_op_gemm(ltx_ctx* ctx, const void* A, const void* B, const float* bias, void* C, int M, int N, int K, int mode,
                int force_bn);
/* The sequence-parallel send layout of the fused q|k|v projection: columns < col_from of A B^T + bias go row-major (pitch col_from)
 * to plain_out, the others leave in blocks of col_block columns, block j to blocks_out + j * block_stride (row pitch col_block);
 * force_bn as above, -2 = the few-row weight-streaming kernel. */
int ltx_op_gemm_blocked(ltx_ctx* ctx, const void* A, const void* B, const float* bias, void* plain_out, void* blocks_out, int M, int N,
                        int K, int col_from, int col_block, int64_t block_stride, int force_bn);
/* x[M,N] (fp32) += (A B^T + bias) * (gate_a[n] + gate_b[n]) * scale ; shadow (bf16, nullable) = new x. */
int ltx_op_gemm_resid(ltx_ctx* ctx, const void* A, const void* B, const float* bias, float* x, const float* gate_a,
                      const float* gate_b, void* shadow, int M, int N, int K, float scale);
/* The weight-streaming kernel on a batch of `items` (1 or 2) items of up to 32 rows each (M <= 32 * items; two items take its
 * 64-row form, the dual model's batched audio stream), or an error: C[M,N] = A[M,K] B[N,K]^T + bias[N] with
 *   mode 0 / 1 / 3 / 4 as ltx_op_gemm (out [M,N]); mode 0 with vt_item_ld > 0: out is V^T [N, items * vt_item_ld], row m of
 *   item i = m / (M / items) in column i * vt_item_ld + m % (M / items);
 *   mode 2: x[M,N] += (A B^T + bias) * (gate_a[(m / rows_per_gate) * N + n] + gate_b[n]) (one gate row per item: rows_per_gate
 *   = M / items; gate_b nullable). */
int ltx_op_gemm_skinny(ltx_ctx* ctx, const void* A, const void* B, const float* bias, void* out, float* x, const float* gate_a,
                       const float* gate_b, int rows_per_gate, int M, int N, int K, int mode, int items, int64_t vt_item_ld);
/* per-64-group affine quantiser / dequantiser and the dequant-fused GEMM (codes [N,K] bytes or [N,K/2] nibbles;
 * scales, biases fp32 [K/64, N]); mode / force_bn as in ltx_op_gemm. */
int ltx_op_quantize(ltx_ctx* ctx, const void* w_bf16, int N, int K, int bits, void* q_out, float* scales_out, float* biases_out);
int ltx_op_dequantize(ltx_ctx* ctx, const void* q, const float* scales, const float* biases, int N, int K, int bits, void* w_bf16);
int ltx_op_gemm_q(ltx_ctx* ctx, const void* A, const void* q, const float* scales, const float* biases, int bits,
                  const float* bias, void* C, int M, int N, int K, int mode, int force_bn);
/* FP8 mode's per-row quantiser: x bf16 [M, K] (row pitch ld elements, ld % 8 == 0, K % 16 == 0) -> e4m3 codes [M, K] and fp32
 * scales [M], s = 2^ceil(log2(amax / 448)) (1 for a zero row), q = e4m3_rn_satfinite(x / s). */
int ltx_op_quantize_fp8(ltx_ctx* ctx, const void* x_bf16, int M, int K, int64_t ld, void* codes, float* scales);
/* FP8 pair GEMM: C[M,N] = (Aq[M,K] Bq[N,K]^T) * sa[m] * sb[n] + bias[n] on e4m3 codes (K % 16 == 0, sb 16-byte aligned);
 * mode as in ltx_op_gemm; force_bn 0 = fitted tile width, else a multiple of 16 in [64, 256]. */
int ltx_op_gemm_fp8(ltx_ctx* ctx, const void* Aq, const float* sa, const void* Bq, const float* sb, const float* bias, void* C, int M,
                    int N, int K, int mode, int force_bn);
/* The same product with the fused q|k|v or residual epilogues.  C != NULL: bf16 output, columns n >= tsplit_col (> 0, a multiple
 * of 32) stored transposed into Ct[(n - tsplit_col) * ldt + m], the others into C [M, tsplit_col] (tsplit_col = 0: C [M, N]).
 * x != NULL (C == NULL): x[M,N] (fp32) += (product + bias) * (gate_a[n] + gate_b[n]) (gates nullable), shadow (bf16, nullable)
 * = new x. */
int ltx_op_gemm_fp8_ex(ltx_ctx* ctx, const void* Aq, const float* sa, const void* Bq, const float* sb, const float* bias, void* C,
                       void* Ct, int tsplit_col, int64_t ldt, float* x, const float* gate_a, const float* gate_b, void* shadow,
                       int M, int N, int K, int force_bn);
/* O = softmax(Q K^T * scale + key_bias) V ; Q [B*Nq, H*128], K [B*Nk, H*128], Vt [H*128, B*ldvb] (batch b owns
 * columns [b*ldvb, b*ldvb + Nk), ldvb % 8 == 0), all bf16. */
int ltx_op_attention(ltx_ctx* ctx, const void* Q, const void* K, const void* Vt, int64_t ldvb, const float* key_bias, void* O,
                     int B, int H, int Nq, int Nk, float scale);
/* the same with head_dim 128 or 64 (64: the audio / cross-modal attentions of the dual block, 32 heads x 64); Q, K [.., H*head_dim],
 * Vt [H*head_dim, B*ldvb] */
int ltx_op_attention_hd(ltx_ctx* ctx, const void* Q, const void* K, const void* Vt, int64_t ldvb, const float* key_bias, void* O,
                        int B, int H, int head_dim, int Nq, int Nk, float scale);
/* head_dim 128, B = 1, output rows scattered in blocks: row r goes to o_blocks[r / rows_per_block] + (r % rows_per_block) * H*128
 * (the Ulysses epilogue that stores each destination rank's token block straight into that rank's buffer; here local pointers) */
int ltx_op_attention_blocks(ltx_ctx* ctx, const void* Q, const void* K, const void* Vt, int64_t ldvb, int H, int Nq, int Nk,
                            float scale, void* const* o_blocks, int n_blocks, int rows_per_block);
int ltx_op_rmsnorm_mod(ltx_ctx* ctx, const float* x, void* out_bf16, int M, int D, const float* tbl_shift,
                       const float* tbl_scale, const float* ada_shift, const float* ada_scale, float eps, int layernorm);
int ltx_op_qknorm_rope(ltx_ctx* ctx, void* x_bf16, int M, int D, const float* w, const float* cos_tab, const float* sin_tab,
                       int rows_per_rope, float eps);
/* What the conv launcher decides for a [T,H,W,Cin] -> Cout convolution (Conv3dFull, Models/VAE/VideoConvolution.swift:238-347)
 * on a device with sm_count SMs; host-only (no context, no GPU).  plan7 = {tile width, CTA pairs, slab stages, bt, bh, bw,
 * tap split}.  Slab stages and the tap split change the order in which the 27 taps are added up, so they depend on H, W and
 * the channel counts only, never on T: a temporal shard of a clip rounds exactly like the whole clip (the multi-GPU decode is
 * bit-identical to the single-GPU one).  mode: 0 plain, 1 depth-to-space, 2 unpatchify, 3 / 4 the fused hand-over epilogues. */
int ltx_conv3d_plan(int T, int H, int W, int Cin, int Cout, int mode, int ntaps, int sm_count, int32_t* plan7);
/* 3x3x3 conv on a channels-last fp32 volume [T,H,W,Cin] -> [T,H,W,Cout] fp32 with reflect/replicate padding. */
int ltx_op_conv3d(ltx_ctx* ctx, const float* x, const void* w_bf16_27_O_I, const float* bias, float* out, int T, int H,
                  int W, int Cin, int Cout, int causal);
/* The convolution's padding prologue: fp32 [T,H,W,C] -> bf16 [T+2,H+2,W+2,C] with the padding materialised.  mode 0 copy,
 * 1 x*a[c] + b[c], 2 silu(pixel_norm(x) * (1 + a[c]) + b[c]) (a, b both NULL: no modulation), 3 silu(x*a[c] + b[c]).
 * pad bits: 1 causal (two leading frame copies), 2 zero padding in H, W instead of reflect, 4 zero padding in T instead of
 * frame replication. */
int ltx_op_vae_prep(ltx_ctx* ctx, const float* x, void* out_pad_bf16, int T, int H, int W, int C, int mode, const float* a,
                    const float* b, int pad);
/* Rewrites the padding voxels of a bf16 [T+2,H+2,W+2,C] volume from its interior, as ltx_op_vae_prep pads (same pad bits). */
int ltx_op_vae_halo_fill(ltx_ctx* ctx, void* vol_bf16, int T, int H, int W, int C, int pad);
/* The implicit-GEMM conv on an already padded bf16 volume [T+2,H+2,W+2,Cin] with weights bf16 [ntaps][Cout][Cin] (27: 3x3x3,
 * 9: the per-frame 3x3 taps dt = 1) and one of its epilogues: 0 out = conv + bias (+ resid, nullable; out == resid allowed)
 * [T,H,W,Cout]; 1 depth-to-space into out [2T-1+t_shift,2H,2W,Cout/8] plus the 4x tiled depth-to-space of resid [T,H,W,Cin];
 * 2 unpatchify 4x4 + (x+1)/2 (clipped to [0,1] unless no_clip) into out [T,4H,4W,3] (Cout = 48); 3 pixel-norm,
 * * (1 + next_scale) + next_shift (both nullable), SiLU of conv + bias into the interior of next_pad [T+2,H+2,W+2,Cout] at frame
 * offset next_tshift (1 or 2); 4 as 0 with resid, and its output also as in 3. */
int ltx_op_conv3d_epi(ltx_ctx* ctx, const void* x_pad_bf16, const void* w_bf16, const float* bias, int T, int H, int W, int Cin,
                      int Cout, int ntaps, int mode, float* out, const float* resid, int t_shift, int no_clip, void* next_pad_bf16,
                      const float* next_scale, const float* next_shift, int next_tshift);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* LTXCUDA_H_ */
