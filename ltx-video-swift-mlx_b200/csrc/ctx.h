// libltxcuda context: device weights, workspaces and caches for one GPU.
#pragma once
#include <atomic>
#include <map>
#include <string>
#include <vector>

#include "../../include/ltxcuda.h"
#include "ltx_internal.h"

namespace ltx {

// Storage of a transformer Linear held as the e4m3 codes of a scaled-FP8 checkpoint (FP8 mode only; never an ltx_dtype): codes
// [N, K] in ptr, fp32 row scales [N] in scales, w[n][k] = e4m3(code) * scales[n].  Two allocations: the scales appended to
// the codes would push every codes allocation past a multiple of the allocator's 2 MB granule.
constexpr int DT_E4M3 = 100;

struct DevTensor {
  void* ptr = nullptr;
  int dtype = LTX_F32;     // storage dtype on the device: LTX_BF16, LTX_F32 or DT_E4M3
  float* scales = nullptr; // DT_E4M3 only
  std::vector<int64_t> shape;
  int64_t numel() const {
    int64_t n = 1;
    for (auto d : shape) n *= d;
    return n;
  }
  const uint8_t* codes() const { return static_cast<const uint8_t*>(ptr); }
  void free_storage() {
    if (ptr) cudaFree(ptr);
    if (scales) cudaFree(scales);
    ptr = nullptr;
    scales = nullptr;
  }
};

// Bumped whenever a DevBuf (re)allocates or frees: captured CUDA graphs hold raw workspace pointers and are only replayed
// while the generation they were captured at is still current.
inline std::atomic<uint64_t>& devbuf_generation() {
  static std::atomic<uint64_t> g{1};
  return g;
}

// Grow-only device buffer.
struct DevBuf {
  void* ptr = nullptr;
  size_t bytes = 0;
  void reserve(size_t n) {
    if (n <= bytes) return;
    devbuf_generation().fetch_add(1, std::memory_order_relaxed);
    if (ptr) LTX_CUDA(cudaFree(ptr));
    ptr = nullptr;
    bytes = 0;
    LTX_CUDA(cudaMalloc(&ptr, n));
    bytes = n;
  }
  void release() {
    if (ptr) { devbuf_generation().fetch_add(1, std::memory_order_relaxed); cudaFree(ptr); }
    ptr = nullptr;
    bytes = 0;
  }
  template <typename T>
  T* as() const { return reinterpret_cast<T*>(ptr); }
};

// The weight of a transformer Linear [n, k] in one of three formats.  dit_quantize / dit_convert_fp8 replace the bf16 matrix
// by its codes in place (w becomes nullptr); linear() in dit.cu picks the kernels from fmt.
enum LinearFormat : int {
  LW_BF16 = 0,     // w: bf16 [n, k] row-major
  LW_AFFINE = 1,   // q: per-64-group affine codes s * q + beta (8 or 4 bit): dequant-fused / panel kernels
  LW_E4M3 = 2,     // q: e4m3 codes with one fp32 scale per row (precision mode 8): the FP8 pair kernel.  A power of two when
                   // dit_convert_fp8 made the codes, the checkpoint's scale when they were loaded from a scaled-FP8 file
};
struct LinearW {
  int fmt = LW_BF16;
  int n = 0, k = 0;
  const bf16* w = nullptr;
  QuantW q;
};

struct AdaLnW {   // AdaLayerNormSingle: Linear(256, dim) -> SiLU -> Linear(dim, dim) ; SiLU -> Linear(dim, n * dim)
  const bf16 *w1 = nullptr, *w2 = nullptr, *wl = nullptr;
  const float *b1 = nullptr, *b2 = nullptr, *bl = nullptr;
  int dim = 0, n = 0;
};

struct AttnWeights {
  // [inner, cdim] (wo: [qdim, inner]).  Video attn1: wq is the packed q|k|v [3D, D] and wv its v rows; wk is unused.  With
  // affine codes wq holds only the q|k rows [2D, D] and wv the v rows as a matrix of their own.
  LinearW wq, wk, wv, wo;
  const float *bq = nullptr, *bk = nullptr, *bv = nullptr, *bo = nullptr;
  const float *q_norm = nullptr, *k_norm = nullptr;
};

struct BlockWeights {
  const float* sst = nullptr;  // scale_shift_table [6, D]
  AttnWeights a1, a2;
  LinearW w_in, w_out;
  const float *b_in = nullptr, *b_out = nullptr;
};

struct TextCache {  // caption projection + per-block cross-attention K / V^T (step-invariant, SURVEY H11)
  uint64_t key = 0;
  uint64_t fingerprint = 0;   // host-buffer entry points: sampled hash of the embedding + mask the entry was built from (0 = not recorded)
  int B = 0, S = 0;
  int64_t ldv = 0;
  DevBuf k;    // [L][B*S, D] bf16
  DevBuf vt;   // [L][D, ldv] bf16
  DevBuf bias; // [B, S] fp32 additive key bias (or unused when no mask)
  bool has_bias = false;
};

// what dit_prepare_text needs to build a stream's text cache: caption projection + per-block cross-attention K / V weights
struct TextProjW {
  LinearW w_c1, w_c2;
  const float *b_c1 = nullptr, *b_c2 = nullptr;
  int D = 0;
  const void* user = nullptr;
  const AttnWeights& (*layer)(const void* user, int i) = nullptr;
};

struct ConvW {
  const bf16* w = nullptr;  // [27][Cout][Cin]
  const float* b = nullptr;
  int cin = 0, cout = 0;
  int taps = 27;            // 27: 3x3x3 ; 9: per-frame 3x3 (upscaler Conv2d)
};
struct VaeResBlock {
  ConvW c1, c2;
  const float* sst = nullptr;  // [4, C] rows shift1, scale1, shift2, scale2
};
struct VaeTimeEmb {   // VAETimestepEmbedder (V/VideoDecoder.swift:37-52): Linear(256,256) -> SiLU -> Linear(256, out)
  const bf16 *w1 = nullptr, *w2 = nullptr;
  const float *b1 = nullptr, *b2 = nullptr;
  int out = 0;
};
struct VaeWeights {
  bool ready = false;
  bool has_time = false;                // timestep-conditioning weights are present
  float ts_mult = 1000.0f;              // timestep_scale_multiplier
  VaeTimeEmb stage_te[4], last_te;
  const float *mean = nullptr, *std = nullptr;
  ConvW conv_in, conv_out;
  std::vector<std::vector<VaeResBlock>> stages;  // 4 stages x blocks_per_stage
  std::vector<ConvW> ups;                        // 3 depth-to-space convs
  const float* last_sst = nullptr;               // [2, C_last] rows shift, scale
};

// dual audio / video model (T/LTX2Transformer.swift, T/LTX2TransformerBlock.swift): the audio stream, the learned norms and the
// cross-modal attentions on top of the video weights held in ltx_ctx::blocks
struct AvBlockW {
  const float *norm1 = nullptr, *norm2 = nullptr, *norm3 = nullptr, *a2v_norm = nullptr;        // video, [D]
  const float *anorm1 = nullptr, *anorm2 = nullptr, *anorm3 = nullptr, *v2a_norm = nullptr;     // audio, [Da]
  AttnWeights aa1, aa2, a2v, v2a;   // audio self / audio text-cross / audio->video / video->audio
  LinearW w_in, w_out;
  const float *b_in = nullptr, *b_out = nullptr;
  const float *asst = nullptr;      // audio_scale_shift_table [6, Da]
  const float *sst_ca_v = nullptr;  // scale_shift_table_a2v_ca_video [5, D]
  const float *sst_ca_a = nullptr;  // scale_shift_table_a2v_ca_audio [5, Da]
};
struct AvWeights {
  bool ready = false;
  int Da = 0, Ha = 0, hd = 0, Cin = 0;
  LinearW w_patch, w_c1, w_c2, w_out;
  const float *b_patch = nullptr, *b_c1 = nullptr, *b_c2 = nullptr, *b_out = nullptr, *sst_out = nullptr;
  AdaLnW ada_a, cv_ss, cv_g, ca_ss, ca_g;
  std::vector<AvBlockW> blocks;
  TextCache text[2];
  int text_rr = 0;
  DevBuf ws;                             // audio / cross-modal activations
  DevBuf a_cos, a_sin, xv_cos, xv_sin;   // 1-D RoPE tables: audio frames [Ta, Da/2], video frames' temporal coordinate [N, Da/2]
  int rope_ta = 0, rope_f = 0, rope_hw = 0;
};

// VAE encoder (V/VideoEncoder.swift:211-268): conv_in 48 -> base, 4 down blocks (res blocks + space-to-depth conv), mid block, conv_out
struct EncResBlock { ConvW c1, c2; };
struct EncStage {
  std::vector<EncResBlock> res;
  ConvW down;       // base_i -> cout / (ft*fh*fw)
  int cout = 0;     // channels after space-to-depth
};
struct EncWeights {
  bool ready = false;
  int base = 0;
  ConvW conv_in, conv_out;
  EncStage stage[4];
  std::vector<EncResBlock> mid;
};
// latent upscaler (Models/Upscaler/SpatialUpscaler.swift:167-258)
struct GnW { const float *w = nullptr, *b = nullptr; };
struct UpsBlock { ConvW c1, c2; GnW n1, n2; };
struct UpsWeights {
  bool ready = false;
  int mid = 0, cin = 0;
  ConvW initial, up2d, final_conv;
  GnW initial_norm;
  std::vector<UpsBlock> pre, post;
};

}  // namespace ltx

namespace ltx {
struct DistState {
  // ---- Ulysses over peer memory (dist.cu: dist_p2p_*): every sp rank's receive buffer is mapped into its peers through
  // CUDA IPC, producers store straight into it over NVLink, a flag barrier replaces the NCCL all-to-all
  bool p2p_tried = false, p2p = false;
  void* p2p_local = nullptr;          // this rank's exported allocation: [recv bytes | flags]
  size_t p2p_bytes = 0;               // recv capacity (bytes) of every rank's allocation
  void* p2p_peer[8] = {};             // base of rank r's allocation in this process (own pointer for r == sp_rank)
  bool p2p_ipc[8] = {};               // mapped through CUDA IPC (another process) rather than a same-process pointer
  void* p2p_pool = nullptr;           // cudaMemPool_t the local buffer comes from when every sp rank lives in this process
                                      // barrier generations (0 = q/k/v landed, 1 = attention output landed) are counted on the
                                      // device, next to the flags, so that a captured step replays with fresh epochs
  void* comm_world = nullptr;  // ncclComm_t
  void* comm_sp = nullptr;     // sequence-parallel sub-communicator (== world when pass_groups == 1)
  bool sp_is_world = true;
  int rank = 0, world = 1, sp = 1, groups = 1, group = 0, sp_rank = 0;
};
// One captured denoise step / forward (api.cu: run_graphed).  state 0: seen once (ran eagerly, buffers are sized), 1: captured.
struct StepGraph {
  int state = 0;
  cudaGraphExec_t exec = nullptr;
  uint64_t launches = 0;     // kernel launches one replay stands for
  uint64_t generation = 0;   // devbuf_generation() at capture
  uint64_t last_use = 0;
};
enum ProfClass { PROF_GEMM = 0, PROF_ATTN = 1, PROF_ROW = 2, PROF_CONV = 3, PROF_PREP = 4, PROF_OTHER = 5, PROF_COMM = 6, PROF_NCLASS = 8 };
struct ProfRec {
  cudaEvent_t a, b;
  int cls;
  double flops, bytes;
};
}  // namespace ltx

struct ltx_ctx {
  ltx_config cfg;
  ltx::DistState dist;
  // ---- optional per-kernel-class timing (CUDA events on the context stream around every launch)
  bool prof_on = false;
  std::vector<ltx::ProfRec> prof_recs;
  std::vector<cudaEvent_t> prof_pool;

  // ---- captured step graphs (keyed by everything that shapes the launch sequence; see run_graphed in api.cu)
  std::map<std::string, ltx::StepGraph> graphs;
  uint64_t graph_clock = 0, graph_replays = 0, graph_captures = 0;
  int graphs_enabled = 1;

  int device = 0;
  cudaStream_t stream = nullptr;
  mutable std::string last_error;
  uint64_t launches = 0;

  std::map<std::string, ltx::DevTensor> tensors;  // raw tensors by post-mapping key
  int quant_bits = 16;
  int quant_materialise = 0;                      // 1: dequantised bf16 values replace the weights at finalize (ltx_set_quant_storage)
  ltx::DevBuf q_panel;                            // bf16 conversion panel of the large-M quantised GEMM path
  ltx::DevBuf gemm_ws;                            // split-K workspace of the weight-streaming GEMM: [counters 64 KB | fp32 partials]
  std::vector<void*> owned;                       // packed allocations made by finalize
  bool dit_ready = false;
  std::vector<ltx::BlockWeights> blocks;
  ltx::LinearW w_patch, w_c1, w_c2, w_out;
  const float *b_patch = nullptr, *b_c1 = nullptr, *b_c2 = nullptr, *b_out = nullptr, *sst_out = nullptr;
  ltx::AdaLnW adaln;   // timestep embedder + AdaLN-single (bf16 weights in every format)
  ltx::VaeWeights vae;
  ltx::AvWeights av;
  ltx::EncWeights enc;
  ltx::UpsWeights ups;

  // ---- DiT workspaces (grow-only)
  ltx::DevBuf lat_in, ctx_in, ts_in, mask_in;      // staged inputs
  ltx::DevBuf api_lat, api_ctx;                    // host-API upload buffers
  ltx::DevBuf x, xb, h, qk, vt, att, q2, ffh, vel;  // activations
  ltx::DevBuf se, t1, emb, ada;                     // timestep path
  ltx::DevBuf c1, c2;                               // caption projection
  ltx::DevBuf rope_cos, rope_sin;
  int rope_f = 0, rope_h = 0, rope_w = 0;
  ltx::TextCache text[2];
  int text_rr = 0;
  ltx::DevBuf scratch;  // small fp64 scratch for reductions
  ltx::DevBuf sp_send, sp_recv, sp_vt, sp_vel;  // Ulysses exchange buffers
  ltx::DevBuf snap_x;                           // residual-stream snapshot for the shared STG prefix
  int snap_rows = 0;

  // ---- fp32 mode (dit_f32.cu): fp32 weights + activations, split-bf16 GEMM operands
  int precision = 16;   // 16: bf16 weights (default), 32: DiT matrices stay fp32 and the forward runs in fp32 mode,
                        // 8: the block Linears run as e4m3 x e4m3 GEMMs (weights converted at finalize, dit_convert_fp8)
  ltx::DevBuf fp8_act;  // mode 8: e4m3 codes + row scales of the current GEMM's A operand
  ltx::DevBuf f_asplit, f_wsplit, f_h, f_q, f_k, f_v, f_att, f_ffh, f_ctx, f_c1, f_c2, f_tk, f_tv, f_lat, f_bias;

  // ---- resident denoise session
  ltx::DevBuf s_latent, s_tok, s_vc, s_vu, s_vs, s_vprev, s_ctx_pos, s_ctx_neg, s_mask_pos, s_mask_neg, s_sigma, s_ts;
  ltx::DevBuf s_ctx_pair, s_mask_pair;   // [2, S, Cc] / [2, S]: positive | negative prompt, for the batched guidance forward
  int s_F = 0, s_H = 0, s_W = 0, s_S = 0;
  bool s_has_neg = false, s_has_mask_pos = false, s_has_mask_neg = false;
  int s_ctx_dtype = LTX_BF16;
  uint64_t s_serial = 0;
  // audio + video session (ltx_av_denoise_*): audio latent / velocities [Ta, Ca] fp32, audio contexts
  ltx::DevBuf s_alat, s_avc, s_avu, s_actx_pos, s_actx_neg;
  ltx::DevBuf s_alat_pair, s_actx_pair;   // [2, Ta, Ca] / [2, S, Cc]: inputs of the batched guidance forward
  int s_Ta = 0;

  // ---- VAE workspaces
  ltx::DevBuf v_a, v_b, v_h, v_pad, v_lat, v_noise, v_frames, v_mix, v_te, v_split, v_pad2;
  ltx::DevBuf v_tile_lat, v_tile_noise, v_tile_frames;   // temporally tiled decode: one gathered chunk and its frames
  ltx::DevBuf v_frames_f32;   // fp32 frames before the 8-bit conversion (tiled u8 decode, host-buffer ltx_frames_to_u8)
  int vae_no_clip = 0;                                    // conv_out stores (x+1)/2 unclipped (tiles are clipped after blending)
  ltx::DevBuf av_in[8];   // host-API staging of the dual model's inputs / outputs
  ltx::DevBuf u_part, u_ab, u_stats, u_in, u_out, u_ref;   // encoder / upscaler / AdaIN scratch and host-API staging
};

namespace ltx {
// split-K workspace of the swap-AB GEMM (gemm_swapab.cu), one per context = per stream: 16 K zeroed arrival counters followed by
// 40 MB of fp32 partial tiles (74 CTA pairs x 256 x 512 x 4 B is the most a launch can use)
void gemm_attach_workspace(ltx_ctx* c, GemmEpi& e);
// RAII scope: times the launches issued inside it when profiling is on, and counts them.
struct ProfScope {
  ltx_ctx* c;
  ProfRec r;
  bool on;
  ProfScope(ltx_ctx* ctx, int cls, double flops, double bytes, int launches = 1) : c(ctx), on(ctx->prof_on) {
    c->launches += launches;
    if (!on) return;
    auto get = [&]() {
      cudaEvent_t e;
      if (!c->prof_pool.empty()) { e = c->prof_pool.back(); c->prof_pool.pop_back(); }
      else LTX_CUDA(cudaEventCreate(&e));
      return e;
    };
    r.a = get(); r.b = get(); r.cls = cls; r.flops = flops; r.bytes = bytes;
    LTX_CUDA(cudaEventRecord(r.a, c->stream));
  }
  ~ProfScope() {
    if (!on) return;
    cudaEventRecord(r.b, c->stream);
    c->prof_recs.push_back(r);
  }
};
// api.cu: drop every captured graph (weights, communicators or precision changed)
void graphs_clear(ltx_ctx* c);
// dit.cu: the transformer Linears.  What a caller's rows imply for the bf16 kernels:
struct LinearOpts {
  int allow_skinny = 0;          // products of up to this many rows may take the weight-streaming kernel (launch_gemm)
  bool split_k = false;          // M <= 512: opt in to the swap-AB kernel by giving it the context's split-K workspace
  int tile_n = 0;                // bf16 / e4m3: forced tile width, 0: fitted (bf16: pair kernel for M > 128; e4m3: always pairs)
  int a_kblock = 0;              // K-blocked A operand (Ulysses receive layout, see launch_gemm); not for e4m3 codes
  int64_t a_kblock_stride = 0;
};
// epi(A[M, K] W[:N]^T): the only place that launches a transformer Linear.  Picks the kernels from W.fmt (e4m3: row quantiser +
// FP8 pair kernel; affine: dequant-fused or panel kernel; bf16: launch_gemm with `o`) and profiles them.  N <= W.n: the first
// N rows of the weight (the q|k rows of a packed q|k|v).
void linear(ltx_ctx* c, const bf16* A, int64_t lda, const LinearW& W, int M, int N, int K, const GemmEpi& e, const LinearOpts& o);
// V^T = (A W^T + bias)^T for `items` batch items of `rows` rows each (A [items * rows, W.k], pitch W.k): item i's [W.n, rows]
// block starts at column i * item_ld of `out` (row pitch ld_out).  bf16: the weight-streaming kernel stores V^T directly when
// o.allow_skinny admits the rows, otherwise the weight is the A operand so the product lands transposed; codes must be the B
// operand: project into tmp [items * rows, W.n], then transpose each item.
void linear_vt(ltx_ctx* c, const bf16* A, int rows, int items, const LinearW& W, const float* bias, bf16* out, int64_t ld_out,
               int64_t item_ld, bf16* tmp, const LinearOpts& o);
// Q [B*Nq, ldq], K [B*Nk, ldk], V^T [D, B*ldv] (item b at column b * ldv), key bias [B, Nk]; head_dim D / H
void attention(ltx_ctx* c, const bf16* Q, int64_t ldq, const bf16* K, int64_t ldk, const bf16* Vt, int64_t ldv, const float* bias,
               bf16* O, int64_t ldo, int B, int H, int Nq, int Nk, int D, const PeerTable* o_blocks = nullptr,
               int rows_per_block = 0);
// AdaLayerNormSingle (T/LTXTimestepEmbedding.swift:96-124) for one sigma per batch item (B rows): emb = L2(silu(L1(se))),
// lin = L(silu(emb)), row pitches dim and n * dim.  se = sincos(sigma * mult) is shared by every embedder of the same stream;
// given `sigma`, it is computed into se first.
void adaln_single(ltx_ctx* c, const AdaLnW& a, float* se, float* t1, float* emb, float* lin, int B, const float* sigma = nullptr,
                  float mult = 0.f);
// The same for R sigmas (one per token): the three Linears as tensor-core GEMMs over the R rows, bf16 operands, the SiLUs in
// the first epilogue / a cast pass.  se_bf [R, 256] bf16; t1_bf [R, dim] bf16 scratch; emb [R, dim] fp32; lin [R, n * dim]
// fp32 with row pitch ld_lin.
void adaln_single_rows(ltx_ctx* c, const AdaLnW& a, const bf16* se_bf, int R, bf16* t1_bf, float* emb, float* lin, int64_t ld_lin,
                       const LinearOpts& o);
// finalize helpers: shape-checked weights by key
const bf16* wbf(ltx_ctx* c, const std::string& k, int64_t r, int64_t cc);
const float* wf(ltx_ctx* c, const std::string& k, int64_t n);
LinearW wlin(ltx_ctx* c, const std::string& k, int64_t n, int64_t kk);
AdaLnW adaln_w(ltx_ctx* c, const std::string& p, int64_t dim, int n);
void dit_finalize(ltx_ctx* c);
void dit_quantize(ltx_ctx* c, int bits);
void dit_convert_fp8(ltx_ctx* c);
// snapshot_block >= 0: save the residual stream at the entry of that block (for a later resume);
// resume_block >= 0: skip the embedding and blocks [0, resume_block) and continue from the saved stream (SURVEY H10:
// the STG-perturbed pass shares every block before the first perturbed one with the conditional pass).
void dit_forward_dev(ltx_ctx* c, const void* latent, int latent_dtype, const void* context, int context_dtype,
                     const float* timesteps_dev, int ts_per_token, const int32_t* mask_dev, int B, int N, int S, int F,
                     int H, int W, const ltx_dit_flags* flags, float* out_velocity_dev, int snapshot_block = -1,
                     int resume_block = -1);
void dit_clear_caches(ltx_ctx* c);
TextCache& dit_prepare_text(ltx_ctx* c, TextCache* slots, int* rr, const TextProjW& src, const void* context, int context_dtype,
                            const int32_t* mask_dev, int B, int S, uint64_t key);
void dit_build_rope(ltx_ctx* c, int F, int H, int W);
// dit_av.cu: dual audio / video model (LTX2Transformer)
void dit_av_finalize(ltx_ctx* c);
void dit_av_forward_dev(ltx_ctx* c, const void* v_latent, int v_dtype, const void* a_latent, int a_dtype, const void* v_context,
                        const void* a_context, int ctx_dtype, const float* v_ts_dev, int v_ts_per_token, const float* a_ts_dev,
                        const int32_t* v_mask_dev, const int32_t* a_mask_dev, int B, int N, int Ta, int S, int F, int H, int W, uint64_t context_key,
                        float* out_v_dev, float* out_a_dev);
// dit_f32.cu
void dit_finalize_f32(ltx_ctx* c);
void dit_forward_f32(ltx_ctx* c, const void* latent, int latent_dtype, const void* context, int context_dtype,
                     const float* timesteps_dev, int ts_per_token, const int32_t* mask_dev, int B, int N, int S, int F, int H,
                     int W, const ltx_dit_flags* flags, float* out_velocity_dev);
// vae.cu
void vae_finalize(ltx_ctx* c);
int vae_tiled_frames(int Fp, int tile_size, int overlap);
// Output formats of the decode: FRAMES_F32 = fp32 [F, H, W, 3] in [0, 1]; otherwise LTX_FRAMES_RGB8 / LTX_FRAMES_I420.
constexpr int FRAMES_F32 = 0;
// bytes of F frames of H x W in an 8-bit format; 0 for a bad format or size (I420: H and W even)
size_t frames_u8_bytes(int64_t F, int64_t H, int64_t W, int format);
// fp32 frames [F, H, W, 3] (clipped to [0, 1] on the way) -> 8-bit frames; the arithmetic of the fused conv_out store
void frames_to_u8_dev(ltx_ctx* c, const float* frames_dev, int F, int H, int W, int format, uint8_t* out_dev);
// returns the number of frames written
int vae_decode_tiled_dev(ltx_ctx* c, const float* latent_dev, int Fp, int Hp, int Wp, float timestep, const float* noise_dev,
                         int causal, int tile_size, int tile_overlap, void* frames_dev, int format = FRAMES_F32);
void vae_decode_dev(ltx_ctx* c, const float* latent_dev, int Fp, int Hp, int Wp, float timestep, const float* noise_dev,
                    int causal, void* frames_dev, int format = FRAMES_F32);
ConvW vae_pack_conv_keys(ltx_ctx* c, const std::string& wkey, const std::string& bkey, int64_t cout, int64_t cin,
                         int64_t cout_use, int taps);
const float* vae_vec(ltx_ctx* c, const std::string& key, int64_t n);
// out: fp32, or the 8-bit frames of epilogue modes CONV_EPI_RGB8 / CONV_EPI_I420
void vae_conv(ltx_ctx* c, const float* x, int prep_mode, const float* a, const float* b, const ConvW& w, int T, int H, int W,
              int pad, int epi_mode, void* out, const float* resid, int n_active = 1, int t_shift = 0);
// vae_extra.cu: VAE encoder (V/VideoEncoder.swift), latent upscaler (Models/Upscaler/SpatialUpscaler.swift), AdaIN, re-noise
void vae_encoder_finalize(ltx_ctx* c);
void vae_encode_dev(ltx_ctx* c, const float* pixels_dev, int T, int H, int W, int normalize, float* latent_dev);
void upscaler_finalize(ltx_ctx* c);
void upscale_latent_dev(ltx_ctx* c, const float* latent_dev, int F, int H, int W, float* out_dev);
void adain_filter_dev(ltx_ctx* c, float* latent_dev, int64_t n_per_channel, const float* ref_dev, int64_t n_ref_per_channel,
                      int C, float factor);
void renoise_dev(ltx_ctx* c, float* latent_dev, const float* noise_dev, int64_t n, float noise_scale);
// dist.cu
void dist_get_unique_id(void* out128);
void dist_init(ltx_ctx* c, const void* unique_id, int rank, int world_size, int sp_size, int pass_groups);
void dist_init_local(ltx_ctx** contexts, int n, int sp_size, int pass_groups);
void dist_destroy(ltx_ctx* c);
void dist_broadcast(ltx_ctx* c, void* buf, size_t bytes, int root_world_rank);
void dist_allgather_sp(ltx_ctx* c, const void* send, void* recv, size_t bytes_per_rank);
void dist_all_to_all_sp(ltx_ctx* c, const void* const* send, void* const* recv, int n_tensors, size_t bytes_per_peer);
// peer-memory Ulysses: (re)registers a receive buffer of >= bytes on every sp rank (collective); false = unavailable
bool dist_p2p_ensure(ltx_ctx* c, size_t bytes);
// all sp ranks: 'my stores of this phase have been issued' + wait for everyone's (kind 0: q/k/v, 1: attention output)
void dist_p2p_barrier(ltx_ctx* c, int kind);
void dist_halo_exchange(ltx_ctx* c, const void* send_prev, void* recv_prev, const void* send_next, void* recv_next,
                        size_t bytes, int n_active);
// safetensors.cu
std::string map_transformer_key(const std::string& file_key, bool include_audio = false);
std::string map_vae_key(const std::string& file_key);
std::string map_vae_encoder_key(const std::string& file_key);
std::string map_upscaler_key(const std::string& file_key);
int load_safetensors(ltx_ctx* c, const char* path, int which);
// weights.cu
const DevTensor& get_tensor(ltx_ctx* c, const std::string& key);
void load_tensor_host(ltx_ctx* c, const std::string& key, const void* host, int dtype, const int64_t* shape, int ndim);
// A transformer Linear [N, K] from e4m3 codes and fp32 scales (n_scales: 1 = per tensor, N = per output channel; validated by the
// caller).  FP8 mode with keep_codes keeps the codes of the block Linears dit_convert_fp8 would convert (DT_E4M3); every other
// case decodes to the storage dtype of the mode.  NaN codes: LTX_ERR_WEIGHTS, and the tensor is not left in the context.
void load_tensor_e4m3_host(ltx_ctx* c, const std::string& key, const uint8_t* codes, const float* scales, int64_t n_scales,
                           const int64_t* shape, bool keep_codes);
// A DT_E4M3 tensor's codes decoded to bf16 storage in place (ltx_fuse_lora merges into the decoded values)
void decode_e4m3_tensor(ltx_ctx* c, DevTensor& t);
void init_random_weights(ltx_ctx* c, int which, uint64_t seed);
void fuse_lora(ltx_ctx* c, const std::string& key, const void* down_host, const void* up_host, int dtype, int rank, float scale);
std::string map_lora_key(const std::string& lora_key);
}  // namespace ltx
