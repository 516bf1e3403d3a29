// Internal declarations shared by the libltxcuda translation units (not part of the C ABI).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <stdexcept>
#include <string>

namespace ltx {

typedef __nv_bfloat16 bf16;

struct LtxError : public std::runtime_error {
  int code;
  LtxError(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define LTX_CHECK(cond, code, msg)                                                                  \
  do {                                                                                              \
    if (!(cond)) throw ::ltx::LtxError((code), std::string(msg) + " [" #cond "] at " __FILE__ ":" + \
                                                   std::to_string(__LINE__));                       \
  } while (0)
#define LTX_CUDA(expr)                                                                                       \
  do {                                                                                                       \
    cudaError_t _e = (expr);                                                                                 \
    if (_e != cudaSuccess)                                                                                   \
      throw ::ltx::LtxError(3, std::string("CUDA error: ") + cudaGetErrorString(_e) + " in " #expr " at " + \
                                   __FILE__ ":" + std::to_string(__LINE__));                                 \
  } while (0)

// ---------------------------------------------------------------- kernel launch with programmatic stream serialization
// The kernel must call griddep_wait() (ptx.cuh) before touching dependent global memory.  LTX_PDL=0 launches normally.
bool pdl_enabled(int cls = 0);   // cls: 0 GEMM, 1 row kernels, 2 attention, 3 VAE (LTX_PDL_MASK bit per class, debugging)
enum { PDL_GEMM = 0, PDL_ROWS = 1, PDL_ATTN = 2, PDL_VAE = 3 };
template <typename... KArgs, typename... Args>
inline void launch_pdl(int cls, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled(cls) ? 1 : 0;
  LTX_CUDA(cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...));
}

// ---------------------------------------------------------------- TMA descriptors (tmap.cu)
// 2-D row-major bf16 matrix [rows, cols] with row pitch `ld` elements; box = [box_rows, 64 cols], 128B swizzle.
CUtensorMap make_tmap_2d(const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                         uint32_t box_cols = 64);
// 4-D channels-last bf16 volume [T, H, W, C] (C fastest); box = [bt, bh, bw, 64 channels], 128B swizzle.
CUtensorMap make_tmap_thwc(const void* base, uint64_t T, uint64_t H, uint64_t W, uint64_t C, uint32_t bt, uint32_t bh,
                           uint32_t bw);
// 3-D bf16 tensor (d0 fastest); strides in elements; box = [box0 (64), box1, 1].
CUtensorMap make_tmap_3d(const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1, uint64_t stride2,
                         uint32_t box0, uint32_t box1);
int device_sm_count();   // of the calling thread's current device (cached per device)
// opt a kernel in to `bytes` of dynamic shared memory on the current device, once per (kernel, device); thread-safe
void ensure_dyn_smem(const void* kernel, size_t bytes);
template <typename K>
inline void ensure_dyn_smem(K* kernel, size_t bytes) { ensure_dyn_smem(reinterpret_cast<const void*>(kernel), bytes); }

// ---------------------------------------------------------------- GEMM (gemm.cu)
enum EpiMode : int {
  EPI_BF16 = 0,        // out_bf16[m,n] = acc + bias
  EPI_GELU_BF16 = 1,   // out_bf16[m,n] = gelu_tanh(acc + bias)
  EPI_GATE_RESID = 2,  // resid[m,n] += (acc + bias) * gate * scale ; optional bf16 shadow of the new resid
  EPI_F32 = 3,         // out_f32[m,n] = acc + bias
  EPI_SILU_BF16 = 4,   // out_bf16[m,n] = silu(acc + bias)
};

// up to 8 destination base pointers (own memory or NVLink-mapped peer memory), indexed by destination rank
constexpr int LTX_MAX_PEERS = 8;
struct PeerTable {
  void* p[LTX_MAX_PEERS];
};

struct GemmEpi {
  int mode = EPI_BF16;
  void* out = nullptr;  // bf16 or f32, row pitch ldo (elements)
  int64_t ldo = 0;
  const float* bias = nullptr;  // [N], or [M] when bias_per_row
  int bias_per_row = 0;
  float* resid = nullptr;  // EPI_GATE_RESID: fp32 [M, ldr]
  int64_t ldr = 0;
  const float* gate_a = nullptr;  // gate = gate_a[(m / rows_per_gate) * gate_ld + n] + gate_b[n]; nullptr -> gate = 1
  const float* gate_b = nullptr;
  int64_t gate_ld = 0;
  int rows_per_gate = 1;
  bf16* shadow = nullptr;  // optional bf16 copy of the updated residual, row pitch lds
  int64_t lds = 0;
  float scale = 1.0f;
  // bf16 outputs only: column-blocked destination (Ulysses send layout): element (m, n) goes to
  // out[(n / col_block) * col_block_stride + m * ldo + n % col_block]; col_block = 0 -> plain row-major.
  int col_block = 0;
  int64_t col_block_stride = 0;
  // column-blocked destination with one base pointer per block (Ulysses over peer memory: block d is written straight into
  // rank d's receive buffer through NVLink): element (m, n) goes to col_ptrs.p[n / col_block][m * ldo + n % col_block]
  int use_col_ptrs = 0;
  PeerTable col_ptrs = {};
  // col_block_from > 0: only columns n >= col_block_from are column-blocked (block index (n - col_block_from) / col_block, base
  // blocked_out -- or col_ptrs -- and row pitch blocked_ld); the columns before it go row-major to `out` / ldo.  Lets the
  // sequence-parallel path run q | k | v as ONE projection: q | k stay local, the v columns leave for their destination ranks.
  // col_block_from % 32 == 0.
  int col_block_from = 0;
  void* blocked_out = nullptr;   // nullptr -> out
  int64_t blocked_ld = 0;        // 0 -> ldo
  // EPI_BF16 only: columns n >= tsplit_col are stored TRANSPOSED: element (m, n) -> out_t[(n - tsplit_col) * ldt + m].
  // Used by the fused q|k|v projection: q|k land row-major in `out`, V lands as V^T (K-major for the PV MMA).  Needs
  // tsplit_col % 32 == 0, a tile width that is a multiple of 32, ldt % 8 == 0.  0 = off.
  int tsplit_col = 0;
  bf16* out_t = nullptr;
  int64_t ldt = 0;
  // weight-streaming kernel only (gemm_skinny.cu), EPI_BF16: element (m, n) is stored at out[n * ldo + m] -- V^T for the PV MMA
  int transpose_out = 0;
  // with transpose_out, a batch of items (64-row form): row m of item m / t_item_rows lands in column
  // (m / t_item_rows) * t_item_ld + m % t_item_rows, so each item's V^T block starts at a padded column.  0 = off.
  int t_item_rows = 0;
  int64_t t_item_ld = 0;
  // Optional split-K workspace of the weight-streaming kernel for M <= 512 (gemm_swapab.cu): fp32 partial tiles + one zeroed
  // arrival counter per (weight tile, CTA).  Owned by the caller's context (one per stream); giving it is also the opt-in to
  // that kernel -- its summation order differs from the tile kernels' when K is split.
  float* ws = nullptr;
  size_t ws_bytes = 0;
  unsigned int* ws_counters = nullptr;
  size_t ws_counter_count = 0;
};

// C[M,N] = A[M,K] * B[N,K]^T ; A, B bf16 K-major (row pitch lda / ldb elements, multiples of 8).
// a_kblock > 0: A is K-blocked (Ulysses receive layout): element (m, k) lives at A[(k / a_kblock) * a_kblock_stride +
// m * lda + k % a_kblock] (a_kblock % 64 == 0, lda = a_kblock).
// allow_skinny: problems of up to that many rows may take the weight-streaming kernel (gemm_skinny.cu) -- opt-in, because its
// summation order differs from the tile kernels' and the sequence-parallel path promises results bit-identical to one GPU.
// 0: never; 32; 64 only for a batch of two items of <= 32 rows each, whose one-item calls take the kernel too.
void launch_gemm(const bf16* A, int64_t lda, const bf16* B, int64_t ldb, int M, int N, int K, const GemmEpi& epi,
                 cudaStream_t stream, int force_bn = 0, int a_kblock = 0, int64_t a_kblock_stride = 0, int allow_skinny = 0);
// weight-streaming Linear for M <= max_rows (32 or 64, gemm_skinny.cu): HBM-bound, mma.sync on 16-byte coalesced weight rows
bool gemm_skinny_eligible(int64_t lda, int64_t ldb, int M, int N, int K, const GemmEpi& epi, int a_kblock, int max_rows = 32);
void launch_gemm_skinny(const bf16* A, int64_t lda, const bf16* W, int64_t ldb, int M, int N, int K, const GemmEpi& epi,
                        cudaStream_t stream);
int gemm_fit_tile_width(int M, int N);
// weight-streaming kernel for M <= 512 (gemm_swapab.cu): the weight tile rides the TMEM lanes, the activation rows are the MMA's
// N dimension; split-K with a deterministic last-arriver reduction when epi.ws is given.  Same contract as launch_gemm.
bool gemm_swapab_eligible(int64_t lda, int64_t ldb, int M, int N, int K, const GemmEpi& epi);
void launch_gemm_swapab(const bf16* A, int64_t lda, const bf16* W, int64_t ldb, int M, int N, int K, const GemmEpi& epi,
                        cudaStream_t stream, int a_kblock = 0, int64_t a_kblock_stride = 0);
// 2-CTA (cta_group::2) pair kernel, same contract as launch_gemm (gemm2.cu)
void launch_gemm_2cta(const bf16* A, int64_t lda, const bf16* B, int64_t ldb, int M, int N, int K, const GemmEpi& epi,
                      cudaStream_t stream, int force_bn, int a_kblock, int64_t a_kblock_stride);
int gemm2_fit_tile_width(int M, int N);
// FP8 form of the pair kernel: C[M,N] = (A[M,K] * B[N,K]^T) * sa[m] * sb[n] (fp32, in that order) + the epilogue of `epi`.
// A, B: e4m3 codes, K-major, row pitch lda / ldb bytes (multiples of 16; K % 16 == 0, the K tail is zero-filled by TMA);
// sa [M], sb [N] fp32 row scales.  force_bn: 0 = gemm2_fit_tile_width, else a multiple of 16 in [64, 256].
void launch_gemm_fp8(const uint8_t* A, int64_t lda, const float* sa, const uint8_t* B, int64_t ldb, const float* sb, int M, int N,
                     int K, const GemmEpi& epi, cudaStream_t stream, int force_bn = 0);
// Per-row e4m3 quantiser (gemm_q.cu): s[m] = 2^ceil(log2(amax_m / 448)) (1 for a zero row), q[m,k] = e4m3_rn_satfinite(x / s).
// x bf16 [M, K] with row pitch ld (elements, multiple of 8; K % 16 == 0); q [M, K] (pitch K), s [M].
void launch_quantize_rows_fp8(const bf16* x, int64_t ld, int M, int K, uint8_t* q, float* s, cudaStream_t stream);
// ---------------------------------------------------------------- quantised weights (gemm_q.cu)
// affine codes (launch_gemm_q) or e4m3 codes (launch_gemm_fp8); which one is the LinearW's format (ctx.h)
struct QuantW {
  const uint8_t* q = nullptr;    // [N, K] codes (8-bit, e4m3) or [N, K/2] packed nibbles (4-bit)
  const float* scales = nullptr; // affine: [K/64, N]; e4m3: [N]
  const float* biases = nullptr; // affine: [K/64, N]; e4m3: unused
  int bits = 0, n = 0, k = 0;
  // optional bf16 [n, k] scratch panel shared by all quantised weights of a context: for M > 256 the weight is converted
  // once per GEMM into it (it stays in the 126 MB L2 for the D x D projections) and the bf16 pair kernel runs on the panel
  bf16* scratch = nullptr;
};
// C[M,N] = A[M,K] * (s*q + beta)[N,K]^T with the epilogues of launch_gemm (group size 64)
void launch_gemm_q(const bf16* A, int64_t lda, const QuantW& W, int M, int N, int K, const GemmEpi& epi, cudaStream_t stream,
                   int force_bn = 0, int a_kblock = 0, int64_t a_kblock_stride = 0);
// whether launch_gemm_q (force_bn = 0) takes an M-row product through the bf16 panel: a dequantize launch + the bf16 GEMM
bool gemm_q_uses_panel(const QuantW& W, int M);
void launch_quantize(const bf16* w, int N, int K, int bits, uint8_t* q, float* scales, float* biases, cudaStream_t s);
void launch_dequantize(const QuantW& W, bf16* w, cudaStream_t s);
// vectorised, PDL-aware conversion of the whole weight into a bf16 panel (same rounding as the fused kernels)
void launch_dequantize_panel(const QuantW& W, bf16* w, cudaStream_t s);
// uint8 matrix [rows, row_bytes], box [box_rows, box_bytes], no swizzle
CUtensorMap make_tmap_u8(const void* base, uint64_t rows, uint64_t row_bytes, uint32_t box_rows, uint32_t box_bytes);
// uint8 matrix [rows, cols] with row pitch row_bytes; box [box_rows, 128 bytes], 128-byte swizzle (the e4m3 GEMM operands)
CUtensorMap make_tmap_u8_sw128(const void* base, uint64_t rows, uint64_t cols, uint64_t row_bytes, uint32_t box_rows);
// bf16 [R, C] (row pitch ld_in) -> [C, R] (row pitch ld_out)
void launch_transpose_bf16(const bf16* in, int64_t ld_in, int R, int C, bf16* out, int64_t ld_out, cudaStream_t s);

// ---------------------------------------------------------------- attention (attention.cu)
// Q [B*Nq, D], K [B*Nk, D] bf16 (head h = columns h*128..h*128+127); Vt [D, B*ldvb] bf16 (row h*128+d, column
// b*ldvb + j, ldvb % 8 == 0); key_bias: optional fp32 [B, Nk] additive logits bias; O [B*Nq, D] bf16.
void launch_attention(const bf16* Q, int64_t ldq, const bf16* K, int64_t ldk, const bf16* Vt, int64_t ldvb,
                      const float* key_bias, bf16* O, int64_t ldo, int B, int H, int Nq, int Nk, int D, float scale,
                      cudaStream_t stream, const PeerTable* o_blocks = nullptr, int rows_per_block = 0);
// o_blocks != nullptr: output row r goes to o_blocks->p[r / rows_per_block] + (r % rows_per_block) * ldo (peer memory)

// ---------------------------------------------------------------- elementwise / row kernels (elementwise.cu)
// out_bf16[m,:] = norm(x[m,:]) * (1 + tbl_scale[n] + ada_scale[g*ada_ld + n]) + tbl_shift[n] + ada_shift[g*ada_ld + n],
// g = m / rows_per_mod; norm = weight-less RMSNorm (layernorm = 0) or affine-less LayerNorm (layernorm = 1).
void launch_rmsnorm_mod(const float* x, bf16* out, int M, int D, const float* tbl_shift, const float* tbl_scale,
                        const float* ada_shift, const float* ada_scale, int64_t ada_ld, int rows_per_mod, float eps,
                        int layernorm, cudaStream_t s);
// In place on bf16 [M, ld]: y = rms(x[:, :D]) * w, then optional split-RoPE with cos/sin [rows_per_rope, D/2] (token-major).
// w_second != nullptr: the same for the second segment x[:, D:2D] with that weight (q | k of the fused projection).
// QkOut (optional): write the result out of place in the head-blocked Ulysses send layout instead of in place:
// head h of segment g goes to out[g][(h / heads_per_block) * block_stride + row * ld + (h % heads_per_block) * 128 + d].
struct QkOut {
  bf16* out[2] = {nullptr, nullptr};
  int heads_per_block = 0;
  int64_t block_stride = 0, ld = 0;
  // use_peer: head block d of segment g goes to peer[g].p[d] + row * ld + ... instead (peer memory, no block_stride)
  int use_peer = 0;
  PeerTable peer[2] = {};
};
void launch_qknorm_rope(bf16* x, int64_t ld, int M, int D, const float* w, const float* cosb, const float* sinb,
                        int rows_per_rope, float eps, cudaStream_t s, const float* w_second = nullptr,
                        const QkOut* blocked = nullptr);
void launch_cast_f32_bf16(const float* in, bf16* out, int64_t n, cudaStream_t s);
void launch_cast_bf16_f32(const bf16* in, float* out, int64_t n, cudaStream_t s);
// y[o] = act_out( sum_i W[o,i] * act_in(x[i]) + b[o] ), bf16 W [O,I]; tiny-M path for the timestep MLP (M rows).
void launch_gemv(const bf16* W, const float* bias, const float* x, float* y, int M, int O, int I, int silu_in,
                 cudaStream_t s);
void launch_mask_to_bias(const int32_t* mask, float* bias, int n, cudaStream_t s);
void launch_scale_f32(float* x, float a, int64_t n, cudaStream_t s);
// lat += dt * (v_cond + (cfg_scale - 1) * (v_cond - v_uncond))   (v_uncond nullable: lat += dt * v_cond)
void launch_audio_cfg_euler(float* lat, const float* v_cond, const float* v_uncond, float cfg_scale, float dt, int64_t n,
                            cudaStream_t s);
void launch_sincos_embed(const float* sigma, float mult, float* out, int M, int dim, cudaStream_t s, bf16* out_bf16 = nullptr);
// out_bf16 = silu(in) (fp32 in)
void launch_silu_cast(const float* in, bf16* out, int64_t n, cudaStream_t s);
// ts[i] = (i % period) < frozen ? 0 : sigma   (per-token timesteps of the image-conditioned denoise loop)
void launch_fill_token_timesteps(float* ts, int n, int period, int frozen, const float* sigma_dev, cudaStream_t s);
// latent [C, T] (channel-major, T = F*H*W tokens) <-> tokens [T, C]
void launch_patchify(const float* latent, bf16* tok_bf16, float* tok_f32, int C, int T, cudaStream_t s);
void launch_unpatchify(const float* tok, float* latent, int C, int T, cudaStream_t s);
void launch_transpose_slice(const float* in, int64_t ld_in, int rows, int cols, float* out, cudaStream_t s);
// guidance + Euler (P/LatentUtils.swift:131-183, P/LTXPipeline.swift:920-927, S/LTXScheduler.swift:305-327)
struct GuidedEulerArgs {
  float* latent;          // in/out fp32 [n]
  const float* v_cond;    // [n]
  const float* v_uncond;  // nullable
  const float* v_stg;     // nullable
  float* v_prev;          // nullable in/out (GE momentum state)
  int use_prev;           // apply GE (step > 0)
  float* v_out;           // nullable: final velocity
  size_t n;
  float cfg, phi, stg, ge_gamma, sigma, sigma_next;
  double* scratch;  // >= 8 doubles of device scratch for the rescale reductions
  size_t period = 0, frozen = 0;  // elements with (i % period) < frozen keep their latent (frame-0 freeze of the I2V loop)
};
void launch_guided_euler(const GuidedEulerArgs& a, cudaStream_t s);
void launch_fill_normal_bf16(bf16* p, int64_t n, float std, float mean, uint64_t seed, cudaStream_t s);
void launch_fill_normal_f32(float* p, int64_t n, float std, float mean, uint64_t seed, cudaStream_t s);

// ---------------------------------------------------------------- VAE kernels (conv3d.cu)
struct ConvEpi {
  int mode;                 // 0: out_f32 = acc + bias (+ resid) ; 1: depth-to-space scatter (+ tiled d2s residual) ; 2: unpatchify+clip to frames
  float* out;               // mode 0: [T,H,W,Cout] fp32 ; mode 1: [2T-1,2H,2W,Cout/8] fp32 ; mode 2: [T,4H,4W,3] fp32
  const float* bias;        // [Cout]
  const float* resid;       // mode 0: nullable [T,H,W,Cout] ; mode 1: conv input x fp32 [T,H,W,Cin]
  int Cin;
  int t_shift = 0;          // mode 1: output frame = 2t + p1 - 1 + t_shift (1 on temporal shards other than the first,
                            // which keep the frame the first shard trims; frames < 0 are dropped)
  // mode 3 (Cout <= tile width): the epilogue is the NEXT conv's padding prologue -- pixel-norm over the voxel's Cout channels
  // of (acc + bias), * (1 + next_scale) + next_shift, SiLU, bf16, stored into the interior of the next conv's padded volume
  // [T+2, H+2, W+2, Cout] (frame offset next_tshift: 1, or 2 when causal); launch_vae_halo_fill completes the padding.
  // The fp32 tensor is never written (VAEResBlock3d conv1 -> conv2, V/VideoDecoder.swift:118-127).
  // mode 4: the same hand-over from conv2 to the NEXT res block's conv1: out = acc + bias + resid is stored as fp32 (the residual
  // stream) and its normalised / modulated / activated bf16 copy goes into next_pad.
  bf16* next_pad = nullptr;
  const float* next_scale = nullptr;
  const float* next_shift = nullptr;
  int next_tshift = 1;
  int no_clip = 0;          // mode 2: store (x+1)/2 unclipped (temporal tiles are blended before the clip)
};
// x_pad: bf16 [T+2, H+2, W+2, Cin] (already padded), w: bf16 [ntaps][Cout][Cin]; 3x3x3 cross-correlation (ntaps = 27) or a
// per-frame 3x3 one (ntaps = 9: only the dt = 1 taps, the upscaler's Conv2d).
bool conv3d_wants_tap_split(int H, int W, int Cin, int Cout);
// what launch_conv3d decides from the shape (pure: no device access); slab and ksplit change the summation order of the taps
// and never depend on T
struct ConvPlan {
  int bn;           // tile width (output channels per tile): 256 | 128 | 64
  int pair;         // CTA pairs (cta_group::2)
  int slab;         // slab stages (pairs, Cout < 256): h-haloed activation slab shared by the three dh taps
  int bt, bh, bw;   // voxel box of one tile (bt * bh * bw == 128)
  int ksplit;       // 3: the taps are split by dt over three work items + a fixed-order reduction pass
};
ConvPlan conv3d_plan(int T, int H, int W, int Cin, int Cout, int mode, int ntaps, bool scratch_ok, int sm_count, bool pair_on,
                     bool slab_on);
bool conv3d_pair_default();   // LTX_CONV_PAIR / LTX_CONV_SLAB as launch_conv3d reads them
bool conv3d_slab_default();
// splitk_scratch (optional, >= 3 * T*H*W*Cout fp32): lets tile-starved mode-0 convs split their taps over 3 work items.
void launch_conv3d(const bf16* x_pad, const bf16* w, int T, int H, int W, int Cin, int Cout, const ConvEpi& epi,
                   cudaStream_t s, int ntaps = 27, float* splitk_scratch = nullptr, size_t splitk_scratch_bytes = 0);
// pad (+ optional pixel-norm * (1+scale) + shift -> SiLU, or per-channel affine) from fp32 [T,H,W,C] into bf16 [T+2,H+2,W+2,C]
// mode 0: copy ; 1: x*a[c]+b[c] (denormalise) ; 2: silu(pn(x)*(1+a[c])+b[c]) (a, b nullable) ; 3: silu(x*a[c]+b[c])
// pad: VAE_PAD_* bits (0 = reflect H/W + one replicated frame each side: the decoder's non-causal convolution)
enum { VAE_PAD_CAUSAL = 1, VAE_PAD_ZERO_HW = 2, VAE_PAD_ZERO_T = 4 };
// fills the padding voxels of a bf16 padded volume [T+2,H+2,W+2,C] whose interior has been written (conv epilogue mode 3):
// reflect / zero in H, W and frame replication / zero in T, as launch_vae_prep would have produced
void launch_vae_halo_fill(bf16* pad_vol, int T, int H, int W, int C, int pad, cudaStream_t s);
void launch_vae_prep(const float* x, bf16* out, int T, int H, int W, int C, int mode, const float* a, const float* b,
                     int pad, cudaStream_t s);

}  // namespace ltx
