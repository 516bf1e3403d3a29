// LTX-2 video DiT forward on one B200: orchestration of the sm_100a kernels.
// Restates LTXTransformer.callAsFunction (Models/Transformer/LTXTransformer.swift:235-486) and
// BasicTransformerBlock.callAsFunction (Models/Transformer/LTXTransformerBlock.swift:187-232).
//
// HBM layout (token-major, rows r = b*N + token):
//   x   fp32 [R, D]   residual stream          xb  bf16 [R, D]  bf16 shadow of x (A operand of the cross-attn q-proj)
//   h   bf16 [R, D]   AdaLN output             qk  bf16 [R, 2D] fused q|k projection (normed + RoPE'd in place)
//   vt  bf16 [D, ldv] V^T (K-major for P V)    att bf16 [R, D]  attention output
//   ffh bf16 [R, 4D]  GELU(FFN in)             text cache: per block K [B*S, D], V^T [D, ldv2] (step-invariant)
#include <algorithm>
#include <cmath>

#include "ctx.h"

namespace ltx {

namespace {

double gemm_bytes(int M, int N, int K) {
  return 2.0 * (static_cast<double>(M) * K + static_cast<double>(N) * K + static_cast<double>(M) * N);
}
// the bf16 kernels (B: the weight, or the activation rows when a V^T projection makes the weight the A operand)
void gemm_bf16(ltx_ctx* c, const bf16* A, int64_t lda, const bf16* B, int64_t ldb, int M, int N, int K, const GemmEpi& e,
               const LinearOpts& o) {
  ProfScope ps(c, PROF_GEMM, 2.0 * M * N * K, gemm_bytes(M, N, K));
  GemmEpi ew = e;
  if (o.split_k && M <= 512) gemm_attach_workspace(c, ew);
  const int force_bn = o.tile_n == 0 ? 0 : M > 128 ? 1000 + o.tile_n : o.tile_n;
  launch_gemm(A, lda, B, ldb, M, N, K, ew, c->stream, force_bn, o.a_kblock, o.a_kblock_stride, o.allow_skinny);
}

}  // namespace

// profiled launch helpers (flop / byte counts are the algorithmic ones used by bench.py's roofline)
void linear(ltx_ctx* c, const bf16* A, int64_t lda, const LinearW& W, int M, int N, int K, const GemmEpi& e, const LinearOpts& o) {
  LTX_CHECK(W.k == K && N >= 1 && N <= W.n, LTX_ERR_INVALID_ARGUMENT, "Linear: weight shape mismatch");
  if (W.fmt == LW_BF16) {
    gemm_bf16(c, A, lda, W.w, K, M, N, K, e, o);
  } else if (W.fmt == LW_AFFINE) {   // dequant-fused kernel, or panel + bf16 kernel for large M
    ProfScope ps(c, PROF_GEMM, 2.0 * M * N * K, gemm_bytes(M, N, K), gemm_q_uses_panel(W.q, M) ? 2 : 1);
    launch_gemm_q(A, lda, W.q, M, N, K, e, c->stream, 0, o.a_kblock, o.a_kblock_stride);
  } else {
    // A's rows become e4m3 codes + power-of-two row scales in one reused scratch buffer, then the FP8 pair kernel runs for
    // every M (no weight-streaming, 1-CTA or swap-AB form), so each row's result depends on that row alone: a batched forward
    // equals its items' forwards bit for bit
    LTX_CHECK(o.a_kblock == 0, LTX_ERR_UNSUPPORTED, "FP8 GEMM: no K-blocked A operand");
    const size_t code_bytes = (static_cast<size_t>(M) * K + 15) / 16 * 16;
    c->fp8_act.reserve(code_bytes + static_cast<size_t>(M) * 4);
    uint8_t* q = c->fp8_act.as<uint8_t>();
    float* s = reinterpret_cast<float*>(q + code_bytes);
    {
      ProfScope ps(c, PROF_ROW, 0.0, 3.0 * M * K + 4.0 * M);
      launch_quantize_rows_fp8(A, lda, M, K, q, s, c->stream);
    }
    ProfScope ps(c, PROF_GEMM, 2.0 * M * N * K, static_cast<double>(M) * K + static_cast<double>(N) * K + 2.0 * M * N);
    launch_gemm_fp8(q, K, s, W.q.q, W.q.k, W.q.scales, M, N, K, e, c->stream, o.tile_n);
  }
}

void linear_vt(ltx_ctx* c, const bf16* A, int rows, int items, const LinearW& W, const float* bias, bf16* out, int64_t ld_out,
               int64_t item_ld, bf16* tmp, const LinearOpts& o) {
  const int N = W.n, K = W.k;
  GemmEpi e;
  e.mode = EPI_BF16; e.bias = bias;
  if (W.fmt != LW_BF16) {
    e.out = tmp; e.ldo = N;
    linear(c, A, K, W, items * rows, N, K, e, o);
    ProfScope ps(c, PROF_OTHER, 0.0, 4.0 * items * rows * N, items);
    for (int i = 0; i < items; ++i)
      launch_transpose_bf16(tmp + static_cast<int64_t>(i) * rows * N, N, rows, N, out + i * item_ld, ld_out, c->stream);
    return;
  }
  e.out = out; e.ldo = ld_out;
  if (items > 1) { e.t_item_rows = rows; e.t_item_ld = item_ld; }
  if (gemm_skinny_eligible(K, K, items * rows, N, K, e, 0, o.allow_skinny)) {
    e.transpose_out = 1;
    linear(c, A, K, W, items * rows, N, K, e, o);
    return;
  }
  e.t_item_rows = 0;
  e.bias_per_row = 1;
  if (items == 1 || rows == item_ld) {   // the items' column blocks are contiguous
    gemm_bf16(c, W.w, K, A, K, N, items * rows, K, e, o);
    return;
  }
  for (int i = 0; i < items; ++i) {
    e.out = out + i * item_ld;
    gemm_bf16(c, W.w, K, A + static_cast<int64_t>(i) * rows * K, K, N, rows, K, e, o);
  }
}

void attention(ltx_ctx* c, const bf16* Q, int64_t ldq, const bf16* K, int64_t ldk, const bf16* Vt, int64_t ldv, const float* bias,
               bf16* O, int64_t ldo, int B, int H, int Nq, int Nk, int D, const PeerTable* o_blocks, int rows_per_block) {
  const int hd = D / H;
  ProfScope ps(c, PROF_ATTN, 4.0 * B * H * static_cast<double>(Nq) * Nk * hd, 2.0 * B * (2.0 * Nq + 2.0 * Nk) * D);
  launch_attention(Q, ldq, K, ldk, Vt, ldv, bias, O, ldo, B, H, Nq, Nk, D, 1.0f / sqrtf(static_cast<float>(hd)), c->stream, o_blocks,
                   rows_per_block);
}

void adaln_single(ltx_ctx* c, const AdaLnW& a, float* se, float* t1, float* emb, float* lin, int B, const float* sigma, float mult) {
  ProfScope ps(c, PROF_OTHER, 2.0 * B * a.dim * (256.0 + (1.0 + a.n) * a.dim), 2.0 * a.dim * (256.0 + (1.0 + a.n) * a.dim),
               sigma ? 4 : 3);
  if (sigma) launch_sincos_embed(sigma, mult, se, B, 256, c->stream);
  launch_gemv(a.w1, a.b1, se, t1, B, a.dim, 256, 0, c->stream);
  launch_gemv(a.w2, a.b2, t1, emb, B, a.dim, a.dim, 1, c->stream);
  launch_gemv(a.wl, a.bl, emb, lin, B, a.n * a.dim, a.dim, 1, c->stream);
}

void adaln_single_rows(ltx_ctx* c, const AdaLnW& a, const bf16* se_bf, int R, bf16* t1_bf, float* emb, float* lin, int64_t ld_lin,
                       const LinearOpts& o) {
  GemmEpi e1;
  e1.mode = EPI_SILU_BF16; e1.out = t1_bf; e1.ldo = a.dim; e1.bias = a.b1;
  gemm_bf16(c, se_bf, 256, a.w1, 256, R, a.dim, 256, e1, o);
  GemmEpi e2;
  e2.mode = EPI_F32; e2.out = emb; e2.ldo = a.dim; e2.bias = a.b2;
  gemm_bf16(c, t1_bf, a.dim, a.w2, a.dim, R, a.dim, a.dim, e2, o);
  {
    ProfScope ps(c, PROF_OTHER, 0.0, 6.0 * R * a.dim);
    launch_silu_cast(emb, t1_bf, static_cast<int64_t>(R) * a.dim, c->stream);
  }
  GemmEpi e3;
  e3.mode = EPI_F32; e3.out = lin; e3.ldo = ld_lin; e3.bias = a.bl;
  gemm_bf16(c, t1_bf, a.dim, a.wl, a.dim, R, a.n * a.dim, a.dim, e3, o);
}

const bf16* wbf(ltx_ctx* c, const std::string& k, int64_t r, int64_t cc) {
  const DevTensor& t = get_tensor(c, k);
  LTX_CHECK(t.dtype == LTX_BF16 && t.shape.size() == 2 && t.shape[0] == r && t.shape[1] == cc, LTX_ERR_WEIGHTS,
            "bad shape for '" + k + "'");
  return reinterpret_cast<const bf16*>(t.ptr);
}
const float* wf(ltx_ctx* c, const std::string& k, int64_t n) {
  const DevTensor& t = get_tensor(c, k);
  LTX_CHECK(t.dtype == LTX_F32 && t.numel() == n, LTX_ERR_WEIGHTS, "bad shape for '" + k + "'");
  return reinterpret_cast<const float*>(t.ptr);
}
LinearW wlin(ltx_ctx* c, const std::string& k, int64_t n, int64_t kk) {
  LinearW w;
  w.n = static_cast<int>(n); w.k = static_cast<int>(kk);
  const DevTensor& t = get_tensor(c, k);
  if (t.dtype == DT_E4M3) {   // codes of a scaled-FP8 checkpoint, kept in FP8 mode
    LTX_CHECK(t.shape.size() == 2 && t.shape[0] == n && t.shape[1] == kk, LTX_ERR_WEIGHTS, "bad shape for '" + k + "'");
    w.fmt = LW_E4M3;
    w.q.q = t.codes(); w.q.scales = t.scales; w.q.bits = 8; w.q.n = w.n; w.q.k = w.k;
    return w;
  }
  w.w = wbf(c, k, n, kk);
  return w;
}
AdaLnW adaln_w(ltx_ctx* c, const std::string& p, int64_t dim, int n) {
  AdaLnW a;
  a.w1 = wbf(c, p + ".emb.linear_1.weight", dim, 256); a.b1 = wf(c, p + ".emb.linear_1.bias", dim);
  a.w2 = wbf(c, p + ".emb.linear_2.weight", dim, dim); a.b2 = wf(c, p + ".emb.linear_2.bias", dim);
  a.wl = wbf(c, p + ".linear.weight", n * dim, dim); a.bl = wf(c, p + ".linear.bias", n * dim);
  a.dim = static_cast<int>(dim); a.n = n;
  return a;
}

namespace {

void norm_mod(ltx_ctx* c, const float* x, bf16* out, int M, int D, const float* ts, const float* tsc, const float* as,
              const float* asc, int64_t ada_ld, int rows_per_mod, float eps, int ln) {
  ProfScope ps(c, PROF_ROW, 0.0, static_cast<double>(M) * D * 6.0);
  launch_rmsnorm_mod(x, out, M, D, ts, tsc, as, asc, ada_ld, rows_per_mod, eps, ln, c->stream);
}
void qknorm(ltx_ctx* c, bf16* x, int64_t ld, int M, int D, const float* w, const float* cs, const float* sn, int rpr,
            float eps, const float* w_second = nullptr, const QkOut* blocked = nullptr) {
  const int segs = w_second ? 2 : 1;
  ProfScope ps(c, PROF_ROW, 0.0, segs * static_cast<double>(M) * D * (4.0 + (cs ? 4.0 : 0.0)), (D == 4096) ? 1 : segs);
  launch_qknorm_rope(x, ld, M, D, w, cs, sn, rpr, eps, c->stream, w_second, blocked);
}

// Host fp64 RoPE table, token-major [N, D/2] (T/LTXRoPE.swift:375-488, 552-610; see oracle.rope_table).
void build_rope(ltx_ctx* c, int F, int H, int W) {
  if (c->rope_f == F && c->rope_h == H && c->rope_w == W && c->rope_cos.ptr) return;
  const ltx_config& g = c->cfg;
  const int D = g.num_heads * g.head_dim;
  const int half = D / 2;
  const int n_idx = std::max(1, D / 6);
  const int pad = std::max(0, half - n_idx * 3);
  const int64_t N = static_cast<int64_t>(F) * H * W;
  std::vector<float> cs(static_cast<size_t>(N) * half), sn(static_cast<size_t>(N) * half);
  std::vector<double> idx(n_idx);
  for (int i = 0; i < n_idx; ++i) {
    const double t = n_idx > 1 ? static_cast<double>(i) / (n_idx - 1) : 0.0;
    idx[i] = std::pow(static_cast<double>(g.rope_theta), t) * (M_PI / 2.0);
  }
  for (int f = 0; f < F; ++f) {
    // pixel-space temporal mid-point with the causal fix, divided by fps = 24 -- all in fp32 like the reference
    const float ts = 8.0f, fi = static_cast<float>(f);
    const float st = std::max(fi * ts + (1.0f - ts), 0.0f), en = std::max((fi + 1.0f) * ts + (1.0f - ts), 0.0f);
    const float pt = ((st + en) / 2.0f) / 24.0f;
    for (int y = 0; y < H; ++y) {
      const float phh = static_cast<float>(y) * 32.0f + 16.0f;
      for (int x = 0; x < W; ++x) {
        const float pw = static_cast<float>(x) * 32.0f + 16.0f;
        const int64_t n = (static_cast<int64_t>(f) * H + y) * W + x;
        const double sc[3] = {static_cast<double>(pt) / g.max_pos[0] * 2.0 - 1.0,
                              static_cast<double>(phh) / g.max_pos[1] * 2.0 - 1.0,
                              static_cast<double>(pw) / g.max_pos[2] * 2.0 - 1.0};
        float* cr = &cs[static_cast<size_t>(n) * half];
        float* sr = &sn[static_cast<size_t>(n) * half];
        for (int p = 0; p < pad; ++p) { cr[p] = 1.0f; sr[p] = 0.0f; }
        for (int k = 0; k < n_idx; ++k)
          for (int d = 0; d < 3; ++d) {
            const int o = pad + k * 3 + d;
            if (o >= half) continue;
            const double a = idx[k] * sc[d];
            cr[o] = static_cast<float>(std::cos(a));
            sr[o] = static_cast<float>(std::sin(a));
          }
      }
    }
  }
  const size_t bytes = cs.size() * sizeof(float);
  c->rope_cos.reserve(bytes);
  c->rope_sin.reserve(bytes);
  LTX_CUDA(cudaMemcpyAsync(c->rope_cos.ptr, cs.data(), bytes, cudaMemcpyHostToDevice, c->stream));
  LTX_CUDA(cudaMemcpyAsync(c->rope_sin.ptr, sn.data(), bytes, cudaMemcpyHostToDevice, c->stream));
  LTX_CUDA(cudaStreamSynchronize(c->stream));  // host vectors go out of scope
  c->rope_f = F; c->rope_h = H; c->rope_w = W;
}

int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

bool in_list(int v, const int32_t* lst, int n) {
  for (int i = 0; i < n; ++i)
    if (lst[i] == v) return true;
  return false;
}

// caption projection + per-block text K / V^T (T/LTXTimestepEmbedding.swift:146-151, T/LTXAttention.swift:171-180)
}  // namespace

// Generic over the stream: `src` names the caption-projection and per-block cross-attention K / V weights (the video stream
// of both models, or the audio stream of the dual model), `slots` / `rr` the two-entry cache it fills.
TextCache& dit_prepare_text(ltx_ctx* c, TextCache* slots, int* rr, const TextProjW& src, const void* context, int context_dtype,
                            const int32_t* mask_dev, int B, int S, uint64_t key) {
  const ltx_config& g = c->cfg;
  const int D = src.D, L = g.num_layers, Cc = g.caption_channels;
  if (key != 0)
    for (int i = 0; i < 2; ++i)
      if (slots[i].key == key && slots[i].B == B && slots[i].S == S) return slots[i];
  // miss: take an un-keyed slot if there is one, otherwise evict round-robin
  int slot = -1;
  for (int i = 0; i < 2; ++i)
    if (slots[i].key == 0) { slot = i; break; }
  if (slot < 0) slot = ((*rr)++) & 1;
  TextCache& tc = slots[slot];
  const int64_t R = static_cast<int64_t>(B) * S;
  tc.key = key; tc.fingerprint = 0; tc.B = B; tc.S = S;
  tc.ldv = round_up(S, 8);  // per-batch pitch of V^T; row pitch is B * ldv
  tc.k.reserve(static_cast<size_t>(L) * R * D * 2);
  tc.vt.reserve(static_cast<size_t>(L) * D * B * tc.ldv * 2);
  cudaStream_t st = c->stream;
  // stage context as bf16
  const bf16* ctx_bf;
  if (context_dtype == LTX_BF16) {
    ctx_bf = reinterpret_cast<const bf16*>(context);
  } else {
    LTX_CHECK(context_dtype == LTX_F32, LTX_ERR_UNSUPPORTED, "context dtype must be bf16 or f32");
    LTX_CHECK((R * Cc) % 4 == 0, LTX_ERR_INVALID_ARGUMENT, "context size");
    c->ctx_in.reserve(static_cast<size_t>(R) * Cc * 2);
    {
      ProfScope ps(c, PROF_OTHER, 0.0, 6.0 * R * Cc);
      launch_cast_f32_bf16(reinterpret_cast<const float*>(context), c->ctx_in.as<bf16>(), R * Cc, st);
    }
    ctx_bf = c->ctx_in.as<bf16>();
  }
  c->c1.reserve(static_cast<size_t>(R) * D * 2);
  c->c2.reserve(static_cast<size_t>(R) * D * 2);
  LinearOpts o;   // both models build their text caches with the video model's rule: split-K for few rows
  o.split_k = true;
  GemmEpi e;
  e.mode = EPI_GELU_BF16; e.out = c->c1.ptr; e.ldo = D; e.bias = src.b_c1;
  linear(c, ctx_bf, Cc, src.w_c1, static_cast<int>(R), D, Cc, e, o);
  e.mode = EPI_BF16; e.out = c->c2.ptr; e.bias = src.b_c2;
  linear(c, c->c1.as<bf16>(), D, src.w_c2, static_cast<int>(R), D, D, e, o);
  for (int i = 0; i < L; ++i) {
    const AttnWeights& a = src.layer(src.user, i);
    bf16* kd = tc.k.as<bf16>() + static_cast<int64_t>(i) * R * D;
    bf16* vd = tc.vt.as<bf16>() + static_cast<int64_t>(i) * D * B * tc.ldv;
    GemmEpi ek;
    ek.mode = EPI_BF16; ek.out = kd; ek.ldo = D; ek.bias = a.bk;
    linear(c, c->c2.as<bf16>(), D, a.wk, static_cast<int>(R), D, D, ek, o);
    qknorm(c, kd, D, static_cast<int>(R), D, a.k_norm, nullptr, nullptr, 1, g.norm_eps);
    for (int b = 0; b < B; ++b)  // V^T[D, S] per batch, one column block each
      linear_vt(c, c->c2.as<bf16>() + static_cast<int64_t>(b) * S * D, S, 1, a.wv, a.bv, vd + b * tc.ldv, B * tc.ldv, tc.ldv,
                c->c1.as<bf16>(), o);
  }
  // An all-ones mask (what the real text connector emits, LTXTextEncoder.swift:514-520) adds a zero bias: skip it.
  bool any_masked = false;
  if (mask_dev) {
    std::vector<int32_t> hm(static_cast<size_t>(R));
    LTX_CUDA(cudaMemcpyAsync(hm.data(), mask_dev, static_cast<size_t>(R) * 4, cudaMemcpyDeviceToHost, st));
    LTX_CUDA(cudaStreamSynchronize(st));
    for (int32_t v : hm) any_masked |= (v == 0);
  }
  tc.has_bias = any_masked;
  if (any_masked) {
    tc.bias.reserve(static_cast<size_t>(R) * 4);
    ProfScope ps(c, PROF_OTHER, 0.0, 8.0 * R);
    launch_mask_to_bias(mask_dev, tc.bias.as<float>(), static_cast<int>(R), st);
  }
  return tc;
}

namespace {
const AttnWeights& video_text_layer(const void* user, int i) { return static_cast<const ltx_ctx*>(user)->blocks[i].a2; }
TextCache& prepare_text(ltx_ctx* c, const void* context, int context_dtype, const int32_t* mask_dev, int B, int S,
                        uint64_t key) {
  TextProjW src;
  src.w_c1 = c->w_c1; src.w_c2 = c->w_c2; src.b_c1 = c->b_c1; src.b_c2 = c->b_c2;
  src.D = c->cfg.num_heads * c->cfg.head_dim; src.user = c; src.layer = video_text_layer;
  return dit_prepare_text(c, c->text, &c->text_rr, src, context, context_dtype, mask_dev, B, S, key);
}
}  // namespace

void dit_build_rope(ltx_ctx* c, int F, int H, int W) { build_rope(c, F, H, W); }

void gemm_attach_workspace(ltx_ctx* c, GemmEpi& e) {
  constexpr size_t kCounters = 16384, kPartials = static_cast<size_t>(40) << 20;
  if (!c->gemm_ws.ptr) {
    c->gemm_ws.reserve(kCounters * 4 + kPartials);
    LTX_CUDA(cudaMemsetAsync(c->gemm_ws.ptr, 0, kCounters * 4, c->stream));
  }
  e.ws_counters = c->gemm_ws.as<unsigned int>();
  e.ws_counter_count = kCounters;
  e.ws = reinterpret_cast<float*>(c->gemm_ws.as<uint8_t>() + kCounters * 4);
  e.ws_bytes = kPartials;
}

void dit_clear_caches(ltx_ctx* c) {
  c->rope_f = c->rope_h = c->rope_w = 0;
  for (auto& t : c->text) { t.key = 0; t.fingerprint = 0; t.B = t.S = 0; }
  for (auto& t : c->av.text) { t.key = 0; t.fingerprint = 0; t.B = t.S = 0; }   // the dual model's audio-stream text cache
  c->av.rope_ta = c->av.rope_f = c->av.rope_hw = 0;
}

// Pack raw tensors into kernel-ready pointers.  attn1 to_q|to_k are concatenated into one [2D, D] operand so the
// q and k projections run as a single N = 2D GEMM (better wave quantisation at M = 1536).
void dit_finalize(ltx_ctx* c) {
  const ltx_config& g = c->cfg;
  LTX_CHECK(g.head_dim == 128, LTX_ERR_INVALID_CONFIGURATION, "head_dim must be 128");
  const int64_t D = static_cast<int64_t>(g.num_heads) * g.head_dim, FF = g.ffn_mult * D;
  LTX_CHECK(g.in_channels % 8 == 0 && g.caption_channels % 8 == 0 && g.out_channels % 8 == 0, LTX_ERR_INVALID_CONFIGURATION,
            "channel counts must be multiples of 8");
  c->w_patch = wlin(c, "patchify_proj.weight", D, g.in_channels);
  c->b_patch = wf(c, "patchify_proj.bias", D);
  c->adaln = adaln_w(c, "adaln_single", D, 6);
  c->w_c1 = wlin(c, "caption_projection.linear_1.weight", D, g.caption_channels);
  c->b_c1 = wf(c, "caption_projection.linear_1.bias", D);
  c->w_c2 = wlin(c, "caption_projection.linear_2.weight", D, D);
  c->b_c2 = wf(c, "caption_projection.linear_2.bias", D);
  c->sst_out = wf(c, "scale_shift_table", 2 * D);
  c->w_out = wlin(c, "proj_out.weight", g.out_channels, D);
  c->b_out = wf(c, "proj_out.bias", g.out_channels);
  c->blocks.assign(g.num_layers, BlockWeights());
  for (int i = 0; i < g.num_layers; ++i) {
    const std::string p = "transformer_blocks." + std::to_string(i) + ".";
    BlockWeights& b = c->blocks[i];
    b.sst = wf(c, p + "scale_shift_table", 6 * D);
    // attn1: pack q|k|v into one [3D, D] operand: the three projections of the block run as ONE GEMM (N = 3D; V leaves its
    // epilogue transposed); the other paths address the q|k rows (wq, N = 2D) and the v rows (wv) of the same buffer
    {
      const LinearW ws[3] = {wlin(c, p + "attn1.to_q.weight", D, D), wlin(c, p + "attn1.to_k.weight", D, D),
                             wlin(c, p + "attn1.to_v.weight", D, D)};
      const float* bq = wf(c, p + "attn1.to_q.bias", D);
      const float* bk = wf(c, p + "attn1.to_k.bias", D);
      const float* bvv = wf(c, p + "attn1.to_v.bias", D);
      float* bqkv = nullptr;
      LTX_CUDA(cudaMalloc(&bqkv, static_cast<size_t>(3) * D * 4));
      c->owned.push_back(bqkv);
      const float* bs[3] = {bq, bk, bvv};
      for (int t = 0; t < 3; ++t)
        LTX_CUDA(cudaMemcpyAsync(bqkv + static_cast<size_t>(t) * D, bs[t], static_cast<size_t>(D) * 4, cudaMemcpyDeviceToDevice, c->stream));
      if (ws[0].fmt == LW_E4M3 || ws[1].fmt == LW_E4M3 || ws[2].fmt == LW_E4M3) {
        // FP8 mode with sources held as e4m3 codes: the packed q|k|v is made as codes + row scales [3D] one [D, D] block per
        // source -- codes and scales copied, a bf16 source converted by dit_convert_fp8's per-row rule (rows are independent)
        uint8_t* q = nullptr;
        float* s = nullptr;
        LTX_CUDA(cudaMalloc(&q, static_cast<size_t>(3) * D * D));
        LTX_CUDA(cudaMalloc(&s, static_cast<size_t>(3) * D * 4));
        c->owned.push_back(q); c->owned.push_back(s);
        for (int t = 0; t < 3; ++t) {
          uint8_t* qt = q + static_cast<size_t>(t) * D * D;
          if (ws[t].fmt == LW_E4M3) {
            LTX_CUDA(cudaMemcpyAsync(qt, ws[t].q.q, static_cast<size_t>(D) * D, cudaMemcpyDeviceToDevice, c->stream));
            LTX_CUDA(cudaMemcpyAsync(s + t * D, ws[t].q.scales, static_cast<size_t>(D) * 4, cudaMemcpyDeviceToDevice, c->stream));
          } else {
            launch_quantize_rows_fp8(ws[t].w, D, static_cast<int>(D), static_cast<int>(D), qt, s + t * D, c->stream);
          }
        }
        b.a1.wq.fmt = LW_E4M3; b.a1.wq.n = 3 * D; b.a1.wq.k = D;
        b.a1.wq.q.q = q; b.a1.wq.q.scales = s; b.a1.wq.q.bits = 8; b.a1.wq.q.n = 3 * D; b.a1.wq.q.k = D;
      } else {
        bf16* wqkv = nullptr;
        LTX_CUDA(cudaMalloc(&wqkv, static_cast<size_t>(3) * D * D * 2));
        c->owned.push_back(wqkv);
        for (int t = 0; t < 3; ++t)
          LTX_CUDA(cudaMemcpyAsync(wqkv + static_cast<size_t>(t) * D * D, ws[t].w, static_cast<size_t>(D) * D * 2, cudaMemcpyDeviceToDevice, c->stream));
        b.a1.wq.n = 3 * D; b.a1.wq.k = D; b.a1.wq.w = wqkv;
        b.a1.wv.n = D; b.a1.wv.k = D; b.a1.wv.w = wqkv + 2 * D * D;
      }
      LTX_CUDA(cudaStreamSynchronize(c->stream));
      // the unpacked copies are no longer needed
      for (const char* k : {"attn1.to_q.weight", "attn1.to_k.weight", "attn1.to_v.weight"}) {
        auto it = c->tensors.find(p + k);
        it->second.free_storage();
        c->tensors.erase(it);
      }
      b.a1.bq = bqkv; b.a1.bk = bqkv + D; b.a1.bv = bqkv + 2 * D;
    }
    b.a1.wo = wlin(c, p + "attn1.to_out.weight", D, D);
    b.a1.bo = wf(c, p + "attn1.to_out.bias", D);
    b.a1.q_norm = wf(c, p + "attn1.q_norm.weight", D);
    b.a1.k_norm = wf(c, p + "attn1.k_norm.weight", D);
    b.a2.wq = wlin(c, p + "attn2.to_q.weight", D, D);
    b.a2.bq = wf(c, p + "attn2.to_q.bias", D);
    b.a2.wk = wlin(c, p + "attn2.to_k.weight", D, D);
    b.a2.bk = wf(c, p + "attn2.to_k.bias", D);
    b.a2.wv = wlin(c, p + "attn2.to_v.weight", D, D);
    b.a2.bv = wf(c, p + "attn2.to_v.bias", D);
    b.a2.wo = wlin(c, p + "attn2.to_out.weight", D, D);
    b.a2.bo = wf(c, p + "attn2.to_out.bias", D);
    b.a2.q_norm = wf(c, p + "attn2.q_norm.weight", D);
    b.a2.k_norm = wf(c, p + "attn2.k_norm.weight", D);
    b.w_in = wlin(c, p + "ff.project_in.proj.weight", FF, D);
    b.b_in = wf(c, p + "ff.project_in.proj.bias", FF);
    b.w_out = wlin(c, p + "ff.project_out.weight", D, FF);
    b.b_out = wf(c, p + "ff.project_out.bias", D);
  }
  c->scratch.reserve(64 * sizeof(double));
  c->dit_ready = true;
}

namespace {
// frees a replaced weight: a loaded tensor or an allocation made by finalize
void release_weight(ltx_ctx* c, const void* p) {
  for (auto it = c->tensors.begin(); it != c->tensors.end(); ++it)
    if (it->second.ptr == p) { cudaFree(it->second.ptr); c->tensors.erase(it); return; }
  for (auto it = c->owned.begin(); it != c->owned.end(); ++it)
    if (*it == p) { cudaFree(*it); c->owned.erase(it); return; }
}
}  // namespace

// Replace every GEMM weight of the DiT by per-64-group affine codes (the reference quantises every Linear,
// P/LTXPipeline.swift:323-333); the bf16 copies are freed.  The M = 1 timestep-MLP GEMVs keep bf16 weights.
void dit_quantize(ltx_ctx* c, int bits) {
  LTX_CHECK(c->dit_ready, LTX_ERR_WEIGHTS, "DiT weights not finalized");
  LTX_CHECK(bits == 8 || bits == 4, LTX_ERR_UNSUPPORTED, "quant_bits must be 16, 8 or 4");
  const ltx_config& g = c->cfg;
  const int D = g.num_heads * g.head_dim;
  std::vector<const void*> to_free;   // freed at the end: attn1's v rows live in the allocation of its packed q|k|v
  std::vector<LinearW*> coded;
  // rows: quantise only the leading rows of the matrix (0: all of them)
  auto qf = [&](LinearW& w, int rows = 0) {
    const int N = rows ? rows : w.n, K = w.k;
    LTX_CHECK(w.fmt == LW_BF16, LTX_ERR_WEIGHTS, "quantisation needs bf16 weights");
    LTX_CHECK(K % 64 == 0, LTX_ERR_INVALID_CONFIGURATION, "quantisation needs every Linear input width to be a multiple of 64");
    uint8_t* q = nullptr;
    float *s = nullptr, *b = nullptr;
    const size_t qbytes = static_cast<size_t>(N) * K * bits / 8, sbytes = static_cast<size_t>(K / 64) * N * 4;
    LTX_CUDA(cudaMalloc(&q, qbytes));
    LTX_CUDA(cudaMalloc(&s, sbytes));
    LTX_CUDA(cudaMalloc(&b, sbytes));
    c->owned.push_back(q); c->owned.push_back(s); c->owned.push_back(b);
    launch_quantize(w.w, N, K, bits, q, s, b, c->stream);
    QuantW r;
    r.q = q; r.scales = s; r.biases = b; r.bits = bits; r.n = N; r.k = K;
    if (c->quant_materialise) {
      // materialised storage: the weight keeps its place and dtype, its values become s * q + beta (the panel conversion's
      // arithmetic and rounding, i.e. exactly what the fused kernels would feed the tensor cores); the codes are dropped
      launch_dequantize_panel(r, const_cast<bf16*>(w.w), c->stream);
      LTX_CUDA(cudaStreamSynchronize(c->stream));
      for (void* ptr : {static_cast<void*>(q), static_cast<void*>(s), static_cast<void*>(b)}) {
        cudaFree(ptr);
        c->owned.erase(std::find(c->owned.begin(), c->owned.end(), ptr));
      }
      return;
    }
    LTX_CUDA(cudaStreamSynchronize(c->stream));
    to_free.push_back(w.w);
    w.fmt = LW_AFFINE; w.n = N; w.w = nullptr; w.q = r;
    coded.push_back(&w);
  };
  qf(c->w_patch); qf(c->w_c1); qf(c->w_c2); qf(c->w_out);
  for (auto& b : c->blocks) {
    qf(b.a1.wq, 2 * D);   // the q|k rows of the packed q|k|v (its v rows are quantised by the next call: rows are independent)
    qf(b.a1.wv); qf(b.a1.wo);
    qf(b.a2.wq); qf(b.a2.wk); qf(b.a2.wv); qf(b.a2.wo);
    qf(b.w_in); qf(b.w_out);
  }
  if (c->av.ready) {
    // the dual model's Linears (quantize(model: ltx2, groupSize: 64, bits:), Pipeline/LTXPipeline.swift:491); the AdaLN-single
    // embedders stay bf16 like the video model's timestep MLP
    AvWeights& a = c->av;
    qf(a.w_patch); qf(a.w_c1); qf(a.w_c2); qf(a.w_out);
    for (auto& b : a.blocks) {
      for (AttnWeights* w : {&b.aa1, &b.aa2, &b.a2v, &b.v2a}) { qf(w->wq); qf(w->wk); qf(w->wv); qf(w->wo); }
      qf(b.w_in); qf(b.w_out);
    }
  }
  c->quant_bits = bits;
  if (c->quant_materialise) return;   // the weights stay bf16 (now dequantised)
  for (const void* p : to_free) release_weight(c, p);
  // one bf16 panel for the large-M path of launch_gemm_q, sized for the largest weight (the FFN matrices)
  size_t max_elems = 0;
  for (const LinearW* w : coded) max_elems = std::max(max_elems, static_cast<size_t>(w->n) * w->k);
  c->q_panel.reserve(max_elems * 2);
  for (LinearW* w : coded) w->q.scratch = c->q_panel.as<bf16>();
}

// Precision mode 8: every Linear inside the transformer blocks becomes e4m3 codes with one power-of-two scale per output
// channel (launch_quantize_rows_fp8: the rule linear() applies to the activation rows); the bf16 copies are freed.  Patchify,
// caption projection, the timestep MLPs / AdaLN and proj_out stay bf16.  Linears loaded as the codes of a scaled-FP8 checkpoint
// (wlin: LW_E4M3 already) keep them and their scales.
void dit_convert_fp8(ltx_ctx* c) {
  LTX_CHECK(c->dit_ready, LTX_ERR_WEIGHTS, "DiT weights not finalized");
  const ltx_config& g = c->cfg;
  const int D = g.num_heads * g.head_dim, FF = g.ffn_mult * D;
  LTX_CHECK(D % 16 == 0 && FF % 16 == 0, LTX_ERR_INVALID_CONFIGURATION, "FP8 mode needs Linear widths that are multiples of 16");
  std::vector<const void*> to_free;
  auto conv = [&](LinearW& w) {
    if (w.fmt == LW_E4M3) return;
    LTX_CHECK(w.fmt == LW_BF16, LTX_ERR_WEIGHTS, "FP8 conversion needs unquantised DiT weights");
    const int N = w.n, K = w.k;
    uint8_t* q = nullptr;
    float* s = nullptr;
    LTX_CUDA(cudaMalloc(&q, static_cast<size_t>(N) * K));
    LTX_CUDA(cudaMalloc(&s, static_cast<size_t>(N) * 4));
    c->owned.push_back(q); c->owned.push_back(s);
    launch_quantize_rows_fp8(w.w, K, N, K, q, s, c->stream);
    to_free.push_back(w.w);
    w.fmt = LW_E4M3; w.w = nullptr;
    w.q.q = q; w.q.scales = s; w.q.bits = 8; w.q.n = N; w.q.k = K;
  };
  for (auto& b : c->blocks) {
    // the packed q|k|v [3D, D] as one matrix, so the fused projection with its V^T epilogue stays one launch; its v rows are a
    // view of it (rows are independent) for the per-batch V^T projections
    conv(b.a1.wq);
    b.a1.wv = b.a1.wq;
    b.a1.wv.n = b.a1.wv.q.n = D;
    b.a1.wv.q.q += static_cast<size_t>(2) * D * D; b.a1.wv.q.scales += 2 * D;
    conv(b.a1.wo);
    conv(b.a2.wq); conv(b.a2.wk); conv(b.a2.wv); conv(b.a2.wo);
    conv(b.w_in); conv(b.w_out);
  }
  LTX_CUDA(cudaStreamSynchronize(c->stream));
  for (const void* p : to_free) release_weight(c, p);
}

void dit_forward_dev(ltx_ctx* c, const void* latent, int latent_dtype, const void* context, int context_dtype,
                     const float* timesteps_dev, int ts_per_token, const int32_t* mask_dev, int B, int N, int S, int F,
                     int H, int W, const ltx_dit_flags* flags, float* out_velocity_dev, int snapshot_block, int resume_block) {
  LTX_CHECK(c->dit_ready, LTX_ERR_WEIGHTS, "DiT weights not finalized");
  LTX_CHECK(B >= 1 && B <= 4 && N >= 1 && S >= 1, LTX_ERR_INVALID_ARGUMENT, "bad B/N/S");
  LTX_CHECK(static_cast<int64_t>(F) * H * W == N, LTX_ERR_INVALID_ARGUMENT, "N must equal F*H*W");
  LTX_CHECK(latent && context && timesteps_dev && out_velocity_dev, LTX_ERR_INVALID_ARGUMENT, "null tensor");
  if (c->precision == 32) {   // fp32 mode: no prefix sharing (a resumed pass is recomputed in full, same values)
    dit_forward_f32(c, latent, latent_dtype, context, context_dtype, timesteps_dev, ts_per_token, mask_dev, B, N, S, F, H, W, flags,
                    out_velocity_dev);
    return;
  }
  const ltx_config& g = c->cfg;
  const int D = g.num_heads * g.head_dim, FFD = g.ffn_mult * D, Hh = g.num_heads, L = g.num_layers;
  const int Cin = g.in_channels, Cout = g.out_channels;
  // ---- Ulysses sequence parallelism: this rank owns tokens [tok0, tok0 + Nl) for every row-wise op
  const int P = (c->dist.comm_world && c->dist.sp > 1) ? c->dist.sp : 1;
  LTX_CHECK(P == 1 || c->precision != 8, LTX_ERR_UNSUPPORTED, "FP8 mode has no sequence-parallel forward");
  LTX_CHECK(P == 1 || (B == 1 && N % P == 0 && Hh % P == 0), LTX_ERR_INVALID_ARGUMENT,
            "sequence parallelism needs B == 1 and N, num_heads divisible by sp_size");
  const int Nl = N / P, tok0 = (P > 1 ? c->dist.sp_rank : 0) * Nl;
  const int R = (P > 1) ? Nl : B * N;      // local rows
  const int Nq = (P > 1) ? Nl : N;         // local query rows per batch
  const int Csp = D / P, Hl = Hh / P;      // per-rank feature slice / heads inside self-attention
  const float eps = g.norm_eps;
  cudaStream_t st = c->stream;
  LinearOpts o;   // few rows (an Ulysses shard, a small clip): opt in to the weight-streaming kernel
  o.split_k = true;
  ltx_dit_flags noflags = {};
  noflags.cross_attn_scale = 1.0f;
  if (!flags) flags = &noflags;
  LTX_CHECK(flags->n_stg_blocks >= 0 && flags->n_stg_blocks <= LTX_MAX_FLAG_BLOCKS && flags->n_cas_blocks >= 0 &&
                flags->n_cas_blocks <= LTX_MAX_FLAG_BLOCKS,
            LTX_ERR_INVALID_ARGUMENT, "bad flag block counts");

  // ---- workspaces
  const int64_t ldv = round_up(N, 8);  // per-batch pitch of V^T
  c->x.reserve(static_cast<size_t>(R) * D * 4);
  c->xb.reserve(static_cast<size_t>(R) * D * 2);
  c->h.reserve(static_cast<size_t>(R) * D * 2);
  c->qk.reserve(static_cast<size_t>(R) * 2 * D * 2);
  c->vt.reserve(static_cast<size_t>(D) * B * ldv * 2);
  c->att.reserve(static_cast<size_t>(R) * D * 2);
  c->q2.reserve(static_cast<size_t>(R) * D * 2);
  c->ffh.reserve(static_cast<size_t>(R) * FFD * 2);
  // timestep rows: one per batch, or one per (local) token when timesteps are per token (I2V, P/LTXPipeline.swift:2237-2252)
  const int TR = ts_per_token ? R : B;
  c->se.reserve(static_cast<size_t>(TR) * 256 * 4);
  c->t1.reserve(static_cast<size_t>(TR) * D * 4);
  c->emb.reserve(static_cast<size_t>(TR) * D * 4);
  c->ada.reserve(static_cast<size_t>(TR) * 6 * D * 4);
  float* x = c->x.as<float>();
  bf16* xb = c->xb.as<bf16>();
  bf16* h = c->h.as<bf16>();
  bf16* qk = c->qk.as<bf16>();
  bf16* vt = c->vt.as<bf16>();
  bf16* att = c->att.as<bf16>();
  bf16* q2 = c->q2.as<bf16>();
  bf16* ffh = c->ffh.as<bf16>();
  float* ada = c->ada.as<float>();
  float* emb = c->emb.as<float>();
  const int64_t blk = static_cast<int64_t>(Nl) * Csp;   // elements one rank sends to one peer per tensor
  bf16 *qsend = nullptr, *ksend = nullptr, *vsend = nullptr, *qrecv = nullptr, *krecv = nullptr, *vrecv = nullptr,
       *osend = nullptr, *orecv = nullptr, *vt_sp = nullptr;
  // Ulysses exchange buffers.  Preferred: every rank's receive buffer [q | k | v | o][P][Nl][Csp] is mapped into its peers
  // (CUDA IPC over NVLink) and the producing kernels store straight into it; otherwise NCCL all-to-all through send buffers.
  bool p2p = false;
  bf16* peer_base[LTX_MAX_PEERS] = {};
  const int me = c->dist.sp_rank;
  if (P > 1) {
    p2p = dist_p2p_ensure(c, static_cast<size_t>(4) * P * blk * 2);
    c->sp_vt.reserve(static_cast<size_t>(Csp) * ldv * 2);
    c->sp_vel.reserve(static_cast<size_t>(Nl) * Cout * 4);
    vt_sp = c->sp_vt.as<bf16>();
    if (p2p) {
      for (int r = 0; r < P; ++r) peer_base[r] = reinterpret_cast<bf16*>(c->dist.p2p_peer[r]);
      qrecv = peer_base[me]; krecv = qrecv + P * blk; vrecv = krecv + P * blk; orecv = vrecv + P * blk;
      osend = orecv;   // placeholder (attention output rows go to the peers' o regions)
    } else {
      c->sp_send.reserve(static_cast<size_t>(3) * P * blk * 2);
      c->sp_recv.reserve(static_cast<size_t>(3) * P * blk * 2);
      qsend = c->sp_send.as<bf16>(); ksend = qsend + P * blk; vsend = ksend + P * blk;
      qrecv = c->sp_recv.as<bf16>(); krecv = qrecv + P * blk; vrecv = krecv + P * blk;
      osend = qsend;   // the attention output [N, Csp] reuses the q send buffer, its exchange lands in the q recv buffer
      orecv = qrecv;
    }
  }

  // ---- step-invariant pieces
  build_rope(c, F, H, W);
  TextCache& tc = prepare_text(c, context, context_dtype, mask_dev, B, S, flags->context_key);
  const float* key_bias = tc.has_bias ? tc.bias.as<float>() : nullptr;
  const float* cos_l = c->rope_cos.as<float>() + static_cast<int64_t>(tok0) * (D / 2);
  const float* sin_l = c->rope_sin.as<float>() + static_cast<int64_t>(tok0) * (D / 2);
  const int rope_period = (P > 1) ? Nl : N;
  const int rows_per_b = ts_per_token ? 1 : rope_period;   // rows sharing one modulation / gate vector

  // ---- patchify_proj (T/LTXTransformer.swift:257); the reference's bf16 Linear output is rounded to bf16
  const bf16* lat_bf;
  if (latent_dtype == LTX_BF16) {
    lat_bf = reinterpret_cast<const bf16*>(latent);
  } else {
    LTX_CHECK(latent_dtype == LTX_F32, LTX_ERR_UNSUPPORTED, "latent dtype must be bf16 or f32");
    c->lat_in.reserve(static_cast<size_t>(B) * N * Cin * 2);
    {
      ProfScope ps(c, PROF_OTHER, 0.0, 6.0 * B * N * Cin);
      launch_cast_f32_bf16(reinterpret_cast<const float*>(latent), c->lat_in.as<bf16>(), static_cast<int64_t>(B) * N * Cin, st);
    }
    lat_bf = c->lat_in.as<bf16>();
  }
  lat_bf += static_cast<int64_t>(tok0) * Cin;
  if (resume_block < 0) {
    GemmEpi e;
    e.mode = EPI_BF16; e.out = xb; e.ldo = D; e.bias = c->b_patch;
    linear(c, lat_bf, Cin, c->w_patch, R, D, Cin, e, o);
    ProfScope ps(c, PROF_OTHER, 0.0, 6.0 * R * D);
    launch_cast_bf16_f32(xb, x, static_cast<int64_t>(R) * D, st);
  } else {
    // resume from the stream saved at the entry of block `resume_block` by an identical-input pass
    // (a snapshot taken by a batched pass holds the rows of every batch entry; entry 0 -- the first R rows -- is the pass resumed)
    LTX_CHECK(resume_block < L && c->snap_x.ptr && c->snap_rows >= R, LTX_ERR_INVALID_ARGUMENT, "no matching snapshot to resume from");
    ProfScope ps(c, PROF_OTHER, 0.0, 14.0 * R * D, 2);
    LTX_CUDA(cudaMemcpyAsync(x, c->snap_x.ptr, static_cast<size_t>(R) * D * 4, cudaMemcpyDeviceToDevice, st));
    launch_cast_f32_bf16(x, xb, static_cast<int64_t>(R) * D, st);
  }
  // ---- timestep path (T/LTXTimestepEmbedding.swift:62-124): fp32 activations, bf16 weights
  if (!ts_per_token) {
    adaln_single(c, c->adaln, c->se.as<float>(), c->t1.as<float>(), emb, ada, B, timesteps_dev, g.timestep_scale_multiplier);
  } else {
    // one embedding per token over the R local rows; timesteps [B, N] are indexed from this rank's first token
    bf16* se_bf = reinterpret_cast<bf16*>(c->se.ptr);      // [R, 256] bf16
    {
      ProfScope ps(c, PROF_OTHER, 0.0, 4.0 * R + 512.0 * R);
      launch_sincos_embed(timesteps_dev + tok0, g.timestep_scale_multiplier, nullptr, R, 256, st, se_bf);
    }
    adaln_single_rows(c, c->adaln, se_bf, R, reinterpret_cast<bf16*>(c->t1.ptr), emb, ada, 6 * D, o);
  }

  const int64_t ada_ld = 6 * static_cast<int64_t>(D);
  for (int i = (resume_block > 0 ? resume_block : 0); i < L; ++i) {
    const BlockWeights& bw = c->blocks[i];
    if (i == snapshot_block) {
      c->snap_x.reserve(static_cast<size_t>(R) * D * 4);
      c->snap_rows = R;
      ProfScope ps(c, PROF_OTHER, 0.0, 8.0 * R * D);
      LTX_CUDA(cudaMemcpyAsync(c->snap_x.ptr, x, static_cast<size_t>(R) * D * 4, cudaMemcpyDeviceToDevice, st));
    }
    const bool flagged = in_list(i, flags->stg_blocks, flags->n_stg_blocks);
    const bool skip_sa = flagged && flags->skip_self_attn;
    const bool skip_ff = flagged && flags->skip_ff;
    const float cas = in_list(i, flags->cas_blocks, flags->n_cas_blocks) ? flags->cross_attn_scale : 1.0f;
    if (!skip_sa) {
      // h = rms(x) * (1 + scale_msa) + shift_msa      (T/LTXTransformerBlock.swift:72-83, rows 0/1 of table+ada)
      norm_mod(c, x, h, R, D, bw.sst, bw.sst + D, ada, ada + D, ada_ld, rows_per_b, eps, 0);
      // q|k|v in one GEMM (N = 3D, 256-wide tiles: 288 tiles = 3.9 rounds of 74 CTA pairs at M = 1536), the V columns stored
      // transposed by the epilogue; separate q|k and V^T GEMMs for batches, sequence parallelism and quantised weights
      // (batches: V^T row = feature, column = b * ldv + token -- the same as the GEMM row b * N + token when ldv == N)
      const bool packed_qkv = bw.a1.wq.fmt != LW_AFFINE;   // the q|k|v rows are one matrix
      const bool fused_qkv = P == 1 && (B == 1 || ldv == N) && packed_qkv && D % 32 == 0;
      GemmEpi e;
      e.mode = EPI_BF16; e.out = qk; e.ldo = 2 * D; e.bias = bw.a1.bq;
      if (fused_qkv) {
        e.tsplit_col = 2 * D; e.out_t = vt; e.ldt = B * ldv;
        LinearOpts ow;
        ow.tile_n = 256;
        linear(c, h, D, bw.a1.wq, R, 3 * D, D, e, ow);
      } else if (P == 1) {
        linear(c, h, D, bw.a1.wq, R, 2 * D, D, e, o);  // fused q|k projection
      }
      if (P == 1) {
        for (int b = 0; b < B && !fused_qkv; ++b)  // V^T, one column block per batch
          linear_vt(c, h + static_cast<int64_t>(b) * N * D, N, 1, bw.a1.wv, bw.a1.bv, vt + b * ldv, B * ldv, ldv, q2, o);
        qknorm(c, qk, 2 * D, R, D, bw.a1.q_norm, cos_l, sin_l, rope_period, eps, bw.a1.k_norm);
        attention(c, qk, 2 * D, qk + D, 2 * D, vt, ldv, nullptr, att, D, B, Hh, N, N, D);
      } else {
        // ---- Ulysses: q/k (normed + RoPE'd, which needs the full feature row) and v leave in a head-blocked layout,
        // one all-to-all turns [Nl tokens, all heads] into [all tokens, Hl heads]; attention runs on the local heads;
        // a second all-to-all returns the output rows to their owners, K-blocked, straight into the to_out GEMM.
        GemmEpi ev;
        ev.mode = EPI_BF16; ev.out = p2p ? vrecv : vsend; ev.ldo = Csp; ev.bias = bw.a1.bv; ev.col_block = Csp; ev.col_block_stride = blk;
        QkOut qo;
        qo.out[0] = qsend; qo.out[1] = ksend; qo.heads_per_block = Hl; qo.block_stride = blk; qo.ld = Csp;
        PeerTable ot = {};
        if (p2p) {   // destination rank d receives this rank's block at [region][me] of its buffer
          ev.use_col_ptrs = 1;
          qo.use_peer = 1;
          for (int d = 0; d < P; ++d) {
            qo.peer[0].p[d] = peer_base[d] + static_cast<int64_t>(0 * P + me) * blk;
            qo.peer[1].p[d] = peer_base[d] + static_cast<int64_t>(1 * P + me) * blk;
            ev.col_ptrs.p[d] = peer_base[d] + static_cast<int64_t>(2 * P + me) * blk;
            ot.p[d] = peer_base[d] + static_cast<int64_t>(3 * P + me) * blk;
          }
        }
        if (packed_qkv) {
          // q | k | v as ONE projection over the packed [3D, D] operand (one launch instead of two at a row count where every
          // launch is latency-bound): q | k stay local (row-major, pitch 2D), the v columns go column-blocked to their
          // destination ranks
          GemmEpi eqkv = ev;
          eqkv.out = qk; eqkv.ldo = 2 * D; eqkv.bias = bw.a1.bq;
          eqkv.col_block_from = 2 * D; eqkv.blocked_out = ev.out; eqkv.blocked_ld = Csp;
          linear(c, h, D, bw.a1.wq, R, 3 * D, D, eqkv, o);
        } else {
          linear(c, h, D, bw.a1.wq, R, 2 * D, D, e, o);  // fused q|k projection
          linear(c, h, D, bw.a1.wv, R, D, D, ev, o);
        }
        qknorm(c, qk, 2 * D, R, D, bw.a1.q_norm, cos_l, sin_l, rope_period, eps, bw.a1.k_norm, &qo);
        if (p2p) {
          ProfScope ps(c, PROF_COMM, 0.0, 3.0 * 2.0 * P * blk * 2.0);
          dist_p2p_barrier(c, 0);   // everyone's q / k / v blocks have landed here, ours at the peers
        } else {
          ProfScope ps(c, PROF_COMM, 0.0, 3.0 * 2.0 * P * blk * 2.0);
          const void* sb[3] = {qsend, ksend, vsend};
          void* rb[3] = {qrecv, krecv, vrecv};
          dist_all_to_all_sp(c, sb, rb, 3, static_cast<size_t>(blk) * 2);
        }
        {
          ProfScope ps(c, PROF_OTHER, 0.0, 4.0 * N * Csp);
          launch_transpose_bf16(vrecv, Csp, N, Csp, vt_sp, ldv, st);
        }
        if (p2p) {
          attention(c, qrecv, Csp, krecv, Csp, vt_sp, ldv, nullptr, osend, Csp, 1, Hl, N, N, Csp, &ot, Nl);
          ProfScope ps(c, PROF_COMM, 0.0, 2.0 * P * blk * 2.0);
          dist_p2p_barrier(c, 1);   // every rank's attention rows for our tokens have landed in the o region
        } else {
          attention(c, qrecv, Csp, krecv, Csp, vt_sp, ldv, nullptr, osend, Csp, 1, Hl, N, N, Csp);
          ProfScope ps(c, PROF_COMM, 0.0, 2.0 * P * blk * 2.0);
          const void* sb[1] = {osend};
          void* rb[1] = {orecv};
          dist_all_to_all_sp(c, sb, rb, 1, static_cast<size_t>(blk) * 2);
        }
      }
      GemmEpi eo;  // x += (att Wo^T + bo) * gate_msa ; refresh the bf16 shadow
      eo.mode = EPI_GATE_RESID; eo.resid = x; eo.ldr = D; eo.bias = bw.a1.bo;
      eo.gate_a = ada + 2 * D; eo.gate_b = bw.sst + 2 * D; eo.gate_ld = ada_ld; eo.rows_per_gate = rows_per_b;
      eo.shadow = xb; eo.lds = D;
      if (P == 1) {
        linear(c, att, D, bw.a1.wo, R, D, D, eo, o);
      } else {   // the exchanged attention rows arrive K-blocked
        LinearOpts ok = o;
        ok.a_kblock = Csp; ok.a_kblock_stride = blk;
        linear(c, orecv, Csp, bw.a1.wo, R, D, D, eo, ok);
      }
    }
    {
      // cross-attention on the UN-normalised stream (T/LTXTransformerBlock.swift:205-214)
      GemmEpi e;
      e.mode = EPI_BF16; e.out = q2; e.ldo = D; e.bias = bw.a2.bq;
      linear(c, xb, D, bw.a2.wq, R, D, D, e, o);
      qknorm(c, q2, D, R, D, bw.a2.q_norm, nullptr, nullptr, 1, eps);
      const bf16* k2 = tc.k.as<bf16>() + static_cast<int64_t>(i) * B * S * D;
      const bf16* v2 = tc.vt.as<bf16>() + static_cast<int64_t>(i) * D * B * tc.ldv;
      attention(c, q2, D, k2, D, v2, tc.ldv, key_bias, att, D, B, Hh, Nq, S, D);
      GemmEpi eo;
      eo.mode = EPI_GATE_RESID; eo.resid = x; eo.ldr = D; eo.bias = bw.a2.bo; eo.scale = cas;
      const bool next_needs_shadow = skip_ff && (i + 1 < L) &&
                                     in_list(i + 1, flags->stg_blocks, flags->n_stg_blocks) && flags->skip_self_attn;
      if (next_needs_shadow) { eo.shadow = xb; eo.lds = D; }
      linear(c, att, D, bw.a2.wo, R, D, D, eo, o);
    }
    if (!skip_ff) {
      norm_mod(c, x, h, R, D, bw.sst + 3 * D, bw.sst + 4 * D, ada + 3 * D, ada + 4 * D, ada_ld, rows_per_b, eps, 0);
      GemmEpi e;
      e.mode = EPI_GELU_BF16; e.out = ffh; e.ldo = FFD; e.bias = bw.b_in;
      linear(c, h, D, bw.w_in, R, FFD, D, e, o);
      GemmEpi eo;
      eo.mode = EPI_GATE_RESID; eo.resid = x; eo.ldr = D; eo.bias = bw.b_out;
      eo.gate_a = ada + 5 * D; eo.gate_b = bw.sst + 5 * D; eo.gate_ld = ada_ld; eo.rows_per_gate = rows_per_b;
      const bool next_needs_shadow =
          (i + 1 < L) && in_list(i + 1, flags->stg_blocks, flags->n_stg_blocks) && flags->skip_self_attn;
      if (next_needs_shadow) { eo.shadow = xb; eo.lds = D; }
      linear(c, ffh, FFD, bw.w_out, R, D, FFD, eo, o);
    }
  }
  // ---- output head (T/LTXTransformer.swift:208-224): LayerNorm(no affine) * (1 + scale) + shift ; proj_out
  norm_mod(c, x, h, R, D, c->sst_out, c->sst_out + D, emb, emb, D, rows_per_b, eps, 1);
  GemmEpi e;
  e.mode = EPI_F32; e.out = (P > 1) ? c->sp_vel.ptr : out_velocity_dev; e.ldo = Cout; e.bias = c->b_out;
  linear(c, h, D, c->w_out, R, Cout, D, e, o);
  if (P > 1) {  // every rank receives the full velocity [N, Cout]
    ProfScope ps(c, PROF_COMM, 0.0, 4.0 * N * Cout);
    dist_allgather_sp(c, c->sp_vel.ptr, out_velocity_dev, static_cast<size_t>(Nl) * Cout * 4);
  }
}

}  // namespace ltx
