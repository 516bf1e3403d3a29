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

// the e4m3 replacement of a weight (precision mode 8), or nullptr
const QuantW* fp8_weight(const ltx_ctx* c, const void* w) {
  if (c->qw.empty()) return nullptr;
  auto it = c->qw.find(w);
  return (it != c->qw.end() && it->second.fmt == QF_E4M3) ? &it->second : nullptr;
}

// Precision mode 8: A's rows become e4m3 codes + power-of-two row scales in one reused scratch buffer, then the FP8 pair kernel
// runs for every M (no weight-streaming, 1-CTA or swap-AB form), so each row's result depends on that row alone: a batched
// forward equals its items' forwards bit for bit.  Rows [0, N) of the weight are used (the q|k rows of the packed q|k|v).
void gemm_fp8(ltx_ctx* c, const bf16* A, int64_t lda, const QuantW& W, int M, int N, int K, const GemmEpi& e, int force_bn) {
  LTX_CHECK(W.k == K && W.n >= N, LTX_ERR_INVALID_ARGUMENT, "FP8 GEMM: weight shape mismatch");
  const size_t code_bytes = (static_cast<size_t>(M) * K + 15) / 16 * 16;
  c->fp8_act.reserve(code_bytes + static_cast<size_t>(M) * 4);
  uint8_t* q = c->fp8_act.as<uint8_t>();
  float* s = reinterpret_cast<float*>(q + code_bytes);
  {
    ProfScope ps(c, PROF_ROW, 0.0, 3.0 * M * K + 4.0 * M);
    launch_quantize_rows_fp8(A, lda, M, K, q, s, c->stream);
  }
  ProfScope ps(c, PROF_GEMM, 2.0 * M * N * K, static_cast<double>(M) * K + static_cast<double>(N) * K + 2.0 * M * N);
  launch_gemm_fp8(q, K, s, W.q, W.k, W.scales, M, N, K, e, c->stream, force_bn);
}

// profiled launch helpers (flop / byte counts are the algorithmic ones used by bench.py's roofline)
void gemm(ltx_ctx* c, const bf16* A, int64_t lda, const bf16* B, int64_t ldb, int M, int N, int K, const GemmEpi& e,
          int a_kblock = 0, int64_t a_kblock_stride = 0) {
  if (const QuantW* w8 = fp8_weight(c, B)) {
    LTX_CHECK(a_kblock == 0, LTX_ERR_UNSUPPORTED, "FP8 GEMM: no K-blocked A operand");
    gemm_fp8(c, A, lda, *w8, M, N, K, e, 0);
    return;
  }
  auto it = c->qw.empty() ? c->qw.end() : c->qw.find(B);
  const bool panel = it != c->qw.end() && gemm_q_uses_panel(it->second, M);
  ProfScope ps(c, PROF_GEMM, 2.0 * M * N * K, 2.0 * (static_cast<double>(M) * K + static_cast<double>(N) * K + static_cast<double>(M) * N),
               panel ? 2 : 1);
  if (it != c->qw.end()) {   // weight was replaced by int8 / int4 codes: dequant-fused kernel, or panel + bf16 kernel for large M
    launch_gemm_q(A, lda, it->second, M, N, K, e, c->stream, 0, a_kblock, a_kblock_stride);
    return;
  }
  if (M <= 512) {   // few rows (an Ulysses shard, a small clip): opt in to the weight-streaming kernel
    GemmEpi ew = e;
    gemm_attach_workspace(c, ew);
    launch_gemm(A, lda, B, ldb, M, N, K, ew, c->stream, 0, a_kblock, a_kblock_stride);
    return;
  }
  launch_gemm(A, lda, B, ldb, M, N, K, e, c->stream, 0, a_kblock, a_kblock_stride);
}
// V^T [D, ncols] (row pitch ld_out) = (h Wv^T + bv)^T for one batch.  bf16 weights: run the projection with the weight as
// the A operand so the result lands transposed; quantised weights must be the B operand: project into `tmp`, transpose.
void v_transposed(ltx_ctx* c, const bf16* wv, const float* bv, const bf16* hrows, int rows, int D, bf16* out, int64_t ld_out,
                  bf16* tmp) {
  if (c->qw.empty() || c->qw.find(wv) == c->qw.end()) {
    GemmEpi ev;
    ev.mode = EPI_BF16; ev.out = out; ev.ldo = ld_out; ev.bias = bv; ev.bias_per_row = 1;
    gemm(c, wv, D, hrows, D, D, rows, D, ev);
    return;
  }
  GemmEpi ev;
  ev.mode = EPI_BF16; ev.out = tmp; ev.ldo = D; ev.bias = bv;
  gemm(c, hrows, D, wv, D, rows, D, D, ev);
  ProfScope ps(c, PROF_OTHER, 0.0, 4.0 * rows * D);
  launch_transpose_bf16(tmp, D, rows, D, out, ld_out, c->stream);
}
void attention(ltx_ctx* c, const bf16* Q, int64_t ldq, const bf16* K, int64_t ldk, const bf16* Vt, int64_t ldvb,
               const float* bias, bf16* O, int64_t ldo, int B, int H, int Nq, int Nk, int D, float scale,
               const PeerTable* o_blocks = nullptr, int rows_per_block = 0) {
  ProfScope ps(c, PROF_ATTN, 4.0 * B * H * static_cast<double>(Nq) * Nk * 128.0,
               2.0 * B * (2.0 * Nq + 2.0 * Nk) * D);
  launch_attention(Q, ldq, K, ldk, Vt, ldvb, bias, O, ldo, B, H, Nq, Nk, D, scale, c->stream, o_blocks, rows_per_block);
}
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
  GemmEpi e;
  e.mode = EPI_GELU_BF16; e.out = c->c1.ptr; e.ldo = D; e.bias = src.b_c1;
  gemm(c, ctx_bf, Cc, src.w_c1, Cc, static_cast<int>(R), D, Cc, e);
  e.mode = EPI_BF16; e.out = c->c2.ptr; e.bias = src.b_c2;
  gemm(c, c->c1.as<bf16>(), D, src.w_c2, D, static_cast<int>(R), D, D, e);
  for (int i = 0; i < L; ++i) {
    const AttnWeights& a = src.layer(src.user, i);
    bf16* kd = tc.k.as<bf16>() + static_cast<int64_t>(i) * R * D;
    bf16* vd = tc.vt.as<bf16>() + static_cast<int64_t>(i) * D * B * tc.ldv;
    GemmEpi ek;
    ek.mode = EPI_BF16; ek.out = kd; ek.ldo = D; ek.bias = a.bk;
    gemm(c, c->c2.as<bf16>(), D, a.wk, D, static_cast<int>(R), D, D, ek);
    qknorm(c, kd, D, static_cast<int>(R), D, a.k_norm, nullptr, nullptr, 1, g.norm_eps);
    for (int b = 0; b < B; ++b)  // V^T[D, S] per batch, one column block each
      v_transposed(c, a.wv, a.bv, c->c2.as<bf16>() + static_cast<int64_t>(b) * S * D, S, D, vd + b * tc.ldv, B * tc.ldv,
                   c->c1.as<bf16>());
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
  c->w_patch = wbf(c, "patchify_proj.weight", D, g.in_channels);
  c->b_patch = wf(c, "patchify_proj.bias", D);
  c->w_t1 = wbf(c, "adaln_single.emb.linear_1.weight", D, 256);
  c->b_t1 = wf(c, "adaln_single.emb.linear_1.bias", D);
  c->w_t2 = wbf(c, "adaln_single.emb.linear_2.weight", D, D);
  c->b_t2 = wf(c, "adaln_single.emb.linear_2.bias", D);
  c->w_ada = wbf(c, "adaln_single.linear.weight", 6 * D, D);
  c->b_ada = wf(c, "adaln_single.linear.bias", 6 * D);
  c->w_c1 = wbf(c, "caption_projection.linear_1.weight", D, g.caption_channels);
  c->b_c1 = wf(c, "caption_projection.linear_1.bias", D);
  c->w_c2 = wbf(c, "caption_projection.linear_2.weight", D, D);
  c->b_c2 = wf(c, "caption_projection.linear_2.bias", D);
  c->sst_out = wf(c, "scale_shift_table", 2 * D);
  c->w_out = wbf(c, "proj_out.weight", g.out_channels, D);
  c->b_out = wf(c, "proj_out.bias", g.out_channels);
  c->blocks.assign(g.num_layers, BlockWeights());
  for (int i = 0; i < g.num_layers; ++i) {
    const std::string p = "transformer_blocks." + std::to_string(i) + ".";
    BlockWeights& b = c->blocks[i];
    b.sst = wf(c, p + "scale_shift_table", 6 * D);
    // attn1: pack q|k|v into one [3D, D] operand: the three projections of the block run as ONE GEMM (N = 3D; V leaves its
    // epilogue transposed); the Ulysses / quantised paths address the q|k rows and the v rows of the same buffer separately
    {
      const bf16* wq = wbf(c, p + "attn1.to_q.weight", D, D);
      const bf16* wk = wbf(c, p + "attn1.to_k.weight", D, D);
      const bf16* wv = wbf(c, p + "attn1.to_v.weight", D, D);
      const float* bq = wf(c, p + "attn1.to_q.bias", D);
      const float* bk = wf(c, p + "attn1.to_k.bias", D);
      const float* bvv = wf(c, p + "attn1.to_v.bias", D);
      bf16* wqkv = nullptr;
      float* bqkv = nullptr;
      LTX_CUDA(cudaMalloc(&wqkv, static_cast<size_t>(3) * D * D * 2));
      c->owned.push_back(wqkv);
      LTX_CUDA(cudaMalloc(&bqkv, static_cast<size_t>(3) * D * 4));
      c->owned.push_back(bqkv);
      const bf16* ws[3] = {wq, wk, wv};
      const float* bs[3] = {bq, bk, bvv};
      for (int t = 0; t < 3; ++t) {
        LTX_CUDA(cudaMemcpyAsync(wqkv + static_cast<size_t>(t) * D * D, ws[t], static_cast<size_t>(D) * D * 2, cudaMemcpyDeviceToDevice, c->stream));
        LTX_CUDA(cudaMemcpyAsync(bqkv + static_cast<size_t>(t) * D, bs[t], static_cast<size_t>(D) * 4, cudaMemcpyDeviceToDevice, c->stream));
      }
      LTX_CUDA(cudaStreamSynchronize(c->stream));
      // the unpacked copies are no longer needed
      for (const char* k : {"attn1.to_q.weight", "attn1.to_k.weight", "attn1.to_v.weight"}) {
        auto it = c->tensors.find(p + k);
        cudaFree(it->second.ptr);
        c->tensors.erase(it);
      }
      b.a1.wq = wqkv; b.a1.wk = wqkv + D * D; b.a1.wv = wqkv + 2 * D * D;
      b.a1.bq = bqkv; b.a1.bk = bqkv + D; b.a1.bv = bqkv + 2 * D;
    }
    b.a1.wo = wbf(c, p + "attn1.to_out.weight", D, D);
    b.a1.bo = wf(c, p + "attn1.to_out.bias", D);
    b.a1.q_norm = wf(c, p + "attn1.q_norm.weight", D);
    b.a1.k_norm = wf(c, p + "attn1.k_norm.weight", D);
    b.a2.wq = wbf(c, p + "attn2.to_q.weight", D, D);
    b.a2.bq = wf(c, p + "attn2.to_q.bias", D);
    b.a2.wk = wbf(c, p + "attn2.to_k.weight", D, D);
    b.a2.bk = wf(c, p + "attn2.to_k.bias", D);
    b.a2.wv = wbf(c, p + "attn2.to_v.weight", D, D);
    b.a2.bv = wf(c, p + "attn2.to_v.bias", D);
    b.a2.wo = wbf(c, p + "attn2.to_out.weight", D, D);
    b.a2.bo = wf(c, p + "attn2.to_out.bias", D);
    b.a2.q_norm = wf(c, p + "attn2.q_norm.weight", D);
    b.a2.k_norm = wf(c, p + "attn2.k_norm.weight", D);
    b.w_in = wbf(c, p + "ff.project_in.proj.weight", FF, D);
    b.b_in = wf(c, p + "ff.project_in.proj.bias", FF);
    b.w_out = wbf(c, p + "ff.project_out.weight", D, FF);
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
  const int D = g.num_heads * g.head_dim, FF = g.ffn_mult * D;
  auto release = [&](const void* p) { release_weight(c, p); };
  // Each quantised weight gets a 16-byte device allocation whose address is its identity from now on: the struct field
  // is repointed to it and gemm() recognises it in c->qw (the freed bf16 address could be handed out again by cudaMalloc).
  std::vector<const void*> to_free;
  auto qf = [&](const bf16*& w, int N, int K) {
    LTX_CHECK(K % 64 == 0, LTX_ERR_INVALID_CONFIGURATION, "quantisation needs every Linear input width to be a multiple of 64");
    uint8_t* q = nullptr;
    float *s = nullptr, *b = nullptr;
    void* handle = nullptr;
    const size_t qbytes = static_cast<size_t>(N) * K * bits / 8, sbytes = static_cast<size_t>(K / 64) * N * 4;
    LTX_CUDA(cudaMalloc(&q, qbytes));
    LTX_CUDA(cudaMalloc(&s, sbytes));
    LTX_CUDA(cudaMalloc(&b, sbytes));
    LTX_CUDA(cudaMalloc(&handle, 16));
    c->owned.push_back(q); c->owned.push_back(s); c->owned.push_back(b); c->owned.push_back(handle);
    launch_quantize(w, N, K, bits, q, s, b, c->stream);
    QuantW r;
    r.q = q; r.scales = s; r.biases = b; r.bits = bits; r.n = N; r.k = K;
    if (c->quant_materialise) {
      // materialised storage: the weight keeps its place and dtype, its values become s * q + beta (the panel conversion's
      // arithmetic and rounding, i.e. exactly what the fused kernels would feed the tensor cores); the codes are dropped
      launch_dequantize_panel(r, const_cast<bf16*>(w), c->stream);
      LTX_CUDA(cudaStreamSynchronize(c->stream));
      for (void* ptr : {static_cast<void*>(q), static_cast<void*>(s), static_cast<void*>(b), handle}) {
        cudaFree(ptr);
        c->owned.erase(std::find(c->owned.begin(), c->owned.end(), ptr));
      }
      return;
    }
    LTX_CUDA(cudaStreamSynchronize(c->stream));
    c->qw[handle] = r;
    to_free.push_back(w);
    w = reinterpret_cast<const bf16*>(handle);
  };
  const bool codes = !c->quant_materialise;
  qf(c->w_patch, D, g.in_channels);
  qf(c->w_c1, D, g.caption_channels);
  qf(c->w_c2, D, D);
  qf(c->w_out, g.out_channels, D);
  for (auto& b : c->blocks) {
    qf(b.a1.wq, 2 * D, D);            // packed q|k (the v rows behind them are quantised by the next call: rows are independent)
    if (codes) b.a1.wk = nullptr;
    qf(b.a1.wv, D, D); qf(b.a1.wo, D, D);
    qf(b.a2.wq, D, D); qf(b.a2.wk, D, D); qf(b.a2.wv, D, D); qf(b.a2.wo, D, D);
    qf(b.w_in, FF, D); qf(b.w_out, D, FF);
  }
  if (c->av.ready) {
    // the dual model's Linears (quantize(model: ltx2, groupSize: 64, bits:), Pipeline/LTXPipeline.swift:491); the AdaLN-single
    // embedders stay bf16 like the video model's timestep MLP
    AvWeights& a = c->av;
    const int Da = a.Da, FFa = g.ffn_mult * Da, Ca = a.Cin;
    qf(a.w_patch, Da, Ca);
    qf(a.w_c1, Da, g.caption_channels);
    qf(a.w_c2, Da, Da);
    qf(a.w_out, Ca, Da);
    auto qattn = [&](AttnWeights& w, int qdim, int cdim, int inner) {
      qf(w.wq, inner, qdim); qf(w.wk, inner, cdim); qf(w.wv, inner, cdim); qf(w.wo, qdim, inner);
    };
    for (auto& b : a.blocks) {
      qattn(b.aa1, Da, Da, Da);
      qattn(b.aa2, Da, Da, Da);
      qattn(b.a2v, D, Da, Da);
      qattn(b.v2a, Da, D, Da);
      qf(b.w_in, FFa, Da); qf(b.w_out, Da, FFa);
    }
  }
  if (!codes) { c->quant_bits = bits; return; }   // materialised: the structs still point at (now dequantised) bf16 weights
  for (const void* p : to_free) release(p);
  // one bf16 panel for the large-M path of launch_gemm_q, sized for the largest weight (the FFN matrices)
  size_t max_elems = 0;
  for (auto& kv : c->qw) max_elems = std::max(max_elems, static_cast<size_t>(kv.second.n) * kv.second.k);
  c->q_panel.reserve(max_elems * 2);
  for (auto& kv : c->qw) kv.second.scratch = c->q_panel.as<bf16>();
  c->quant_bits = bits;
}

// Precision mode 8: every Linear inside the transformer blocks becomes e4m3 codes with one power-of-two scale per output
// channel (launch_quantize_rows_fp8: the rule gemm() applies to the activation rows); the bf16 copies are freed.  Patchify,
// caption projection, the timestep MLPs / AdaLN and proj_out stay bf16.  The weights are found through dit_quantize's
// handles, with the e4m3 format in their map entry.
void dit_convert_fp8(ltx_ctx* c) {
  LTX_CHECK(c->dit_ready && c->qw.empty(), LTX_ERR_WEIGHTS, "FP8 conversion needs finalized, unquantised DiT weights");
  const ltx_config& g = c->cfg;
  const int D = g.num_heads * g.head_dim, FF = g.ffn_mult * D;
  LTX_CHECK(D % 16 == 0 && FF % 16 == 0, LTX_ERR_INVALID_CONFIGURATION, "FP8 mode needs Linear widths that are multiples of 16");
  std::vector<const void*> to_free;
  auto handle_for = [&](const QuantW& r) {
    void* handle = nullptr;
    LTX_CUDA(cudaMalloc(&handle, 16));
    c->owned.push_back(handle);
    c->qw[handle] = r;
    return reinterpret_cast<const bf16*>(handle);
  };
  auto conv = [&](const bf16*& w, int N, int K) {
    uint8_t* q = nullptr;
    float* s = nullptr;
    LTX_CUDA(cudaMalloc(&q, static_cast<size_t>(N) * K));
    LTX_CUDA(cudaMalloc(&s, static_cast<size_t>(N) * 4));
    c->owned.push_back(q); c->owned.push_back(s);
    launch_quantize_rows_fp8(w, K, N, K, q, s, c->stream);
    QuantW r;
    r.fmt = QF_E4M3; r.q = q; r.scales = s; r.bits = 8; r.n = N; r.k = K;
    to_free.push_back(w);
    w = handle_for(r);
    return r;
  };
  for (auto& b : c->blocks) {
    // the packed q|k|v [3D, D] as one matrix, so the fused projection with its V^T epilogue stays one launch; its v rows get
    // a handle of their own (rows are independent) for the per-batch V^T projections
    QuantW v = conv(b.a1.wq, 3 * D, D);
    v.q += static_cast<size_t>(2) * D * D; v.scales += 2 * D; v.n = D;
    b.a1.wk = nullptr;
    b.a1.wv = handle_for(v);
    conv(b.a1.wo, D, D);
    conv(b.a2.wq, D, D); conv(b.a2.wk, D, D); conv(b.a2.wv, D, D); conv(b.a2.wo, D, D);
    conv(b.w_in, FF, D); conv(b.w_out, D, FF);
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
  const float att_scale = 1.0f / sqrtf(static_cast<float>(g.head_dim));
  cudaStream_t st = c->stream;
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
    gemm(c, lat_bf, Cin, c->w_patch, Cin, R, D, Cin, e);
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
    ProfScope ps(c, PROF_OTHER, 2.0 * B * D * (256.0 + 7.0 * D), 2.0 * D * (256.0 + 7.0 * D), 4);
    launch_sincos_embed(timesteps_dev, g.timestep_scale_multiplier, c->se.as<float>(), B, 256, st);
    launch_gemv(c->w_t1, c->b_t1, c->se.as<float>(), c->t1.as<float>(), B, D, 256, 0, st);
    launch_gemv(c->w_t2, c->b_t2, c->t1.as<float>(), emb, B, D, D, 1, st);
    launch_gemv(c->w_ada, c->b_ada, emb, ada, B, 6 * D, D, 1, st);
  } else {
    // one embedding per token: the same three Linears as tensor-core GEMMs over the R local rows (bf16 operands, the
    // SiLUs fused into the first epilogue / a cast pass); timesteps [B, N] are indexed from this rank's first token
    bf16* se_bf = reinterpret_cast<bf16*>(c->se.ptr);      // [R, 256] bf16
    bf16* t1_bf = reinterpret_cast<bf16*>(c->t1.ptr);      // [R, D] bf16 = silu(linear_1), later silu(emb)
    {
      ProfScope ps(c, PROF_OTHER, 0.0, 4.0 * R + 512.0 * R);
      launch_sincos_embed(timesteps_dev + tok0, g.timestep_scale_multiplier, nullptr, R, 256, st, se_bf);
    }
    GemmEpi e1;
    e1.mode = EPI_SILU_BF16; e1.out = t1_bf; e1.ldo = D; e1.bias = c->b_t1;
    gemm(c, se_bf, 256, c->w_t1, 256, R, D, 256, e1);
    GemmEpi e2;
    e2.mode = EPI_F32; e2.out = emb; e2.ldo = D; e2.bias = c->b_t2;
    gemm(c, t1_bf, D, c->w_t2, D, R, D, D, e2);
    {
      ProfScope ps(c, PROF_OTHER, 0.0, 6.0 * R * D);
      launch_silu_cast(emb, t1_bf, static_cast<int64_t>(R) * D, st);
    }
    GemmEpi e3;
    e3.mode = EPI_F32; e3.out = ada; e3.ldo = 6 * D; e3.bias = c->b_ada;
    gemm(c, t1_bf, D, c->w_ada, D, R, 6 * D, D, e3);
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
      const QuantW* qkv8 = fp8_weight(c, bw.a1.wq);
      const bool fused_qkv = P == 1 && (B == 1 || ldv == N) && (c->qw.empty() || qkv8) && D % 32 == 0;
      GemmEpi e;
      e.mode = EPI_BF16; e.out = qk; e.ldo = 2 * D; e.bias = bw.a1.bq;
      if (fused_qkv && qkv8) {
        e.tsplit_col = 2 * D; e.out_t = vt; e.ldt = B * ldv;
        gemm_fp8(c, h, D, *qkv8, R, 3 * D, D, e, 256);
      } else if (fused_qkv) {
        e.tsplit_col = 2 * D; e.out_t = vt; e.ldt = B * ldv;
        ProfScope ps(c, PROF_GEMM, 2.0 * R * 3.0 * D * D, 2.0 * (static_cast<double>(R) * D + 3.0 * D * D + 3.0 * R * D));
        launch_gemm(h, D, bw.a1.wq, D, R, 3 * D, D, e, st, R > 128 ? 1256 : 256);
      } else if (P == 1) {
        gemm(c, h, D, bw.a1.wq, D, R, 2 * D, D, e);  // fused q|k projection
      }
      if (P == 1) {
        for (int b = 0; b < B && !fused_qkv; ++b)  // V^T, one column block per batch
          v_transposed(c, bw.a1.wv, bw.a1.bv, h + static_cast<int64_t>(b) * N * D, N, D, vt + b * ldv, B * ldv, q2);
        qknorm(c, qk, 2 * D, R, D, bw.a1.q_norm, cos_l, sin_l, rope_period, eps, bw.a1.k_norm);
        attention(c, qk, 2 * D, qk + D, 2 * D, vt, ldv, nullptr, att, D, B, Hh, N, N, D, att_scale);
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
        if (c->qw.empty()) {
          // bf16 weights: q | k | v as ONE projection over the packed [3D, D] operand (one launch instead of two at a row count
          // where every launch is latency-bound): q | k stay local (row-major, pitch 2D), the v columns go column-blocked to
          // their destination ranks
          GemmEpi eqkv = ev;
          eqkv.out = qk; eqkv.ldo = 2 * D; eqkv.bias = bw.a1.bq;
          eqkv.col_block_from = 2 * D; eqkv.blocked_out = ev.out; eqkv.blocked_ld = Csp;
          gemm(c, h, D, bw.a1.wq, D, R, 3 * D, D, eqkv);
        } else {
          gemm(c, h, D, bw.a1.wq, D, R, 2 * D, D, e);  // fused q|k projection
          gemm(c, h, D, bw.a1.wv, D, R, D, D, ev);
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
          attention(c, qrecv, Csp, krecv, Csp, vt_sp, ldv, nullptr, osend, Csp, 1, Hl, N, N, Csp, att_scale, &ot, Nl);
          ProfScope ps(c, PROF_COMM, 0.0, 2.0 * P * blk * 2.0);
          dist_p2p_barrier(c, 1);   // every rank's attention rows for our tokens have landed in the o region
        } else {
          attention(c, qrecv, Csp, krecv, Csp, vt_sp, ldv, nullptr, osend, Csp, 1, Hl, N, N, Csp, att_scale);
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
      if (P == 1)
        gemm(c, att, D, bw.a1.wo, D, R, D, D, eo);
      else
        gemm(c, orecv, Csp, bw.a1.wo, D, R, D, D, eo, Csp, blk);
    }
    {
      // cross-attention on the UN-normalised stream (T/LTXTransformerBlock.swift:205-214)
      GemmEpi e;
      e.mode = EPI_BF16; e.out = q2; e.ldo = D; e.bias = bw.a2.bq;
      gemm(c, xb, D, bw.a2.wq, D, R, D, D, e);
      qknorm(c, q2, D, R, D, bw.a2.q_norm, nullptr, nullptr, 1, eps);
      const bf16* k2 = tc.k.as<bf16>() + static_cast<int64_t>(i) * B * S * D;
      const bf16* v2 = tc.vt.as<bf16>() + static_cast<int64_t>(i) * D * B * tc.ldv;
      attention(c, q2, D, k2, D, v2, tc.ldv, key_bias, att, D, B, Hh, Nq, S, D, att_scale);
      GemmEpi eo;
      eo.mode = EPI_GATE_RESID; eo.resid = x; eo.ldr = D; eo.bias = bw.a2.bo; eo.scale = cas;
      const bool next_needs_shadow = skip_ff && (i + 1 < L) &&
                                     in_list(i + 1, flags->stg_blocks, flags->n_stg_blocks) && flags->skip_self_attn;
      if (next_needs_shadow) { eo.shadow = xb; eo.lds = D; }
      gemm(c, att, D, bw.a2.wo, D, R, D, D, eo);
    }
    if (!skip_ff) {
      norm_mod(c, x, h, R, D, bw.sst + 3 * D, bw.sst + 4 * D, ada + 3 * D, ada + 4 * D, ada_ld, rows_per_b, eps, 0);
      GemmEpi e;
      e.mode = EPI_GELU_BF16; e.out = ffh; e.ldo = FFD; e.bias = bw.b_in;
      gemm(c, h, D, bw.w_in, D, R, FFD, D, e);
      GemmEpi eo;
      eo.mode = EPI_GATE_RESID; eo.resid = x; eo.ldr = D; eo.bias = bw.b_out;
      eo.gate_a = ada + 5 * D; eo.gate_b = bw.sst + 5 * D; eo.gate_ld = ada_ld; eo.rows_per_gate = rows_per_b;
      const bool next_needs_shadow =
          (i + 1 < L) && in_list(i + 1, flags->stg_blocks, flags->n_stg_blocks) && flags->skip_self_attn;
      if (next_needs_shadow) { eo.shadow = xb; eo.lds = D; }
      gemm(c, ffh, FFD, bw.w_out, FFD, R, D, FFD, eo);
    }
  }
  // ---- output head (T/LTXTransformer.swift:208-224): LayerNorm(no affine) * (1 + scale) + shift ; proj_out
  norm_mod(c, x, h, R, D, c->sst_out, c->sst_out + D, emb, emb, D, rows_per_b, eps, 1);
  GemmEpi e;
  e.mode = EPI_F32; e.out = (P > 1) ? c->sp_vel.ptr : out_velocity_dev; e.ldo = Cout; e.bias = c->b_out;
  gemm(c, h, D, c->w_out, D, R, Cout, D, e);
  if (P > 1) {  // every rank receives the full velocity [N, Cout]
    ProfScope ps(c, PROF_COMM, 0.0, 4.0 * N * Cout);
    dist_allgather_sp(c, c->sp_vel.ptr, out_velocity_dev, static_cast<size_t>(Nl) * Cout * 4);
  }
}

}  // namespace ltx
