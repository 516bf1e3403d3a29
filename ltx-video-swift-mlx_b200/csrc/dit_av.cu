// Dual audio / video DiT forward (SURVEY 8f-1): LTX2Transformer.callAsFunction (Models/Transformer/LTX2Transformer.swift:240-392)
// and LTX2TransformerBlock.callAsFunction (Models/Transformer/LTX2TransformerBlock.swift:174-297) on the kernels of the
// video-only path -- the "19 B" model: a second, 2048-wide token stream (32 heads x 64) for the audio latent, learned
// RMSNorms in front of every sub-layer, and two cross-modal attentions per block (audio -> video, video -> audio) whose
// queries / keys carry temporal-only RoPE and whose modulation comes from four extra AdaLN-single embedders.
//
// Streams (token-major rows):  video x fp32 [B*N, D] (D = 4096),  audio ax fp32 [B*Ta, Da] (Da = 2048), B = 1 or 2 items
// (the conditional and unconditional passes of a CFG step as one batched forward).
// Everything GEMM-shaped runs on gemm_bf16_tcgen05 / gemm_bf16_2cta, every attention on attention_fwd_tcgen05 (head_dim 128
// for the video stream, 64 for audio and cross-modal); the learned-weight norm + modulation and the head_dim-generic q/k
// norm + RoPE are the two row kernels below.  Text K / V of both streams are step-invariant and cached like the video-only
// model's.  The video sigma is one scalar, or one value per video token (the image-to-video mode feeds sigma * (1 - mask),
// Pipeline/LTXPipeline.swift:1293-1298; every video-side embedder then runs per token, LTX2Transformer.swift:273-298).
// Weights: bf16, or int8 / int4 codes through the dequant-fused GEMM (quantize(model: ltx2, ...), Pipeline/LTXPipeline.swift:491).
// Every per-row kernel and GEMM row gives each item the arithmetic of its B = 1 forward: at B = 2 the audio stream's
// 2 x Ta <= 64 rows take the 64-row form of the weight-streaming GEMM, and every modulation / gate / RoPE row is looked
// up per item (or per token).  Restrictions of this version: B <= 2, single GPU.
#include <algorithm>
#include <cmath>

#include "ctx.h"
#include "ptx.cuh"

namespace ltx {

namespace {

__device__ __forceinline__ float block_sum_256(float v, float* red) {
  v = warp_sum(v);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = 0.f;
  for (int w = 0; w < (blockDim.x >> 5); ++w) t += red[w];
  return t;
}

// out_bf16[m, :] = rms(x[m, :]) * w * (1 + sc_t + sc_a) + sh_t + sh_a   (any of w, sc_*, sh_* may be null)
// RMSNorm(dims:eps:) with a learned weight (T/LTXAttention.swift:12-25) followed by the AdaLN modulation of
// T/LTX2TransformerBlock.swift:208-281; one row per CTA.
__global__ void __launch_bounds__(256) rmsnorm_w_mod_kernel(const float* x, bf16* out, int D, const float* w, const float* sc_t,
                                                             const float* sc_a, const float* sh_t, const float* sh_a, int64_t a_ld,
                                                             int a_rpr, float eps) {
  __shared__ float red[8];
  griddep_launch();
  griddep_wait();
  const int row = blockIdx.x;
  if (sc_a) {   // a_ld > 0: one modulation row per a_rpr rows (1: per token, N / Ta: per batch item)
    sc_a += (row / a_rpr) * a_ld;
    sh_a += (row / a_rpr) * a_ld;
  }
  const float4* xr = reinterpret_cast<const float4*>(x + static_cast<int64_t>(row) * D);
  const int nv = D >> 2;
  float ss = 0.f;
  for (int i = threadIdx.x; i < nv; i += blockDim.x) {
    const float4 v = xr[i];
    ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  const float rstd = rsqrtf(block_sum_256(ss, red) / D + eps);
  bf16* orow = out + static_cast<int64_t>(row) * D;
  auto ld4 = [](const float* p, int i, float dflt) {
    return p ? reinterpret_cast<const float4*>(p)[i] : make_float4(dflt, dflt, dflt, dflt);
  };
  for (int i = threadIdx.x; i < nv; i += blockDim.x) {
    const float4 v = xr[i];
    const float4 ww = ld4(w, i, 1.f), a = ld4(sc_t, i, 0.f), b = ld4(sc_a, i, 0.f), cc = ld4(sh_t, i, 0.f), d = ld4(sh_a, i, 0.f);
    const float y0 = v.x * rstd * ww.x * (1.f + a.x + b.x) + cc.x + d.x;
    const float y1 = v.y * rstd * ww.y * (1.f + a.y + b.y) + cc.y + d.y;
    const float y2 = v.z * rstd * ww.z * (1.f + a.z + b.z) + cc.z + d.z;
    const float y3 = v.w * rstd * ww.w * (1.f + a.w + b.w) + cc.w + d.w;
    reinterpret_cast<uint2*>(orow)[i] = make_uint2(pack_bf16(y0, y1), pack_bf16(y2, y3));
  }
}

// Fast path of the same op for D == 4 * VPT * 256 (4096: video, 2048: audio): a CTA owns ROWS rows whose loads are all issued
// up front and whose sums of squares are reduced together; the combined per-channel scale w * (1 + sc_t + sc_a) and shift are
// formed once per CTA.  NOUT = 2 writes two differently modulated copies of the same normalised rows (the cross-modal
// attentions use each stream once as query and once as context, T/LTX2TransformerBlock.swift:244-268): one read of x.
struct ModSet {
  const float *sc_t, *sc_a, *sh_t, *sh_a;
  bf16* out;
  int64_t a_ld;   // 0: sc_a / sh_a are one vector shared by all rows; > 0: row r uses sc_a + (r / rpr) * a_ld
  int rpr;        // rows per modulation row: 1 (per-token sigmas) or the rows of one batch item
};
template <int VPT, int ROWS, int NOUT>
__global__ void __launch_bounds__(256) rmsnorm_w_mod_fast_kernel(const float* x, int M, const float* w, const ModSet m0,
                                                                  const ModSet m1, float eps) {
  __shared__ float red[8 * ROWS];
  constexpr int D = 4 * VPT * 256;
  const int row0 = blockIdx.x * ROWS;
  griddep_launch();
  griddep_wait();
  float4 v[ROWS][VPT];
#pragma unroll
  for (int rr = 0; rr < ROWS; ++rr) {
    const float4* xr = reinterpret_cast<const float4*>(x + static_cast<int64_t>(row0 + rr) * D);
#pragma unroll
    for (int k = 0; k < VPT; ++k)
      v[rr][k] = (row0 + rr < M) ? xr[threadIdx.x + k * 256] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float s2[ROWS];
#pragma unroll
  for (int rr = 0; rr < ROWS; ++rr) {
    s2[rr] = 0.f;
#pragma unroll
    for (int k = 0; k < VPT; ++k)
      s2[rr] += v[rr][k].x * v[rr][k].x + v[rr][k].y * v[rr][k].y + v[rr][k].z * v[rr][k].z + v[rr][k].w * v[rr][k].w;
  }
  {   // ROWS sums at once, fixed summation order
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int rr = 0; rr < ROWS; ++rr) s2[rr] = warp_sum(s2[rr]);
    if (lane == 0) {
#pragma unroll
      for (int rr = 0; rr < ROWS; ++rr) red[warp * ROWS + rr] = s2[rr];
    }
    __syncthreads();
#pragma unroll
    for (int rr = 0; rr < ROWS; ++rr) {
      float t = 0.f;
      for (int ww = 0; ww < 8; ++ww) t += red[ww * ROWS + rr];
      s2[rr] = rsqrtf(t / D + eps);
    }
  }
  auto ld4 = [](const float* p, int i, float dflt) {
    return p ? reinterpret_cast<const float4*>(p)[i] : make_float4(dflt, dflt, dflt, dflt);
  };
#pragma unroll
  for (int o = 0; o < NOUT; ++o) {
    const ModSet& m = o == 0 ? m0 : m1;
    float4 sc[VPT], sh[VPT];
    auto combine = [&](int64_t aoff) {
#pragma unroll
      for (int k = 0; k < VPT; ++k) {
        const int i = threadIdx.x + k * 256;
        const float4 ww = ld4(w, i, 1.f), a = ld4(m.sc_t, i, 0.f), b = ld4(m.sc_a ? m.sc_a + aoff : nullptr, i, 0.f),
                     cc = ld4(m.sh_t, i, 0.f), d = ld4(m.sh_a ? m.sh_a + aoff : nullptr, i, 0.f);
        sc[k] = make_float4(ww.x * (1.f + a.x + b.x), ww.y * (1.f + a.y + b.y), ww.z * (1.f + a.z + b.z), ww.w * (1.f + a.w + b.w));
        sh[k] = make_float4(cc.x + d.x, cc.y + d.y, cc.z + d.z, cc.w + d.w);
      }
    };
    if (m.a_ld == 0) combine(0);
#pragma unroll
    for (int rr = 0; rr < ROWS; ++rr) {
      const int row = row0 + rr;
      if (row >= M) break;
      // a new modulation row: the first row of the CTA, and every row whose token (rpr = 1) or batch item differs
      if (m.a_ld != 0 && (rr == 0 || row / m.rpr != (row - 1) / m.rpr)) combine(static_cast<int64_t>(row / m.rpr) * m.a_ld);
      uint2* orow = reinterpret_cast<uint2*>(m.out + static_cast<int64_t>(row) * D);
#pragma unroll
      for (int k = 0; k < VPT; ++k)
        orow[threadIdx.x + k * 256] =
            make_uint2(pack_bf16(v[rr][k].x * s2[rr] * sc[k].x + sh[k].x, v[rr][k].y * s2[rr] * sc[k].y + sh[k].y),
                       pack_bf16(v[rr][k].z * s2[rr] * sc[k].z + sh[k].z, v[rr][k].w * s2[rr] * sc[k].w + sh[k].w));
    }
  }
}

// q / k RMSNorm across all heads (learned weight) + split RoPE for any head_dim that is a multiple of 16, in place on bf16
// rows (T/LTXAttention.swift:179-189, T/LTXRoPE.swift:84-149): head h holds (x1 | x2) halves of hd/2; cos / sin
// [rows_per_rope, D/2] fp32 with index h * hd/2 + j.
__global__ void __launch_bounds__(256) qknorm_rope_hd_kernel(bf16* x, int64_t ld, int D, int hd, const float* w, const float* cosb,
                                                              const float* sinb, int rows_per_rope, float eps) {
  __shared__ float red[8];
  griddep_launch();
  griddep_wait();
  const int row = blockIdx.x;
  bf16* xr = x + static_cast<int64_t>(row) * ld;
  const int nchunk = D >> 3;
  float ss = 0.f;
  for (int i = threadIdx.x; i < nchunk; i += blockDim.x) {
    const uint4 u = reinterpret_cast<const uint4*>(xr)[i];
    const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const float2 f = __bfloat1622float2(h2[t]);
      ss += f.x * f.x + f.y * f.y;
    }
  }
  const float rstd = rsqrtf(block_sum_256(ss, red) / D + eps);
  const int half = hd >> 1, cph = half >> 3;   // 8-element chunks per half head
  const int npair = D >> 4;
  const float* cr = cosb ? cosb + static_cast<int64_t>(row % rows_per_rope) * (D >> 1) : nullptr;
  const float* sr = sinb ? sinb + static_cast<int64_t>(row % rows_per_rope) * (D >> 1) : nullptr;
  for (int pc = threadIdx.x; pc < npair; pc += blockDim.x) {
    const int hh = pc / cph, jc = (pc % cph) * 8;
    const int c1 = hh * hd + jc, c2 = c1 + half;
    const uint4 u1 = *reinterpret_cast<const uint4*>(xr + c1);
    const uint4 u2 = *reinterpret_cast<const uint4*>(xr + c2);
    const __nv_bfloat162* a2 = reinterpret_cast<const __nv_bfloat162*>(&u1);
    const __nv_bfloat162* b2 = reinterpret_cast<const __nv_bfloat162*>(&u2);
    float x1[8], x2[8], y1[8], y2[8];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const float2 fa = __bfloat1622float2(a2[t]), fb = __bfloat1622float2(b2[t]);
      x1[2 * t] = fa.x * rstd * w[c1 + 2 * t];
      x1[2 * t + 1] = fa.y * rstd * w[c1 + 2 * t + 1];
      x2[2 * t] = fb.x * rstd * w[c2 + 2 * t];
      x2[2 * t + 1] = fb.y * rstd * w[c2 + 2 * t + 1];
    }
    if (cr) {
      const int fi = hh * half + jc;
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const float cs = cr[fi + t], sn = sr[fi + t];
        y1[t] = x1[t] * cs - x2[t] * sn;
        y2[t] = x2[t] * cs + x1[t] * sn;
      }
    } else {
#pragma unroll
      for (int t = 0; t < 8; ++t) { y1[t] = x1[t]; y2[t] = x2[t]; }
    }
    *reinterpret_cast<uint4*>(xr + c1) =
        make_uint4(pack_bf16(y1[0], y1[1]), pack_bf16(y1[2], y1[3]), pack_bf16(y1[4], y1[5]), pack_bf16(y1[6], y1[7]));
    *reinterpret_cast<uint4*>(xr + c2) =
        make_uint4(pack_bf16(y2[0], y2[1]), pack_bf16(y2[2], y2[3]), pack_bf16(y2[4], y2[5]), pack_bf16(y2[6], y2[7]));
  }
}

// ---------------------------------------------------------------- profiled launch helpers
// out_bf16[M, N] = A W^T + b
void proj(ltx_ctx* c, const bf16* A, int M, int K, const LinearW& W, const float* b, int N, bf16* out, int mode,
          const LinearOpts& o) {
  GemmEpi e;
  e.mode = mode; e.out = out; e.ldo = N; e.bias = b;
  linear(c, A, K, W, M, N, K, e, o);
}
// x[M, N] (fp32) += (A W^T + b) * (gate_a[(m / gate_rows) * gate_ld + n] + gate_b[n])   (null gates: 1); gate_ld = 0: one
// gate row for all M rows
void proj_resid(ltx_ctx* c, const bf16* A, int M, int K, const LinearW& W, const float* b, int N, float* x, const float* gate_a,
                const float* gate_b, int64_t gate_ld, int gate_rows, const LinearOpts& o) {
  GemmEpi e;
  e.mode = EPI_GATE_RESID; e.resid = x; e.ldr = N; e.bias = b; e.gate_a = gate_a; e.gate_b = gate_b; e.gate_ld = gate_ld;
  e.rows_per_gate = gate_ld > 0 ? gate_rows : (M > 0 ? M : 1);
  linear(c, A, K, W, M, N, K, e, o);
}
// a_ld > 0: row r takes its modulation rows sc_a / sh_a + (r / a_rpr) * a_ld (one per token, or one per batch item)
void normw(ltx_ctx* c, const float* x, bf16* out, int M, int D, const float* w, const float* sc_t, const float* sc_a,
           const float* sh_t, const float* sh_a, float eps, int64_t a_ld = 0, int a_rpr = 1) {
  ProfScope ps(c, PROF_ROW, 0.0, static_cast<double>(M) * D * 6.0);
  const ModSet m{sc_t, sc_a, sh_t, sh_a, out, a_ld, a_rpr};
  if (D == 4096)
    launch_pdl(PDL_ROWS, rmsnorm_w_mod_fast_kernel<4, 4, 1>, dim3((M + 3) / 4), dim3(256), 0, c->stream, x, M, w, m, m, eps);
  else if (D == 2048)
    launch_pdl(PDL_ROWS, rmsnorm_w_mod_fast_kernel<2, 4, 1>, dim3((M + 3) / 4), dim3(256), 0, c->stream, x, M, w, m, m, eps);
  else
    launch_pdl(PDL_ROWS, rmsnorm_w_mod_kernel, dim3(M), dim3(256), 0, c->stream, x, out, D, w, sc_t, sc_a, sh_t, sh_a, a_ld, a_rpr,
               eps);
  LTX_CUDA(cudaGetLastError());
}
// two modulations of the same normalised rows: out0 with (sc0, sh0), out1 with (sc1, sh1); tbl rows r*D of `tbl`, `ada`
void normw2(ltx_ctx* c, const float* x, bf16* out0, bf16* out1, int M, int D, const float* w, const float* tbl, const float* ada,
            float eps, int64_t a_ld = 0, int a_rpr = 1) {
  // rows: 0 a2v scale, 1 a2v shift, 2 v2a scale, 3 v2a shift
  const ModSet m0{tbl, ada, tbl + D, ada + D, out0, a_ld, a_rpr},
      m1{tbl + 2 * D, ada + 2 * D, tbl + 3 * D, ada + 3 * D, out1, a_ld, a_rpr};
  if (D == 4096 || D == 2048) {
    ProfScope ps(c, PROF_ROW, 0.0, static_cast<double>(M) * D * 8.0);
    if (D == 4096)
      launch_pdl(PDL_ROWS, rmsnorm_w_mod_fast_kernel<4, 4, 2>, dim3((M + 3) / 4), dim3(256), 0, c->stream, x, M, w, m0, m1, eps);
    else
      launch_pdl(PDL_ROWS, rmsnorm_w_mod_fast_kernel<2, 4, 2>, dim3((M + 3) / 4), dim3(256), 0, c->stream, x, M, w, m0, m1, eps);
    LTX_CUDA(cudaGetLastError());
    return;
  }
  normw(c, x, out0, M, D, w, m0.sc_t, m0.sc_a, m0.sh_t, m0.sh_a, eps, a_ld, a_rpr);
  normw(c, x, out1, M, D, w, m1.sc_t, m1.sc_a, m1.sh_t, m1.sh_a, eps, a_ld, a_rpr);
}
void qknorm_hd(ltx_ctx* c, bf16* x, int M, int D, int hd, const float* w, const float* cs, const float* sn, int rpr, float eps) {
  ProfScope ps(c, PROF_ROW, 0.0, static_cast<double>(M) * D * (4.0 + (cs ? 4.0 : 0.0)));
  launch_pdl(PDL_ROWS, qknorm_rope_hd_kernel, dim3(M), dim3(256), 0, c->stream, x, static_cast<int64_t>(D), D, hd, w, cs, sn,
             rpr > 0 ? rpr : 1, eps);
  LTX_CUDA(cudaGetLastError());
}

AttnWeights attn_w(ltx_ctx* c, const std::string& p, int64_t qdim, int64_t cdim, int64_t inner) {
  AttnWeights a;
  a.wq = wlin(c, p + ".to_q.weight", inner, qdim); a.bq = wf(c, p + ".to_q.bias", inner);
  a.wk = wlin(c, p + ".to_k.weight", inner, cdim); a.bk = wf(c, p + ".to_k.bias", inner);
  a.wv = wlin(c, p + ".to_v.weight", inner, cdim); a.bv = wf(c, p + ".to_v.bias", inner);
  a.wo = wlin(c, p + ".to_out.weight", qdim, inner); a.bo = wf(c, p + ".to_out.bias", qdim);
  a.q_norm = wf(c, p + ".q_norm.weight", inner);
  a.k_norm = wf(c, p + ".k_norm.weight", inner);
  return a;
}
// 1-D RoPE table, token-major [T, dim/2] (precomputeFreqsCis with a [1, T] grid, T/LTXRoPE.swift:375-488): all dim/2
// frequencies come from the single axis, no identity padding.
void build_rope_1d(ltx_ctx* c, DevBuf& cosb, DevBuf& sinb, const std::vector<float>& pos, int dim, float theta, int max_pos) {
  const int half = dim / 2, n_idx = std::max(1, dim / 2);
  const size_t T = pos.size();
  std::vector<float> cs(T * half), sn(T * half);
  std::vector<double> idx(n_idx);
  for (int i = 0; i < n_idx; ++i)
    idx[i] = std::pow(static_cast<double>(theta), n_idx > 1 ? static_cast<double>(i) / (n_idx - 1) : 0.0) * (M_PI / 2.0);
  for (size_t t = 0; t < T; ++t) {
    const double sc = static_cast<double>(pos[t]) / max_pos * 2.0 - 1.0;
    for (int k = 0; k < half; ++k) {
      const double a = idx[k] * sc;
      cs[t * half + k] = static_cast<float>(std::cos(a));
      sn[t * half + k] = static_cast<float>(std::sin(a));
    }
  }
  cosb.reserve(cs.size() * 4);
  sinb.reserve(sn.size() * 4);
  LTX_CUDA(cudaMemcpyAsync(cosb.ptr, cs.data(), cs.size() * 4, cudaMemcpyHostToDevice, c->stream));
  LTX_CUDA(cudaMemcpyAsync(sinb.ptr, sn.data(), sn.size() * 4, cudaMemcpyHostToDevice, c->stream));
  LTX_CUDA(cudaStreamSynchronize(c->stream));
}

const AttnWeights& audio_text_layer(const void* user, int i) { return static_cast<const ltx_ctx*>(user)->av.blocks[i].aa2; }

int64_t round_up8(int64_t v) { return (v + 7) / 8 * 8; }

}  // namespace

void dit_av_finalize(ltx_ctx* c) {
  const ltx_config& g = c->cfg;
  LTX_CHECK(c->dit_ready && c->precision == 16 && c->w_patch.fmt == LW_BF16, LTX_ERR_WEIGHTS,
            "the dual model is finalized on the bf16 video weights (quantisation follows)");
  AvWeights& a = c->av;
  const int64_t D = static_cast<int64_t>(g.num_heads) * g.head_dim;
  const int Ha = g.audio_num_heads > 0 ? g.audio_num_heads : 32, hd = g.audio_head_dim > 0 ? g.audio_head_dim : 64;
  LTX_CHECK(hd == 64 || hd == 128, LTX_ERR_INVALID_CONFIGURATION, "audio_head_dim must be 64 or 128");
  const int64_t Da = static_cast<int64_t>(Ha) * hd, FFa = g.ffn_mult * Da;
  LTX_CHECK(Da % 128 == 0, LTX_ERR_INVALID_CONFIGURATION, "audio inner dim must be a multiple of 128");
  const int Ca = g.audio_in_channels > 0 ? g.audio_in_channels : 128;
  a.Da = static_cast<int>(Da); a.Ha = Ha; a.hd = hd; a.Cin = Ca;
  a.w_patch = wlin(c, "audio_patchify_proj.weight", Da, Ca); a.b_patch = wf(c, "audio_patchify_proj.bias", Da);
  a.w_c1 = wlin(c, "audio_caption_projection.linear_1.weight", Da, g.caption_channels);
  a.b_c1 = wf(c, "audio_caption_projection.linear_1.bias", Da);
  a.w_c2 = wlin(c, "audio_caption_projection.linear_2.weight", Da, Da);
  a.b_c2 = wf(c, "audio_caption_projection.linear_2.bias", Da);
  a.sst_out = wf(c, "audio_scale_shift_table", 2 * Da);
  a.w_out = wlin(c, "audio_proj_out.weight", Ca, Da); a.b_out = wf(c, "audio_proj_out.bias", Ca);
  a.ada_a = adaln_w(c, "audio_adaln_single", Da, 6);
  a.cv_ss = adaln_w(c, "av_ca_video_scale_shift_adaln_single", D, 4);
  a.cv_g = adaln_w(c, "av_ca_a2v_gate_adaln_single", D, 1);
  a.ca_ss = adaln_w(c, "av_ca_audio_scale_shift_adaln_single", Da, 4);
  a.ca_g = adaln_w(c, "av_ca_v2a_gate_adaln_single", Da, 1);
  a.blocks.assign(g.num_layers, AvBlockW());
  for (int i = 0; i < g.num_layers; ++i) {
    const std::string p = "transformer_blocks." + std::to_string(i) + ".";
    AvBlockW& b = a.blocks[i];
    b.norm1 = wf(c, p + "norm1.weight", D); b.norm2 = wf(c, p + "norm2.weight", D); b.norm3 = wf(c, p + "norm3.weight", D);
    b.a2v_norm = wf(c, p + "audio_to_video_norm.weight", D);
    b.anorm1 = wf(c, p + "audio_norm1.weight", Da); b.anorm2 = wf(c, p + "audio_norm2.weight", Da);
    b.anorm3 = wf(c, p + "audio_norm3.weight", Da); b.v2a_norm = wf(c, p + "video_to_audio_norm.weight", Da);
    b.aa1 = attn_w(c, p + "audio_attn1", Da, Da, Da);
    b.aa2 = attn_w(c, p + "audio_attn2", Da, Da, Da);
    b.a2v = attn_w(c, p + "audio_to_video_attn", D, Da, Da);
    b.v2a = attn_w(c, p + "video_to_audio_attn", Da, D, Da);
    b.w_in = wlin(c, p + "audio_ff.project_in.proj.weight", FFa, Da); b.b_in = wf(c, p + "audio_ff.project_in.proj.bias", FFa);
    b.w_out = wlin(c, p + "audio_ff.project_out.weight", Da, FFa); b.b_out = wf(c, p + "audio_ff.project_out.bias", Da);
    b.asst = wf(c, p + "audio_scale_shift_table", 6 * Da);
    b.sst_ca_v = wf(c, p + "scale_shift_table_a2v_ca_video", 5 * D);
    b.sst_ca_a = wf(c, p + "scale_shift_table_a2v_ca_audio", 5 * Da);
  }
  a.ready = true;
}

void dit_av_forward_dev(ltx_ctx* c, const void* v_latent, int v_dtype, const void* a_latent, int a_dtype, const void* v_context,
                        const void* a_context, int ctx_dtype, const float* v_ts_dev, int v_ts_per_token, const float* a_ts_dev,
                        const int32_t* v_mask_dev, const int32_t* a_mask_dev, int B, int N, int Ta, int S, int F, int H, int W, uint64_t context_key,
                        float* out_v_dev, float* out_a_dev) {
  AvWeights& av = c->av;
  LTX_CHECK(av.ready, LTX_ERR_WEIGHTS, "dual audio/video weights not loaded / finalized");
  LTX_CHECK(!(c->dist.comm_world && c->dist.sp > 1), LTX_ERR_UNSUPPORTED, "the dual model is single-GPU in this version");
  LTX_CHECK(B >= 1 && B <= 2, LTX_ERR_UNSUPPORTED, "dual forward: batches of 1 or 2 items");
  LTX_CHECK(N >= 1 && Ta >= 1 && S >= 1 && static_cast<int64_t>(F) * H * W == N, LTX_ERR_INVALID_ARGUMENT,
            "dual forward: N = F*H*W");
  LTX_CHECK(v_latent && a_latent && v_context && a_context && v_ts_dev && a_ts_dev && out_v_dev && out_a_dev,
            LTX_ERR_INVALID_ARGUMENT, "null tensor");
  LTX_CHECK((v_dtype == LTX_BF16 || v_dtype == LTX_F32) && (a_dtype == LTX_BF16 || a_dtype == LTX_F32), LTX_ERR_UNSUPPORTED,
            "latent dtype must be bf16 or f32");
  const ltx_config& g = c->cfg;
  const int D = g.num_heads * g.head_dim, FFD = g.ffn_mult * D, Hv = g.num_heads, L = g.num_layers, hdv = g.head_dim;
  const int Da = av.Da, Ha = av.Ha, hda = av.hd, FFa = g.ffn_mult * Da, Cv = g.in_channels, Ca = av.Cin;
  const float eps = g.norm_eps;
  cudaStream_t st = c->stream;
  const int64_t ldv = round_up8(N), lda = round_up8(Ta);   // per-item column pitches of the V^T operands
  const int R = B * N, Ra = B * Ta;                         // rows of the two streams
  LinearOpts o;   // the weight-streaming kernel takes up to 32 rows per item: a row of a two-item product runs on the kernel its
  o.allow_skinny = 32 * B;   // one-item product runs on (the audio stream's Linears stream their weights)

  // ---- workspaces: the video stream reuses the video-only model's buffers
  c->x.reserve(static_cast<size_t>(R) * D * 4);
  c->h.reserve(static_cast<size_t>(R) * D * 2);
  c->q2.reserve(static_cast<size_t>(R) * D * 2);
  c->qk.reserve(static_cast<size_t>(R) * 2 * D * 2);
  c->vt.reserve(static_cast<size_t>(D) * B * ldv * 2);
  c->att.reserve(static_cast<size_t>(R) * D * 2);
  c->ffh.reserve(static_cast<size_t>(R) * FFD * 2);
  c->xb.reserve(static_cast<size_t>(R) * D * 2);
  DevBuf& wsb = av.ws;
  // rows of the video-side modulation tensors: one per item, or one per token (per-token sigmas)
  const int VR = v_ts_per_token ? R : B;
  // Modulation / gate rows and their pitches.  Row r of a stream reads row r / *_rpr; a pitch of 0 (B = 1 with one sigma)
  // shares one row among all rows.  The cross-modal tables are [scale/shift rows 0-3 | gate row 4]: interleaved per token
  // ([R, 5, D]) with per-token sigmas, otherwise all items' rows 0-3 ([B, 4, D]) followed by all items' gates ([B, D]).
  const bool per_item = B > 1;
  const int v_rpr = v_ts_per_token ? 1 : N;
  const int64_t vada_ld = (v_ts_per_token || per_item) ? 6 * static_cast<int64_t>(D) : 0;
  const int64_t cv_ld = v_ts_per_token ? 5 * static_cast<int64_t>(D) : per_item ? 4 * static_cast<int64_t>(D) : 0;
  const int64_t cvg_ld = v_ts_per_token ? 5 * static_cast<int64_t>(D) : per_item ? static_cast<int64_t>(D) : 0;
  const int64_t aada_ld = per_item ? 6 * static_cast<int64_t>(Da) : 0, ca_ld = per_item ? 4 * static_cast<int64_t>(Da) : 0,
                cag_ld = per_item ? static_cast<int64_t>(Da) : 0;
  // audio / cross-modal workspace carved out of one allocation
  size_t off = 0;
  auto carve = [&](size_t bytes) { const size_t at = off; off += (bytes + 255) / 256 * 256; return at; };
  const size_t o_ax = carve(static_cast<size_t>(Ra) * Da * 4), o_ah = carve(static_cast<size_t>(Ra) * Da * 2),
               o_ah2 = carve(static_cast<size_t>(Ra) * Da * 2), o_aq = carve(static_cast<size_t>(Ra) * Da * 2),
               o_ak = carve(static_cast<size_t>(Ra) * Da * 2), o_avt = carve(static_cast<size_t>(Da) * B * lda * 2),
               o_aatt = carve(static_cast<size_t>(Ra) * Da * 2), o_affh = carve(static_cast<size_t>(Ra) * FFa * 2),
               o_cq = carve(static_cast<size_t>(R) * Da * 2), o_catt = carve(static_cast<size_t>(R) * Da * 2),
               o_vt2 = carve(static_cast<size_t>(Da) * B * ldv * 2),
               o_lat = carve(static_cast<size_t>(std::max(R * Cv, Ra * Ca)) * 2),
               o_se = carve(static_cast<size_t>(B) * 2 * 256 * 4), o_t1 = carve(static_cast<size_t>(B) * D * 4),
               o_vemb = carve(static_cast<size_t>(VR) * D * 4), o_aemb = carve(static_cast<size_t>(B) * Da * 4),
               o_vada = carve(static_cast<size_t>(VR) * 6 * D * 4), o_aada = carve(static_cast<size_t>(B) * 6 * Da * 4),
               o_cv = carve(static_cast<size_t>(VR) * 5 * D * 4), o_ca = carve(static_cast<size_t>(B) * 5 * Da * 4),
               o_scr = carve(static_cast<size_t>(VR) * D * 4),
               o_tq = carve(c->w_patch.fmt == LW_BF16 ? 0 : static_cast<size_t>(std::max(R, Ra)) * D * 2),   // codes: projection before the V^T transpose
               o_sev = carve(v_ts_per_token ? static_cast<size_t>(R) * 256 * 2 : 0),
               o_t1v = carve(v_ts_per_token ? static_cast<size_t>(R) * D * 2 : 0);
  wsb.reserve(off);
  uint8_t* wbase = wsb.as<uint8_t>();
  float* x = c->x.as<float>();
  bf16 *h = c->h.as<bf16>(), *h2 = c->q2.as<bf16>(), *qk = c->qk.as<bf16>(), *vt = c->vt.as<bf16>(), *att = c->att.as<bf16>(),
       *ffh = c->ffh.as<bf16>(), *q2 = c->xb.as<bf16>();
  float* ax = reinterpret_cast<float*>(wbase + o_ax);
  bf16 *ah = reinterpret_cast<bf16*>(wbase + o_ah), *ah2 = reinterpret_cast<bf16*>(wbase + o_ah2),
       *aq = reinterpret_cast<bf16*>(wbase + o_aq), *ak = reinterpret_cast<bf16*>(wbase + o_ak),
       *avt = reinterpret_cast<bf16*>(wbase + o_avt), *aatt = reinterpret_cast<bf16*>(wbase + o_aatt),
       *affh = reinterpret_cast<bf16*>(wbase + o_affh), *cq = reinterpret_cast<bf16*>(wbase + o_cq),
       *catt = reinterpret_cast<bf16*>(wbase + o_catt), *vt2 = reinterpret_cast<bf16*>(wbase + o_vt2),
       *lat_bf = reinterpret_cast<bf16*>(wbase + o_lat), *tq = reinterpret_cast<bf16*>(wbase + o_tq);
  float *se = reinterpret_cast<float*>(wbase + o_se), *t1 = reinterpret_cast<float*>(wbase + o_t1),
        *vemb = reinterpret_cast<float*>(wbase + o_vemb), *aemb = reinterpret_cast<float*>(wbase + o_aemb),
        *vada = reinterpret_cast<float*>(wbase + o_vada), *aada = reinterpret_cast<float*>(wbase + o_aada),
        *cv = reinterpret_cast<float*>(wbase + o_cv), *ca = reinterpret_cast<float*>(wbase + o_ca),
        *scr = reinterpret_cast<float*>(wbase + o_scr);

  // ---- step-invariant pieces: RoPE tables (video 3-D; audio 1-D; video temporal-only for the cross-modal attention) and
  // the text K / V of both streams
  dit_build_rope(c, F, H, W);
  if (av.rope_ta != Ta || av.rope_f != F || av.rope_hw != H * W || !av.a_cos.ptr) {
    std::vector<float> pa(Ta), pv(static_cast<size_t>(N));
    for (int i = 0; i < Ta; ++i) {   // createAudioPositionGrid (T/LTXRoPE.swift:627-655), fp32 like the reference
      const float fi = static_cast<float>(i), sc = 4.0f, of = 1.0f;
      const float s0 = std::max(0.0f, fi * sc + of - sc), e0 = std::max(0.0f, (fi + 1.0f) * sc + of - sc);
      pa[i] = (s0 + e0) / 2.0f * 160.0f / 16000.0f;
    }
    for (int f = 0; f < F; ++f) {    // temporal coordinate of createPositionGrid (:552-610)
      const float ts = 8.0f, fi = static_cast<float>(f);
      const float s0 = std::max(fi * ts + (1.0f - ts), 0.0f), e0 = std::max((fi + 1.0f) * ts + (1.0f - ts), 0.0f);
      const float pt = ((s0 + e0) / 2.0f) / 24.0f;
      for (int k = 0; k < H * W; ++k) pv[static_cast<size_t>(f) * H * W + k] = pt;
    }
    const int amax = g.audio_max_pos > 0 ? g.audio_max_pos : 20;
    build_rope_1d(c, av.a_cos, av.a_sin, pa, Da, g.rope_theta, amax);
    build_rope_1d(c, av.xv_cos, av.xv_sin, pv, Da, g.rope_theta, amax);
    av.rope_ta = Ta; av.rope_f = F; av.rope_hw = H * W;
  }
  const float *cos_v = c->rope_cos.as<float>(), *sin_v = c->rope_sin.as<float>();
  const float *cos_a = av.a_cos.as<float>(), *sin_a = av.a_sin.as<float>();
  const float *cos_xv = av.xv_cos.as<float>(), *sin_xv = av.xv_sin.as<float>();
  TextProjW vsrc;
  vsrc.w_c1 = c->w_c1; vsrc.w_c2 = c->w_c2; vsrc.b_c1 = c->b_c1; vsrc.b_c2 = c->b_c2; vsrc.D = D; vsrc.user = c;
  vsrc.layer = [](const void* u, int i) -> const AttnWeights& { return static_cast<const ltx_ctx*>(u)->blocks[i].a2; };
  TextCache& tcv = dit_prepare_text(c, c->text, &c->text_rr, vsrc, v_context, ctx_dtype, v_mask_dev, B, S, context_key);
  TextProjW asrc;
  asrc.w_c1 = av.w_c1; asrc.w_c2 = av.w_c2; asrc.b_c1 = av.b_c1; asrc.b_c2 = av.b_c2; asrc.D = Da; asrc.user = c;
  asrc.layer = audio_text_layer;
  TextCache& tca = dit_prepare_text(c, av.text, &av.text_rr, asrc, a_context, ctx_dtype, a_mask_dev, B, S, context_key);
  const float* vbias = tcv.has_bias ? tcv.bias.as<float>() : nullptr;
  const float* abias = tca.has_bias ? tca.bias.as<float>() : nullptr;

  // ---- patchify projections (T/LTX2Transformer.swift:255, 262); the reference's bf16 Linear output is rounded to bf16
  auto embed = [&](const void* lat, int dt, int rows, int Cin, const LinearW& w, const float* b, int Dout, float* xout, bf16* tmp) {
    const bf16* src = reinterpret_cast<const bf16*>(lat);
    if (dt == LTX_F32) {
      LTX_CHECK((static_cast<int64_t>(rows) * Cin) % 4 == 0, LTX_ERR_INVALID_ARGUMENT, "latent size");
      ProfScope ps(c, PROF_OTHER, 0.0, 6.0 * rows * Cin);
      launch_cast_f32_bf16(reinterpret_cast<const float*>(lat), lat_bf, static_cast<int64_t>(rows) * Cin, st);
      src = lat_bf;
    }
    proj(c, src, rows, Cin, w, b, Dout, tmp, EPI_BF16, o);
    ProfScope ps(c, PROF_OTHER, 0.0, 6.0 * rows * Dout);
    launch_cast_bf16_f32(tmp, xout, static_cast<int64_t>(rows) * Dout, st);
  };
  embed(v_latent, v_dtype, R, Cv, c->w_patch, c->b_patch, D, x, h);
  embed(a_latent, a_dtype, Ra, Ca, av.w_patch, av.b_patch, Da, ax, ah);

  // ---- timestep embedders: one sinusoidal embedding per stream and item feeds that stream's three AdaLN-singles (:256-298)
  float* se_a = se + B * 256;
  {
    ProfScope ps(c, PROF_OTHER, 0.0, 2048.0 * B, 2);
    launch_sincos_embed(v_ts_dev, g.timestep_scale_multiplier, se, B, 256, st);
    launch_sincos_embed(a_ts_dev, g.timestep_scale_multiplier, se_a, B, 256, st);
  }
  float* cvg = v_ts_per_token ? cv + 4 * D : cv + static_cast<int64_t>(B) * 4 * D;   // gate rows (see the pitches above)
  float* cag = ca + static_cast<int64_t>(B) * 4 * Da;
  if (!v_ts_per_token) {
    adaln_single(c, c->adaln, se, t1, vemb, vada, B);
    adaln_single(c, av.cv_ss, se, t1, scr, cv, B);              // rows 0-3: a2v scale, a2v shift, v2a scale, v2a shift
    adaln_single(c, av.cv_g, se, t1, scr, cvg, B);              // row 4: a2v gate
  } else {
    bf16 *sev = reinterpret_cast<bf16*>(wbase + o_sev), *t1v = reinterpret_cast<bf16*>(wbase + o_t1v);
    {
      ProfScope ps(c, PROF_OTHER, 0.0, 4.0 * R + 512.0 * R);
      launch_sincos_embed(v_ts_dev, g.timestep_scale_multiplier, nullptr, R, 256, st, sev);
    }
    adaln_single_rows(c, c->adaln, sev, R, t1v, vemb, vada, vada_ld, o);
    adaln_single_rows(c, av.cv_ss, sev, R, t1v, scr, cv, cv_ld, o);         // [R, 5, D]: rows 0-3 of every token
    adaln_single_rows(c, av.cv_g, sev, R, t1v, scr, cvg, cvg_ld, o);        // row 4 of every token
  }
  adaln_single(c, av.ada_a, se_a, t1, aemb, aada, B);
  adaln_single(c, av.ca_ss, se_a, t1, scr, ca, B);
  adaln_single(c, av.ca_g, se_a, t1, scr, cag, B);

  for (int i = 0; i < L; ++i) {
    const BlockWeights& bv = c->blocks[i];
    const AvBlockW& ba = av.blocks[i];
    // ---- 1: video self-attention (T/LTX2TransformerBlock.swift:208-211)
    normw(c, x, h, R, D, ba.norm1, bv.sst + D, vada + D, bv.sst, vada, eps, vada_ld, v_rpr);
    proj(c, h, R, D, bv.a1.wq, bv.a1.bq, 2 * D, qk, EPI_BF16, o);   // packed q|k projection
    linear_vt(c, h, N, B, bv.a1.wv, bv.a1.bv, vt, B * ldv, ldv, tq, o);
    {
      ProfScope ps(c, PROF_ROW, 0.0, 2.0 * R * D * 8.0, (D == 4096) ? 1 : 2);
      launch_qknorm_rope(qk, 2 * D, R, D, bv.a1.q_norm, cos_v, sin_v, N, eps, st, bv.a1.k_norm);
    }
    attention(c, qk, 2 * D, qk + D, 2 * D, vt, ldv, nullptr, att, D, B, Hv, N, N, D);
    proj_resid(c, att, R, D, bv.a1.wo, bv.a1.bo, D, x, vada + 2 * D, bv.sst + 2 * D, vada_ld, v_rpr, o);
    // ---- 2: audio self-attention (:213-216)
    normw(c, ax, ah, Ra, Da, ba.anorm1, ba.asst + Da, aada + Da, ba.asst, aada, eps, aada_ld, Ta);
    proj(c, ah, Ra, Da, ba.aa1.wq, ba.aa1.bq, Da, aq, EPI_BF16, o);
    proj(c, ah, Ra, Da, ba.aa1.wk, ba.aa1.bk, Da, ak, EPI_BF16, o);
    linear_vt(c, ah, Ta, B, ba.aa1.wv, ba.aa1.bv, avt, B * lda, lda, tq, o);
    qknorm_hd(c, aq, Ra, Da, hda, ba.aa1.q_norm, cos_a, sin_a, Ta, eps);
    qknorm_hd(c, ak, Ra, Da, hda, ba.aa1.k_norm, cos_a, sin_a, Ta, eps);
    attention(c, aq, Da, ak, Da, avt, lda, nullptr, aatt, Da, B, Ha, Ta, Ta, Da);
    proj_resid(c, aatt, Ra, Da, ba.aa1.wo, ba.aa1.bo, Da, ax, aada + 2 * Da, ba.asst + 2 * Da, aada_ld, Ta, o);
    // ---- 3: video text cross-attention on norm2(x), no RoPE, no gate (:218-221)
    normw(c, x, h, R, D, ba.norm2, nullptr, nullptr, nullptr, nullptr, eps);
    proj(c, h, R, D, bv.a2.wq, bv.a2.bq, D, q2, EPI_BF16, o);
    qknorm_hd(c, q2, R, D, hdv, bv.a2.q_norm, nullptr, nullptr, 1, eps);
    attention(c, q2, D, tcv.k.as<bf16>() + static_cast<int64_t>(i) * B * S * D, D,
              tcv.vt.as<bf16>() + static_cast<int64_t>(i) * D * B * tcv.ldv, tcv.ldv, vbias, att, D, B, Hv, N, S, D);
    proj_resid(c, att, R, D, bv.a2.wo, bv.a2.bo, D, x, nullptr, nullptr, 0, 1, o);
    // ---- 4: audio text cross-attention (:223-226)
    normw(c, ax, ah, Ra, Da, ba.anorm2, nullptr, nullptr, nullptr, nullptr, eps);
    proj(c, ah, Ra, Da, ba.aa2.wq, ba.aa2.bq, Da, aq, EPI_BF16, o);
    qknorm_hd(c, aq, Ra, Da, hda, ba.aa2.q_norm, nullptr, nullptr, 1, eps);
    attention(c, aq, Da, tca.k.as<bf16>() + static_cast<int64_t>(i) * B * S * Da, Da,
              tca.vt.as<bf16>() + static_cast<int64_t>(i) * Da * B * tca.ldv, tca.ldv, abias, aatt, Da, B, Ha, Ta, S, Da);
    proj_resid(c, aatt, Ra, Da, ba.aa2.wo, ba.aa2.bo, Da, ax, nullptr, nullptr, 0, 1, o);
    // ---- 5-6: cross-modal attention; both directions read the streams as they are here (:228-271).  Table / embedding
    // rows: 0 a2v scale, 1 a2v shift, 2 v2a scale, 3 v2a shift, 4 gate.  Each item attends within itself only.
    normw2(c, x, h, h2, R, D, ba.a2v_norm, ba.sst_ca_v, cv, eps, cv_ld, v_rpr);   // video as a2v query (h) and v2a context (h2)
    normw2(c, ax, ah, ah2, Ra, Da, ba.v2a_norm, ba.sst_ca_a, ca, eps, ca_ld, Ta);  // audio as a2v context (ah) and v2a query (ah2)
    // A2V: Q from video (temporal RoPE of the video frames), K / V from audio
    proj(c, h, R, D, ba.a2v.wq, ba.a2v.bq, Da, cq, EPI_BF16, o);
    proj(c, ah, Ra, Da, ba.a2v.wk, ba.a2v.bk, Da, ak, EPI_BF16, o);
    linear_vt(c, ah, Ta, B, ba.a2v.wv, ba.a2v.bv, avt, B * lda, lda, tq, o);
    qknorm_hd(c, cq, R, Da, hda, ba.a2v.q_norm, cos_xv, sin_xv, N, eps);
    qknorm_hd(c, ak, Ra, Da, hda, ba.a2v.k_norm, cos_a, sin_a, Ta, eps);
    attention(c, cq, Da, ak, Da, avt, lda, nullptr, catt, Da, B, Ha, N, Ta, Da);
    // V2A: Q from audio, K / V from video (projected before the a2v update lands in x: h2 was taken above)
    proj(c, ah2, Ra, Da, ba.v2a.wq, ba.v2a.bq, Da, aq, EPI_BF16, o);
    proj(c, h2, R, D, ba.v2a.wk, ba.v2a.bk, Da, cq, EPI_BF16, o);
    linear_vt(c, h2, N, B, ba.v2a.wv, ba.v2a.bv, vt2, B * ldv, ldv, tq, o);
    qknorm_hd(c, aq, Ra, Da, hda, ba.v2a.q_norm, cos_a, sin_a, Ta, eps);
    qknorm_hd(c, cq, R, Da, hda, ba.v2a.k_norm, cos_xv, sin_xv, N, eps);
    attention(c, aq, Da, cq, Da, vt2, ldv, nullptr, aatt, Da, B, Ha, Ta, N, Da);
    proj_resid(c, catt, R, Da, ba.a2v.wo, ba.a2v.bo, D, x, cvg, ba.sst_ca_v + 4 * D, cvg_ld, v_rpr, o);
    proj_resid(c, aatt, Ra, Da, ba.v2a.wo, ba.v2a.bo, Da, ax, cag, ba.sst_ca_a + 4 * Da, cag_ld, Ta, o);
    // ---- 7-8: feed-forward on both streams (:273-281)
    normw(c, x, h, R, D, ba.norm3, bv.sst + 4 * D, vada + 4 * D, bv.sst + 3 * D, vada + 3 * D, eps, vada_ld, v_rpr);
    proj(c, h, R, D, bv.w_in, bv.b_in, FFD, ffh, EPI_GELU_BF16, o);
    proj_resid(c, ffh, R, FFD, bv.w_out, bv.b_out, D, x, vada + 5 * D, bv.sst + 5 * D, vada_ld, v_rpr, o);
    normw(c, ax, ah, Ra, Da, ba.anorm3, ba.asst + 4 * Da, aada + 4 * Da, ba.asst + 3 * Da, aada + 3 * Da, eps, aada_ld, Ta);
    proj(c, ah, Ra, Da, ba.w_in, ba.b_in, FFa, affh, EPI_GELU_BF16, o);
    proj_resid(c, affh, Ra, FFa, ba.w_out, ba.b_out, Da, ax, aada + 5 * Da, ba.asst + 5 * Da, aada_ld, Ta, o);
  }
  // ---- output heads (T/LTX2Transformer.swift:370-388): LayerNorm(no affine) * (1 + scale) + shift ; proj_out
  // emb: one row per item (rpr = rows of an item) or per token (rpr = 1)
  auto head = [&](const float* xs, int rows, int Dx, const float* sst, const float* emb, int rpr, bf16* tmp, const LinearW& w,
                  const float* b, int Cout, float* out) {
    {
      ProfScope ps(c, PROF_ROW, 0.0, static_cast<double>(rows) * Dx * 6.0);
      launch_rmsnorm_mod(xs, tmp, rows, Dx, sst, sst + Dx, emb, emb, Dx, rpr, eps, 1, st);
    }
    GemmEpi e;
    e.mode = EPI_F32; e.out = out; e.ldo = Cout; e.bias = b;
    linear(c, tmp, Dx, w, rows, Cout, Dx, e, o);
  };
  head(x, R, D, c->sst_out, vemb, v_rpr, h, c->w_out, c->b_out, g.out_channels, out_v_dev);
  head(ax, Ra, Da, av.sst_out, aemb, Ta, ah, av.w_out, av.b_out, Ca, out_a_dev);
}

}  // namespace ltx
