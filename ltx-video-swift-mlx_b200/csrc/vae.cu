// Video-VAE decoder on one B200.  Restates VideoDecoder.callAsFunction (Models/VAE/VideoDecoder.swift:358-449) and
// decodeVideo's untiled path (:466-508) on top of the implicit-GEMM conv kernel (conv3d.cu).
//
// HBM layout: every activation is channels-last fp32 [T, H, W, C] (the residual stream stays fp32); each conv reads a
// bf16 padded copy produced by the fused pixel-norm/scale-shift/SiLU prologue and writes fp32 through its epilogue
// (+bias, +residual, depth-to-space scatter, or unpatchify+clip straight into the [F, H, W, 3] frame buffer).
#include "ctx.h"
#include "frames_u8.cuh"

namespace ltx {

namespace {

__global__ void permute_conv_weight_kernel(const bf16* __restrict__ in, bf16* __restrict__ out, int O, int I, int taps,
                                           int Ou, int Ip) {
  // in [O][I][taps] -> out [taps][Ou][Ip]: the first Ou <= O output channels, input channels zero-padded to Ip >= I
  const int64_t n = static_cast<int64_t>(Ou) * Ip * taps;
  for (int64_t idx = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; idx < n;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(idx % Ip);
    const int o = static_cast<int>((idx / Ip) % Ou);
    const int tap = static_cast<int>(idx / (static_cast<int64_t>(Ip) * Ou));
    out[idx] = i < I ? in[(static_cast<int64_t>(o) * I + i) * taps + tap] : __float2bfloat16(0.f);
  }
}

__global__ void noise_mix_kernel(float* __restrict__ x, const float* __restrict__ nz, int64_t n, float scale) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    x[i] = nz[i] * scale + (1.0f - scale) * x[i];
}

__global__ void add_vec_kernel(float* __restrict__ out, const float* __restrict__ a, const float* __restrict__ b, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = a[i] + b[i];
}
// temporal tiling (V/VideoDecoder.swift:560-585): the first `po` frames of the next tile are cross-faded into the last `po`
// frames of the result, weight j / po on the next tile
__global__ void tile_blend_kernel(float* __restrict__ dst, const float* __restrict__ src, int64_t frame_elems, int po) {
  const int64_t n4 = frame_elems * po / 4, fe4 = frame_elems / 4;
  const float inv = 1.0f / static_cast<float>(po);
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n4; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float w = static_cast<float>(i / fe4) * inv;
    float4 a = reinterpret_cast<float4*>(dst)[i];
    const float4 b = reinterpret_cast<const float4*>(src)[i];
    a.x = a.x * (1.f - w) + b.x * w; a.y = a.y * (1.f - w) + b.y * w;
    a.z = a.z * (1.f - w) + b.z * w; a.w = a.w * (1.f - w) + b.w * w;
    reinterpret_cast<float4*>(dst)[i] = a;
  }
}
__global__ void clip01_kernel(float* __restrict__ x, int64_t n4) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n4; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float4 a = reinterpret_cast<float4*>(x)[i];
    a.x = fminf(fmaxf(a.x, 0.f), 1.f); a.y = fminf(fmaxf(a.y, 0.f), 1.f);
    a.z = fminf(fmaxf(a.z, 0.f), 1.f); a.w = fminf(fmaxf(a.w, 0.f), 1.f);
    reinterpret_cast<float4*>(x)[i] = a;
  }
}

// fp32 frames -> 8-bit frames (frames_u8.cuh), the converter beside the fused conv_out store: one sample (RGB8) or one 2x2
// chroma cell (I420) per thread and iteration
__global__ void frames_rgb8_kernel(const float* __restrict__ x, uint8_t* __restrict__ out, int64_t n) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    out[i] = static_cast<uint8_t>(rgb8_code(fminf(fmaxf(x[i], 0.f), 1.f)));
}
__global__ void frames_i420_kernel(const float* __restrict__ x, uint8_t* __restrict__ out, int F, int H, int W) {
  const int Hc = H / 2, Wc = W / 2;
  const int64_t plane = static_cast<int64_t>(H) * W, ncell = static_cast<int64_t>(F) * Hc * Wc;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < ncell; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int cx = static_cast<int>(i % Wc), cy = static_cast<int>((i / Wc) % Hc);
    const int64_t f = i / (static_cast<int64_t>(Wc) * Hc);
    float p[4][3];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float* src = x + ((f * H + 2 * cy + (k >> 1)) * W + 2 * cx + (k & 1)) * 3;
#pragma unroll
      for (int c = 0; c < 3; ++c) p[k][c] = fminf(fmaxf(src[c], 0.f), 1.f);
    }
    uint32_t y[4], cb, cr;
    i420_cell(p, y, cb, cr);
    uint8_t* yp = out + f * (plane + plane / 2);
#pragma unroll
    for (int k = 0; k < 4; ++k) yp[static_cast<int64_t>(2 * cy + (k >> 1)) * W + 2 * cx + (k & 1)] = static_cast<uint8_t>(y[k]);
    const int64_t off = static_cast<int64_t>(cy) * Wc + cx;
    yp[plane + off] = static_cast<uint8_t>(cb);
    yp[plane + plane / 4 + off] = static_cast<uint8_t>(cr);
  }
}

}  // namespace

size_t frames_u8_bytes(int64_t F, int64_t H, int64_t W, int format) {
  if (F <= 0 || H <= 0 || W <= 0) return 0;
  if (format == LTX_FRAMES_RGB8) return static_cast<size_t>(F * H * W * 3);
  if (format == LTX_FRAMES_I420 && H % 2 == 0 && W % 2 == 0) return static_cast<size_t>(F * (H * W + H * W / 2));
  return 0;
}

void frames_to_u8_dev(ltx_ctx* c, const float* frames_dev, int F, int H, int W, int format, uint8_t* out_dev) {
  const size_t bytes = frames_u8_bytes(F, H, W, format);
  LTX_CHECK(bytes > 0 && frames_dev != nullptr && out_dev != nullptr, LTX_ERR_INVALID_ARGUMENT,
            "frames_to_u8: bad format, size or buffer (I420 needs even H and W)");
  const int64_t work = format == LTX_FRAMES_RGB8 ? static_cast<int64_t>(bytes) : static_cast<int64_t>(F) * (H / 2) * (W / 2);
  const int grid = static_cast<int>(std::min<int64_t>((work + 255) / 256, 148 * 16));
  ProfScope ps(c, PROF_OTHER, 0.0, 4.0 * F * H * W * 3 + static_cast<double>(bytes));
  if (format == LTX_FRAMES_RGB8) frames_rgb8_kernel<<<grid, 256, 0, c->stream>>>(frames_dev, out_dev, work);
  else frames_i420_kernel<<<grid, 256, 0, c->stream>>>(frames_dev, out_dev, F, H, W);
  LTX_CUDA(cudaGetLastError());
}

// Repacks a conv kernel stored in the checkpoint layout (O, I, 3, 3, 3) -- or (O, I, 3, 3) for the per-frame Conv2d of the
// upscaler -- into the implicit GEMM's [taps][Cout][Cin] bf16 matrix.  cout_use < cout keeps the leading output channels
// (encoder conv_out: 129 -> the 128 mean channels); cin is zero-padded to a multiple of 64 (encoder conv_in: 48 -> 64).
ConvW vae_pack_conv_keys(ltx_ctx* c, const std::string& wkey, const std::string& bkey, int64_t cout, int64_t cin, int64_t cout_use,
                         int taps) {
  const DevTensor& w = get_tensor(c, wkey);
  const bool ok3 = taps == 27 && w.shape.size() == 5 && w.shape[2] == 3 && w.shape[3] == 3 && w.shape[4] == 3;
  const bool ok2 = taps == 9 && w.shape.size() == 4 && w.shape[2] == 3 && w.shape[3] == 3;
  LTX_CHECK(w.dtype == LTX_BF16 && (ok3 || ok2) && w.shape[0] == cout && w.shape[1] == cin && cout_use <= cout, LTX_ERR_WEIGHTS,
            "bad shape for '" + wkey + "'");
  const DevTensor& b = get_tensor(c, bkey);
  LTX_CHECK(b.dtype == LTX_F32 && b.numel() == cout, LTX_ERR_WEIGHTS, "bad shape for '" + bkey + "'");
  const int64_t cin_pad = (cin + 63) / 64 * 64;
  bf16* packed = nullptr;
  const int64_t n = cout_use * cin_pad * taps;
  LTX_CUDA(cudaMalloc(&packed, static_cast<size_t>(n) * 2));
  c->owned.push_back(packed);
  int64_t blocks = (n + 255) / 256;
  if (blocks > 8192) blocks = 8192;
  permute_conv_weight_kernel<<<static_cast<int>(blocks), 256, 0, c->stream>>>(
      reinterpret_cast<const bf16*>(w.ptr), packed, static_cast<int>(cout), static_cast<int>(cin), taps,
      static_cast<int>(cout_use), static_cast<int>(cin_pad));
  LTX_CUDA(cudaGetLastError());
  LTX_CUDA(cudaStreamSynchronize(c->stream));
  auto it = c->tensors.find(wkey);
  cudaFree(it->second.ptr);
  c->tensors.erase(it);
  ConvW r;
  r.w = packed; r.b = reinterpret_cast<const float*>(b.ptr); r.cin = static_cast<int>(cin_pad); r.cout = static_cast<int>(cout_use);
  r.taps = taps;
  return r;
}

namespace {

ConvW pack_conv(ltx_ctx* c, const std::string& name, int64_t cout, int64_t cin) {
  return vae_pack_conv_keys(c, name + ".conv.weight", name + ".conv.bias", cout, cin, cout, 27);
}

}  // namespace

const float* vae_vec(ltx_ctx* c, const std::string& k, int64_t n) {
  const DevTensor& t = get_tensor(c, k);
  LTX_CHECK(t.dtype == LTX_F32 && t.numel() == n, LTX_ERR_WEIGHTS, "bad shape for '" + k + "'");
  return reinterpret_cast<const float*>(t.ptr);
}

// One convolution = padding prologue (fp32 [T,H,W,Cin] -> activated bf16 [T+2,H+2,W+2,Cin]) + implicit-GEMM kernel.
// pad: VAE_PAD_* bits.  n_active > 1: this rank holds a temporal slab; the two time-padding frames of the conv input come
// from the neighbouring ranks (the global first / last slab keep the replicated frame the prologue wrote).
void vae_conv(ltx_ctx* c, const float* x, int prep_mode, const float* a, const float* b, const ConvW& w, int T, int H, int W,
              int pad, int epi_mode, void* out, const float* resid, int n_active, int t_shift) {
  c->v_pad.reserve(static_cast<size_t>(T + 2) * (H + 2) * (W + 2) * w.cin * 2);
  const double vox = static_cast<double>(T) * H * W;
  {
    ProfScope ps(c, PROF_PREP, 0.0, vox * w.cin * 4.0 + static_cast<double>(T + 2) * (H + 2) * (W + 2) * w.cin * 2.0);
    launch_vae_prep(x, c->v_pad.as<bf16>(), T, H, W, w.cin, prep_mode, a, b, pad, c->stream);
  }
  if (n_active > 1) {
    const size_t frame = static_cast<size_t>(H + 2) * (W + 2) * w.cin;  // one padded frame, contiguous in v_pad
    bf16* padv = c->v_pad.as<bf16>();
    ProfScope ps(c, PROF_COMM, 0.0, 4.0 * frame * 2.0);
    dist_halo_exchange(c, padv + frame, padv, padv + static_cast<size_t>(T) * frame, padv + static_cast<size_t>(T + 1) * frame,
                       frame * 2, n_active);
  }
  ConvEpi e;
  e.mode = epi_mode; e.bias = w.b; e.resid = resid; e.Cin = w.cin; e.t_shift = t_shift;
  if (epi_mode == CONV_EPI_RGB8 || epi_mode == CONV_EPI_I420) e.out_u8 = static_cast<uint8_t*>(out);
  else e.out = static_cast<float*>(out);
  e.no_clip = c->vae_no_clip;
  ProfScope ps(c, PROF_CONV, 2.0 * w.taps * w.cin * w.cout * vox,
               vox * (w.cin * 2.0 + w.cout * 4.0) + static_cast<double>(w.taps) * w.cin * w.cout * 2.0);
  // scratch for the tap-split of tile-starved convs (three partial-sum slabs)
  const size_t slab3 = static_cast<size_t>(3) * T * H * W * w.cout * 4;
  float* scratch = nullptr;
  if (epi_mode == 0 && w.taps == 27 && conv3d_wants_tap_split(H, W, w.cin, w.cout)) {
    c->v_split.reserve(slab3);
    scratch = c->v_split.as<float>();
  }
  launch_conv3d(c->v_pad.as<bf16>(), w.w, T, H, W, w.cin, w.cout, e, c->stream, w.taps, scratch, scratch ? slab3 : 0);
}

// A group of VAEResBlock3d (V/VideoDecoder.swift:93-130, 152-167) with both hand-overs fused into the producing conv's epilogue
// (conv3d.cu modes 3 and 4): only the first conv1 of the group runs the padding prologue kernel; afterwards
//   conv1 epilogue -> bf16 interior of conv2's padded volume (pixel-norm, scale2/shift2, SiLU; the fp32 h is never written)
//   conv2 epilogue -> x += ... as fp32 AND the bf16 interior of the next block's conv1 input (scale1/shift1 of that block)
// a halo-fill pass completes each padded volume (+ the neighbour exchange on temporal shards).  tables[j] = block j's
// [shift1 | scale1 | shift2 | scale2] rows.  Requires 64 < C <= 256 (one tile = all channels of a voxel).
void vae_resgroup_fused(ltx_ctx* c, float* x, const std::vector<VaeResBlock>& blocks, const std::vector<const float*>& tables, int T,
                        int H, int W, int pad, int n_active) {
  const int C = blocks[0].c1.cout;
  const size_t padded = static_cast<size_t>(T + 2) * (H + 2) * (W + 2);
  c->v_pad.reserve(padded * C * 2);
  c->v_pad2.reserve(padded * C * 2);
  bf16* padA = c->v_pad.as<bf16>();
  bf16* padB = c->v_pad2.as<bf16>();
  const double vox = static_cast<double>(T) * H * W;
  const int tshift = (pad & VAE_PAD_CAUSAL) ? 2 : 1;
  auto exchange = [&](bf16* pv) {
    if (n_active <= 1) return;
    const size_t frame = static_cast<size_t>(H + 2) * (W + 2) * C;
    ProfScope ps(c, PROF_COMM, 0.0, 4.0 * frame * 2.0);
    dist_halo_exchange(c, pv + frame, pv, pv + static_cast<size_t>(T) * frame, pv + static_cast<size_t>(T + 1) * frame, frame * 2, n_active);
  };
  auto halo = [&](bf16* pv) {
    {
      ProfScope ps(c, PROF_PREP, 0.0, static_cast<double>(padded - vox) * C * 4.0);
      launch_vae_halo_fill(pv, T, H, W, C, pad, c->stream);
    }
    exchange(pv);
  };
  {
    ProfScope ps(c, PROF_PREP, 0.0, vox * C * 4.0 + static_cast<double>(padded) * C * 2.0);
    launch_vae_prep(x, padA, T, H, W, C, 2, tables[0] + C, tables[0], pad, c->stream);
  }
  exchange(padA);
  const double cflops = 2.0 * 27.0 * C * C * vox, wbytes = 27.0 * C * C * 2.0;
  // conv2 -> next conv1 hand-over (mode 4, in the coalesced epilogue domain).  Measured: 25-frame decode 16.26 -> 16.14 ms
  // (prologue 3.1 -> 2.3 ms, convs +1.5 ms: the second epilogue pass is exposed at the short 128-channel main loops), 121 frames
  // 76.7 -> 72.3 ms.
  for (size_t j = 0; j < blocks.size(); ++j) {
    const VaeResBlock& rb = blocks[j];
    const float* tb = tables[j];
    {
      ConvEpi e;
      e.mode = 3; e.out = nullptr; e.bias = rb.c1.b; e.resid = nullptr; e.Cin = C;
      e.next_pad = padB; e.next_scale = tb + 3 * C; e.next_shift = tb + 2 * C; e.next_tshift = tshift;
      ProfScope ps(c, PROF_CONV, cflops, vox * C * 4.0 + wbytes);
      launch_conv3d(padA, rb.c1.w, T, H, W, C, C, e, c->stream, 27);
    }
    halo(padB);
    const bool last = j + 1 == blocks.size();
    ConvEpi e;
    e.mode = last ? 0 : 4; e.out = x; e.bias = rb.c2.b; e.resid = x; e.Cin = C;
    if (!last) { e.next_pad = padA; e.next_scale = tables[j + 1] + C; e.next_shift = tables[j + 1]; e.next_tshift = tshift; }
    {
      ProfScope ps(c, PROF_CONV, cflops, vox * C * (last ? 10.0 : 12.0) + wbytes);
      launch_conv3d(padB, rb.c2.w, T, H, W, C, C, e, c->stream, 27);
    }
    if (!last) {
      halo(padA);
    } else if (j + 1 < blocks.size()) {   // next block's conv1 input through the prologue kernel
      {
        ProfScope ps(c, PROF_PREP, 0.0, vox * C * 4.0 + static_cast<double>(padded) * C * 2.0);
        launch_vae_prep(x, padA, T, H, W, C, 2, tables[j + 1] + C, tables[j + 1], pad, c->stream);
      }
      exchange(padA);
    }
  }
}

namespace {
inline const float* vf(ltx_ctx* c, const std::string& k, int64_t n) { return vae_vec(c, k, n); }
inline void conv(ltx_ctx* c, const float* x, int prep_mode, const float* a, const float* b, const ConvW& w, int T, int H, int W,
                 int causal, int epi_mode, void* out, const float* resid, int n_active = 1, int t_shift = 0) {
  vae_conv(c, x, prep_mode, a, b, w, T, H, W, causal ? VAE_PAD_CAUSAL : 0, epi_mode, out, resid, n_active, t_shift);
}
}  // namespace

void vae_finalize(ltx_ctx* c) {
  const ltx_config& g = c->cfg;
  LTX_CHECK(g.vae_base_channels % 512 == 0 || g.vae_base_channels % 64 == 0, LTX_ERR_INVALID_CONFIGURATION, "vae channels");
  LTX_CHECK((g.vae_base_channels / 8) % 64 == 0, LTX_ERR_INVALID_CONFIGURATION,
            "vae_base_channels / 8 must be a multiple of 64");
  LTX_CHECK(g.vae_latent_channels % 64 == 0, LTX_ERR_INVALID_CONFIGURATION, "vae_latent_channels must be a multiple of 64");
  VaeWeights& v = c->vae;
  const int64_t C = g.vae_latent_channels;
  v.mean = vf(c, "vae.mean_of_means", C);
  v.std = vf(c, "vae.std_of_means", C);
  int64_t ch = g.vae_base_channels;
  v.conv_in = pack_conv(c, "vae.conv_in", ch, C);
  v.stages.clear();
  v.ups.clear();
  for (int st = 0; st < 4; ++st) {
    const std::string blk = "vae.up_blocks_" + std::to_string(2 * st);
    std::vector<VaeResBlock> rbs;
    for (int j = 0; j < g.vae_blocks_per_stage; ++j) {
      const std::string rb = blk + ".res_blocks." + std::to_string(j);
      VaeResBlock r;
      r.c1 = pack_conv(c, rb + ".conv1", ch, ch);
      r.c2 = pack_conv(c, rb + ".conv2", ch, ch);
      r.sst = vf(c, rb + ".scale_shift_table", 4 * ch);
      rbs.push_back(r);
    }
    v.stages.push_back(rbs);
    if (st < 3) {
      v.ups.push_back(pack_conv(c, "vae.up_blocks_" + std::to_string(2 * st + 1) + ".conv", 4 * ch, ch));
      ch /= 2;
    }
  }
  v.last_sst = vf(c, "vae.last_scale_shift_table", 2 * ch);
  // optional timestep conditioning (V/VideoDecoder.swift:136-167, 311-318, 419-436)
  v.has_time = c->tensors.count("vae.last_time_embedder.timestep_embedder.linear_1.weight") > 0;
  if (v.has_time) {
    auto te = [&](const std::string& pfx, int out) {
      VaeTimeEmb t;
      const DevTensor& w1 = get_tensor(c, pfx + ".timestep_embedder.linear_1.weight");
      const DevTensor& w2 = get_tensor(c, pfx + ".timestep_embedder.linear_2.weight");
      LTX_CHECK(w1.dtype == LTX_BF16 && w1.shape.size() == 2 && w1.shape[0] == 256 && w1.shape[1] == 256 && w2.dtype == LTX_BF16 &&
                    w2.shape.size() == 2 && w2.shape[0] == out && w2.shape[1] == 256,
                LTX_ERR_WEIGHTS, "bad time embedder shape under '" + pfx + "'");
      t.w1 = reinterpret_cast<const bf16*>(w1.ptr); t.w2 = reinterpret_cast<const bf16*>(w2.ptr);
      t.b1 = vf(c, pfx + ".timestep_embedder.linear_1.bias", 256);
      t.b2 = vf(c, pfx + ".timestep_embedder.linear_2.bias", out);
      t.out = out;
      return t;
    };
    int64_t cc = g.vae_base_channels;
    for (int st = 0; st < 4; ++st) {
      v.stage_te[st] = te("vae.up_blocks_" + std::to_string(2 * st) + ".time_embedder", static_cast<int>(4 * cc));
      if (st < 3) cc /= 2;
    }
    v.last_te = te("vae.last_time_embedder", static_cast<int>(2 * cc));
    if (c->tensors.count("vae.timestep_scale_multiplier")) {
      const DevTensor& m = get_tensor(c, "vae.timestep_scale_multiplier");
      LTX_CHECK(m.dtype == LTX_F32 && m.numel() == 1, LTX_ERR_WEIGHTS, "bad timestep_scale_multiplier");
      LTX_CUDA(cudaMemcpy(&v.ts_mult, m.ptr, 4, cudaMemcpyDeviceToHost));
    }
  }
  v.conv_out = pack_conv(c, "vae.conv_out", 3 * g.vae_patch_size * g.vae_patch_size, ch);
  LTX_CHECK(g.vae_patch_size == 4, LTX_ERR_INVALID_CONFIGURATION, "vae_patch_size must be 4");
  v.ready = true;
}

void vae_decode_dev(ltx_ctx* c, const float* latent_dev, int Fp, int Hp, int Wp, float timestep, const float* noise_dev,
                    int causal, void* frames_dev, int format) {
  VaeWeights& v = c->vae;
  LTX_CHECK(format == FRAMES_F32 || format == LTX_FRAMES_RGB8 || format == LTX_FRAMES_I420, LTX_ERR_INVALID_ARGUMENT,
            "bad frame format");
  LTX_CHECK(v.ready, LTX_ERR_WEIGHTS, "VAE weights not finalized");
  LTX_CHECK(latent_dev && frames_dev && Fp > 0 && Hp > 1 && Wp > 1, LTX_ERR_INVALID_ARGUMENT, "bad vae_decode arguments");
  LTX_CHECK(format == FRAMES_F32 || reinterpret_cast<uintptr_t>(frames_dev) % 4 == 0, LTX_ERR_INVALID_ARGUMENT,
            "8-bit frames need a 4-byte aligned output buffer");
  const bool timed = timestep >= 0.f;
  LTX_CHECK(!timed || v.has_time, LTX_ERR_WEIGHTS, "timestep-conditioned decode needs the VAE time-embedder weights");
  LTX_CHECK(!timed || noise_dev != nullptr, LTX_ERR_INVALID_ARGUMENT, "decode_noise is required when timestep >= 0");
  const ltx_config& g = c->cfg;
  cudaStream_t st = c->stream;
  const int C0 = g.vae_latent_channels;
  // ---- timestep conditioning (:368-375): x = 0.025 * noise + 0.975 * x on the normalised latent; every res-block table and
  // the last table get + time_emb(sincos(t * multiplier)).  te_buf: [sincos 256 | hidden 256 | emb 4C] scratch + effective tables.
  const float* latent_in = latent_dev;
  float* te_base = nullptr;
  if (timed) {
    const size_t n = static_cast<size_t>(C0) * Fp * Hp * Wp;
    c->v_mix.reserve(n * 4);
    LTX_CUDA(cudaMemcpyAsync(c->v_mix.ptr, latent_dev, n * 4, cudaMemcpyDeviceToDevice, st));
    {
      ProfScope ps(c, PROF_OTHER, 0.0, 12.0 * n);
      int64_t blocks = (static_cast<int64_t>(n) + 255) / 256;
      if (blocks > 4096) blocks = 4096;
      noise_mix_kernel<<<static_cast<int>(blocks), 256, 0, st>>>(c->v_mix.as<float>(), noise_dev, static_cast<int64_t>(n), 0.025f);
      LTX_CUDA(cudaGetLastError());
    }
    latent_in = c->v_mix.as<float>();
    c->v_te.reserve((1 + 256 + 256 + 4 * static_cast<size_t>(g.vae_base_channels) * (1 + std::max(1, g.vae_blocks_per_stage)) + 64) * 4);
    te_base = c->v_te.as<float>();
    const float ts_host = timestep;
    LTX_CUDA(cudaMemcpyAsync(te_base, &ts_host, 4, cudaMemcpyHostToDevice, st));
    launch_sincos_embed(te_base, v.ts_mult, te_base + 16, 1, 256, st);
    c->launches++;
  }
  // effective scale-shift table of a block: table (+ time embedding of its stage)
  auto time_emb = [&](const VaeTimeEmb& te, float* out) {   // out[te.out]
    ProfScope ps(c, PROF_OTHER, 0.0, 2.0 * 256 * (256 + te.out), 2);
    launch_gemv(te.w1, te.b1, te_base + 16, te_base + 16 + 256, 1, 256, 256, 0, st);
    launch_gemv(te.w2, te.b2, te_base + 16 + 256, out, 1, te.out, 256, 1, st);
  };
  float* te_stage = timed ? te_base + 16 + 512 : nullptr;                                   // [4C]
  float* tbl_eff = timed ? te_stage + 4 * static_cast<size_t>(g.vae_base_channels) : nullptr;   // [4C]
  auto eff_table = [&](const float* sst, int n) -> const float* {
    if (!timed) return sst;
    ProfScope ps(c, PROF_OTHER, 0.0, 12.0 * n);
    add_vec_kernel<<<(n + 255) / 256, 256, 0, st>>>(tbl_eff, sst, te_stage, n);
    LTX_CUDA(cudaGetLastError());
    return tbl_eff;
  };
  // ---- temporal sharding: the first n_active ranks own contiguous slabs of latent frames [f0, f1)
  const int world = c->dist.world, rank = c->dist.rank;
  const int n_active = (c->dist.comm_world && world > 1) ? std::min(world, Fp) : 1;
  LTX_CHECK(n_active == 1 || !causal, LTX_ERR_UNSUPPORTED, "temporally sharded decode supports the non-causal decoder only");
  auto slab = [&](int r, int& f0, int& f1) {
    const int base = Fp / n_active, rem = Fp % n_active;
    f0 = r * base + std::min(r, rem);
    f1 = f0 + base + (r < rem ? 1 : 0);
  };
  int f0 = 0, f1 = Fp;
  if (n_active > 1 && rank < n_active) slab(rank, f0, f1);
  const bool active = rank < n_active;
  const int Ho = 32 * Hp, Wo = 32 * Wp;
  const size_t frame_bytes = format == FRAMES_F32 ? static_cast<size_t>(Ho) * Wo * 3 * 4 : frames_u8_bytes(1, Ho, Wo, format);
  uint8_t* frames = static_cast<uint8_t*>(frames_dev);
  if (active) {
    int T = f1 - f0, H = Hp, W = Wp;
    const int t_shift = (n_active > 1 && rank > 0) ? 1 : 0;
    // worst-case activation sizes over the stages: x at stage s has ch_s channels on a (T_s, H_s, W_s) grid
    size_t max_x = 0;
    {
      int t = T, h = Hp, w = Wp;
      int64_t ch = g.vae_base_channels;
      for (int s = 0; s < 4; ++s) {
        max_x = std::max(max_x, static_cast<size_t>(t) * h * w * ch);
        if (s < 3) { t = 2 * t - 1 + t_shift; h *= 2; w *= 2; ch /= 2; }
      }
      max_x = std::max(max_x, static_cast<size_t>(T) * Hp * Wp * C0);
    }
    c->v_a.reserve(max_x * 4);
    c->v_b.reserve(max_x * 4);
    c->v_h.reserve(max_x * 4);
    float* x = c->v_a.as<float>();
    float* y = c->v_b.as<float>();
    float* hbuf = c->v_h.as<float>();
    // [C, F*H*W] (frames f0..f1) -> channels-last [T*H*W, C]
    {
      ProfScope ps(c, PROF_OTHER, 0.0, 8.0 * C0 * T * H * W);
      launch_transpose_slice(latent_in + static_cast<size_t>(f0) * H * W, static_cast<int64_t>(Fp) * H * W, C0, T * H * W, hbuf,
                             st);
    }
    // denormalise (x*std + mean, :379-381) fused into conv_in's padding prologue
    conv(c, hbuf, 1, v.std, v.mean, v.conv_in, T, H, W, causal, 0, x, nullptr, n_active);
    int64_t ch = g.vae_base_channels;
    for (int s = 0; s < 4; ++s) {
      if (timed) time_emb(v.stage_te[s], te_stage);   // one embedding per res-block group (:152-160)
      const bool fuse = ch > 64 && ch <= 256 && ch % 32 == 0 && !v.stages[s].empty();
      if (fuse) {
        // every block's effective table is needed at once: a conv2 epilogue applies the NEXT block's scale1 / shift1
        std::vector<const float*> tabs;
        for (size_t j = 0; j < v.stages[s].size(); ++j) {
          const VaeResBlock& rb = v.stages[s][j];
          if (!timed) { tabs.push_back(rb.sst); continue; }
          float* dstt = tbl_eff + j * 4 * ch;
          ProfScope ps(c, PROF_OTHER, 0.0, 12.0 * 4 * ch);
          add_vec_kernel<<<static_cast<int>((4 * ch + 255) / 256), 256, 0, st>>>(dstt, rb.sst, te_stage, static_cast<int>(4 * ch));
          LTX_CUDA(cudaGetLastError());
          tabs.push_back(dstt);
        }
        vae_resgroup_fused(c, x, v.stages[s], tabs, T, H, W, causal ? VAE_PAD_CAUSAL : 0, n_active);
      } else {
        for (const VaeResBlock& rb : v.stages[s]) {
          // h = conv1(silu(pn(x) * (1 + scale1) + shift1)) ; x = x + conv2(silu(pn(h) * (1 + scale2) + shift2))   (:93-130)
          const float* tb = eff_table(rb.sst, static_cast<int>(4 * ch));
          conv(c, x, 2, tb + ch, tb, rb.c1, T, H, W, causal, 0, hbuf, nullptr, n_active);
          conv(c, hbuf, 2, tb + 3 * ch, tb + 2 * ch, rb.c2, T, H, W, causal, 0, x, x, n_active);
        }
      }
      if (s < 3) {
        // conv -> d2s -> drop frame 0 (first slab only) -> + tiled d2s(x)
        conv(c, x, 0, nullptr, nullptr, v.ups[s], T, H, W, causal, 1, y, x, n_active, t_shift);
        std::swap(x, y);
        T = 2 * T - 1 + t_shift; H *= 2; W *= 2; ch /= 2;
      }
    }
    // pn * (1 + scale) + shift -> SiLU -> conv_out -> unpatchify -> (x+1)/2 clip -> [F, H, W, 3]   (:419-444, 501-505),
    // or straight on to 8-bit frames (tensorToImages, U/VideoExporter.swift:543-580, or I420) in the same store
    const int out_f0 = f0 == 0 ? 0 : 8 * (f0 - 1) + 1;
    if (timed) time_emb(v.last_te, te_stage);
    const float* lt = eff_table(v.last_sst, static_cast<int>(2 * ch));
    const int out_mode = format == LTX_FRAMES_RGB8 ? CONV_EPI_RGB8 : (format == LTX_FRAMES_I420 ? CONV_EPI_I420 : 2);
    conv(c, x, 2, lt + ch, lt, v.conv_out, T, H, W, causal, out_mode, frames + static_cast<size_t>(out_f0) * frame_bytes,
         nullptr, n_active);
  }
  if (n_active > 1) {
    // all ranks receive every slab (an all-gather with unequal counts, as one broadcast per owner)
    ProfScope ps(c, PROF_COMM, 0.0, static_cast<double>(frame_bytes) * (8.0 * (Fp - 1) + 1), n_active);
    for (int r = 0; r < n_active; ++r) {
      int a0, a1;
      slab(r, a0, a1);
      const int o0 = a0 == 0 ? 0 : 8 * (a0 - 1) + 1, o1 = 8 * (a1 - 1) + 1;
      dist_broadcast(c, frames + static_cast<size_t>(o0) * frame_bytes, static_cast<size_t>(o1 - o0) * frame_bytes, r);
    }
  }
}

// decodeWithTemporalTiling (V/VideoDecoder.swift:517-602): overlapping chunks of `tile_size` latent frames (stride
// tile_size - overlap) are decoded independently and their 8 * overlap boundary frames cross-faded; the result is clipped
// afterwards.  The chunk decodes store (x + 1) / 2 unclipped -- the blend is linear, so blending those equals blending x.
// Returns the number of frames written (the reference's chunk arithmetic, not 8 (F' - 1) + 1 in general).
int vae_tiled_frames(int Fp, int tile_size, int overlap) {
  if (tile_size <= 0 || Fp <= tile_size) return 8 * (Fp - 1) + 1;
  const int stride = tile_size - overlap, po = 8 * overlap;
  int total = 0;
  for (int start = 0;; start += stride) {
    const int end = std::min(start + tile_size, Fp), nf = 8 * (end - start - 1) + 1;
    if (total == 0) total = nf;
    else total += (po > 0 && po < total && po < nf) ? nf - po : nf;
    if (end >= Fp) break;
  }
  return total;
}

// 8-bit formats: the fp32 chunks are blended and clipped in v_frames_f32 and converted at the end (frames_to_u8_dev).
int vae_decode_tiled_dev(ltx_ctx* c, const float* latent_dev, int Fp, int Hp, int Wp, float timestep, const float* noise_dev,
                         int causal, int tile_size, int overlap, void* out_dev, int format) {
  LTX_CHECK(format == FRAMES_F32 || format == LTX_FRAMES_RGB8 || format == LTX_FRAMES_I420, LTX_ERR_INVALID_ARGUMENT,
            "bad frame format");
  LTX_CHECK(latent_dev && out_dev && Fp > 0 && Hp > 1 && Wp > 1, LTX_ERR_INVALID_ARGUMENT, "bad vae_decode arguments");
  if (tile_size <= 0 || Fp <= tile_size) {   // decodeVideo's single-pass branch (:482, 496)
    vae_decode_dev(c, latent_dev, Fp, Hp, Wp, timestep, noise_dev, causal, out_dev, format);
    return 8 * (Fp - 1) + 1;
  }
  LTX_CHECK(overlap >= 0 && overlap < tile_size, LTX_ERR_INVALID_ARGUMENT, "temporal tile overlap must be in [0, tile size)");
  const bool timed = timestep >= 0.f;
  LTX_CHECK(!timed || noise_dev != nullptr, LTX_ERR_INVALID_ARGUMENT, "decode_noise is required when timestep >= 0");
  const int C0 = c->cfg.vae_latent_channels, stride = tile_size - overlap, po = 8 * overlap;
  const size_t hw = static_cast<size_t>(Hp) * Wp, fe = static_cast<size_t>(32 * Hp) * (32 * Wp) * 3;
  cudaStream_t st = c->stream;
  c->v_tile_lat.reserve(static_cast<size_t>(C0) * tile_size * hw * 4);
  if (timed) c->v_tile_noise.reserve(static_cast<size_t>(C0) * tile_size * hw * 4);
  c->v_tile_frames.reserve(static_cast<size_t>(8 * (tile_size - 1) + 1) * fe * 4);
  float* frames_dev = static_cast<float*>(out_dev);
  if (format != FRAMES_F32) {
    c->v_frames_f32.reserve(static_cast<size_t>(vae_tiled_frames(Fp, tile_size, overlap)) * fe * 4);
    frames_dev = c->v_frames_f32.as<float>();
  }
  struct NoClip {   // the chunk decodes leave the clip to the end; restored on every exit path
    ltx_ctx* c;
    explicit NoClip(ltx_ctx* cc) : c(cc) { c->vae_no_clip = 1; }
    ~NoClip() { c->vae_no_clip = 0; }
  } guard(c);
  auto grid_for = [](int64_t n4) { return static_cast<int>(std::min<int64_t>((n4 + 255) / 256, 148 * 16)); };
  int total = 0;
  for (int start = 0;; start += stride) {
    const int end = std::min(start + tile_size, Fp), Fc = end - start, nf = 8 * (Fc - 1) + 1;
    // gather frames [start, end) of every channel: [C, F', H'W'] -> [C, Fc, H'W']
    {
      ProfScope ps(c, PROF_OTHER, 0.0, 8.0 * C0 * Fc * hw * (timed ? 2 : 1), timed ? 2 : 1);
      LTX_CUDA(cudaMemcpy2DAsync(c->v_tile_lat.ptr, Fc * hw * 4, latent_dev + start * hw, static_cast<size_t>(Fp) * hw * 4, Fc * hw * 4,
                                 C0, cudaMemcpyDeviceToDevice, st));
      if (timed)
        LTX_CUDA(cudaMemcpy2DAsync(c->v_tile_noise.ptr, Fc * hw * 4, noise_dev + start * hw, static_cast<size_t>(Fp) * hw * 4,
                                   Fc * hw * 4, C0, cudaMemcpyDeviceToDevice, st));
    }
    float* dst = total == 0 ? frames_dev : c->v_tile_frames.as<float>();
    vae_decode_dev(c, c->v_tile_lat.as<float>(), Fc, Hp, Wp, timestep, timed ? c->v_tile_noise.as<float>() : nullptr, causal, dst);
    if (total == 0) {
      total = nf;
    } else if (po > 0 && po < total && po < nf) {
      ProfScope ps(c, PROF_OTHER, 0.0, 4.0 * fe * (3.0 * po + 2.0 * (nf - po)), 2);
      tile_blend_kernel<<<grid_for(static_cast<int64_t>(fe) * po / 4), 256, 0, st>>>(frames_dev + static_cast<size_t>(total - po) * fe,
                                                                                   dst, static_cast<int64_t>(fe), po);
      LTX_CUDA(cudaGetLastError());
      LTX_CUDA(cudaMemcpyAsync(frames_dev + static_cast<size_t>(total) * fe, dst + static_cast<size_t>(po) * fe,
                               static_cast<size_t>(nf - po) * fe * 4, cudaMemcpyDeviceToDevice, st));
      total += nf - po;
    } else {
      ProfScope ps(c, PROF_OTHER, 0.0, 8.0 * fe * nf);
      LTX_CUDA(cudaMemcpyAsync(frames_dev + static_cast<size_t>(total) * fe, dst, static_cast<size_t>(nf) * fe * 4,
                               cudaMemcpyDeviceToDevice, st));
      total += nf;
    }
    if (end >= Fp) break;
  }
  {
    const int64_t n4 = static_cast<int64_t>(total) * fe / 4;
    ProfScope ps(c, PROF_OTHER, 0.0, 8.0 * fe * total);
    clip01_kernel<<<grid_for(n4), 256, 0, st>>>(frames_dev, n4);
    LTX_CUDA(cudaGetLastError());
  }
  if (format != FRAMES_F32) frames_to_u8_dev(c, frames_dev, total, 32 * Hp, 32 * Wp, format, static_cast<uint8_t*>(out_dev));
  return total;
}

}  // namespace ltx
