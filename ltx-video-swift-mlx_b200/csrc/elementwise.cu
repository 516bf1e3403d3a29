// HBM-bound row / elementwise kernels of the DiT step: AdaLN-modulated RMSNorm / LayerNorm, q/k RMSNorm-across-heads
// fused with split RoPE, the timestep-embedding GEMV chain, patchify / unpatchify, and the fused
// CFG + rescale + STG + GE + Euler update.  All vectorised 16-byte accesses, fp32 math.
// The two row kernels of a DiT block take D = 4096 in a streaming form (rmsnorm_mod_stream_kernel, qknorm_rope_stream_kernel:
// persistent CTAs whose rows arrive in shared memory by cp.async.bulk, all of a CTA's rows requested up front) and other
// widths in the generic one-row-per-CTA kernels.
#include <algorithm>

#include "ltx_internal.h"
#include "ptx.cuh"

namespace ltx {

namespace {

__device__ __forceinline__ float block_sum(float v, float* red) {
  // red: >= 33 floats of shared memory
  v = warp_sum(v);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  if (warp == 0) {
    float t = lane < nw ? red[lane] : 0.f;
    t = warp_sum(t);
    if (lane == 0) red[32] = t;
  }
  __syncthreads();
  return red[32];
}

// ---------------------------------------------------------------------------------------------
// AdaLN: out = norm(x) * (1 + scale) + shift      (T/LTXTransformerBlock.swift:72-83, T/LTXTransformer.swift:208-221)
// norm = RMSNorm without weight (layernorm = 0) or LayerNorm without affine (layernorm = 1).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) rmsnorm_mod_kernel(const float* __restrict__ x, bf16* __restrict__ out, int D,
                                                           const float* __restrict__ tbl_shift,
                                                           const float* __restrict__ tbl_scale,
                                                           const float* __restrict__ ada_shift,
                                                           const float* __restrict__ ada_scale, int64_t ada_ld,
                                                           int rows_per_mod, float eps, int layernorm) {
  __shared__ float red[33];
  const int row = blockIdx.x;
  const float* xr = x + static_cast<int64_t>(row) * D;
  const int nv = D >> 2;
  float s1 = 0.f, s2 = 0.f;
  for (int i = threadIdx.x; i < nv; i += blockDim.x) {
    float4 v = reinterpret_cast<const float4*>(xr)[i];
    s1 += v.x + v.y + v.z + v.w;
    s2 += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  float mean = 0.f, rstd;
  if (layernorm) {
    mean = block_sum(s1, red) / D;
    float sv = 0.f;
    for (int i = threadIdx.x; i < nv; i += blockDim.x) {
      float4 v = reinterpret_cast<const float4*>(xr)[i];
      float a = v.x - mean, b = v.y - mean, c = v.z - mean, d = v.w - mean;
      sv += a * a + b * b + c * c + d * d;
    }
    rstd = rsqrtf(block_sum(sv, red) / D + eps);
  } else {
    rstd = rsqrtf(block_sum(s2, red) / D + eps);
  }
  const int64_t aoff = static_cast<int64_t>(row / rows_per_mod) * ada_ld;
  const float4* sh_t = reinterpret_cast<const float4*>(tbl_shift);
  const float4* sc_t = reinterpret_cast<const float4*>(tbl_scale);
  const float4* sh_a = reinterpret_cast<const float4*>(ada_shift + aoff);
  const float4* sc_a = reinterpret_cast<const float4*>(ada_scale + aoff);
  bf16* orow = out + static_cast<int64_t>(row) * D;
  for (int i = threadIdx.x; i < nv; i += blockDim.x) {
    float4 v = reinterpret_cast<const float4*>(xr)[i];
    float4 a = sh_t[i], b = sh_a[i], c = sc_t[i], d = sc_a[i];
    float y0 = (v.x - mean) * rstd * (1.f + c.x + d.x) + a.x + b.x;
    float y1 = (v.y - mean) * rstd * (1.f + c.y + d.y) + a.y + b.y;
    float y2 = (v.z - mean) * rstd * (1.f + c.z + d.z) + a.z + b.z;
    float y3 = (v.w - mean) * rstd * (1.f + c.w + d.w) + a.w + b.w;
    reinterpret_cast<uint2*>(orow)[i] = make_uint2(pack_bf16(y0, y1), pack_bf16(y2, y3));
  }
}

// Streaming form (D = 4096): persistent CTAs, three per SM, each with a ring of NST row buffers in shared memory
// that ONE thread fills with 16 KB bulk copies (cp.async.bulk + mbarrier) -- every row a CTA will ever touch is requested
// before the first one is reduced, at no register cost: 3 x NST x 16 KB in flight per SM against 64 KB for a form that
// staged 4 rows per CTA in registers (146 registers -> one CTA per SM: load phase, reduce phase, store phase in turn:
// 2.9 TB/s at M = 1536).  The modulation vectors stay in registers for the CTA's whole life (one L2 read per CTA).
// Reduction scratch alternates between two slots, so one __syncthreads per reduction is enough; the same barrier tells
// the filling thread that every thread has taken its part of the stage out of shared memory.
__device__ __forceinline__ float block_sum_256(float v, float* red, int& slot) {
  v = warp_sum(v);
  float* r = red + (slot & 1) * 8;
  ++slot;
  if ((threadIdx.x & 31) == 0) r[threadIdx.x >> 5] = v;
  __syncthreads();
  return ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
}

template <int NST>
__global__ void __launch_bounds__(256, 3) rmsnorm_mod_stream_kernel(const float* x, bf16* out, int M,
                                                                     const float* __restrict__ tbl_shift,
                                                                     const float* __restrict__ tbl_scale,
                                                                     const float* ada_shift, const float* ada_scale,
                                                                     int64_t ada_ld, int rows_per_mod, float eps, int layernorm) {
  constexpr int D = 4096, ROW_BYTES = D * 4;
  extern __shared__ __align__(128) uint8_t smem_rows[];
  const float4* stage = reinterpret_cast<const float4*>(smem_rows);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_rows + NST * ROW_BYTES);
  float* red = reinterpret_cast<float*>(full + NST);   // 2 x 8 floats
  const int t = threadIdx.x;
  const int first = blockIdx.x, stride = gridDim.x;
  const int n_my = (M - first + stride - 1) / stride;   // first < M: the launcher never starts more CTAs than rows
  if (t == 0) {
#pragma unroll
    for (int s = 0; s < NST; ++s) mbar_init(&full[s], 1);
    fence_mbar_init();
  }
  __syncthreads();
  griddep_launch();
  griddep_wait();   // x and the ada vectors come from preceding kernels
  if (t == 0) {
    for (int i = 0; i < NST && i < n_my; ++i) {
      mbar_arrive_expect_tx(&full[i], ROW_BYTES);
      bulk_load_1d(smem_rows + i * ROW_BYTES, x + static_cast<int64_t>(first + i * stride) * D, ROW_BYTES, &full[i]);
    }
  }
  int cur_mod = -1, slot = 0;
  float4 sc[4], sh[4];
  for (int i = 0; i < n_my; ++i) {
    const int s = i % NST;
    const int row = first + i * stride;
    const int mod = row / rows_per_mod;
    if (mod != cur_mod) {   // while the row is in flight
      cur_mod = mod;
      const int64_t aoff = static_cast<int64_t>(mod) * ada_ld;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int c = t + k * 256;
        const float4 a = reinterpret_cast<const float4*>(tbl_scale)[c], b = reinterpret_cast<const float4*>(ada_scale + aoff)[c];
        const float4 e = reinterpret_cast<const float4*>(tbl_shift)[c], f = reinterpret_cast<const float4*>(ada_shift + aoff)[c];
        sc[k] = make_float4(1.f + a.x + b.x, 1.f + a.y + b.y, 1.f + a.z + b.z, 1.f + a.w + b.w);
        sh[k] = make_float4(e.x + f.x, e.y + f.y, e.z + f.z, e.w + f.w);
      }
    }
    mbar_wait(&full[s], (i / NST) & 1);
    float4 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = stage[s * (D / 4) + t + k * 256];
    float mean = 0.f, part = 0.f;
    if (layernorm) {
#pragma unroll
      for (int k = 0; k < 4; ++k) part += (v[k].x + v[k].y) + (v[k].z + v[k].w);
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k) part += (v[k].x * v[k].x + v[k].y * v[k].y) + (v[k].z * v[k].z + v[k].w * v[k].w);
    }
    float tot = block_sum_256(part, red, slot);
    // every thread holds its part of the stage in registers: refill it with the row NST steps ahead
    if (t == 0 && i + NST < n_my) {
      mbar_arrive_expect_tx(&full[s], ROW_BYTES);
      bulk_load_1d(smem_rows + s * ROW_BYTES, x + static_cast<int64_t>(row + NST * stride) * D, ROW_BYTES, &full[s]);
    }
    if (layernorm) {
      mean = tot / D;
      part = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float a = v[k].x - mean, b = v[k].y - mean, c = v[k].z - mean, d = v[k].w - mean;
        part += (a * a + b * b) + (c * c + d * d);
      }
      tot = block_sum_256(part, red, slot);
    }
    const float rstd = rsqrtf(tot / D + eps);
    uint2* orow = reinterpret_cast<uint2*>(out + static_cast<int64_t>(row) * D);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float y0 = (v[k].x - mean) * rstd * sc[k].x + sh[k].x;
      const float y1 = (v[k].y - mean) * rstd * sc[k].y + sh[k].y;
      const float y2 = (v[k].z - mean) * rstd * sc[k].z + sh[k].z;
      const float y3 = (v[k].w - mean) * rstd * sc[k].w + sh[k].w;
      orow[t + k * 256] = make_uint2(pack_bf16(y0, y1), pack_bf16(y2, y3));
    }
  }
}

// ---------------------------------------------------------------------------------------------
// q/k RMSNorm across all heads (learned weight) + split RoPE, in place on bf16 rows.
// T/LTXAttention.swift:179-189, T/LTXRoPE.swift:84-149.  cos/sin: [rows_per_rope, D/2] fp32, index h*64 + j.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) qknorm_rope_kernel(bf16* __restrict__ x, int64_t ld, int D,
                                                           const float* __restrict__ w, const float* __restrict__ cosb,
                                                           const float* __restrict__ sinb, int rows_per_rope, float eps,
                                                           bf16* __restrict__ bout, int hpb, int64_t bstride, int64_t bld,
                                                           int use_peer, const PeerTable peer) {
  __shared__ float red[33];
  const int row = blockIdx.x;
  bf16* xr = x + static_cast<int64_t>(row) * ld;
  const int nchunk = D >> 3;  // 8 bf16 per 16-byte chunk
  float ss = 0.f;
  for (int i = threadIdx.x; i < nchunk; i += blockDim.x) {
    uint4 u = reinterpret_cast<const uint4*>(xr)[i];
    const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      float2 f = __bfloat1622float2(h2[t]);
      ss += f.x * f.x + f.y * f.y;
    }
  }
  const float rstd = rsqrtf(block_sum(ss, red) / D + eps);
  // pair-chunks: head hh, 8 consecutive j in [0,64): x1 at hh*128 + j, x2 at hh*128 + 64 + j
  const int npair = D >> 4;
  const float* cr = cosb ? cosb + static_cast<int64_t>(row % rows_per_rope) * (D >> 1) : nullptr;
  const float* sr = sinb ? sinb + static_cast<int64_t>(row % rows_per_rope) * (D >> 1) : nullptr;
  for (int pc = threadIdx.x; pc < npair; pc += blockDim.x) {
    const int hh = pc >> 3, jc = (pc & 7) * 8;
    const int c1 = hh * 128 + jc, c2 = c1 + 64;
    uint4 u1 = *reinterpret_cast<const uint4*>(xr + c1);
    uint4 u2 = *reinterpret_cast<const uint4*>(xr + c2);
    const __nv_bfloat162* a2 = reinterpret_cast<const __nv_bfloat162*>(&u1);
    const __nv_bfloat162* b2 = reinterpret_cast<const __nv_bfloat162*>(&u2);
    float x1[8], x2[8], y1[8], y2[8];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      float2 fa = __bfloat1622float2(a2[t]), fb = __bfloat1622float2(b2[t]);
      x1[2 * t] = fa.x * rstd * w[c1 + 2 * t];
      x1[2 * t + 1] = fa.y * rstd * w[c1 + 2 * t + 1];
      x2[2 * t] = fb.x * rstd * w[c2 + 2 * t];
      x2[2 * t + 1] = fb.y * rstd * w[c2 + 2 * t + 1];
    }
    if (cr) {
      const int fi = hh * 64 + jc;
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const float c = cr[fi + t], s = sr[fi + t];
        y1[t] = x1[t] * c - x2[t] * s;
        y2[t] = x2[t] * c + x1[t] * s;
      }
    } else {
#pragma unroll
      for (int t = 0; t < 8; ++t) { y1[t] = x1[t]; y2[t] = x2[t]; }
    }
    bf16* o1 = xr + c1;
    bf16* o2 = xr + c2;
    if (use_peer) {
      bf16* ob = reinterpret_cast<bf16*>(peer.p[hh / hpb]) + static_cast<int64_t>(row) * bld + (hh % hpb) * 128 + jc;
      o1 = ob;
      o2 = ob + 64;
    } else if (bout) {
      bf16* ob = bout + static_cast<int64_t>(hh / hpb) * bstride + static_cast<int64_t>(row) * bld + (hh % hpb) * 128 + jc;
      o1 = ob;
      o2 = ob + 64;
    }
    *reinterpret_cast<uint4*>(o1) =
        make_uint4(pack_bf16(y1[0], y1[1]), pack_bf16(y1[2], y1[3]), pack_bf16(y1[4], y1[5]), pack_bf16(y1[6], y1[7]));
    *reinterpret_cast<uint4*>(o2) =
        make_uint4(pack_bf16(y2[0], y2[1]), pack_bf16(y2[2], y2[3]), pack_bf16(y2[4], y2[5]), pack_bf16(y2[6], y2[7]));
  }
}

// Streaming form of the q/k norm (D = 4096): as rmsnorm_mod_stream_kernel.  A stage holds one row: the nseg
// (1 | 2) bf16 segments -- contiguous in the fused q|k projection output -- and, with RoPE, its cos and sin rows, so the
// rotation tables are fetched once per row for both segments.  Two CTAs per SM, STAGES_BYTES of bulk copies in flight each.
constexpr int QK_STREAM_BYTES = 96 * 1024;

template <bool ROPE>
__global__ void __launch_bounds__(256, 2) qknorm_rope_stream_kernel(bf16* x, int64_t ld, int M, int nseg,
                                                                     const float* __restrict__ w0, const float* __restrict__ w1,
                                                                     const float* __restrict__ cosb, const float* __restrict__ sinb,
                                                                     int rows_per_rope, float eps, bf16* bout0, bf16* bout1, int hpb,
                                                                     int64_t bstride, int64_t bld, int use_peer,
                                                                     const PeerTable peer0, const PeerTable peer1) {
  constexpr int D = 4096, SEG_BYTES = D * 2, TAB_BYTES = (D / 2) * 4;
  extern __shared__ __align__(128) uint8_t smem_rows[];
  const int x_bytes = nseg * SEG_BYTES;
  const int stage_bytes = x_bytes + (ROPE ? 2 * TAB_BYTES : 0);
  const int nst = min(8, QK_STREAM_BYTES / stage_bytes);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_rows + QK_STREAM_BYTES);
  float* red = reinterpret_cast<float*>(full + 8);   // 2 slots x 2 segments x 8 warps
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int first = blockIdx.x, stride = gridDim.x;
  const int n_my = (M - first + stride - 1) / stride;
  const int hh = t >> 3, jc = (t & 7) * 8;
  const int c1 = hh * 128 + jc, c2 = c1 + 64;
  float wa[2][8], wb[2][8];
#pragma unroll
  for (int sg = 0; sg < 2; ++sg) {
    const float* w = sg == 0 ? w0 : w1;
    if (sg < nseg) {
#pragma unroll
      for (int e = 0; e < 8; e += 4) {
        const float4 a = *reinterpret_cast<const float4*>(w + c1 + e), b = *reinterpret_cast<const float4*>(w + c2 + e);
        wa[sg][e] = a.x; wa[sg][e + 1] = a.y; wa[sg][e + 2] = a.z; wa[sg][e + 3] = a.w;
        wb[sg][e] = b.x; wb[sg][e + 1] = b.y; wb[sg][e + 2] = b.z; wb[sg][e + 3] = b.w;
      }
    }
  }
  if (t == 0) {
    for (int s = 0; s < nst; ++s) mbar_init(&full[s], 1);
    fence_mbar_init();
  }
  __syncthreads();
  griddep_launch();
  griddep_wait();   // x comes from the preceding GEMM
  auto fill = [&](int s, int row) {
    uint8_t* dst = smem_rows + s * stage_bytes;
    mbar_arrive_expect_tx(&full[s], stage_bytes);
    bulk_load_1d(dst, x + static_cast<int64_t>(row) * ld, x_bytes, &full[s]);
    if (ROPE) {
      const int64_t fo = static_cast<int64_t>(row % rows_per_rope) * (D / 2);
      bulk_load_1d(dst + x_bytes, cosb + fo, TAB_BYTES, &full[s]);
      bulk_load_1d(dst + x_bytes + TAB_BYTES, sinb + fo, TAB_BYTES, &full[s]);
    }
  };
  if (t == 0)
    for (int i = 0; i < nst && i < n_my; ++i) fill(i, first + i * stride);
  int slot = 0;
  for (int i = 0; i < n_my; ++i) {
    const int s = i % nst;
    const int row = first + i * stride;
    const uint8_t* src = smem_rows + s * stage_bytes;
    mbar_wait(&full[s], (i / nst) & 1);
    uint4 u1[2], u2[2];
    float ss[2] = {0.f, 0.f};
#pragma unroll
    for (int sg = 0; sg < 2; ++sg) {
      if (sg < nseg) {
        u1[sg] = *reinterpret_cast<const uint4*>(src + sg * SEG_BYTES + c1 * 2);
        u2[sg] = *reinterpret_cast<const uint4*>(src + sg * SEG_BYTES + c2 * 2);
        const __nv_bfloat162* a2 = reinterpret_cast<const __nv_bfloat162*>(&u1[sg]);
        const __nv_bfloat162* b2 = reinterpret_cast<const __nv_bfloat162*>(&u2[sg]);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 fa = __bfloat1622float2(a2[e]), fb = __bfloat1622float2(b2[e]);
          ss[sg] += fa.x * fa.x + fa.y * fa.y + fb.x * fb.x + fb.y * fb.y;
        }
      }
    }
    float cs[8], sn[8];
    if (ROPE) {
      const float* ct = reinterpret_cast<const float*>(src + x_bytes) + hh * 64 + jc;
      const float* stb = ct + D / 2;
#pragma unroll
      for (int e = 0; e < 8; e += 4) {
        const float4 a = *reinterpret_cast<const float4*>(ct + e), b = *reinterpret_cast<const float4*>(stb + e);
        cs[e] = a.x; cs[e + 1] = a.y; cs[e + 2] = a.z; cs[e + 3] = a.w;
        sn[e] = b.x; sn[e + 1] = b.y; sn[e + 2] = b.z; sn[e + 3] = b.w;
      }
    }
    // both segments' sums of squares in one barrier; scratch alternates between two slots
    ss[0] = warp_sum(ss[0]);
    ss[1] = warp_sum(ss[1]);
    float* r = red + (slot & 1) * 16;
    ++slot;
    if (lane == 0) { r[warp] = ss[0]; r[8 + warp] = ss[1]; }
    __syncthreads();
    if (t == 0 && i + nst < n_my) fill(s, row + nst * stride);   // the stage is in registers everywhere
#pragma unroll
    for (int sg = 0; sg < 2; ++sg) {
      if (sg >= nseg) break;
      const float* rr = r + sg * 8;
      const float tot = ((rr[0] + rr[1]) + (rr[2] + rr[3])) + ((rr[4] + rr[5]) + (rr[6] + rr[7]));
      const float rstd = rsqrtf(tot / D + eps);
      const __nv_bfloat162* a2 = reinterpret_cast<const __nv_bfloat162*>(&u1[sg]);
      const __nv_bfloat162* b2 = reinterpret_cast<const __nv_bfloat162*>(&u2[sg]);
      float y1[8], y2[8];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 fa = __bfloat1622float2(a2[e]), fb = __bfloat1622float2(b2[e]);
        const float xa[2] = {fa.x, fa.y}, xb[2] = {fb.x, fb.y};
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int j = 2 * e + h;
          const float a = xa[h] * rstd * wa[sg][j], b = xb[h] * rstd * wb[sg][j];
          if (ROPE) {
            y1[j] = a * cs[j] - b * sn[j];
            y2[j] = b * cs[j] + a * sn[j];
          } else {
            y1[j] = a; y2[j] = b;
          }
        }
      }
      bf16* xr = x + static_cast<int64_t>(row) * ld + static_cast<int64_t>(sg) * D;
      bf16* o1 = xr + c1;
      bf16* o2 = xr + c2;
      bf16* bout = sg == 0 ? bout0 : bout1;
      if (use_peer) {   // Ulysses over peer memory: head block hh / hpb lives in that rank's receive buffer
        bf16* base = reinterpret_cast<bf16*>(sg == 0 ? peer0.p[hh / hpb] : peer1.p[hh / hpb]);
        bf16* ob = base + static_cast<int64_t>(row) * bld + (hh % hpb) * 128 + jc;
        o1 = ob;
        o2 = ob + 64;
      } else if (bout) {
        bf16* ob = bout + static_cast<int64_t>(hh / hpb) * bstride + static_cast<int64_t>(row) * bld + (hh % hpb) * 128 + jc;
        o1 = ob;
        o2 = ob + 64;
      }
      *reinterpret_cast<uint4*>(o1) =
          make_uint4(pack_bf16(y1[0], y1[1]), pack_bf16(y1[2], y1[3]), pack_bf16(y1[4], y1[5]), pack_bf16(y1[6], y1[7]));
      *reinterpret_cast<uint4*>(o2) =
          make_uint4(pack_bf16(y2[0], y2[1]), pack_bf16(y2[2], y2[3]), pack_bf16(y2[4], y2[5]), pack_bf16(y2[6], y2[7]));
    }
  }
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ in, bf16* __restrict__ out, int64_t n4) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float4 v = reinterpret_cast<const float4*>(in)[i];
    reinterpret_cast<uint2*>(out)[i] = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
  }
}
__global__ void cast_bf16_f32_kernel(const bf16* __restrict__ in, float* __restrict__ out, int64_t n) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    out[i] = __bfloat162float(in[i]);
}

// ---------------------------------------------------------------------------------------------
// Timestep path (T/LTXTimestepEmbedding.swift:17-124): sinusoidal embedding and small-M linear layers.
// ---------------------------------------------------------------------------------------------
__global__ void sincos_embed_kernel(const float* __restrict__ sigma, float mult, float* __restrict__ out, int dim,
                                    bf16* __restrict__ out_bf16) {
  const int m = blockIdx.x, half = dim >> 1;
  const float t = sigma[m] * mult;
  for (int k = threadIdx.x; k < half; k += blockDim.x) {
    const float f = expf(-logf(10000.0f) * (static_cast<float>(k) / static_cast<float>(half)));
    const float a = t * f;
    const float cv = cosf(a), sv = sinf(a);
    if (out) {
      out[static_cast<int64_t>(m) * dim + k] = cv;
      out[static_cast<int64_t>(m) * dim + half + k] = sv;
    }
    if (out_bf16) {
      out_bf16[static_cast<int64_t>(m) * dim + k] = __float2bfloat16(cv);
      out_bf16[static_cast<int64_t>(m) * dim + half + k] = __float2bfloat16(sv);
    }
  }
}
__global__ void silu_cast_kernel(const float* __restrict__ in, bf16* __restrict__ out, int64_t n4) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(in)[i];
    reinterpret_cast<uint2*>(out)[i] = make_uint2(pack_bf16(silu(v.x), silu(v.y)), pack_bf16(silu(v.z), silu(v.w)));
  }
}
__global__ void fill_token_timesteps_kernel(float* __restrict__ ts, int n, int period, int frozen, const float* __restrict__ sigma) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) ts[i] = (i % period) < frozen ? 0.f : sigma[0];
}

// one warp per output feature; x rows staged through registers; W streamed once with 16-byte loads.
template <int MAXM>
__global__ void __launch_bounds__(256) gemv_kernel(const bf16* __restrict__ W, const float* __restrict__ bias,
                                                    const float* __restrict__ x, float* __restrict__ y, int M, int O, int I,
                                                    int silu_in) {
  const int o = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (o >= O) return;
  const bf16* wr = W + static_cast<int64_t>(o) * I;
  float acc[MAXM];
#pragma unroll
  for (int m = 0; m < MAXM; ++m) acc[m] = 0.f;
  for (int i = lane * 8; i < I; i += 256) {
    uint4 u = *reinterpret_cast<const uint4*>(wr + i);
    const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&u);
    float wv[8];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      float2 f = __bfloat1622float2(h2[t]);
      wv[2 * t] = f.x;
      wv[2 * t + 1] = f.y;
    }
#pragma unroll
    for (int m = 0; m < MAXM; ++m) {
      if (m < M) {
        const float* xr = x + static_cast<int64_t>(m) * I + i;
        float4 a = *reinterpret_cast<const float4*>(xr), b = *reinterpret_cast<const float4*>(xr + 4);
        float xv[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          float v = silu_in ? silu(xv[t]) : xv[t];
          acc[m] += wv[t] * v;
        }
      }
    }
  }
#pragma unroll
  for (int m = 0; m < MAXM; ++m) {
    float v = warp_sum(acc[m]);
    if (lane == 0 && m < M) y[static_cast<int64_t>(m) * O + o] = v + (bias ? bias[o] : 0.f);
  }
}

// ---------------------------------------------------------------------------------------------
// patchify / unpatchify (P/LatentUtils.swift:20-54): [C, T] <-> [T, C] transposes through a padded smem tile.
// ---------------------------------------------------------------------------------------------
__global__ void transpose_kernel(const float* __restrict__ in, float* __restrict__ out_f32, bf16* __restrict__ out_bf16,
                                 int R, int Cc, int64_t ld_in) {
  // in [R, Cc] (row pitch ld_in) -> out [Cc, R]
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < R && c < Cc) ? in[static_cast<int64_t>(r) * ld_in + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < Cc && r < R) {
      const float v = tile[threadIdx.x][i];
      if (out_f32) out_f32[static_cast<int64_t>(c) * R + r] = v;
      if (out_bf16) out_bf16[static_cast<int64_t>(c) * R + r] = __float2bfloat16(v);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Guidance + Euler (one pass; a preceding reduction pass only when guidance-rescale is on).
//   v = vc + (g-1)(vc - vu)                      P/LatentUtils.swift:131-141
//   v = phi * v * std(vc)/std(v) + (1-phi) * v   P/LatentUtils.swift:164-183 (population variance, eps 1e-8)
//   v += stg * (v - vp)                          P/LTXPipeline.swift:920
//   v = gamma * (v - v_prev) + v_prev            P/LTXPipeline.swift:924-927
//   x' = sigma' > 0 ? d + sigma' (x - d) / sigma : d,  d = x - sigma v      S/LTXScheduler.swift:305-327
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) guidance_stats_kernel(const float* __restrict__ vc, const float* __restrict__ vu,
                                                              size_t n, float cfg, double* __restrict__ acc) {
  // acc[0..3] = sum(vc), sum(vc^2), sum(v), sum(v^2) with v = cfg-combined velocity
  double s[4] = {0, 0, 0, 0};
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float c = vc[i], u = vu[i];
    const float v = c + (cfg - 1.0f) * (c - u);
    s[0] += c; s[1] += static_cast<double>(c) * c; s[2] += v; s[3] += static_cast<double>(v) * v;
  }
  __shared__ double red[4][8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    double v = s[k];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[k][warp] = v;
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    double t = 0;
    for (int w = 0; w < (blockDim.x >> 5); ++w) t += red[threadIdx.x][w];
    atomicAdd(&acc[threadIdx.x], t);
  }
}

__global__ void __launch_bounds__(256) guided_euler_kernel(GuidedEulerArgs a) {
  float rescale = 1.0f;
  const bool has_cfg = a.v_uncond != nullptr;
  if (has_cfg && a.phi > 0.f) {
    const double n = static_cast<double>(a.n);
    const double mc = a.scratch[0] / n, mv = a.scratch[2] / n;
    const double var_c = a.scratch[1] / n - mc * mc, var_v = a.scratch[3] / n - mv * mv;
    const float std_c = sqrtf(static_cast<float>(var_c) + 1e-8f), std_v = sqrtf(static_cast<float>(var_v) + 1e-8f);
    rescale = std_c / std_v;
  }
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < a.n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    float v = a.v_cond[i];
    if (has_cfg) {
      v = v + (a.cfg - 1.0f) * (v - a.v_uncond[i]);
      if (a.phi > 0.f) v = a.phi * (v * rescale) + (1.0f - a.phi) * v;
    }
    if (a.v_stg != nullptr && a.stg > 0.f) v = v + a.stg * (v - a.v_stg[i]);
    if (a.v_prev != nullptr) {
      if (a.ge_gamma > 0.f && a.use_prev) {
        const float pv = a.v_prev[i];
        v = a.ge_gamma * (v - pv) + pv;
      }
      a.v_prev[i] = v;
    }
    if (a.v_out) a.v_out[i] = v;
    if (a.period != 0 && (i % a.period) < a.frozen) continue;   // slice Euler: the conditioned first frame stays clean
    const float x = a.latent[i];
    const float den = x - a.sigma * v;
    a.latent[i] = (a.sigma_next > 0.f) ? den + a.sigma_next * (x - den) / a.sigma : den;
  }
}

// ---------------------------------------------------------------------------------------------
// Counter-based normal fill (random-init weights for the benchmark: no checkpoints in this environment).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__device__ __forceinline__ float2 normal_pair(uint64_t seed, uint64_t idx) {
  const uint64_t r = splitmix64(seed ^ splitmix64(idx));
  const float u1 = (static_cast<float>(r >> 40) + 1.0f) * (1.0f / 16777217.0f);
  const float u2 = static_cast<float>((r >> 8) & 0xFFFFFF) * (1.0f / 16777216.0f);
  const float rad = sqrtf(-2.0f * __logf(u1));
  float sn, cs;
  __sincosf(6.283185307179586f * u2, &sn, &cs);
  return make_float2(rad * cs, rad * sn);
}
template <typename T>
__global__ void fill_normal_kernel(T* __restrict__ p, int64_t n, float stdv, float mean, uint64_t seed) {
  const int64_t npair = (n + 1) >> 1;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < npair;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float2 z = normal_pair(seed, static_cast<uint64_t>(i));
    const float a = z.x * stdv + mean, b = z.y * stdv + mean;
    if (sizeof(T) == 2) {
      reinterpret_cast<bf16*>(p)[2 * i] = __float2bfloat16(a);
      if (2 * i + 1 < n) reinterpret_cast<bf16*>(p)[2 * i + 1] = __float2bfloat16(b);
    } else {
      reinterpret_cast<float*>(p)[2 * i] = a;
      if (2 * i + 1 < n) reinterpret_cast<float*>(p)[2 * i + 1] = b;
    }
  }
}

inline int grid_for(int64_t work, int threads) {
  int64_t blocks = (work + threads - 1) / threads;
  const int64_t cap = static_cast<int64_t>(device_sm_count()) * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

}  // namespace

void launch_rmsnorm_mod(const float* x, bf16* out, int M, int D, const float* tbl_shift, const float* tbl_scale,
                        const float* ada_shift, const float* ada_scale, int64_t ada_ld, int rows_per_mod, float eps,
                        int layernorm, cudaStream_t s) {
  LTX_CHECK(D % 4 == 0 && M > 0 && ada_ld % 4 == 0, 2, "rmsnorm_mod: D must be a multiple of 4");
  if (D == 4096) {   // rows arrive by 16 KB bulk copies
    LTX_CHECK((reinterpret_cast<uintptr_t>(x) & 15) == 0, 2, "rmsnorm_mod: x must be 16-byte aligned");
    constexpr int NST = 4;
    const size_t smem = NST * 4096 * 4 + NST * 8 + 64;
    auto kern = rmsnorm_mod_stream_kernel<NST>;
    ensure_dyn_smem(reinterpret_cast<const void*>(kern), smem);
    launch_pdl(PDL_ROWS, kern, dim3(std::min(M, 3 * device_sm_count())), dim3(256), smem, s, x, out, M, tbl_shift, tbl_scale,
               ada_shift, ada_scale, ada_ld, rows_per_mod > 0 ? rows_per_mod : 1, eps, layernorm);
    return;
  }
  rmsnorm_mod_kernel<<<M, 256, 0, s>>>(x, out, D, tbl_shift, tbl_scale, ada_shift, ada_scale, ada_ld,
                                       rows_per_mod > 0 ? rows_per_mod : 1, eps, layernorm);
  LTX_CUDA(cudaGetLastError());
}

void launch_qknorm_rope(bf16* x, int64_t ld, int M, int D, const float* w, const float* cosb, const float* sinb,
                        int rows_per_rope, float eps, cudaStream_t s, const float* w_second, const QkOut* blocked) {
  // w_second != nullptr: also normalise the second segment x[:, D:2D] with that weight (fused q|k projection output)
  LTX_CHECK(D % 128 == 0 && ld % 8 == 0 && M > 0, 2, "qknorm_rope: D must be a multiple of 128");
  const int rpr = rows_per_rope > 0 ? rows_per_rope : 1;
  bf16* b0 = blocked ? blocked->out[0] : nullptr;
  bf16* b1 = blocked ? blocked->out[1] : nullptr;
  const int hpb = blocked ? blocked->heads_per_block : 1;
  const int64_t bs = blocked ? blocked->block_stride : 0, bld = blocked ? blocked->ld : 0;
  const int use_peer = blocked ? blocked->use_peer : 0;
  const PeerTable pt0 = blocked ? blocked->peer[0] : PeerTable{}, pt1 = blocked ? blocked->peer[1] : PeerTable{};
  LTX_CHECK(!blocked || (hpb > 0 && (D / 128) % hpb == 0 && (use_peer || (b0 && (!w_second || b1)))), 2, "qknorm_rope: bad blocked output");
  if (D == 4096) {   // a row's segments and its cos / sin rows arrive by bulk copies: one contiguous, 16-byte aligned piece each
    LTX_CHECK((reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
                  (!cosb || ((reinterpret_cast<uintptr_t>(cosb) | reinterpret_cast<uintptr_t>(sinb)) & 15) == 0),
              2, "qknorm_rope: x, cos and sin must be 16-byte aligned");
    const size_t smem = QK_STREAM_BYTES + 8 * 8 + 128;
    const int nseg = w_second ? 2 : 1;
    const dim3 grid(std::min(M, 2 * device_sm_count()));
    if (cosb) {
      auto kern = qknorm_rope_stream_kernel<true>;
      ensure_dyn_smem(reinterpret_cast<const void*>(kern), smem);
      launch_pdl(PDL_ROWS, kern, grid, dim3(256), smem, s, x, ld, M, nseg, w, w_second, cosb, sinb, rpr, eps, b0, b1, hpb, bs, bld,
                 use_peer, pt0, pt1);
    } else {
      auto kern = qknorm_rope_stream_kernel<false>;
      ensure_dyn_smem(reinterpret_cast<const void*>(kern), smem);
      launch_pdl(PDL_ROWS, kern, grid, dim3(256), smem, s, x, ld, M, nseg, w, w_second, cosb, sinb, rpr, eps, b0, b1, hpb, bs, bld,
                 use_peer, pt0, pt1);
    }
    return;
  }
  qknorm_rope_kernel<<<M, 256, 0, s>>>(x, ld, D, w, cosb, sinb, rpr, eps, b0, hpb, bs, bld, use_peer, pt0);
  LTX_CUDA(cudaGetLastError());
  if (w_second) {
    qknorm_rope_kernel<<<M, 256, 0, s>>>(x + D, ld, D, w_second, cosb, sinb, rpr, eps, b1, hpb, bs, bld, use_peer, pt1);
    LTX_CUDA(cudaGetLastError());
  }
}

__global__ void transpose_bf16_kernel(const bf16* __restrict__ in, int64_t ld_in, int R, int Cc, bf16* __restrict__ out,
                                      int64_t ld_out) {
  __shared__ bf16 tile[32][34];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < R && c < Cc) ? in[static_cast<int64_t>(r) * ld_in + c] : __float2bfloat16(0.f);
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < Cc && r < R) out[static_cast<int64_t>(c) * ld_out + r] = tile[threadIdx.x][i];
  }
}
void launch_transpose_bf16(const bf16* in, int64_t ld_in, int R, int C, bf16* out, int64_t ld_out, cudaStream_t s) {
  dim3 grid((C + 31) / 32, (R + 31) / 32), block(32, 8);
  transpose_bf16_kernel<<<grid, block, 0, s>>>(in, ld_in, R, C, out, ld_out);
  LTX_CUDA(cudaGetLastError());
}

void launch_cast_f32_bf16(const float* in, bf16* out, int64_t n, cudaStream_t s) {
  LTX_CHECK(n % 4 == 0, 2, "cast: n must be a multiple of 4");
  cast_f32_bf16_kernel<<<grid_for(n / 4, 256), 256, 0, s>>>(in, out, n / 4);
  LTX_CUDA(cudaGetLastError());
}
void launch_cast_bf16_f32(const bf16* in, float* out, int64_t n, cudaStream_t s) {
  cast_bf16_f32_kernel<<<grid_for(n, 256), 256, 0, s>>>(in, out, n);
  LTX_CUDA(cudaGetLastError());
}

void launch_gemv(const bf16* W, const float* bias, const float* x, float* y, int M, int O, int I, int silu_in,
                 cudaStream_t s) {
  LTX_CHECK(I % 8 == 0, 2, "gemv: input width must be a multiple of 8");
  LTX_CHECK(M >= 1 && M <= 4, 2, "gemv: 1..4 rows (larger M goes through the GEMM)");
  const int wpb = 8;
  gemv_kernel<4><<<(O + wpb - 1) / wpb, wpb * 32, 0, s>>>(W, bias, x, y, M, O, I, silu_in);
  LTX_CUDA(cudaGetLastError());
}

__global__ void mask_to_bias_kernel(const int32_t* __restrict__ mask, float* __restrict__ bias, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) bias[i] = (1.0f - static_cast<float>(mask[i])) * -10000.0f;  // T/LTXTransformer.swift:141-156
}
__global__ void scale_f32_kernel(float* __restrict__ x, float a, int64_t n) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    x[i] *= a;
}
// audio latent of the audio + video loop: applyCFG on the audio velocity, then a += dt * v (P/LTXPipeline.swift:1340-1362,
// 1402); separate roundings (no FMA contraction) so the result equals the reference's op-by-op fp32 arithmetic
__global__ void audio_cfg_euler_kernel(float* __restrict__ lat, const float* __restrict__ vc, const float* __restrict__ vu,
                                       float cfg_m1, float dt, int64_t n) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float v = vc[i];
    if (vu) v = __fadd_rn(v, __fmul_rn(cfg_m1, __fsub_rn(v, vu[i])));
    lat[i] = __fadd_rn(lat[i], __fmul_rn(dt, v));
  }
}
void launch_audio_cfg_euler(float* lat, const float* v_cond, const float* v_uncond, float cfg_scale, float dt, int64_t n,
                            cudaStream_t s) {
  int64_t blocks = (n + 255) / 256;
  if (blocks > 4096) blocks = 4096;
  audio_cfg_euler_kernel<<<static_cast<int>(blocks), 256, 0, s>>>(lat, v_cond, v_uncond, cfg_scale - 1.0f, dt, n);
  LTX_CUDA(cudaGetLastError());
}
void launch_mask_to_bias(const int32_t* mask, float* bias, int n, cudaStream_t s) {
  mask_to_bias_kernel<<<(n + 255) / 256, 256, 0, s>>>(mask, bias, n);
  LTX_CUDA(cudaGetLastError());
}
void launch_scale_f32(float* x, float a, int64_t n, cudaStream_t s) {
  int64_t blocks = (n + 255) / 256;
  if (blocks > 4096) blocks = 4096;
  scale_f32_kernel<<<static_cast<int>(blocks), 256, 0, s>>>(x, a, n);
  LTX_CUDA(cudaGetLastError());
}

void launch_sincos_embed(const float* sigma, float mult, float* out, int M, int dim, cudaStream_t s, bf16* out_bf16) {
  sincos_embed_kernel<<<M, 128, 0, s>>>(sigma, mult, out, dim, out_bf16);
  LTX_CUDA(cudaGetLastError());
}
void launch_silu_cast(const float* in, bf16* out, int64_t n, cudaStream_t s) {
  LTX_CHECK(n % 4 == 0, 2, "silu_cast: n must be a multiple of 4");
  silu_cast_kernel<<<grid_for(n / 4, 256), 256, 0, s>>>(in, out, n / 4);
  LTX_CUDA(cudaGetLastError());
}
void launch_fill_token_timesteps(float* ts, int n, int period, int frozen, const float* sigma_dev, cudaStream_t s) {
  fill_token_timesteps_kernel<<<(n + 255) / 256, 256, 0, s>>>(ts, n, period, frozen, sigma_dev);
  LTX_CUDA(cudaGetLastError());
}

void launch_patchify(const float* latent, bf16* tok_bf16, float* tok_f32, int C, int T, cudaStream_t s) {
  dim3 grid((T + 31) / 32, (C + 31) / 32), block(32, 8);
  transpose_kernel<<<grid, block, 0, s>>>(latent, tok_f32, tok_bf16, C, T, T);
  LTX_CUDA(cudaGetLastError());
}
void launch_transpose_slice(const float* in, int64_t ld_in, int rows, int cols, float* out, cudaStream_t s) {
  // in [rows, cols] with row pitch ld_in -> out [cols, rows]
  dim3 grid((cols + 31) / 32, (rows + 31) / 32), block(32, 8);
  transpose_kernel<<<grid, block, 0, s>>>(in, out, nullptr, rows, cols, ld_in);
  LTX_CUDA(cudaGetLastError());
}
void launch_unpatchify(const float* tok, float* latent, int C, int T, cudaStream_t s) {
  dim3 grid((C + 31) / 32, (T + 31) / 32), block(32, 8);
  transpose_kernel<<<grid, block, 0, s>>>(tok, latent, nullptr, T, C, C);
  LTX_CUDA(cudaGetLastError());
}

void launch_guided_euler(const GuidedEulerArgs& a, cudaStream_t s) {
  LTX_CHECK(a.n > 0 && a.latent && a.v_cond, 2, "guided_euler: missing tensors");
  LTX_CHECK(a.sigma > 0.f, 2, "guided_euler: sigma must be > 0");
  if (a.v_uncond != nullptr && a.phi > 0.f) {
    LTX_CHECK(a.scratch != nullptr, 2, "guided_euler: rescale needs scratch");
    LTX_CUDA(cudaMemsetAsync(a.scratch, 0, 4 * sizeof(double), s));
    guidance_stats_kernel<<<grid_for(static_cast<int64_t>(a.n), 256), 256, 0, s>>>(a.v_cond, a.v_uncond, a.n, a.cfg,
                                                                                   a.scratch);
    LTX_CUDA(cudaGetLastError());
  }
  guided_euler_kernel<<<grid_for(static_cast<int64_t>(a.n), 256), 256, 0, s>>>(a);
  LTX_CUDA(cudaGetLastError());
}

void launch_fill_normal_bf16(bf16* p, int64_t n, float stdv, float mean, uint64_t seed, cudaStream_t s) {
  fill_normal_kernel<bf16><<<grid_for((n + 1) / 2, 256), 256, 0, s>>>(p, n, stdv, mean, seed);
  LTX_CUDA(cudaGetLastError());
}
void launch_fill_normal_f32(float* p, int64_t n, float stdv, float mean, uint64_t seed, cudaStream_t s) {
  fill_normal_kernel<float><<<grid_for((n + 1) / 2, 256), 256, 0, s>>>(p, n, stdv, mean, seed);
  LTX_CUDA(cudaGetLastError());
}

}  // namespace ltx
