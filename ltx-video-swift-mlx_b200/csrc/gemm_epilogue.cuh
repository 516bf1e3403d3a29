// Fused GEMM epilogues shared by the bf16 (1-CTA, 2-CTA, 4-CTA) and the dequant-fused kernels.
//
// One epilogue warp owns 32 accumulator rows (its TMEM lane quarter).  tcgen05.ld hands each THREAD one row, which is the
// wrong shape for global memory (32 rows x 16 B per instruction = 32 L1 wavefronts).  Each 32x32 fp32 chunk is therefore
// transposed through a warp-private 4 KB shared-memory tile (float4 slots XOR-swizzled by row, conflict-free both ways),
// after which 8 lanes cover 128 contiguous bytes of one row and one instruction touches 4 rows = 4 wavefronts.  Per-column
// operands (bias, gate) are loaded once per chunk per lane.  The TMEM load of chunk c+1 is issued before the global traffic
// of chunk c, so it overlaps it.
#pragma once
#include "ltx_internal.h"
#include "ptx.cuh"

namespace ltx {

constexpr int EPI_STAGE_BYTES = 32 * 32 * 4;  // per epilogue warp

// thread = row: park this thread's 32 columns in the swizzled staging tile
__device__ __forceinline__ void epi_stage_write(float* stage, int lane, const uint32_t (&r)[32]) {
  float4* st4 = reinterpret_cast<float4*>(stage) + lane * 8;
#pragma unroll
  for (int j = 0; j < 8; ++j)
    st4[j ^ (lane & 7)] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                                      __uint_as_float(r[4 * j + 3]));
}

__device__ __forceinline__ float4 ld4_guard(const float* p, int nvalid) {
  if (nvalid >= 4) return *reinterpret_cast<const float4*>(p);
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (nvalid > 0) v.x = p[0];
  if (nvalid > 1) v.y = p[1];
  if (nvalid > 2) v.z = p[2];
  return v;
}

// Global side of one staged chunk: rows [row0, row0+32), columns [col0, col0+ncols), ncols = 32 or 16.
// Lane l owns columns col0 + 4*(l&7) .. +3 of rows (l>>3) + 4*i, i = 0..7.
template <int MODE>
__device__ __forceinline__ void epi_store_chunk(const float* stage, int lane, int row0, int col0, int ncols, int M, int N,
                                                const GemmEpi& ep, const float4 (&xin)[8]) {
  const int cg = lane & 7, rs = lane >> 3;
  const int c = col0 + cg * 4;
  const int nlim = (col0 + ncols < N) ? col0 + ncols : N;   // never touch the next tile's columns from a 16-wide tail chunk
  const int nvalid = nlim - c;                               // columns of this lane's group that exist (<= 0: none)
  if (nvalid <= 0 || row0 >= M) return;
  const float4* st4 = reinterpret_cast<const float4*>(stage);
  float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
  if (ep.bias && !ep.bias_per_row) bv = ld4_guard(ep.bias + c, nvalid);

  if (MODE == EPI_GATE_RESID) {
    float4 gb = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ep.gate_a && ep.gate_b) gb = ld4_guard(ep.gate_b + c, nvalid);
    // rows of this chunk usually share one gate vector (rows_per_gate >= 32): fetch it once
    const int last_row = (row0 + 31 < M ? row0 + 31 : M - 1);
    const bool uniform_gate = ep.gate_a && (row0 / ep.rows_per_gate == last_row / ep.rows_per_gate);
    float4 gu = make_float4(1.f, 1.f, 1.f, 1.f);
    if (uniform_gate) {
      const float4 t = ld4_guard(ep.gate_a + static_cast<int64_t>(row0 / ep.rows_per_gate) * ep.gate_ld + c, nvalid);
      gu = make_float4(t.x + gb.x, t.y + gb.y, t.z + gb.z, t.w + gb.w);
    }
    // the residual values xin[] were prefetched by epi_prefetch_resid (all loads issued before any store of the chunk:
    // the compiler cannot prove that stores do not alias later loads, interleaving would serialise the memory latencies)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int rr = rs + 4 * i, row = row0 + rr;
      if (row >= M) break;
      const float4 a = st4[rr * 8 + (cg ^ (rr & 7))];
      float4 g = gu;
      if (ep.gate_a && !uniform_gate) {   // per-token gates (per-token timesteps): one gate row per output row
        const float4 t = ld4_guard(ep.gate_a + static_cast<int64_t>(row / ep.rows_per_gate) * ep.gate_ld + c, nvalid);
        g = make_float4(t.x + gb.x, t.y + gb.y, t.z + gb.z, t.w + gb.w);
      }
      const float rb = (ep.bias && ep.bias_per_row) ? ep.bias[row] : 0.f;
      float4 xv = xin[i];
      xv.x += (a.x + bv.x + rb) * g.x * ep.scale;
      xv.y += (a.y + bv.y + rb) * g.y * ep.scale;
      xv.z += (a.z + bv.z + rb) * g.z * ep.scale;
      xv.w += (a.w + bv.w + rb) * g.w * ep.scale;
      float* xr = ep.resid + static_cast<int64_t>(row) * ep.ldr + c;
      bf16* sh = ep.shadow ? ep.shadow + static_cast<int64_t>(row) * ep.lds + c : nullptr;
      if (nvalid >= 4) {
        *reinterpret_cast<float4*>(xr) = xv;
        if (sh) *reinterpret_cast<uint2*>(sh) = make_uint2(pack_bf16(xv.x, xv.y), pack_bf16(xv.z, xv.w));
      } else {
        const float v[3] = {xv.x, xv.y, xv.z};
        for (int j = 0; j < nvalid; ++j) {
          xr[j] = v[j];
          if (sh) sh[j] = __float2bfloat16(v[j]);
        }
      }
    }
  } else if (MODE == EPI_F32) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int rr = rs + 4 * i, row = row0 + rr;
      if (row >= M) break;
      const float4 a = st4[rr * 8 + (cg ^ (rr & 7))];
      const float rb = (ep.bias && ep.bias_per_row) ? ep.bias[row] : 0.f;
      const float4 v = make_float4(a.x + bv.x + rb, a.y + bv.y + rb, a.z + bv.z + rb, a.w + bv.w + rb);
      float* o = reinterpret_cast<float*>(ep.out) + static_cast<int64_t>(row) * ep.ldo + c;
      if (nvalid >= 4) {
        *reinterpret_cast<float4*>(o) = v;
      } else {
        const float vv[3] = {v.x, v.y, v.z};
        for (int j = 0; j < nvalid; ++j) o[j] = vv[j];
      }
    }
  } else {  // EPI_BF16 / EPI_GELU_BF16 / EPI_SILU_BF16
    // column-blocked destination (Ulysses send layout): a 4-column group never straddles a block (col_block % 32 == 0)
    bf16* obase = reinterpret_cast<bf16*>(ep.out) + c;
    int64_t old = ep.ldo;
    if (ep.col_block > 0 && c >= ep.col_block_from) {
      const int cb = c - ep.col_block_from;
      if (ep.blocked_ld) old = ep.blocked_ld;
      if (ep.use_col_ptrs)   // one base per destination rank: the store goes over NVLink when the block is a peer's
        obase = reinterpret_cast<bf16*>(ep.col_ptrs.p[cb / ep.col_block]) + (cb % ep.col_block);
      else
        obase = reinterpret_cast<bf16*>(ep.blocked_out ? ep.blocked_out : ep.out) + static_cast<int64_t>(cb / ep.col_block) * ep.col_block_stride +
                (cb % ep.col_block);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int rr = rs + 4 * i, row = row0 + rr;
      if (row >= M) break;
      const float4 a = st4[rr * 8 + (cg ^ (rr & 7))];
      const float rb = (ep.bias && ep.bias_per_row) ? ep.bias[row] : 0.f;
      float v[4] = {a.x + bv.x + rb, a.y + bv.y + rb, a.z + bv.z + rb, a.w + bv.w + rb};
      if (MODE == EPI_GELU_BF16) {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = gelu_tanh(v[j]);
      }
      if (MODE == EPI_SILU_BF16) {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = silu(v[j]);
      }
      bf16* o = obase + static_cast<int64_t>(row) * old;
      if (nvalid >= 4) {
        *reinterpret_cast<uint2*>(o) = make_uint2(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]));
      } else {
        for (int j = 0; j < nvalid; ++j) o[j] = __float2bfloat16(v[j]);
      }
    }
  }
}

// Transposed store of one staged chunk (bf16): lane l owns column col0 + l and gathers its 32 rows from the staging tile
// (bank = ((l >> 2) ^ (rr & 7)) * 4 + (l & 3): a permutation of the 32 banks for every rr), adds the bias, and writes 64
// contiguous bytes of row (n - tsplit_col) of the transposed output.
__device__ __forceinline__ void epi_store_chunk_t(const float* stage, int lane, int row0, int col0, int ncols, int M, int N,
                                                  const GemmEpi& ep) {
  const int n = col0 + lane;
  if (lane >= ncols || n >= N || row0 >= M) return;
  const float b = (ep.bias && !ep.bias_per_row) ? ep.bias[n] : 0.f;
  bf16* dst = ep.out_t + static_cast<int64_t>(n - ep.tsplit_col) * ep.ldt + row0;
  const int nrows = (M - row0 < 32) ? M - row0 : 32;
  float v[32];
#pragma unroll
  for (int rr = 0; rr < 32; ++rr) v[rr] = stage[(rr * 8 + ((lane >> 2) ^ (rr & 7))) * 4 + (lane & 3)] + b;
  if (nrows == 32) {
#pragma unroll
    for (int q4 = 0; q4 < 4; ++q4)
      *reinterpret_cast<uint4*>(dst + q4 * 8) = make_uint4(pack_bf16(v[q4 * 8], v[q4 * 8 + 1]), pack_bf16(v[q4 * 8 + 2], v[q4 * 8 + 3]),
                                                           pack_bf16(v[q4 * 8 + 4], v[q4 * 8 + 5]), pack_bf16(v[q4 * 8 + 6], v[q4 * 8 + 7]));
  } else {
    for (int rr = 0; rr < nrows; ++rr) dst[rr] = __float2bfloat16(v[rr]);
  }
}

// EPI_GATE_RESID: fetch this lane's 8 residual float4 of chunk [row0, +32) x [col0, +ncols) (same ownership as above)
__device__ __forceinline__ void epi_prefetch_resid(float4 (&xin)[8], int lane, int row0, int col0, int ncols, int M, int N,
                                                   const GemmEpi& ep) {
  const int cg = lane & 7, rs = lane >> 3;
  const int c = col0 + cg * 4;
  const int nlim = (col0 + ncols < N) ? col0 + ncols : N;
  const int nvalid = nlim - c;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int row = row0 + rs + 4 * i;
    xin[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < M && nvalid > 0) xin[i] = ld4_guard(ep.resid + static_cast<int64_t>(row) * ep.ldr + c, nvalid);
  }
}

// SCALED (the FP8 pair kernel): this thread's accumulator row times sa[row], then times sb[column], in fp32 and in that order,
// before anything else of the epilogue.  Columns past N read no scale (their results are never stored).
__device__ __forceinline__ void epi_scale_chunk(uint32_t (&r)[32], float sa, const float* sb, int col0, int N) {
  float s[32];
  if (col0 + 32 <= N) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 t = reinterpret_cast<const float4*>(sb + col0)[j];
      s[4 * j] = t.x; s[4 * j + 1] = t.y; s[4 * j + 2] = t.z; s[4 * j + 3] = t.w;
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) s[j] = col0 + j < N ? sb[col0 + j] : 0.f;
  }
#pragma unroll
  for (int j = 0; j < 32; ++j) r[j] = __float_as_uint((__uint_as_float(r[j]) * sa) * s[j]);
}

// Whole-tile epilogue of one warp: accumulator lanes [taddr.lane, +32) x BN columns starting at TMEM address `taddr`;
// output rows [row0, row0+32), columns [col_base, col_base+BN).  BN is a multiple of 16.  Must be called by all 32 lanes.
template <int MODE, bool SCALED = false>
__device__ __forceinline__ void epilogue_tile(uint32_t taddr, int BN, float* stage, int lane, int row0, int col_base, int M,
                                              int N, const GemmEpi& ep, const float* sa = nullptr, const float* sb = nullptr) {
  const int nfull = BN >> 5;
  const int nch = nfull + ((BN & 16) ? 1 : 0);
  uint32_t r[32];
  float4 xcur[8], xnext[8];   // residual prefetch, one chunk ahead (EPI_GATE_RESID only; dead code otherwise)
  if (nfull > 0) tmem_ld32(taddr, r);
  else tmem_ld16(taddr, r);
  if (MODE == EPI_GATE_RESID) epi_prefetch_resid(xcur, lane, row0, col_base, nfull > 0 ? 32 : 16, M, N, ep);
  float row_s = 0.f;
  if (SCALED && row0 + lane < M) row_s = sa[row0 + lane];
#pragma unroll 1
  for (int c = 0; c < nch; ++c) {
    tmem_ld_wait();
    if (SCALED) epi_scale_chunk(r, row_s, sb, col_base + c * 32, N);
    epi_stage_write(stage, lane, r);
    __syncwarp();
    if (c + 1 < nch) {   // next chunk's TMEM read and residual loads overlap this chunk's global traffic
      if (c + 1 < nfull) tmem_ld32(taddr + (c + 1) * 32, r);
      else tmem_ld16(taddr + (c + 1) * 32, r);
      if (MODE == EPI_GATE_RESID)
        epi_prefetch_resid(xnext, lane, row0, col_base + (c + 1) * 32, (c + 1 < nfull) ? 32 : 16, M, N, ep);
    }
    if (MODE == EPI_BF16 && ep.tsplit_col > 0 && col_base + c * 32 >= ep.tsplit_col)
      epi_store_chunk_t(stage, lane, row0, col_base + c * 32, (c < nfull) ? 32 : 16, M, N, ep);
    else
      epi_store_chunk<MODE>(stage, lane, row0, col_base + c * 32, (c < nfull) ? 32 : 16, M, N, ep, xcur);
    __syncwarp();
    if (MODE == EPI_GATE_RESID) {
#pragma unroll
      for (int i = 0; i < 8; ++i) xcur[i] = xnext[i];
    }
  }
}

}  // namespace ltx
