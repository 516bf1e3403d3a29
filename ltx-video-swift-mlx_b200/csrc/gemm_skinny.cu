// Weight-streaming Linear for M <= 32 (or 64) activation rows: C[M, N] = A[M, K] * W[N, K]^T with the fused epilogues of launch_gemm.
//
// The dual model's audio stream (26 tokens, T/LTX2TransformerBlock.swift:213-281) runs twelve Linears per block against
// 2048..8192-wide weights.  At 26 flop per weight byte they sit far below the tensor-core ridge: the roof is HBM, and the
// tcgen05 tile kernel -- 128 x 32 tiles whose TMA boxes are 32 separate 128-byte segments per k-block -- streams weights
// at ~1 TB/s (profiles/r01e_launches_av_forward_summary.md).  Here every warp walks whole weight rows instead:
//
//   block = 16 output columns, 8 warps; the K axis is dealt to the warps in steps of 32 (step s -> warp s % 8), so the block
//   reads 8 weight rows x 512 contiguous bytes at a time.  Lane (g = lane / 4, c = lane % 4) loads 16 bytes of weight row
//   n0 + g (and n0 + 8 + g) at k0 + 8c and the same 16 bytes of activation rows g, g + 8, g + 16, g + 24; two
//   mma.sync.m16n8k16 per (row block, column group) consume them.  The MMA's k order inside a step is a fixed permutation
//   of the physical one (logical 2c, 2c+1 | 2c+8, 2c+9  <-  physical 8c+0, 8c+1 | 8c+2, 8c+3, then 8c+4.. for the second
//   MMA), applied to A and W alike, so every load is a 16-byte vector and the dot products are unchanged.
//   The 64-row form (a batch of two audio streams, 2 x 26 rows) adds row blocks 2 and 3 (rows g + 32 .. g + 56): every
//   row goes through the same MMA sequence, k permutation and warp-order reduction as in the 32-row form, so row r of a
//   two-item product equals, bit for bit, row r (or r - M/2) of the one-item products.  It fetches activations two steps
//   at a time (the grouping only changes when loads are issued, not the order of the MMAs).
//   Weight loads of the first steps are issued BEFORE griddepcontrol.wait (weights are constants): under programmatic
//   dependent launch they overlap the producer's tail.  Partial sums of the 8 warps meet in shared memory and are added in
//   warp order (deterministic); 256 threads then apply bias / GELU / SiLU / gate * residual and store two columns each.
//
// Supported: a_kblock = 0, row-major outputs (no column blocking, no split transposed columns) or, for the bf16 epilogue, the
// whole output transposed (V^T; in the 64-row form optionally one padded column block per batch item), K % 32 == 0,
// N % 16 == 0.
// launch_gemm falls back to the tensor-core kernels otherwise (and for M above the caller's limit, 32 or 64).
#include "ltx_internal.h"
#include "ptx.cuh"

namespace ltx {

namespace {

constexpr int SK_WARPS = 8;
constexpr int SK_COLS = 16;
constexpr int SK_THREADS = SK_WARPS * 32;
constexpr int SK_UNROLL = 8;   // k-steps of weights in flight per warp (16 x 16 B per lane: 64 KB per block)
constexpr int SK_AGROUP = 4;   // activation fragments are fetched (from L2) four steps at a time (two in the 64-row form)

__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                               uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};\n"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// RB = 16-row MMA blocks: 2 (M <= 32) or 4 (M <= 64)
template <int MODE, int RB>
__global__ void __launch_bounds__(SK_THREADS)
gemm_skinny_kernel(const bf16* A, int64_t lda, const bf16* W, int64_t ldb, int M, int N, int K, const GemmEpi ep) {
  constexpr int AR = 2 * RB;                         // activation rows per lane: g + 8 i
  constexpr int AGROUP = RB == 2 ? SK_AGROUP : 2;    // keeps the 64-row form's fragments in registers
  __shared__ float part[SK_WARPS][16 * RB][SK_COLS + 2];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, c = lane & 3;
  const int n0 = blockIdx.x * SK_COLS;
  const int steps = K >> 5;
  const bool two_blocks = M > 16, three_blocks = M > 32, four_blocks = M > 48;
  auto block_on = [&](int rb) { return rb == 0 || (rb == 1 ? two_blocks : rb == 2 ? three_blocks : four_blocks); };
  float acc[RB][2][4];
#pragma unroll
  for (int rb = 0; rb < RB; ++rb)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[rb][j][e] = 0.f;

  const uint4* w0 = reinterpret_cast<const uint4*>(W + static_cast<int64_t>(n0 + g) * ldb + c * 8);
  const uint4* w1 = reinterpret_cast<const uint4*>(W + static_cast<int64_t>(n0 + 8 + g) * ldb + c * 8);
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
  // activation rows of this lane: g, g + 8 (row block 0), g + 16, g + 24 (row block 1), ...; rows >= M read as zero
  const bf16* arow[AR];
  bool aok[AR];
#pragma unroll
  for (int i = 0; i < AR; ++i) {
    const int r = g + 8 * i;
    aok[i] = r < M;
    arow[i] = A + static_cast<int64_t>(aok[i] ? r : 0) * lda + c * 8;
  }

  uint4 wv[SK_UNROLL][2];
  auto load_w = [&](int s0) {
#pragma unroll
    for (int u = 0; u < SK_UNROLL; ++u) {
      const int s = s0 + u * SK_WARPS;
      if (s < steps) {
        wv[u][0] = __ldg(w0 + s * 4);   // 32 bf16 = 4 uint4 per step
        wv[u][1] = __ldg(w1 + s * 4);
      } else {
        wv[u][0] = zero4;
        wv[u][1] = zero4;
      }
    }
  };
  load_w(warp);      // constants: may run ahead of the producer kernel
  griddep_launch();
  griddep_wait();    // activations, gates and the residual are the producer's output: only touched from here on

  for (int s0 = warp; s0 < steps; s0 += SK_WARPS * SK_UNROLL) {
#pragma unroll
    for (int h = 0; h < SK_UNROLL / AGROUP; ++h) {
      uint4 av[AGROUP][AR];
#pragma unroll
      for (int u = 0; u < AGROUP; ++u) {
        const int s = s0 + (h * AGROUP + u) * SK_WARPS;
#pragma unroll
        for (int i = 0; i < AR; ++i) {
          av[u][i] = zero4;
          if (s < steps && aok[i] && (i < 2 || block_on(i >> 1))) av[u][i] = *reinterpret_cast<const uint4*>(arow[i] + s * 32);
        }
      }
#pragma unroll
      for (int u = 0; u < AGROUP; ++u) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const uint4 w = wv[h * AGROUP + u][j];
          mma_bf16_16816(acc[0][j], av[u][0].x, av[u][1].x, av[u][0].y, av[u][1].y, w.x, w.y);
          mma_bf16_16816(acc[0][j], av[u][0].z, av[u][1].z, av[u][0].w, av[u][1].w, w.z, w.w);
#pragma unroll
          for (int rb = 1; rb < RB; ++rb) {
            if (block_on(rb)) {
              mma_bf16_16816(acc[rb][j], av[u][2 * rb].x, av[u][2 * rb + 1].x, av[u][2 * rb].y, av[u][2 * rb + 1].y, w.x, w.y);
              mma_bf16_16816(acc[rb][j], av[u][2 * rb].z, av[u][2 * rb + 1].z, av[u][2 * rb].w, av[u][2 * rb + 1].w, w.z, w.w);
            }
          }
        }
      }
    }
    if (s0 + SK_WARPS * SK_UNROLL < steps) load_w(s0 + SK_WARPS * SK_UNROLL);
  }

  // accumulator fragment: regs 0, 1 -> (row g, cols 2c, 2c + 1); regs 2, 3 -> (row g + 8, same cols)
#pragma unroll
  for (int rb = 0; rb < RB; ++rb)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      part[warp][rb * 16 + g][j * 8 + 2 * c] = acc[rb][j][0];
      part[warp][rb * 16 + g][j * 8 + 2 * c + 1] = acc[rb][j][1];
      part[warp][rb * 16 + g + 8][j * 8 + 2 * c] = acc[rb][j][2];
      part[warp][rb * 16 + g + 8][j * 8 + 2 * c + 1] = acc[rb][j][3];
    }
  __syncthreads();
  const int col = (threadIdx.x & 7) * 2;
#pragma unroll
  for (int pass = 0; pass < RB / 2; ++pass) {   // 32 rows per pass
    const int row = (threadIdx.x >> 3) + 32 * pass;
    if (row >= M) return;
    float v[2] = {0.f, 0.f};
#pragma unroll
    for (int w = 0; w < SK_WARPS; ++w) {
      v[0] += part[w][row][col];
      v[1] += part[w][row][col + 1];
    }
    const int n = n0 + col;
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      float b = 0.f;
      if (ep.bias) b = ep.bias_per_row ? ep.bias[row] : ep.bias[n + e];
      v[e] += b;
    }
    if (MODE == EPI_GATE_RESID) {
      float* xr = ep.resid + static_cast<int64_t>(row) * ep.ldr + n;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        float gt = 1.f;
        if (ep.gate_a) {
          gt = ep.gate_a[static_cast<int64_t>(row / ep.rows_per_gate) * ep.gate_ld + n + e];
          if (ep.gate_b) gt += ep.gate_b[n + e];
        }
        const float x = xr[e] + v[e] * gt * ep.scale;
        xr[e] = x;
        if (ep.shadow) ep.shadow[static_cast<int64_t>(row) * ep.lds + n + e] = __float2bfloat16(x);
      }
    } else if (MODE == EPI_F32) {
      float* o = reinterpret_cast<float*>(ep.out) + static_cast<int64_t>(row) * ep.ldo + n;
      o[0] = v[0];
      o[1] = v[1];
    } else {
      if (MODE == EPI_GELU_BF16) { v[0] = gelu_tanh(v[0]); v[1] = gelu_tanh(v[1]); }
      if (MODE == EPI_SILU_BF16) { v[0] = silu(v[0]); v[1] = silu(v[1]); }
      if (MODE == EPI_BF16 && ep.transpose_out) {
        int64_t m = row;
        if constexpr (RB == 4) {
          if (ep.t_item_rows) m = static_cast<int64_t>(row / ep.t_item_rows) * ep.t_item_ld + row % ep.t_item_rows;
        }
        bf16* o = reinterpret_cast<bf16*>(ep.out) + static_cast<int64_t>(n) * ep.ldo + m;
        o[0] = __float2bfloat16(v[0]);
        o[ep.ldo] = __float2bfloat16(v[1]);
      } else {
        bf16* o = reinterpret_cast<bf16*>(ep.out) + static_cast<int64_t>(row) * ep.ldo + n;
        o[0] = __float2bfloat16(v[0]);
        o[1] = __float2bfloat16(v[1]);
      }
    }
  }
}

template <int MODE>
void launch_impl(const bf16* A, int64_t lda, const bf16* W, int64_t ldb, int M, int N, int K, const GemmEpi& epi,
                 cudaStream_t stream) {
  if (M <= 32 && epi.t_item_rows == 0)
    launch_pdl(PDL_GEMM, gemm_skinny_kernel<MODE, 2>, dim3(N / SK_COLS), dim3(SK_THREADS), 0, stream, A, lda, W, ldb, M, N, K, epi);
  else
    launch_pdl(PDL_GEMM, gemm_skinny_kernel<MODE, 4>, dim3(N / SK_COLS), dim3(SK_THREADS), 0, stream, A, lda, W, ldb, M, N, K, epi);
}

}  // namespace

bool gemm_skinny_eligible(int64_t lda, int64_t ldb, int M, int N, int K, const GemmEpi& epi, int a_kblock, int max_rows) {
  return M >= 1 && M <= max_rows && (max_rows == 32 || max_rows == 64) && a_kblock == 0 && K % 32 == 0 && N % SK_COLS == 0 && lda % 8 == 0 && ldb % 8 == 0 &&
         epi.col_block == 0 && epi.tsplit_col == 0 && epi.mode >= EPI_BF16 && epi.mode <= EPI_SILU_BF16 &&
         (epi.transpose_out == 0 || epi.mode == EPI_BF16) && (epi.t_item_rows == 0 || (max_rows == 64 && epi.t_item_ld >= epi.t_item_rows));
}

void launch_gemm_skinny(const bf16* A, int64_t lda, const bf16* W, int64_t ldb, int M, int N, int K, const GemmEpi& epi,
                        cudaStream_t stream) {
  LTX_CHECK((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0, 2,
            "skinny GEMM: operands must be 16-byte aligned");
  switch (epi.mode) {
    case EPI_BF16: launch_impl<EPI_BF16>(A, lda, W, ldb, M, N, K, epi, stream); break;
    case EPI_GELU_BF16: launch_impl<EPI_GELU_BF16>(A, lda, W, ldb, M, N, K, epi, stream); break;
    case EPI_GATE_RESID: launch_impl<EPI_GATE_RESID>(A, lda, W, ldb, M, N, K, epi, stream); break;
    case EPI_F32: launch_impl<EPI_F32>(A, lda, W, ldb, M, N, K, epi, stream); break;
    case EPI_SILU_BF16: launch_impl<EPI_SILU_BF16>(A, lda, W, ldb, M, N, K, epi, stream); break;
    default: LTX_CHECK(false, 2, "bad GEMM epilogue mode");
  }
  LTX_CUDA(cudaGetLastError());
}

}  // namespace ltx
