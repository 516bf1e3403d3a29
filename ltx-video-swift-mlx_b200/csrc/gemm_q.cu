// Dequant-fused GEMM for sm_100a: C[M,N] = A[M,K] * dequant(Wq)[N,K]^T with the fused epilogues of gemm.cu.
//
// Replaces MLX `QuantizedLinear` after quantize(model:groupSize:64,bits:8|4) (P/LTXPipeline.swift:323-333,
// C/LTXQuantizationConfig.swift:19-62; SURVEY K15): affine per-64-group weights w ~= s * q + beta, q in [0, 2^bits - 1].
// The quantisation rule itself lives in MLX (not in the reference tree) -> parity for this kernel is pinned as
// "dequant-fused GEMM == bf16 GEMM on the dequantised weights" (SURVEY H8); the device quantiser below is ours.
//
// Storage: q as bytes [N, K] (8-bit) or packed nibbles [N, K/2] (4-bit, even k in the low nibble); scale / bias fp32
// (bf16-representable, like MLX's bf16 scales) transposed to [K/64, N] so one k-block's 64-wide group row is contiguous.
//
// Kernel = gemm.cu's pipeline plus a dequant stage between TMA and MMA (group size 64 == BK, one scale per row per k-block):
//   warp 0     : TMA producer -- A tile (bf16, swizzled) + raw q tile (bytes, unswizzled) per stage
//   warps 6-13 : dequant      -- 16 codes per thread-chunk: byte -> fp32 via PRMT magic (0x4B000000 | q) - 2^23, one FFMA with
//                                (s, beta), cvt to bf16x2, 16-byte stores into the 128B-swizzled K-major B operand buffer,
//                                fence.proxy.async, arrive
//   warp 1     : MMA issuer (tcgen05.mma, TMEM accumulators, two stages)      warps 2-5: epilogue
// HBM / L2 traffic for weights drops 2x (int8) / 4x (int4); the tensor core still runs bf16 x bf16 -> fp32.
#include <cuda_fp8.h>

#include "gemm_epilogue.cuh"
#include "ltx_internal.h"
#include "ptx.cuh"

namespace ltx {

namespace {

constexpr int QBM = 128, QBK = 64;
constexpr int Q_THREADS = 448;      // 14 warps
constexpr int Q_DEQ_WARPS = 8;
constexpr int Q_STAGES = 3;
constexpr int Q_BN_MAX = 256;
constexpr uint32_t QA_BYTES = QBM * QBK * 2;           // 16 KB
constexpr uint32_t QR_STRIDE = Q_BN_MAX * QBK;         // raw codes, up to 16 KB
constexpr uint32_t QB_STRIDE = Q_BN_MAX * QBK * 2;     // dequantised bf16 operand, up to 32 KB
constexpr size_t Q_SMEM = 1024 + Q_STAGES * (QA_BYTES + QR_STRIDE + QB_STRIDE) + (3 * Q_STAGES + 4) * 8 + 16 + 128 + 4 * EPI_STAGE_BYTES;

__device__ __forceinline__ uint32_t deq2(uint32_t word, int i0, int i1, float s, float bm) {
  // two codes (bytes i0, i1 of `word`) -> s*q+beta -> packed bf16x2.  PRMT drops the code byte into mantissa bits [15:8]
  // of 0x47000000 = 2^15, giving the fp32 value 2^15 + q exactly; one FFMA with bm = beta - s*2^15 then yields s*q + beta
  // with a single rounding (s, beta are bf16 values, so bm is exact in fp32).
  const uint32_t sel0 = 0x7604u + (i0 << 4), sel1 = 0x7604u + (i1 << 4);
  const float f0 = __uint_as_float(__byte_perm(word, 0x47000000u, sel0));
  const float f1 = __uint_as_float(__byte_perm(word, 0x47000000u, sel1));
  return pack_bf16_alu(fmaf(f0, s, bm), fmaf(f1, s, bm));
}

template <int MODE, int BITS>
__global__ void __launch_bounds__(Q_THREADS, 1)
gemm_q_tcgen05(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmQ, int M, int N, int K, int BN,
               const float* __restrict__ scales, const float* __restrict__ biases, int a_kblock, const GemmEpi ep) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* sA = smem;
  uint8_t* sB = sA + Q_STAGES * QA_BYTES;
  uint8_t* sR = sB + Q_STAGES * QB_STRIDE;
  uint64_t* full_raw = reinterpret_cast<uint64_t*>(sR + Q_STAGES * QR_STRIDE);
  uint64_t* full_deq = full_raw + Q_STAGES;
  uint64_t* empty = full_deq + Q_STAGES;
  uint64_t* tfull = empty + Q_STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  float* epi_stage = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 127) & ~static_cast<uintptr_t>(127));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_m = (M + QBM - 1) / QBM;
  const int num_n = (N + BN - 1) / BN;
  const int num_tiles = num_m * num_n;
  const int num_k = (K + QBK - 1) / QBK;
  constexpr int ROW_BYTES = (BITS == 8) ? 64 : 32;       // raw bytes per row per k-block
  const uint32_t raw_bytes = static_cast<uint32_t>(BN) * ROW_BYTES;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmQ);
    for (int i = 0; i < Q_STAGES; ++i) {
      mbar_init(&full_raw[i], 1);
      mbar_init(&full_deq[i], Q_DEQ_WARPS);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 4); }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // PDL: everything above overlapped the previous kernel's tail; global memory is touched only from here on
  griddep_launch();
  griddep_wait();

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m_blk = tile % num_m, n_blk = tile / num_m;
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_raw[stage], QA_BYTES + raw_bytes);
          if (a_kblock > 0)   // K-blocked A (Ulysses receive layout): 3-D map (k in block, row, block)
            tma_load_3d(sA + stage * QA_BYTES, &tmA, &full_raw[stage], (kb * QBK) % a_kblock, m_blk * QBM, (kb * QBK) / a_kblock);
          else
            tma_load_2d(sA + stage * QA_BYTES, &tmA, &full_raw[stage], kb * QBK, m_blk * QBM);
          tma_load_2d(sR + stage * QR_STRIDE, &tmQ, &full_raw[stage], kb * ROW_BYTES, n_blk * BN);
          if (++stage == Q_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16(QBM, BN);
      int stage = 0;
      uint32_t phase = 0;
      int t = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++t) {
        const int as = t & 1;
        const uint32_t aphase = (t >> 1) & 1;
        mbar_wait(&tempty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * Q_BN_MAX;
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&full_deq[stage], phase);   // dequant warps waited on the TMA barrier first: A has landed too
          tc_fence_after();
          const uint32_t a_addr = smem_u32(sA + stage * QA_BYTES);
          const uint32_t b_addr = smem_u32(sB + stage * QB_STRIDE);
#pragma unroll
          for (int k = 0; k < QBK / 16; ++k)
            umma_bf16(d_tmem, umma_desc_sw128(a_addr + k * 32), umma_desc_sw128(b_addr + k * 32), idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit(&empty[stage]);
          if (++stage == Q_STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull[as]);
      }
    }
  } else if (warp < 6) {
    const int q = warp & 3;
    int t = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++t) {
      const int m_blk = tile % num_m, n_blk = tile / num_m;
      const int as = t & 1;
      const uint32_t aphase = (t >> 1) & 1;
      mbar_wait(&tfull[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * Q_BN_MAX;
      epilogue_tile<MODE>(taddr, BN, epi_stage + (warp - 2) * (EPI_STAGE_BYTES / 4), lane, m_blk * QBM + q * 32, n_blk * BN, M, N, ep);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[as]);
    }
  } else {
    // ---- dequant warps: raw codes -> bf16 operand tile (K-major, 128 B per row, 128B swizzle)
    const int dt = threadIdx.x - 6 * 32;                 // 0..255
    constexpr int CH_PER_ROW = ROW_BYTES / 16;           // 16-byte raw chunks per row: 4 (int8) / 2 (int4)
    constexpr int MAX_IT = 4;                            // BN * CH_PER_ROW <= 1024 chunks over 256 threads
    const int chunks = BN * CH_PER_ROW;
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int n0 = (tile / num_m) * BN;
      // the rows this thread converts are the same for every k-block of the tile; their (scale, bias) for the NEXT
      // k-block are fetched while the current one is converted, so the L2 latency is off the critical path
      float sc[MAX_IT], bm[MAX_IT];
      auto fetch = [&](int kb, float (&so)[MAX_IT], float (&bo)[MAX_IT]) {
        const float* srow = scales + static_cast<int64_t>(kb) * N;
        const float* brow = biases + static_cast<int64_t>(kb) * N;
#pragma unroll
        for (int it = 0; it < MAX_IT; ++it) {
          const int c = dt + it * (Q_DEQ_WARPS * 32);
          const int n = n0 + c / CH_PER_ROW;
          const bool ok = c < chunks && n < N;
          const float sv = ok ? __ldg(srow + n) : 0.f, bv = ok ? __ldg(brow + n) : 0.f;
          so[it] = sv;
          bo[it] = fmaf(-32768.0f, sv, bv);
        }
      };
      fetch(0, sc, bm);
      for (int kb = 0; kb < num_k; ++kb) {
        float sn[MAX_IT], bn[MAX_IT];
        if (kb + 1 < num_k) fetch(kb + 1, sn, bn);
        mbar_wait(&full_raw[stage], phase);
        const uint8_t* raw = sR + stage * QR_STRIDE;
        uint8_t* dst = sB + stage * QB_STRIDE;
        uint4 u[MAX_IT];
#pragma unroll
        for (int it = 0; it < MAX_IT; ++it) {
          const int c = dt + it * (Q_DEQ_WARPS * 32);
          if (c < chunks) u[it] = *reinterpret_cast<const uint4*>(raw + (c / CH_PER_ROW) * ROW_BYTES + (c % CH_PER_ROW) * 16);
        }
#pragma unroll
        for (int it = 0; it < MAX_IT; ++it) {
          const int c = dt + it * (Q_DEQ_WARPS * 32);
          if (c >= chunks) continue;
          const int row = c / CH_PER_ROW, part = c % CH_PER_ROW;
          const float s = sc[it], b = bm[it];
          const uint32_t w[4] = {u[it].x, u[it].y, u[it].z, u[it].w};
          uint8_t* drow = dst + row * 128;
          if (BITS == 8) {
            // 16 codes -> logical 16-byte chunks 2*part, 2*part+1 of the row
            uint32_t o[8];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              o[2 * i] = deq2(w[i], 0, 1, s, b);
              o[2 * i + 1] = deq2(w[i], 2, 3, s, b);
            }
            *reinterpret_cast<uint4*>(drow + (((2 * part) ^ (row & 7)) * 16)) = make_uint4(o[0], o[1], o[2], o[3]);
            *reinterpret_cast<uint4*>(drow + (((2 * part + 1) ^ (row & 7)) * 16)) = make_uint4(o[4], o[5], o[6], o[7]);
          } else {
            // 32 codes (nibbles, even k low) -> logical chunks 4*part .. 4*part+3
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const uint32_t lo = w[i] & 0x0F0F0F0Fu, hi = (w[i] >> 4) & 0x0F0F0F0Fu;   // codes k = 8i + {0,2,4,6} / {1,3,5,7}
              const uint32_t e01 = __byte_perm(lo, hi, 0x5140);   // bytes: lo0, hi0, lo1, hi1  (k order)
              const uint32_t e23 = __byte_perm(lo, hi, 0x7362);   // bytes: lo2, hi2, lo3, hi3
              const uint4 v = make_uint4(deq2(e01, 0, 1, s, b), deq2(e01, 2, 3, s, b), deq2(e23, 0, 1, s, b), deq2(e23, 2, 3, s, b));
              *reinterpret_cast<uint4*>(drow + (((4 * part + i) ^ (row & 7)) * 16)) = v;
            }
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&full_deq[stage]);
        if (++stage == Q_STAGES) { stage = 0; phase ^= 1; }
        if (kb + 1 < num_k) {
#pragma unroll
          for (int it = 0; it < MAX_IT; ++it) { sc[it] = sn[it]; bm[it] = bn[it]; }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------
// Device quantiser: one warp per (row, 64-group).  Affine min/max: s = (max - min) / (2^bits - 1), beta = min,
// q = clamp(rint((w - beta) / s)); s and beta are rounded to bf16 (MLX keeps them in the weight dtype).
// ---------------------------------------------------------------------------------------------
template <int BITS>
__global__ void quantize_kernel(const bf16* __restrict__ w, int N, int K, uint8_t* __restrict__ q, float* __restrict__ scales,
                                float* __restrict__ biases) {
  const int groups = K / 64;
  const int64_t gid = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (gid >= static_cast<int64_t>(N) * groups) return;
  const int n = static_cast<int>(gid / groups), g = static_cast<int>(gid % groups);
  const bf16* src = w + static_cast<int64_t>(n) * K + g * 64 + lane * 2;
  const float v0 = __bfloat162float(src[0]), v1 = __bfloat162float(src[1]);
  const float mn = -warp_max(-fminf(v0, v1)), mx = warp_max(fmaxf(v0, v1));
  constexpr float LEVELS = (BITS == 8) ? 255.f : 15.f;
  float s = (mx - mn) / LEVELS;
  if (!(s > 0.f)) s = 1.0f;
  s = __bfloat162float(__float2bfloat16(s));
  const float beta = __bfloat162float(__float2bfloat16(mn));
  const int q0 = static_cast<int>(fminf(fmaxf(rintf((v0 - beta) / s), 0.f), LEVELS));
  const int q1 = static_cast<int>(fminf(fmaxf(rintf((v1 - beta) / s), 0.f), LEVELS));
  if (BITS == 8) {
    uint8_t* dst = q + static_cast<int64_t>(n) * K + g * 64 + lane * 2;
    dst[0] = static_cast<uint8_t>(q0);
    dst[1] = static_cast<uint8_t>(q1);
  } else {
    q[static_cast<int64_t>(n) * (K / 2) + g * 32 + lane] = static_cast<uint8_t>(q0 | (q1 << 4));
  }
  if (lane == 0) {
    scales[static_cast<int64_t>(g) * N + n] = s;
    biases[static_cast<int64_t>(g) * N + n] = beta;
  }
}

template <int BITS>
__global__ void dequantize_kernel(const uint8_t* __restrict__ q, const float* __restrict__ scales,
                                  const float* __restrict__ biases, int N, int K, bf16* __restrict__ w) {
  const int64_t total = static_cast<int64_t>(N) * K;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int n = static_cast<int>(i / K), k = static_cast<int>(i % K);
    int code;
    if (BITS == 8) code = q[i];
    else {
      const uint8_t b = q[static_cast<int64_t>(n) * (K / 2) + k / 2];
      code = (k & 1) ? (b >> 4) : (b & 15);
    }
    const int g = k / 64;
    // identical arithmetic to the fused kernel's deq2(): (2^15 + q) * s + (beta - s * 2^15), one rounding each
    const float sv = scales[static_cast<int64_t>(g) * N + n], bv = biases[static_cast<int64_t>(g) * N + n];
    // ... and the same fp32 -> bf16 rounding (pack_bf16_alu)
    const float v = fmaf(32768.0f + static_cast<float>(code), sv, fmaf(-32768.0f, sv, bv));
    const uint32_t pk = pack_bf16_alu(v, 0.f);
    w[i] = __ushort_as_bfloat16(static_cast<unsigned short>(pk & 0xFFFFu));
  }
}

// Whole-weight conversion into a bf16 panel [N, K]: one thread per 16 output values (16 int8 codes = one uint4, or 16 int4
// codes = one uint2), 32-byte coalesced stores.  Same arithmetic and rounding as deq2().  Runs right before the bf16 GEMM
// that consumes the panel; the panel is reused by every weight, so the kernel waits for its predecessor (the previous
// consumer) before its first store.
template <int BITS>
__global__ void __launch_bounds__(256) dequantize_panel_kernel(const uint8_t* __restrict__ q, const float* __restrict__ scales,
                                                                const float* __restrict__ biases, int N, int K, bf16* w) {
  griddep_launch();
  griddep_wait();
  const int cpr = K >> 4;                                  // 16-value chunks per row
  const int64_t total = static_cast<int64_t>(N) * cpr;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int n = static_cast<int>(i / cpr), ch = static_cast<int>(i - static_cast<int64_t>(n) * cpr);
    const int g = ch >> 2;                                 // 64-value group
    const float sv = __ldg(scales + static_cast<int64_t>(g) * N + n), bv = __ldg(biases + static_cast<int64_t>(g) * N + n);
    const float bm = fmaf(-32768.0f, sv, bv);
    uint32_t o[8];
    if (BITS == 8) {
      const uint4 u = *reinterpret_cast<const uint4*>(q + static_cast<int64_t>(n) * K + ch * 16);
      const uint32_t wv[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        o[2 * j] = deq2(wv[j], 0, 1, sv, bm);
        o[2 * j + 1] = deq2(wv[j], 2, 3, sv, bm);
      }
    } else {
      const uint2 u = *reinterpret_cast<const uint2*>(q + static_cast<int64_t>(n) * (K >> 1) + ch * 8);
      const uint32_t wv[2] = {u.x, u.y};
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const uint32_t lo = wv[j] & 0x0F0F0F0Fu, hi = (wv[j] >> 4) & 0x0F0F0F0Fu;
        const uint32_t e01 = __byte_perm(lo, hi, 0x5140), e23 = __byte_perm(lo, hi, 0x7362);
        o[4 * j] = deq2(e01, 0, 1, sv, bm); o[4 * j + 1] = deq2(e01, 2, 3, sv, bm);
        o[4 * j + 2] = deq2(e23, 0, 1, sv, bm); o[4 * j + 3] = deq2(e23, 2, 3, sv, bm);
      }
    }
    uint4* dst = reinterpret_cast<uint4*>(w + static_cast<int64_t>(n) * K + ch * 16);
    dst[0] = make_uint4(o[0], o[1], o[2], o[3]);
    dst[1] = make_uint4(o[4], o[5], o[6], o[7]);
  }
}

template <int MODE, int BITS>
void launch_q(const CUtensorMap& tmA, const CUtensorMap& tmQ, int M, int N, int K, int BN, const float* s, const float* b,
              int a_kblock, const GemmEpi& epi, cudaStream_t stream) {
  auto kern = gemm_q_tcgen05<MODE, BITS>;
  ensure_dyn_smem(kern, Q_SMEM);
  const int tiles = ((M + QBM - 1) / QBM) * ((N + BN - 1) / BN);
  const int grid = tiles < device_sm_count() ? tiles : device_sm_count();
  launch_pdl(PDL_GEMM, kern, dim3(grid), dim3(Q_THREADS), Q_SMEM, stream, tmA, tmQ, M, N, K, BN, s, b, a_kblock, epi);
  LTX_CUDA(cudaGetLastError());
}

template <int BITS>
void launch_q_mode(const CUtensorMap& tmA, const CUtensorMap& tmQ, int M, int N, int K, int BN, const float* s, const float* b,
                   int a_kblock, const GemmEpi& epi, cudaStream_t stream) {
  switch (epi.mode) {
    case EPI_BF16: launch_q<EPI_BF16, BITS>(tmA, tmQ, M, N, K, BN, s, b, a_kblock, epi, stream); break;
    case EPI_GELU_BF16: launch_q<EPI_GELU_BF16, BITS>(tmA, tmQ, M, N, K, BN, s, b, a_kblock, epi, stream); break;
    case EPI_GATE_RESID: launch_q<EPI_GATE_RESID, BITS>(tmA, tmQ, M, N, K, BN, s, b, a_kblock, epi, stream); break;
    case EPI_F32: launch_q<EPI_F32, BITS>(tmA, tmQ, M, N, K, BN, s, b, a_kblock, epi, stream); break;
    case EPI_SILU_BF16: launch_q<EPI_SILU_BF16, BITS>(tmA, tmQ, M, N, K, BN, s, b, a_kblock, epi, stream); break;
    default: LTX_CHECK(false, 2, "bad GEMM epilogue mode");
  }
}

// ---------------------------------------------------------------- per-row e4m3 quantiser (precision mode 8)
// One CTA per row.  Pass 1 takes the row's amax, pass 2 writes the codes; both read 8 bf16 per thread and step.  The scale is
// a power of two, so x / s is exact and each code is a function of its element and the row's amax alone: the codes do not
// depend on the launch shape, and a row's codes do not depend on the other rows.
constexpr int QF8_THREADS = 256;

__global__ void __launch_bounds__(QF8_THREADS) quantize_rows_fp8_kernel(const bf16* x, int64_t ld, int K, uint8_t* q, float* s) {
  __shared__ float red[QF8_THREADS / 32];
  __shared__ float row_scale;
  griddep_wait();
  griddep_launch();
  const int m = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bf16* xr = x + static_cast<int64_t>(m) * ld;
  const int nvec = K / 8;
  float amax = 0.f;
  for (int v = threadIdx.x; v < nvec; v += QF8_THREADS) {
    const uint4 u = *reinterpret_cast<const uint4*>(xr + v * 8);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __bfloat1622float2(h[j]);
      amax = fmaxf(amax, fmaxf(fabsf(f.x), fabsf(f.y)));
    }
  }
  amax = warp_max(amax);
  if (lane == 0) red[warp] = amax;
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f;
#pragma unroll
    for (int w = 0; w < QF8_THREADS / 32; ++w) a = fmaxf(a, red[w]);
    // the least power of two 2^e with a <= 448 * 2^e: a = f * 2^E (f in [0.5, 1)), 448 = 0.875 * 2^9
    float sc = 1.f;
    if (a > 0.f) {
      int E;
      const float f = frexpf(a, &E);
      sc = ldexpf(1.f, f <= 0.875f ? E - 9 : E - 8);
    }
    row_scale = sc;
    s[m] = sc;
  }
  __syncthreads();
  const float sc = row_scale;
  uint8_t* qr = q + static_cast<int64_t>(m) * K;
  for (int v = threadIdx.x; v < nvec; v += QF8_THREADS) {
    const uint4 u = *reinterpret_cast<const uint4*>(xr + v * 8);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
    uint32_t packed[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const float2 f0 = __bfloat1622float2(h[2 * j]), f1 = __bfloat1622float2(h[2 * j + 1]);
      const uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(f0.x / sc, f0.y / sc), __NV_SATFINITE, __NV_E4M3);
      const uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(f1.x / sc, f1.y / sc), __NV_SATFINITE, __NV_E4M3);
      packed[j] = lo | (hi << 16);
    }
    *reinterpret_cast<uint2*>(qr + v * 8) = make_uint2(packed[0], packed[1]);
  }
}

}  // namespace

void launch_quantize_rows_fp8(const bf16* x, int64_t ld, int M, int K, uint8_t* q, float* s, cudaStream_t stream) {
  LTX_CHECK(M > 0 && K > 0 && K % 16 == 0 && ld % 8 == 0 && ld >= K, 2, "FP8 quantiser: K % 16 == 0, ld % 8 == 0, ld >= K");
  LTX_CHECK((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(q) & 15) == 0, 2,
            "FP8 quantiser: 16-byte aligned input and codes");
  launch_pdl(PDL_ROWS, quantize_rows_fp8_kernel, dim3(M), dim3(QF8_THREADS), 0, stream, x, ld, K, q, s);
}

// Large M: the fused kernels redo the code -> bf16 conversion once per 128 / 256-row M tile (12x / 6x at M = 1536) and are
// bound by its instruction issue (~450 TFLOP/s); converting the weight ONCE into the context's bf16 panel and running the
// bf16 pair kernel on it is ~2x faster there.  The fused kernels keep the small-M regime, where weight bytes dominate.
bool gemm_q_uses_panel(const QuantW& W, int M) { return W.scratch != nullptr && M >= 257; }

void launch_gemm_q(const bf16* A, int64_t lda, const QuantW& W, int M, int N, int K, const GemmEpi& epi, cudaStream_t stream,
                   int force_bn, int a_kblock, int64_t a_kblock_stride) {
  LTX_CHECK(M > 0 && N > 0 && K > 0 && K % 64 == 0, 2, "quantised GEMM: K must be a multiple of the group size 64");
  LTX_CHECK(W.bits == 8 || W.bits == 4, 2, "quantised GEMM: 8 or 4 bits");
  LTX_CHECK(W.n == N && W.k == K && W.q && W.scales && W.biases, 2, "quantised GEMM: weight shape mismatch");
  LTX_CHECK(lda % 8 == 0, 2, "quantised GEMM: lda must be a multiple of 8");
  if (force_bn == 0 && gemm_q_uses_panel(W, M)) {
    launch_dequantize_panel(W, W.scratch, stream);
    launch_gemm(A, lda, W.scratch, K, M, N, K, epi, stream, 0, a_kblock, a_kblock_stride);
    return;
  }
  int bn = force_bn ? force_bn : gemm_fit_tile_width(M, N);
  LTX_CHECK(bn >= 32 && bn <= 256 && bn % 16 == 0, 2, "quantised GEMM: bad tile width");
  const uint64_t row_bytes = W.bits == 8 ? K : K / 2;
  CUtensorMap tmA;
  if (a_kblock > 0) {
    LTX_CHECK(a_kblock % QBK == 0 && K % a_kblock == 0 && lda == a_kblock, 2, "quantised GEMM: bad K-blocked A layout");
    tmA = make_tmap_3d(A, a_kblock, M, K / a_kblock, lda, a_kblock_stride, 64, QBM);
  } else {
    tmA = make_tmap_2d(A, M, K, lda, QBM);
  }
  CUtensorMap tmQ = make_tmap_u8(W.q, N, row_bytes, bn, W.bits == 8 ? 64 : 32);
  if (W.bits == 8)
    launch_q_mode<8>(tmA, tmQ, M, N, K, bn, W.scales, W.biases, a_kblock, epi, stream);
  else
    launch_q_mode<4>(tmA, tmQ, M, N, K, bn, W.scales, W.biases, a_kblock, epi, stream);
}

void launch_dequantize_panel(const QuantW& W, bf16* w, cudaStream_t s) {
  LTX_CHECK(W.k % 64 == 0 && (W.bits == 8 || W.bits == 4), 2, "dequantize: K % 64 == 0 and bits in {4, 8}");
  const int64_t chunks = static_cast<int64_t>(W.n) * (W.k / 16);
  int64_t blocks = (chunks + 255) / 256;
  const int64_t cap = static_cast<int64_t>(device_sm_count()) * 16;
  if (blocks > cap) blocks = cap;
  if (W.bits == 8)
    launch_pdl(PDL_GEMM, dequantize_panel_kernel<8>, dim3(static_cast<int>(blocks)), dim3(256), 0, s, W.q, W.scales, W.biases, W.n, W.k, w);
  else
    launch_pdl(PDL_GEMM, dequantize_panel_kernel<4>, dim3(static_cast<int>(blocks)), dim3(256), 0, s, W.q, W.scales, W.biases, W.n, W.k, w);
}

void launch_quantize(const bf16* w, int N, int K, int bits, uint8_t* q, float* scales, float* biases, cudaStream_t s) {
  LTX_CHECK(K % 64 == 0 && (bits == 8 || bits == 4), 2, "quantize: K % 64 == 0 and bits in {4, 8}");
  const int64_t warps = static_cast<int64_t>(N) * (K / 64);
  const int blocks = static_cast<int>((warps * 32 + 255) / 256);
  if (bits == 8)
    quantize_kernel<8><<<blocks, 256, 0, s>>>(w, N, K, q, scales, biases);
  else
    quantize_kernel<4><<<blocks, 256, 0, s>>>(w, N, K, q, scales, biases);
  LTX_CUDA(cudaGetLastError());
}

void launch_dequantize(const QuantW& W, bf16* w, cudaStream_t s) {
  int64_t blocks = (static_cast<int64_t>(W.n) * W.k + 255) / 256;
  if (blocks > 16384) blocks = 16384;
  if (W.bits == 8)
    dequantize_kernel<8><<<static_cast<int>(blocks), 256, 0, s>>>(W.q, W.scales, W.biases, W.n, W.k, w);
  else
    dequantize_kernel<4><<<static_cast<int>(blocks), 256, 0, s>>>(W.q, W.scales, W.biases, W.n, W.k, w);
  LTX_CUDA(cudaGetLastError());
}

}  // namespace ltx
