// bf16 GEMM for sm_100a: C[M,N] = A[M,K] * B[N,K]^T with fused epilogues.
//
// Replaces the MLX `Linear`/`addMM` calls on the DiT path (SURVEY K1,K3,K5,K9,K10,K12,K13,K14;
// T/LTXAttention.swift:171-175,217, T/LTXFeedForward.swift:47-51, T/LTXTransformer.swift:223,257).
//
// Structure (one persistent CTA per SM, 192 threads):
//   warp 0   : TMA producer  -- cp.async.bulk.tensor 2-D boxes [128|BN rows x 64 cols] into a 128B-swizzled smem ring
//   warp 1   : MMA issuer    -- one elected lane issues tcgen05.mma (M=128, N=BN, K=16), accumulators in TMEM,
//                               two accumulator stages so the epilogue of tile i overlaps the mainloop of tile i+1
//   warps 2-5: epilogue      -- tcgen05.ld (thread = output row, 32 columns at a time) -> bias / GELU / gate*residual
// Edges: TMA zero-fills out-of-bounds rows/columns (M, N, K tails); the epilogue masks rows >= M and columns >= N.
//
// Tile width BN is a RUNTIME parameter (any multiple of 16 in [32, 256]: it only changes the TMA box, the UMMA
// instruction descriptor and the epilogue trip count).  The launcher picks the width that fits the output into whole
// waves of 148 CTAs ("wave-fitted" tiles): at M = 1536 an N = 4096 GEMM runs as 12 x 24 tiles of 128x176 (2 waves, 97 %
// full) instead of 12 x 16 tiles of 128x256 (2 waves, 65 % full); N = 8192 / 16384 use 128x224 (3 / 6 waves, 99 % full).
// A stream-K variant (split last wave + fp32 partial fix-up) was measured slower than this on B200 and was dropped.
#include "gemm_epilogue.cuh"
#include "ltx_internal.h"
#include "ptx.cuh"

namespace ltx {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int GEMM_THREADS = 192;

struct GemmCfg {
  static constexpr int STAGES_MIN = 4;                   // ring depth at the widest tile
  static constexpr int STAGES_MAX = 9;                   // ... and at the narrowest (the ring's bytes are fixed, see ring_stages)
  static constexpr int BN_MAX = 256;
  static constexpr uint32_t A_BYTES = BM * BK * 2;
  static constexpr uint32_t RING_BYTES = STAGES_MIN * (A_BYTES + BN_MAX * BK * 2);   // 192 KB of operand stages
  static constexpr uint32_t TMEM_COLS = 512;             // two accumulator stages of up to 256 columns
  static constexpr size_t SMEM = 1024 /*align slack*/ + RING_BYTES + (2 * STAGES_MAX + 4) * 8 + 16 + 128 +
                                 4 * EPI_STAGE_BYTES;  // + per-warp epilogue staging tiles
};
// A stage holds one A tile (16 KB) and one B tile of bn rows (bn * 128 B, a multiple of the 1024-B swizzle atom): narrow
// tiles get a deeper ring out of the same bytes.  The small-M GEMMs that pick them (the dual model's audio stream: M = 26
// rows against 2048..8192-wide weights) are bound by TMA latency x bytes in flight, not by the tensor pipe.
__host__ __device__ inline int ring_stages(int bn) {
  const int s = static_cast<int>(GemmCfg::RING_BYTES / (GemmCfg::A_BYTES + static_cast<uint32_t>(bn) * BK * 2));
  return s > GemmCfg::STAGES_MAX ? GemmCfg::STAGES_MAX : s;
}

template <int MODE>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_tcgen05(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, int M, int N, int K,
                  int BN, int a_kblock, const GemmEpi ep) {
  using Cfg = GemmCfg;
  const int STAGES = ring_stages(BN);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  const uint32_t b_bytes = static_cast<uint32_t>(BN) * BK * 2;   // B stage pitch = the tile itself
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * Cfg::A_BYTES;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + Cfg::RING_BYTES);
  uint64_t* empty = full + Cfg::STAGES_MAX;
  uint64_t* tfull = empty + Cfg::STAGES_MAX;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  float* epi_stage = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 127) & ~static_cast<uintptr_t>(127));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_m = (M + BM - 1) / BM;
  const int num_n = (N + BN - 1) / BN;
  const int num_tiles = num_m * num_n;
  const int num_k = (K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 4);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
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
          mbar_arrive_expect_tx(&full[stage], Cfg::A_BYTES + b_bytes);
          if (a_kblock > 0)   // K-blocked A: 3-D map (k in block, row, block)
            tma_load_3d(sA + stage * Cfg::A_BYTES, &tmA, &full[stage], (kb * BK) % a_kblock, m_blk * BM, (kb * BK) / a_kblock);
          else
            tma_load_2d(sA + stage * Cfg::A_BYTES, &tmA, &full[stage], kb * BK, m_blk * BM);
          tma_load_2d(sB + stage * b_bytes, &tmB, &full[stage], kb * BK, n_blk * BN);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16(BM, BN);
      int stage = 0;
      uint32_t phase = 0;
      int t = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++t) {
        const int as = t & 1;
        const uint32_t aphase = (t >> 1) & 1;
        mbar_wait(&tempty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * Cfg::BN_MAX;
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(sA + stage * Cfg::A_BYTES);
          const uint32_t b_addr = smem_u32(sB + stage * b_bytes);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            umma_bf16(d_tmem, umma_desc_sw128(a_addr + k * 32), umma_desc_sw128(b_addr + k * 32), idesc,
                      (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(&empty[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull[as]);
      }
    }
  } else {
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    int t = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++t) {
      const int m_blk = tile % num_m, n_blk = tile / num_m;
      const int as = t & 1;
      const uint32_t aphase = (t >> 1) & 1;
      mbar_wait(&tfull[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * Cfg::BN_MAX;
      epilogue_tile<MODE>(taddr, BN, epi_stage + (warp - 2) * (EPI_STAGE_BYTES / 4), lane, m_blk * BM + q * 32, n_blk * BN, M, N, ep);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[as]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

template <int MODE>
void launch_impl(const CUtensorMap& tmA, const CUtensorMap& tmB, int M, int N, int K, int BN, int a_kblock,
                 const GemmEpi& epi, cudaStream_t stream) {
  using Cfg = GemmCfg;
  auto kern = gemm_bf16_tcgen05<MODE>;
  ensure_dyn_smem(kern, Cfg::SMEM);
  const int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);
  const int grid = tiles < device_sm_count() ? tiles : device_sm_count();
  launch_pdl(PDL_GEMM, kern, dim3(grid), dim3(GEMM_THREADS), Cfg::SMEM, stream, tmA, tmB, M, N, K, BN, a_kblock, epi);
}

// Tile width that minimises (waves x width): time ~ ceil(tiles / #SM) * (BN + c0), c0 = fixed per-tile cost in columns.
int fit_tile_width(int M, int N, int sms) {
  const int num_m = (M + BM - 1) / BM;
  int best = 256;
  double best_cost = 1e30;
  for (int bn = 256; bn >= 32; bn -= 16) {
    const int num_n = (N + bn - 1) / bn;
    const long long tiles = static_cast<long long>(num_m) * num_n;
    const long long waves = (tiles + sms - 1) / sms;
    // narrow tiles re-read A more often and are smem-bandwidth bound below ~176 columns: penalise them mildly
    const double eff = bn >= 176 ? 1.0 : (bn >= 128 ? 0.92 : 0.75);
    const double cost = static_cast<double>(waves) * (bn + 12.0) / eff;
    if (cost < best_cost - 1e-9) { best_cost = cost; best = bn; }
  }
  return best;
}

}  // namespace

int gemm_fit_tile_width(int M, int N) { return fit_tile_width(M, N, device_sm_count()); }

void launch_gemm(const bf16* A, int64_t lda, const bf16* B, int64_t ldb, int M, int N, int K, const GemmEpi& epi,
                 cudaStream_t stream, int force_bn, int a_kblock, int64_t a_kblock_stride, int allow_skinny) {
  LTX_CHECK(M > 0 && N > 0 && K > 0, 2, "GEMM: empty problem");
  LTX_CHECK(K % 8 == 0 && lda % 8 == 0 && ldb % 8 == 0, 2, "GEMM: K and leading dims must be multiples of 8");
  if (epi.mode == EPI_GATE_RESID) {
    LTX_CHECK(epi.resid != nullptr && epi.ldr % 4 == 0, 2, "GEMM: residual epilogue needs fp32 resid with ld % 4 == 0");
    LTX_CHECK(epi.shadow == nullptr || epi.lds % 4 == 0, 2, "GEMM: shadow ld must be a multiple of 4");
  } else {
    LTX_CHECK(epi.out != nullptr, 2, "GEMM: missing output");
    LTX_CHECK(epi.ldo % (epi.mode == EPI_F32 ? 4 : 8) == 0, 2, "GEMM: output ld alignment");
  }
  // force_bn >= 1000 selects the 2-CTA pair kernel (gemm2.cu) with width force_bn - 1000 (0 = fitted); by default the
  // pair kernel is used whenever the problem has more than one 128-row tile
  const bool skinny = allow_skinny && force_bn == 0 && gemm_skinny_eligible(lda, ldb, M, N, K, epi, a_kblock, allow_skinny);
  LTX_CHECK(epi.transpose_out == 0 || skinny, 2, "GEMM: transpose_out is served by the weight-streaming kernel only");
  if (skinny) {
    launch_gemm_skinny(A, lda, B, ldb, M, N, K, epi, stream);
    return;
  }
  // few activation rows (Ulysses shards, small clips): stream the weights through the swap-AB kernel when the caller opted in
  // by passing a split-K workspace; force_bn == -2 forces it (tests)
  if ((force_bn == 0 && epi.ws != nullptr && gemm_swapab_eligible(lda, ldb, M, N, K, epi)) || force_bn == -2) {
    launch_gemm_swapab(A, lda, B, ldb, M, N, K, epi, stream, a_kblock, a_kblock_stride);
    return;
  }
  if (force_bn >= 1000 || (force_bn == 0 && M > 128)) {
    launch_gemm_2cta(A, lda, B, ldb, M, N, K, epi, stream, force_bn >= 1000 ? force_bn - 1000 : 0, a_kblock, a_kblock_stride);
    return;
  }
  // force_bn: 0 = wave-fitted width (see fit_tile_width); otherwise a multiple of 16 in [32, 256]
  int bn = force_bn;
  if (bn == 0) bn = fit_tile_width(M, N, device_sm_count());
  LTX_CHECK(bn >= 32 && bn <= 256 && bn % 16 == 0, 2, "GEMM: tile width must be a multiple of 16 in [32, 256]");
  LTX_CHECK(epi.tsplit_col == 0 || (epi.mode == EPI_BF16 && bn % 32 == 0 && epi.tsplit_col % 32 == 0 && epi.out_t != nullptr &&
                                    epi.ldt % 8 == 0 && epi.col_block == 0),
            2, "GEMM: transposed-column output needs the bf16 epilogue, a tile width and split column that are multiples of 32");
  LTX_CHECK(epi.col_block == 0 || ((epi.mode == EPI_BF16 || epi.mode == EPI_GELU_BF16 || epi.mode == EPI_SILU_BF16) && epi.col_block % 32 == 0 &&
                                   epi.col_block_from % 32 == 0 && (N - epi.col_block_from) % epi.col_block == 0),
            2, "GEMM: column-blocked output needs a bf16 epilogue and col_block % 32 == 0");
  CUtensorMap tmA;
  if (a_kblock > 0) {
    LTX_CHECK(a_kblock % BK == 0 && K % a_kblock == 0 && lda == a_kblock, 2, "GEMM: bad K-blocked A layout");
    tmA = make_tmap_3d(A, a_kblock, M, K / a_kblock, lda, a_kblock_stride, 64, BM);
  } else {
    tmA = make_tmap_2d(A, M, K, lda, BM);
  }
  CUtensorMap tmB = make_tmap_2d(B, N, K, ldb, bn);
  switch (epi.mode) {
    case EPI_BF16: launch_impl<EPI_BF16>(tmA, tmB, M, N, K, bn, a_kblock, epi, stream); break;
    case EPI_GELU_BF16: launch_impl<EPI_GELU_BF16>(tmA, tmB, M, N, K, bn, a_kblock, epi, stream); break;
    case EPI_GATE_RESID: launch_impl<EPI_GATE_RESID>(tmA, tmB, M, N, K, bn, a_kblock, epi, stream); break;
    case EPI_F32: launch_impl<EPI_F32>(tmA, tmB, M, N, K, bn, a_kblock, epi, stream); break;
    case EPI_SILU_BF16: launch_impl<EPI_SILU_BF16>(tmA, tmB, M, N, K, bn, a_kblock, epi, stream); break;
    default: LTX_CHECK(false, 2, "bad GEMM epilogue mode");
  }
}

}  // namespace ltx
