// 2-CTA (cta_group::2) variant of the bf16 GEMM: a cluster of two CTAs on one TPC computes a 256 x BN tile.
//
// Why: the 1-CTA kernel (gemm.cu) is bound by operand delivery L2 -> SM (48 KB per k-block per CTA at 128x256).  In pair
// mode each CTA loads its own 128 rows of A but only HALF of the B tile (BN/2 rows); tcgen05.mma.cta_group::2 (M = 256)
// reads both halves across the pair, so a CTA moves 16 + BN/4 KB per k-block (32 KB at BN = 256) for the same flops, and
// the smem freed by the half-size B stage buys a deeper TMA ring (3 stages of 128 k).
//
// Protocol (mirrors the CUTLASS / DeepGEMM 2-SM pattern):
//   * both CTAs run every warp role; only the leader (cluster rank 0) issues tcgen05.mma
//   * TMA loads use the .cta_group::2 form and signal the LEADER's full barrier (mbarrier address with the peer bit
//     cleared); the leader arms it with expect_tx for both CTAs' bytes, the peer adds a remote arrive
//   * tcgen05.commit ... .multicast::cluster (mask 0b11) releases the smem stage / publishes the accumulator in BOTH CTAs
//   * each CTA's epilogue drains its own 128 TMEM lanes and arrives remotely on the leader's tmem-empty barrier
//   * TMEM is allocated with cta_group::2 by the same warp of both CTAs; cluster barriers bracket setup and teardown
#include "gemm_epilogue.cuh"
#include "ltx_internal.h"
#include "ptx.cuh"

namespace ltx {

namespace {

constexpr int BM2 = 128;          // rows per CTA (256 per pair)
constexpr int BK2 = 64;           // k of one 128-byte swizzle atom (bf16; 128 e4m3 codes fill the same atom)
constexpr int G2_THREADS = 192;
constexpr int G2_BN_MAX = 256;
constexpr uint32_t G2_A_BYTES = BM2 * BK2 * 2;                 // 16 KB: one atom of A
constexpr uint32_t G2_B_STRIDE = (G2_BN_MAX / 2) * BK2 * 2;    // 16 KB: one atom of half the B tile
// A pipeline stage holds 128 k (two swizzle atoms per operand), so the issuing thread waits on / commits to half as many
// barriers per k as with 64-wide stages and has 8 MMAs in flight per wait; 3 stages of 64 KB.  -4..7 % on every DiT GEMM
// shape at M = 1536 against 64-wide stages on the same box (profiles/r02_gemm_kstage_sweep.txt).
constexpr int G2_KSUB = 2;        // swizzle atoms per operand and stage
constexpr int G2_STAGES = 3;
constexpr uint32_t G2_A_STAGE = G2_KSUB * G2_A_BYTES, G2_B_STAGE = G2_KSUB * G2_B_STRIDE;
constexpr size_t G2_SMEM = 1024 + G2_STAGES * (G2_A_STAGE + G2_B_STAGE) + (2 * G2_STAGES + 4) * 8 + 16 + 128 + 4 * EPI_STAGE_BYTES;

// FP8: the operands are e4m3 codes (kind::f8f6f4).  A swizzle atom then holds 128 k instead of 64, so a stage holds 256 k;
// the byte layout of the stages, the four 32-byte MMA steps per atom and the barrier protocol are the same.  The epilogue
// scales the accumulator by sa[m] * sb[n] (gemm_epilogue.cuh) before the epilogue of `ep`.
template <int MODE, bool FP8>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(G2_THREADS, 1)
gemm_bf16_2cta(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, int M, int N, int K, int BN,
               int a_kblock, const GemmEpi ep, const float* sa, const float* sb) {
  constexpr int AK = FP8 ? 2 * BK2 : BK2;   // k of one swizzle atom
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + G2_STAGES * G2_A_STAGE;
  uint64_t* full = reinterpret_cast<uint64_t*>(sB + G2_STAGES * G2_B_STAGE);
  uint64_t* empty = full + G2_STAGES;
  uint64_t* tfull = empty + G2_STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  float* epi_stage = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 127) & ~static_cast<uintptr_t>(127));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  const int num_mp = (M + 2 * BM2 - 1) / (2 * BM2);   // 256-row pair tiles
  const int num_n = (N + BN - 1) / BN;
  const int num_tiles = num_mp * num_n;
  const int num_k = (K + G2_KSUB * AK - 1) / (G2_KSUB * AK);   // pipeline steps of 128 k (256 k with FP8)
  const int half_bn = BN >> 1;
  const uint32_t b_bytes = static_cast<uint32_t>(half_bn) * BK2 * 2;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < G2_STAGES; ++i) {
      mbar_init(&full[i], 2);    // leader's expect_tx arrive + the peer's remote arrive (only the leader's copy is used)
      mbar_init(&empty[i], 1);   // multicast tcgen05.commit
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);   // multicast tcgen05.commit
      mbar_init(&tempty[i], 8);  // 4 epilogue warps of each CTA (only the leader's copy is used)
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc_2cta<512>(tmem_slot);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // PDL: everything above overlapped the previous kernel's tail; global memory is touched only from here on
  griddep_launch();
  griddep_wait();

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
        const int mp = tile % num_mp, n_blk = tile / num_mp;
        const int m0 = (mp * 2 + static_cast<int>(rank)) * BM2;
        const int n0 = n_blk * BN + static_cast<int>(rank) * half_bn;
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          if (leader) mbar_arrive_expect_tx(&full[stage], 2 * G2_KSUB * (G2_A_BYTES + b_bytes));
          else mbar_arrive_remote(&full[stage], 0);
#pragma unroll
          for (int ks = 0; ks < G2_KSUB; ++ks) {   // k past K (a ragged tail) is zero-filled by TMA
            const int k0 = (kb * G2_KSUB + ks) * AK;
            if (a_kblock > 0)
              tma_load_3d_2sm(sA + stage * G2_A_STAGE + ks * G2_A_BYTES, &tmA, &full[stage], k0 % a_kblock, m0, k0 / a_kblock);
            else
              tma_load_2d_2sm(sA + stage * G2_A_STAGE + ks * G2_A_BYTES, &tmA, &full[stage], k0, m0);
            tma_load_2d_2sm(sB + stage * G2_B_STAGE + ks * G2_B_STRIDE, &tmB, &full[stage], k0, n0);
          }
          if (++stage == G2_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {
      const uint32_t idesc = FP8 ? umma_idesc_e4m3(2 * BM2, BN) : umma_idesc_bf16(2 * BM2, BN);
      const uint64_t a_desc0 = umma_desc_sw128(smem_u32(sA)), b_desc0 = umma_desc_sw128(smem_u32(sB));
      int stage = 0;
      uint32_t phase = 0;
      int t = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters, ++t) {
        const int as = t & 1;
        const uint32_t aphase = (t >> 1) & 1;
        mbar_wait(&tempty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * G2_BN_MAX;
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          // descriptors: stage base + a compile-time offset (the start-address field counts 16-byte units and cannot carry
          // out of its 14 bits: all operand buffers sit below 256 KB) -- the issuing thread spends one add per operand
          const uint64_t a_desc = a_desc0 + static_cast<uint64_t>(stage) * (G2_A_STAGE >> 4);
          const uint64_t b_desc = b_desc0 + static_cast<uint64_t>(stage) * (G2_B_STAGE >> 4);
#pragma unroll
          for (int ks = 0; ks < G2_KSUB; ++ks)
#pragma unroll
            for (int k = 0; k < BK2 / 16; ++k) {
              const uint64_t ad = a_desc + ((ks * G2_A_BYTES + k * 32) >> 4), bd = b_desc + ((ks * G2_B_STRIDE + k * 32) >> 4);
              if (FP8) umma_f8_2cta(d_tmem, ad, bd, idesc, (kb | ks | k) != 0 ? 1u : 0u);
              else umma_bf16_2cta(d_tmem, ad, bd, idesc, (kb | ks | k) != 0 ? 1u : 0u);
            }
          umma_commit_2cta(&empty[stage]);
          if (++stage == G2_STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit_2cta(&tfull[as]);
      }
    }
  } else {
    const int q = warp & 3;
    int t = 0;
    for (int tile = cluster_id; tile < num_tiles; tile += num_clusters, ++t) {
      const int mp = tile % num_mp, n_blk = tile / num_mp;
      const int as = t & 1;
      const uint32_t aphase = (t >> 1) & 1;
      mbar_wait(&tfull[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * G2_BN_MAX;
      epilogue_tile<MODE, FP8>(taddr, BN, epi_stage + (warp - 2) * (EPI_STAGE_BYTES / 4), lane,
                               (mp * 2 + static_cast<int>(rank)) * BM2 + q * 32, n_blk * BN, M, N, ep, sa, sb);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(&tempty[as], 0);
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2cta<512>(tmem_base);
  }
}

template <int MODE, bool FP8 = false>
void launch2(const CUtensorMap& tmA, const CUtensorMap& tmB, int M, int N, int K, int BN, int a_kblock, const GemmEpi& epi,
             cudaStream_t stream, const float* sa = nullptr, const float* sb = nullptr) {
  auto kern = gemm_bf16_2cta<MODE, FP8>;
  ensure_dyn_smem(kern, G2_SMEM);
  const int tiles = ((M + 2 * BM2 - 1) / (2 * BM2)) * ((N + BN - 1) / BN);
  const int clusters = device_sm_count() / 2;
  const int grid = 2 * (tiles < clusters ? tiles : clusters);
  launch_pdl(PDL_GEMM, kern, dim3(grid), dim3(G2_THREADS), G2_SMEM, stream, tmA, tmB, M, N, K, BN, a_kblock, epi, sa, sb);
}

template <bool FP8>
void launch2_mode(const CUtensorMap& tmA, const CUtensorMap& tmB, int M, int N, int K, int bn, int a_kblock, const GemmEpi& epi,
                  cudaStream_t stream, const float* sa, const float* sb) {
  switch (epi.mode) {
    case EPI_BF16: launch2<EPI_BF16, FP8>(tmA, tmB, M, N, K, bn, a_kblock, epi, stream, sa, sb); break;
    case EPI_GELU_BF16: launch2<EPI_GELU_BF16, FP8>(tmA, tmB, M, N, K, bn, a_kblock, epi, stream, sa, sb); break;
    case EPI_GATE_RESID: launch2<EPI_GATE_RESID, FP8>(tmA, tmB, M, N, K, bn, a_kblock, epi, stream, sa, sb); break;
    case EPI_F32: launch2<EPI_F32, FP8>(tmA, tmB, M, N, K, bn, a_kblock, epi, stream, sa, sb); break;
    case EPI_SILU_BF16: launch2<EPI_SILU_BF16, FP8>(tmA, tmB, M, N, K, bn, a_kblock, epi, stream, sa, sb); break;
    default: LTX_CHECK(false, 2, "bad GEMM epilogue mode");
  }
}

void check_tsplit(const GemmEpi& epi, int bn) {
  LTX_CHECK(epi.tsplit_col == 0 || (epi.mode == EPI_BF16 && bn % 32 == 0 && epi.tsplit_col % 32 == 0 && epi.out_t != nullptr &&
                                    epi.ldt % 8 == 0 && epi.col_block == 0),
            2, "GEMM: transposed-column output needs the bf16 epilogue, a tile width and split column that are multiples of 32");
}

}  // namespace

// tile width for the pair kernel: whole waves of (#SM / 2) clusters over 256-row tiles; widths are multiples of 16 (the
// tcgen05.mma N granularity at cta_group::2), so each CTA's half (BN / 2) is a whole number of 8-row swizzle atoms of B
int gemm2_fit_tile_width(int M, int N) {
  const int clusters = device_sm_count() / 2;
  const int num_mp = (M + 255) / 256;
  int best = 256;
  double best_cost = 1e30;
  for (int bn = 256; bn >= 64; bn -= 16) {
    const long long tiles = static_cast<long long>(num_mp) * ((N + bn - 1) / bn);
    const long long waves = (tiles + clusters - 1) / clusters;
    // per-tile time = a fixed part per k step (operand delivery of the 16 KB A block, barrier round trips of the issuing
    // thread) + a part proportional to the width: ~ bn + 100 with 128-wide k stages (round-2 sweep: 256 / 224 / 176 columns
    // take 27.1 / 23.4 / 20.6 us per wave at K = 4096); it was bn + 257 with 64-wide stages
    const double cost = static_cast<double>(waves) * (bn + 100.0);
    if (cost < best_cost - 1e-9) { best_cost = cost; best = bn; }
  }
  return best;
}

void launch_gemm_2cta(const bf16* A, int64_t lda, const bf16* B, int64_t ldb, int M, int N, int K, const GemmEpi& epi,
                      cudaStream_t stream, int force_bn, int a_kblock, int64_t a_kblock_stride) {
  int bn = force_bn ? force_bn : gemm2_fit_tile_width(M, N);
  LTX_CHECK(bn >= 64 && bn <= 256 && bn % 16 == 0, 2, "2-CTA GEMM: tile width must be a multiple of 16 in [64, 256]");
  check_tsplit(epi, bn);
  CUtensorMap tmA;
  if (a_kblock > 0) {
    LTX_CHECK(a_kblock % BK2 == 0 && K % a_kblock == 0 && lda == a_kblock, 2, "GEMM: bad K-blocked A layout");
    tmA = make_tmap_3d(A, a_kblock, M, K / a_kblock, lda, a_kblock_stride, 64, BM2);
  } else {
    tmA = make_tmap_2d(A, M, K, lda, BM2);
  }
  CUtensorMap tmB = make_tmap_2d(B, N, K, ldb, bn / 2);
  launch2_mode<false>(tmA, tmB, M, N, K, bn, a_kblock, epi, stream, nullptr, nullptr);
}

void launch_gemm_fp8(const uint8_t* A, int64_t lda, const float* sa, const uint8_t* B, int64_t ldb, const float* sb, int M, int N,
                     int K, const GemmEpi& epi, cudaStream_t stream, int force_bn) {
  LTX_CHECK(M > 0 && N > 0 && K > 0, 2, "GEMM: empty problem");
  LTX_CHECK(K % 16 == 0 && lda % 16 == 0 && ldb % 16 == 0 && lda >= K && ldb >= K, 2,
            "FP8 GEMM: K and the row pitches must be multiples of 16 bytes");
  LTX_CHECK(sa != nullptr && sb != nullptr && (reinterpret_cast<uintptr_t>(sb) & 15) == 0, 2,
            "FP8 GEMM: row scales of both operands needed (sb 16-byte aligned)");
  LTX_CHECK(epi.col_block == 0 && epi.transpose_out == 0, 2, "FP8 GEMM: no column-blocked or transposed-row output");
  if (epi.mode == EPI_GATE_RESID) {
    LTX_CHECK(epi.resid != nullptr && epi.ldr % 4 == 0, 2, "GEMM: residual epilogue needs fp32 resid with ld % 4 == 0");
    LTX_CHECK(epi.shadow == nullptr || epi.lds % 4 == 0, 2, "GEMM: shadow ld must be a multiple of 4");
  } else {
    LTX_CHECK(epi.out != nullptr, 2, "GEMM: missing output");
    LTX_CHECK(epi.ldo % (epi.mode == EPI_F32 ? 4 : 8) == 0, 2, "GEMM: output ld alignment");
  }
  const int bn = force_bn ? force_bn : gemm2_fit_tile_width(M, N);
  LTX_CHECK(bn >= 64 && bn <= 256 && bn % 16 == 0, 2, "2-CTA GEMM: tile width must be a multiple of 16 in [64, 256]");
  check_tsplit(epi, bn);
  const CUtensorMap tmA = make_tmap_u8_sw128(A, M, K, lda, BM2);
  const CUtensorMap tmB = make_tmap_u8_sw128(B, N, K, ldb, bn / 2);
  launch2_mode<true>(tmA, tmB, M, N, K, bn, 0, epi, stream, sa, sb);
}

}  // namespace ltx
