// Weight-streaming ("swap-AB") bf16 GEMM for few activation rows: C[M,N] = A[M,K] * W[N,K]^T with M <= 512.
//
// Why: under Ulysses sequence parallelism a rank owns N_tokens / P rows (192 at P = 8, 384 at P = 4) but still streams every
// weight (26 GB per step).  The tile kernels (gemm.cu / gemm2.cu) put the ACTIVATIONS on the 128 TMEM lanes: at M = 192 a CTA
// pair re-loads its 32 KB activation k-block for every 64..112 weight rows, 5 bytes of L2 -> SM traffic per weight byte, and
// the chip-wide L2 delivery cap (~6300 B/clk) holds the weights to 1.6 TB/s (profiles/r01c_bench_8gpu.json: 14.6 ms of GEMM per
// step for 4.3 TFLOP).  Here the operands trade places: the WEIGHT tile is the UMMA "A" operand -- 256 rows per CTA pair, 128 TMEM
// lanes each -- and the activation rows are the UMMA "N" dimension (one 256 x MC x 16 tcgen05.mma.cta_group::2 per k-step,
// MC = the row count rounded up to 16, at most 256), split between the two CTAs.  Per k-block a CTA now moves 16 KB of weights
// + MC/2 x 128 B of activations: 1.75 bytes per weight byte at M = 192.  (Measured: without the K split this alone buys nothing --
// both kernels sit at ~60 GB/s of ingest per SM and the tile kernel uses more SMs; the K split below is what pays.)
//
//   * unit of work = (256-row weight tile, K split, activation chunk); persistent CTA pairs, units dealt round-robin with the
//     chunks / splits of one weight tile adjacent, so they run at the same time and the tile's second read hits L2
//   * weight tiles are few when N is small (4096 / 256 = 16): K is split so that ~all 74 pairs stream.  Every split stores its
//     fp32 partial tile to an L2-resident workspace ([row][128 features]: 128-byte lines per warp access) and takes a ticket on
//     the tile's counter.  When all units of the launch are resident at once (units <= CTA pairs, the usual case) the S splits
//     of a tile wait for each other and each one reduces and finishes 1/S of the rows; otherwise the LAST arriver reduces the
//     whole tile.  Either way the partials are added in split order: bit-reproducible whatever the arrival order.
//     Measured (B200, M = 192, cold weights): D x D 26.0 -> 20.4 us, FFN-out (K = 16384) 82.8 -> 39.8 us against the tile kernel
//   * TMEM lane = output feature n, column = activation row m: for a fixed m a warp's 32 lanes own 32 consecutive n, so the
//     epilogue stores straight from registers, 128 B (fp32) / 64 B (bf16) per instruction, no shared-memory transpose
//   * 8-stage TMA ring (224 KB), double-buffered accumulators, PDL prologue overlap, TMA zero-fill for ragged M / N / K
// Same epilogue contract as launch_gemm (bias, GELU / SiLU, gate * residual + bf16 shadow, fp32, column-blocked and peer-memory
// destinations, K-blocked A); transposed-column output (tsplit_col) stays with the tile kernels.
#include "ltx_internal.h"
#include "ptx.cuh"

namespace ltx {

namespace {

constexpr int SW_BK = 64;
constexpr int SW_THREADS = 192;
constexpr int SW_WROWS = 128;                       // weight rows per CTA (256 per pair)
constexpr int SW_MC_MAX = 256;                      // activation rows per unit
constexpr uint32_t SW_W_BYTES = SW_WROWS * SW_BK * 2;   // 16 KB
constexpr int SW_MAX_STAGES = 8;
constexpr size_t SW_SMEM_LIMIT = 227 * 1024;
constexpr size_t SW_SMEM_FIXED = 1024 + (2 * SW_MAX_STAGES + 4) * 8 + 64;

// Fused epilogue of `lim` (<= 32) activation rows [m0, m0 + lim) of output feature n (one thread): v[i] = accumulator of (m0 + i, n).
// lim < 32 on the 16-column tail of a chunk: the rows behind it belong to the next activation chunk (another unit).
template <int MODE>
__device__ __forceinline__ void swap_epilogue32(const float (&v)[32], int m0, int lim, int n, int M, int N, const GemmEpi& ep) {
  if (n >= N || m0 >= M) return;
  const int cnt = (M - m0 < lim) ? M - m0 : lim;
  const float bn = (ep.bias && !ep.bias_per_row) ? __ldg(ep.bias + n) : 0.f;
  if (MODE == EPI_GATE_RESID) {
    float x[32];
#pragma unroll
    for (int i = 0; i < 32; ++i)   // all residual loads in flight before the first store (the compiler cannot reorder them itself)
      x[i] = (i < cnt) ? ep.resid[static_cast<int64_t>(m0 + i) * ep.ldr + n] : 0.f;
    const float gb = (ep.gate_a && ep.gate_b) ? __ldg(ep.gate_b + n) : 0.f;
    const bool uniform = ep.gate_a && (m0 / ep.rows_per_gate == (m0 + cnt - 1) / ep.rows_per_gate);
    const float gu = ep.gate_a ? (uniform ? ep.gate_a[static_cast<int64_t>(m0 / ep.rows_per_gate) * ep.gate_ld + n] + gb : 0.f) : 1.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      if (i >= cnt) break;
      const int m = m0 + i;
      float g = gu;
      if (ep.gate_a && !uniform) g = ep.gate_a[static_cast<int64_t>(m / ep.rows_per_gate) * ep.gate_ld + n] + gb;
      const float rb = (ep.bias && ep.bias_per_row) ? ep.bias[m] : 0.f;
      const float xv = x[i] + (v[i] + bn + rb) * g * ep.scale;
      ep.resid[static_cast<int64_t>(m) * ep.ldr + n] = xv;
      if (ep.shadow) ep.shadow[static_cast<int64_t>(m) * ep.lds + n] = __float2bfloat16(xv);
    }
  } else if (MODE == EPI_F32) {
    float* o = reinterpret_cast<float*>(ep.out) + n;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      if (i >= cnt) break;
      const int m = m0 + i;
      const float rb = (ep.bias && ep.bias_per_row) ? ep.bias[m] : 0.f;
      o[static_cast<int64_t>(m) * ep.ldo] = v[i] + bn + rb;
    }
  } else {
    bf16* o = reinterpret_cast<bf16*>(ep.out) + n;
    int64_t old = ep.ldo;
    if (ep.col_block > 0 && n >= ep.col_block_from) {
      const int nb = n - ep.col_block_from;
      if (ep.blocked_ld) old = ep.blocked_ld;
      if (ep.use_col_ptrs) o = reinterpret_cast<bf16*>(ep.col_ptrs.p[nb / ep.col_block]) + (nb % ep.col_block);
      else o = reinterpret_cast<bf16*>(ep.blocked_out ? ep.blocked_out : ep.out) + static_cast<int64_t>(nb / ep.col_block) * ep.col_block_stride +
               (nb % ep.col_block);
    }
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      if (i >= cnt) break;
      const int m = m0 + i;
      const float rb = (ep.bias && ep.bias_per_row) ? ep.bias[m] : 0.f;
      float a = v[i] + bn + rb;
      if (MODE == EPI_GELU_BF16) a = gelu_tanh(a);
      if (MODE == EPI_SILU_BF16) a = silu(a);
      o[static_cast<int64_t>(m) * old] = __float2bfloat16(a);
    }
  }
}

struct SwapParams {
  int M, N, K;
  int MC;        // activation rows per unit (multiple of 16, <= 256)
  int num_mc;    // activation chunks
  int S;         // K splits
  int kps;       // k-blocks per split
  int stages;
  int a_kblock;
  int spin;      // every unit is resident at once (units <= CTA pairs): the S splits of a tile wait for each other and share the reduction
  float* ws;             // [tile][rank][split][MC * num_mc... see slot()] fp32 partial tiles (S > 1)
  unsigned int* counters;
};

template <int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(SW_THREADS, 1)
gemm_swapab_2cta(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmA, const SwapParams p, const GemmEpi ep) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  const uint32_t a_bytes = static_cast<uint32_t>(p.MC >> 1) * SW_BK * 2;   // this CTA's half of the activation k-block
  const uint32_t stage_bytes = SW_W_BYTES + ((a_bytes + 1023u) & ~1023u);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + static_cast<size_t>(p.stages) * stage_bytes);
  uint64_t* empty = full + SW_MAX_STAGES;
  uint64_t* tfull = empty + SW_MAX_STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  volatile uint32_t* ticket = tmem_slot + 2;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  const int num_nt = (p.N + 2 * SW_WROWS - 1) / (2 * SW_WROWS);
  const int num_k = (p.K + SW_BK - 1) / SW_BK;
  const int num_units = num_nt * p.S * p.num_mc;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmA);
    for (int i = 0; i < p.stages; ++i) {
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
  griddep_launch();
  griddep_wait();   // PDL: global memory is touched only from here on

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = cluster_id; u < num_units; u += num_clusters) {
        const int mc = u % p.num_mc, s = (u / p.num_mc) % p.S, nt = u / (p.num_mc * p.S);
        const int n0 = nt * 2 * SW_WROWS + static_cast<int>(rank) * SW_WROWS;
        const int m0 = mc * p.MC + static_cast<int>(rank) * (p.MC >> 1);
        const int kb0 = s * p.kps, kb1 = min(num_k, kb0 + p.kps);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          if (leader) mbar_arrive_expect_tx(&full[stage], 2 * (SW_W_BYTES + a_bytes));
          else mbar_arrive_remote(&full[stage], 0);
          uint8_t* sW = smem + static_cast<size_t>(stage) * stage_bytes;
          tma_load_2d_2sm(sW, &tmW, &full[stage], kb * SW_BK, n0);
          if (p.a_kblock > 0)
            tma_load_3d_2sm(sW + SW_W_BYTES, &tmA, &full[stage], (kb * SW_BK) % p.a_kblock, m0, (kb * SW_BK) / p.a_kblock);
          else
            tma_load_2d_2sm(sW + SW_W_BYTES, &tmA, &full[stage], kb * SW_BK, m0);
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {
      const uint32_t idesc = umma_idesc_bf16(2 * SW_WROWS, p.MC);
      int stage = 0;
      uint32_t phase = 0;
      int t = 0;
      for (int u = cluster_id; u < num_units; u += num_clusters, ++t) {
        const int s = (u / p.num_mc) % p.S;
        const int kb0 = s * p.kps, kb1 = min(num_k, kb0 + p.kps);
        const int as = t & 1;
        const uint32_t aphase = (t >> 1) & 1;
        mbar_wait(&tempty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * SW_MC_MAX;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t w_addr = smem_u32(smem + static_cast<size_t>(stage) * stage_bytes);
          const uint32_t a_addr = w_addr + SW_W_BYTES;
#pragma unroll
          for (int k = 0; k < SW_BK / 16; ++k)
            umma_bf16_2cta(d_tmem, umma_desc_sw128(w_addr + k * 32), umma_desc_sw128(a_addr + k * 32), idesc,
                           (kb != kb0 || k != 0) ? 1u : 0u);
          umma_commit_2cta(&empty[stage]);
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
        umma_commit_2cta(&tfull[as]);
      }
    }
  } else {
    const int q = warp & 3;
    const int et = threadIdx.x - 64;   // 0..127 among the epilogue threads
    int t = 0;
    for (int u = cluster_id; u < num_units; u += num_clusters, ++t) {
      const int mc = u % p.num_mc, s = (u / p.num_mc) % p.S, nt = u / (p.num_mc * p.S);
      const int n_loc = q * 32 + lane;                                        // feature inside this CTA's 128
      const int n = nt * 2 * SW_WROWS + static_cast<int>(rank) * SW_WROWS + n_loc;
      const int mbase = mc * p.MC;
      const int as = t & 1;
      const uint32_t aphase = (t >> 1) & 1;
      mbar_wait(&tfull[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * SW_MC_MAX;
      const int nch = (p.MC + 31) >> 5;
      if (p.S == 1) {
        uint32_t r[32];
#pragma unroll 1
        for (int c = 0; c < nch; ++c) {
          if (p.MC - c * 32 >= 32) tmem_ld32(taddr + c * 32, r);
          else tmem_ld16(taddr + c * 32, r);
          tmem_ld_wait();
          float v[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
          swap_epilogue32<MODE>(v, mbase + c * 32, min(32, p.MC - c * 32), n, p.M, p.N, ep);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(&tempty[as], 0);
      } else {
        // ---- split-K: park this split's partial tile in the workspace, [activation row][128 features] so that a warp's
        // store / load of one row is one 128-byte line, then take a ticket on the tile's arrival counter
        const int tile_slot = (nt * p.num_mc + mc) * 2 + static_cast<int>(rank);
        const size_t slot_sz = static_cast<size_t>(SW_WROWS) * p.MC;
        float* slot0 = p.ws + static_cast<size_t>(tile_slot) * p.S * slot_sz;
        float* mine = slot0 + static_cast<size_t>(s) * slot_sz + n_loc;
        unsigned int* arrived = p.counters + 2 * tile_slot;
        unsigned int* finished = arrived + 1;
        uint32_t r[32];
#pragma unroll 1
        for (int c = 0; c < nch; ++c) {
          if (p.MC - c * 32 >= 32) tmem_ld32(taddr + c * 32, r);
          else tmem_ld16(taddr + c * 32, r);
          tmem_ld_wait();
          const int lim = min(32, p.MC - c * 32);
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (i < lim) __stcg(mine + static_cast<size_t>(c * 32 + i) * SW_WROWS, __uint_as_float(r[i]));
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(&tempty[as], 0);   // the accumulator buffer is free again
        __threadfence();
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (et == 0) {
          uint32_t tk = atomicAdd(arrived, 1u);
          if (p.spin) {
            // every split of this tile is resident right now (one unit per CTA pair): wait for all of them, then each split
            // reduces and finishes ITS share of the rows -- the reduction reads are spread over S CTAs instead of one
            unsigned long long spins = 0;
            while (tk + 1 < static_cast<uint32_t>(p.S)) {
              asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(tk) : "l"(arrived) : "memory");
              tk -= 1;
              if (++spins > (1ull << 24)) {
                printf("ltxcuda: split-K partner timeout block %d tile %d split %d\n", blockIdx.x, tile_slot, s);
                __trap();
              }
            }
          }
          *ticket = tk;
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        const uint32_t tk = *ticket;
        asm volatile("bar.sync 1, 128;" ::: "memory");   // everyone has read the ticket before the next unit overwrites it
        // rows this CTA reduces: all of them if it is the last arriver (no partner guaranteed to be resident), its 1/S share
        // when all splits are known to be there
        int row_lo = 0, row_hi = 0;
        if (p.spin) {
          const int share = ((p.MC + p.S - 1) / p.S + 15) & ~15;
          row_lo = min(p.MC, s * share);
          row_hi = min(p.MC, row_lo + share);
        } else if (tk == static_cast<uint32_t>(p.S - 1)) {
          row_hi = p.MC;
        }
        if (row_hi > row_lo) {
          __threadfence();
#pragma unroll 1
          for (int c0 = row_lo; c0 < row_hi; c0 += 32) {
            const int lim = min(32, row_hi - c0);
            float v[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = 0.f;
#pragma unroll 1
            for (int ss = 0; ss < p.S; ++ss) {   // fixed order: the sum does not depend on the arrival order
              const float* src = slot0 + static_cast<size_t>(ss) * slot_sz + static_cast<size_t>(c0) * SW_WROWS + n_loc;
              float t[32];
#pragma unroll
              for (int i = 0; i < 32; ++i) t[i] = (i < lim) ? __ldcg(src + static_cast<size_t>(i) * SW_WROWS) : 0.f;
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] += t[i];
            }
            swap_epilogue32<MODE>(v, mbase + c0, lim, n, p.M, p.N, ep);
          }
        }
        // the last CTA to finish with the tile's partials re-arms its counters for the next launch
        if (p.spin) {
          asm volatile("bar.sync 1, 128;" ::: "memory");
          if (et == 0 && atomicAdd(finished, 1u) == static_cast<uint32_t>(p.S - 1)) { *arrived = 0; *finished = 0; }
        } else if (et == 0 && tk == static_cast<uint32_t>(p.S - 1)) {
          *arrived = 0;
        }
      }
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2cta<512>(tmem_base);
  }
}

template <int MODE>
void launch_sw(const CUtensorMap& tmW, const CUtensorMap& tmA, const SwapParams& p, size_t smem, int units, const GemmEpi& epi,
               cudaStream_t stream) {
  auto kern = gemm_swapab_2cta<MODE>;
  ensure_dyn_smem(kern, SW_SMEM_LIMIT);
  const int clusters = device_sm_count() / 2;
  const int grid = 2 * (units < clusters ? units : clusters);
  launch_pdl(PDL_GEMM, kern, dim3(grid), dim3(SW_THREADS), smem, stream, tmW, tmA, p, epi);
}

}  // namespace

bool gemm_swapab_eligible(int64_t lda, int64_t ldb, int M, int N, int K, const GemmEpi& epi) {
  if (M > 2 * SW_MC_MAX || M < 1 || N < 1 || K < 8) return false;
  if (epi.tsplit_col != 0 || epi.transpose_out != 0) return false;
  if (K % 8 != 0 || lda % 8 != 0 || ldb % 8 != 0) return false;
  return true;
}

void launch_gemm_swapab(const bf16* A, int64_t lda, const bf16* W, int64_t ldb, int M, int N, int K, const GemmEpi& epi,
                        cudaStream_t stream, int a_kblock, int64_t a_kblock_stride) {
  LTX_CHECK(gemm_swapab_eligible(lda, ldb, M, N, K, epi), 2, "swap-AB GEMM: unsupported problem");
  SwapParams p = {};
  p.M = M; p.N = N; p.K = K;
  p.num_mc = (M + SW_MC_MAX - 1) / SW_MC_MAX;
  p.MC = (((M + p.num_mc - 1) / p.num_mc) + 15) / 16 * 16;
  const int num_nt = (N + 2 * SW_WROWS - 1) / (2 * SW_WROWS);
  const int num_k = (K + SW_BK - 1) / SW_BK;
  const int clusters = device_sm_count() / 2;
  // K splits: enough units for every CTA pair to stream weights, at least 8 k-blocks each, and the partials must fit the workspace
  int S = 1;
  const int base_units = num_nt * p.num_mc;
  if (epi.ws != nullptr && epi.ws_counters != nullptr && base_units * 4 < clusters * 3) {
    S = clusters / base_units;
    if (S > 8) S = 8;
    while (S > 1 && num_k / S < 8) --S;
    const size_t per_split = static_cast<size_t>(base_units) * 2 * SW_WROWS * p.MC * 4;
    while (S > 1 && per_split * S > epi.ws_bytes) --S;
    if (static_cast<size_t>(base_units) * 4 > epi.ws_counter_count) S = 1;
  }
  p.S = S;
  p.kps = (num_k + S - 1) / S;
  while (p.S > 1 && (p.S - 1) * p.kps >= num_k) --p.S;   // no empty split
  p.a_kblock = a_kblock;
  p.ws = epi.ws;
  p.counters = epi.ws_counters;
  const uint32_t a_bytes = static_cast<uint32_t>(p.MC / 2) * SW_BK * 2;
  const size_t stage_bytes = SW_W_BYTES + ((a_bytes + 1023u) & ~1023u);
  int stages = static_cast<int>((SW_SMEM_LIMIT - SW_SMEM_FIXED) / stage_bytes);
  if (stages > SW_MAX_STAGES) stages = SW_MAX_STAGES;
  p.stages = stages;
  const size_t smem = SW_SMEM_FIXED + stages * stage_bytes;
  CUtensorMap tmW = make_tmap_2d(W, N, K, ldb, SW_WROWS);
  CUtensorMap tmA;
  if (a_kblock > 0) {
    LTX_CHECK(a_kblock % SW_BK == 0 && K % a_kblock == 0 && lda == a_kblock, 2, "GEMM: bad K-blocked A layout");
    tmA = make_tmap_3d(A, a_kblock, M, K / a_kblock, lda, a_kblock_stride, 64, p.MC / 2);
  } else {
    tmA = make_tmap_2d(A, M, K, lda, p.MC / 2);
  }
  const int units = num_nt * p.S * p.num_mc;
  p.spin = (p.S > 1 && units <= clusters) ? 1 : 0;
  switch (epi.mode) {
    case EPI_BF16: launch_sw<EPI_BF16>(tmW, tmA, p, smem, units, epi, stream); break;
    case EPI_GELU_BF16: launch_sw<EPI_GELU_BF16>(tmW, tmA, p, smem, units, epi, stream); break;
    case EPI_GATE_RESID: launch_sw<EPI_GATE_RESID>(tmW, tmA, p, smem, units, epi, stream); break;
    case EPI_F32: launch_sw<EPI_F32>(tmW, tmA, p, smem, units, epi, stream); break;
    case EPI_SILU_BF16: launch_sw<EPI_SILU_BF16>(tmW, tmA, p, smem, units, epi, stream); break;
    default: LTX_CHECK(false, 2, "bad GEMM epilogue mode");
  }
}

}  // namespace ltx
