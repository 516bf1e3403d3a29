// 3x3x3 convolution of the video-VAE decoder as an implicit GEMM on tcgen05 (sm_100a), channels-last.
//
// Replaces Conv3dFull.callAsFunction (Models/VAE/VideoConvolution.swift:238-347: three MLX.conv2d calls over shifted
// temporal slices) and the ops fused around it in the decoder (Models/VAE/VideoDecoder.swift): pixel-norm +
// scale/shift + SiLU (:118-126, 419-436) as a padding prologue kernel, depth-to-space + first-frame trim + tiled
// residual (:201-251) and the final unpatchify + (x+1)/2 clip (:257-275, 501-505) as epilogue stores.
//
// Layout: activations fp32 [T, H, W, C]; the prologue writes a bf16 copy with the conv's own padding materialised
// ([T+2, H+2, W+2, C]: reflect in H/W, frame replication in T), so the implicit GEMM needs no boundary logic:
//   M = output voxels, tiled as TMA boxes bt x bh x bw = 128 voxels;  N = Cout;  K = 27 taps x Cin.
//   A tile (tap, k-chunk) = 4-D TMA box at (t0+dt, h0+dh, w0+dw, k0) of the padded volume -> [128 rows x 64 ch], 128B swizzle
//   B tile               = rows [tap*Cout + n0, +BN) x cols [k0, +64) of the [27*Cout, Cin] weight matrix.
// Warp roles and pipelines are those of gemm.cu (TMA producer / MMA issuer / 4 epilogue warps, 2 TMEM stages).
// Three forms of the main loop share the epilogues (ConvCfg below): one CTA per voxel tile (conv3d_tcgen05), CTA pairs on
// cta_group::2 (conv3d_pair_tcgen05: whenever Cin comes in 128-channel stages) and pairs with slab stages
// (conv3d_slab_tcgen05: Cout < 256).  conv3d_plan() picks; slab stages and the tap split add the taps up in another order
// than the rest, so those two choices never look at T (a temporal shard must round like the whole clip).
#include <cstdlib>

#include "frames_u8.cuh"
#include "gemm_epilogue.cuh"
#include "ltx_internal.h"
#include "ptx.cuh"

namespace ltx {

namespace {

constexpr int CBM = 128, CBK = 64, CONV_THREADS = 192;

// KS = 64-channel k chunks per pipeline stage.  KS = 2 (Cin a multiple of 128): a stage holds both halves of a 128-channel
// slice of one tap, so the issuing thread waits on / commits to half as many barriers per k -- the same change that bought
// 4-7 % on the DiT GEMMs (profiles/r02_gemm_kstage_sweep.txt).
// PAIR: two CTAs of a cluster (the two SMs of a TPC) compute two adjacent voxel tiles against the same weight tile with
// tcgen05.mma.cta_group::2 (M = 256): each CTA loads its own A tile and HALF of the weight tile.  Why: one CTA per tile is bound
// by shared-memory traffic -- per 128-channel stage of the 128 -> 128 convs 64 KB of TMA writes + 64 KB of operand reads against
// 512 clk x 128 B/clk of port bandwidth; in a pair the B half drops out of both: 96 KB.
// SLAB (pairs, tiles up to 128 columns): a stage holds, for one (dt, dw) and 64 channels, the voxel tile's rows WITH their
// two halo rows in h -- a [bh + 2, bw] slab, bt = 1 -- and the weight tiles of the three taps dh = 0, 1, 2.  Tap dh reads the
// 128 rows starting bw * dh rows into the slab (a whole number of 8-row swizzle atoms: only the descriptor's start address
// moves), so the activations come in once for three taps: (bh + 2) / (3 bh) of the A traffic (0.375-0.5).  Why: an SM takes
// operands in at ~64 B/clk; at 128 output channels the per-tap form needs 94 B per tensor-clock (A 32 KB + half a weight
// tile 16 KB per 512 clk), the GEMM at 256 columns 62.5 -- the 128 -> 128 convs (41 % of a decode) ran at ~900 TFLOP/s.
constexpr int SLAB_ROWS_MAX = 192;

template <int BN, int KS = 1, bool PAIR = false, bool SLAB = false>
struct ConvCfg {
  static constexpr int BROWS = PAIR ? BN / 2 : BN;   // weight rows this CTA stages
  static constexpr int STAGES = SLAB ? (BN == 128 ? 4 : 5) : (PAIR ? (BN == 256 ? 6 : 8) : ((BN == 256) ? 4 : (BN == 128 ? 6 : 8))) / KS;
  static constexpr uint32_t A_BYTES = (SLAB ? SLAB_ROWS_MAX : CBM) * CBK * 2;
  static constexpr uint32_t B_TAP_BYTES = BROWS * CBK * 2;
  static constexpr uint32_t B_BYTES = (SLAB ? 3 : 1) * B_TAP_BYTES;
  static constexpr uint32_t A_STAGE = KS * A_BYTES, B_STAGE = KS * B_BYTES;
  static constexpr uint32_t TMEM_COLS = 2 * BN;
  static constexpr size_t SMEM = 1024 + STAGES * (A_STAGE + B_STAGE) + (2 * STAGES + 4) * 8 + 16 + 128 + 4 * EPI_STAGE_BYTES;
};

struct ConvGeom {
  int T, H, W, Cin, Cout;
  int bt, bh, bw;     // voxel box of one M tile (bt*bh*bw == 128)
  int nt, nh, nw;     // tiles per axis
  int tap0, ntaps;    // taps [tap0, tap0 + ntaps) of the 3x3x3 stencil (27: Conv3d; 9 starting at 9: per-frame Conv2d, dt = 1)
  int slab;           // 1: slab stages (conv3d_slab_tcgen05): bt == 1, the A box is [bh + 2, bw] voxels
  int ksplit;         // > 1: the taps are split into ksplit groups, each an own work item writing raw partial sums to
                      // out + ks * T*H*W*Cout (MODE 0, no bias / residual); conv_splitk_reduce_kernel adds them up in a fixed order
};

__device__ __forceinline__ float clip01(float v) { return fminf(fmaxf(v, 0.f), 1.f); }

template <int MODE>
__device__ __forceinline__ void conv_epilogue_chunk(const uint32_t (&r)[32], int t, int h, int w, int col0,
                                                    const ConvGeom& g, const ConvEpi& ep) {
  if (col0 >= g.Cout) return;
  const int64_t vox = (static_cast<int64_t>(t) * g.H + h) * g.W + w;
  if (MODE == 0) {
    float* o = ep.out + vox * g.Cout + col0;
    const float* rs = ep.resid ? ep.resid + vox * g.Cout + col0 : nullptr;
    if (col0 + 32 <= g.Cout) {
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        float4 b = *reinterpret_cast<const float4*>(ep.bias + col0 + j);
        float4 v = make_float4(__uint_as_float(r[j]) + b.x, __uint_as_float(r[j + 1]) + b.y,
                               __uint_as_float(r[j + 2]) + b.z, __uint_as_float(r[j + 3]) + b.w);
        if (rs) {
          float4 x = *reinterpret_cast<const float4*>(rs + j);
          v.x += x.x; v.y += x.y; v.z += x.z; v.w += x.w;
        }
        *reinterpret_cast<float4*>(o + j) = v;
      }
    } else {
      for (int j = 0; j < 32 && col0 + j < g.Cout; ++j)
        o[j] = __uint_as_float(r[j]) + ep.bias[col0 + j] + (rs ? rs[j] : 0.f);
    }
  } else if (MODE == 1) {
    // depth-to-space (2,2,2): conv channel co = c*8 + p1*4 + p2*2 + p3 -> out[2t+p1-1, 2h+p2, 2w+p3, c]
    // residual: x[t,h,w,(c mod Cin/8)*8 + p]   (VideoDecoder.swift:201-251)
    const int Cf = g.Cout >> 3;        // output channels
    const int Cr = g.Cin >> 3;         // residual d2s channels (tiled x4)
    const int Ho = 2 * g.H, Wo = 2 * g.W;
    const float* xr = ep.resid + vox * g.Cin;
    const int c0 = col0 >> 3;          // first of 4 output channels covered by these 32 columns
#pragma unroll
    for (int p = 0; p < 8; ++p) {
      const int p1 = p >> 2, p2 = (p >> 1) & 1, p3 = p & 1;
      const int to = 2 * t + p1 - 1 + ep.t_shift;
      if (to < 0) continue;
      float v[4];
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        const int co = col0 + cc * 8 + p;
        const int c = c0 + cc;
        v[cc] = __uint_as_float(r[cc * 8 + p]) + ep.bias[co] + xr[(c % Cr) * 8 + p];
      }
      float* o = ep.out + ((static_cast<int64_t>(to) * Ho + (2 * h + p2)) * Wo + (2 * w + p3)) * Cf + c0;
      *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
    }
  } else {
    // unpatchify 4x4: conv channel co = c*16 + pa*4 + pb -> frames[t, 4h + pb, 4w + pa, c], (x+1)/2 clipped to [0,1]
    const int Ho = 4 * g.H, Wo = 4 * g.W;
    for (int j = 0; j < 32 && col0 + j < g.Cout; ++j) {
      const int co = col0 + j;
      const int c = co >> 4, pa = (co >> 2) & 3, pb = co & 3;
      const float v = (__uint_as_float(r[j]) + ep.bias[co] + 1.0f) * 0.5f;
      ep.out[((static_cast<int64_t>(t) * Ho + (4 * h + pb)) * Wo + (4 * w + pa)) * 3 + c] = ep.no_clip ? v : clip01(v);
    }
  }
}

// Modes 5 / 6: the voxel's 48 conv channels are 3 colours x one 4x4 pixel block (co = c*16 + pa*4 + pb -> pixel row pb,
// column pa); r0 holds channels 0-31, r1 channels 32-47.  The values are mode 2's, clipped; the block is four whole 2x2
// chroma cells, so I420 needs nothing from a neighbouring voxel.
template <int MODE>
__device__ __forceinline__ void conv_store_frames_u8(const uint32_t (&r0)[32], const uint32_t (&r1)[32], int t, int h, int w,
                                                     const ConvGeom& g, const ConvEpi& ep) {
  const int Ho = 4 * g.H, Wo = 4 * g.W;
  float px[4][4][3];   // [row pb][column pa][colour]
#pragma unroll
  for (int co = 0; co < 48; ++co) {
    const float v = (__uint_as_float(co < 32 ? r0[co] : r1[co - 32]) + ep.bias[co] + 1.0f) * 0.5f;
    px[co & 3][(co >> 2) & 3][co >> 4] = clip01(v);
  }
  if (MODE == CONV_EPI_RGB8) {
#pragma unroll
    for (int pb = 0; pb < 4; ++pb) {   // 12 bytes per pixel row: 3 aligned words
      uint32_t b[12];
#pragma unroll
      for (int i = 0; i < 12; ++i) b[i] = rgb8_code(px[pb][i / 3][i % 3]);
      uint32_t* o = reinterpret_cast<uint32_t*>(ep.out_u8 + ((static_cast<int64_t>(t) * Ho + 4 * h + pb) * Wo + 4 * w) * 3);
#pragma unroll
      for (int k = 0; k < 3; ++k) o[k] = b[4 * k] | (b[4 * k + 1] << 8) | (b[4 * k + 2] << 16) | (b[4 * k + 3] << 24);
    }
  } else {
    const int64_t plane = static_cast<int64_t>(Ho) * Wo;
    uint8_t* yp = ep.out_u8 + static_cast<int64_t>(t) * (plane + plane / 2);
    uint8_t* up = yp + plane;
    uint8_t* vp = up + plane / 4;
    uint32_t y[4][4], cb[2][2], cr[2][2];
#pragma unroll
    for (int cy = 0; cy < 2; ++cy)
#pragma unroll
      for (int cx = 0; cx < 2; ++cx) {
        float p[4][3];
        uint32_t yc[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int c = 0; c < 3; ++c) p[i][c] = px[2 * cy + (i >> 1)][2 * cx + (i & 1)][c];
        i420_cell(p, yc, cb[cy][cx], cr[cy][cx]);
#pragma unroll
        for (int i = 0; i < 4; ++i) y[2 * cy + (i >> 1)][2 * cx + (i & 1)] = yc[i];
      }
#pragma unroll
    for (int pb = 0; pb < 4; ++pb)
      *reinterpret_cast<uint32_t*>(yp + static_cast<int64_t>(4 * h + pb) * Wo + 4 * w) =
          y[pb][0] | (y[pb][1] << 8) | (y[pb][2] << 16) | (y[pb][3] << 24);
#pragma unroll
    for (int cy = 0; cy < 2; ++cy) {
      const int64_t off = static_cast<int64_t>(2 * h + cy) * (Wo / 2) + 2 * w;
      *reinterpret_cast<uint16_t*>(up + off) = static_cast<uint16_t>(cb[cy][0] | (cb[cy][1] << 8));
      *reinterpret_cast<uint16_t*>(vp + off) = static_cast<uint16_t>(cr[cy][0] | (cr[cy][1] << 8));
    }
  }
}

template <int BN, int MODE, int KS, bool PAIR, bool SLAB = false>
__device__ __forceinline__ void conv3d_body(const CUtensorMap& tmX, const CUtensorMap& tmW, const ConvGeom& g, const ConvEpi& ep) {
  static_assert(!SLAB || (PAIR && KS == 1 && BN <= 128), "slab stages: CTA pairs, 64-channel stages, tiles up to 128 columns");
  using Cfg = ConvCfg<BN, KS, PAIR, SLAB>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * Cfg::A_STAGE;
  uint64_t* full = reinterpret_cast<uint64_t*>(sB + STAGES * Cfg::B_STAGE);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  float* epi_stage = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 127) & ~static_cast<uintptr_t>(127));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const bool leader = rank == 0;
  const int worker = PAIR ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
  const int num_workers = PAIR ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);
  const int num_vox_tiles = g.nt * g.nh * g.nw;
  // PAIR: a work item covers voxel tiles 2 * mp and 2 * mp + 1 (the second may lie past the volume when the count is odd: its
  // TMA boxes are zero-filled, its rows masked by the epilogue)
  const int num_m = PAIR ? (num_vox_tiles + 1) / 2 : num_vox_tiles;
  const int num_n = (g.Cout + BN - 1) / BN;
  const int num_mn = num_m * num_n;
  const int num_tiles = num_mn * g.ksplit;
  const int kchunks = g.Cin / (CBK * KS);   // pipeline steps per tap (KS * 64 channels each)
  const int taps_per_split = g.ntaps / g.ksplit;
  // SLAB: a pipeline step covers the three dh taps of one (dt, dw)
  const int num_k = (SLAB ? taps_per_split / 3 : taps_per_split) * kchunks;
  const uint32_t slab_bytes = static_cast<uint32_t>((g.bh + 2) * g.bw) * CBK * 2;   // SLAB: A bytes of one stage

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmW);
    // PAIR (protocol of gemm2.cu): full = the leader's expect_tx arrive + the peer's remote arrive, the 2-SM TMA loads of both
    // CTAs report their bytes to the leader's copy; empty / tfull are released in BOTH CTAs by the multicast tcgen05.commit;
    // tempty (leader's copy) collects the 4 epilogue warps of each CTA
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], PAIR ? 2 : 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], PAIR ? 8 : 4); }
    fence_mbar_init();
  }
  if (warp == 1) {
    if (PAIR) tmem_alloc_2cta<Cfg::TMEM_COLS>(tmem_slot);
    else tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all();
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  griddep_launch();
  griddep_wait();   // PDL: the prologue above overlapped the previous kernel's tail

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = worker; tile < num_tiles; tile += num_workers) {
        const int ks = tile / num_mn, mn = tile % num_mn;
        const int m_blk = PAIR ? 2 * (mn % num_m) + static_cast<int>(rank) : mn % num_m, n_blk = mn / num_m;
        const int iw = m_blk % g.nw, ih = (m_blk / g.nw) % g.nh, it = m_blk / (g.nw * g.nh);
        const int t0 = it * g.bt, h0 = ih * g.bh, w0 = iw * g.bw;
        for (int kb = 0; kb < num_k; ++kb) {
          if constexpr (SLAB) {
            // group gi = (dt_local, dw); its taps are wt0 + 3 * dh in the weight matrix
            const int gi = ks * (taps_per_split / 3) + kb / kchunks, kc = kb % kchunks;
            const int dtl = gi / 3, dw = gi % 3;
            const int dt = g.tap0 / 9 + dtl, wt0 = dtl * 9 + dw;
            mbar_wait(&empty[stage], phase ^ 1);
            if (leader) mbar_arrive_expect_tx(&full[stage], 2 * (slab_bytes + Cfg::B_BYTES));
            else mbar_arrive_remote(&full[stage], 0);
            tma_load_4d_2sm(sA + stage * Cfg::A_STAGE, &tmX, &full[stage], kc * CBK, w0 + dw, h0, t0 + dt);
#pragma unroll
            for (int dh = 0; dh < 3; ++dh)
              tma_load_2d_2sm(sB + stage * Cfg::B_STAGE + dh * Cfg::B_TAP_BYTES, &tmW, &full[stage], kc * CBK,
                              (wt0 + 3 * dh) * g.Cout + n_blk * BN + static_cast<int>(rank) * Cfg::BROWS);
          } else {
            const int wtap = ks * taps_per_split + kb / kchunks, kc = kb % kchunks;
            const int tap = g.tap0 + wtap;
            const int dt = tap / 9, dh = (tap / 3) % 3, dw = tap % 3;
            mbar_wait(&empty[stage], phase ^ 1);
            if (!PAIR) mbar_arrive_expect_tx(&full[stage], Cfg::A_STAGE + Cfg::B_STAGE);
            else if (leader) mbar_arrive_expect_tx(&full[stage], 2 * (Cfg::A_STAGE + Cfg::B_STAGE));
            else mbar_arrive_remote(&full[stage], 0);
            const int wrow = wtap * g.Cout + n_blk * BN + static_cast<int>(rank) * Cfg::BROWS;   // PAIR: this CTA's half of the weight tile
#pragma unroll
            for (int s2 = 0; s2 < KS; ++s2) {
              uint8_t* a_dst = sA + stage * Cfg::A_STAGE + s2 * Cfg::A_BYTES;
              uint8_t* b_dst = sB + stage * Cfg::B_STAGE + s2 * Cfg::B_BYTES;
              const int c0 = (kc * KS + s2) * CBK;
              if (PAIR) {
                tma_load_4d_2sm(a_dst, &tmX, &full[stage], c0, w0 + dw, h0 + dh, t0 + dt);
                tma_load_2d_2sm(b_dst, &tmW, &full[stage], c0, wrow);
              } else {
                tma_load_4d(a_dst, &tmX, &full[stage], c0, w0 + dw, h0 + dh, t0 + dt);
                tma_load_2d(b_dst, &tmW, &full[stage], c0, wrow);
              }
            }
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = umma_idesc_bf16(PAIR ? 2 * CBM : CBM, BN);
      // operand descriptors: built ONCE; per stage one add, per MMA a compile-time offset (the start-address field counts
      // 16-byte units and cannot carry out of its 14 bits below 256 KB).  At 128 columns an MMA lasts 64 clk: a descriptor
      // built from scratch for each operand kept the single issuing thread busier than the tensor pipe.
      const uint64_t a_desc0 = umma_desc_sw128(smem_u32(sA)), b_desc0 = umma_desc_sw128(smem_u32(sB));
      const uint64_t slab_row = static_cast<uint64_t>((g.bw * CBK * 2) >> 4);   // SLAB: one h row of the slab, in 16-byte units
      int stage = 0;
      uint32_t phase = 0;
      int t = 0;
      for (int tile = worker; tile < num_tiles; tile += num_workers, ++t) {
        const int as = t & 1;
        const uint32_t aphase = (t >> 1) & 1;
        mbar_wait(&tempty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint64_t a_desc = a_desc0 + static_cast<uint64_t>(stage) * (Cfg::A_STAGE >> 4);
          const uint64_t b_desc = b_desc0 + static_cast<uint64_t>(stage) * (Cfg::B_STAGE >> 4);
          if constexpr (SLAB) {
#pragma unroll
            for (int dh = 0; dh < 3; ++dh) {
              const uint64_t a_tap = a_desc + dh * slab_row;   // tap dh: the tile's rows start dh h-rows into the slab
#pragma unroll
              for (int k = 0; k < CBK / 16; ++k)
                umma_bf16_2cta(d_tmem, a_tap + ((k * 32) >> 4), b_desc + ((dh * Cfg::B_TAP_BYTES + k * 32) >> 4), idesc,
                               (kb | dh | k) != 0 ? 1u : 0u);
            }
            umma_commit_2cta(&empty[stage]);
          } else {
#pragma unroll
            for (int s2 = 0; s2 < KS; ++s2)
#pragma unroll
              for (int k = 0; k < CBK / 16; ++k) {
                const uint64_t ad = a_desc + ((s2 * Cfg::A_BYTES + k * 32) >> 4), bd = b_desc + ((s2 * Cfg::B_BYTES + k * 32) >> 4);
                if (PAIR) umma_bf16_2cta(d_tmem, ad, bd, idesc, (kb | s2 | k) != 0 ? 1u : 0u);
                else umma_bf16(d_tmem, ad, bd, idesc, (kb | s2 | k) != 0 ? 1u : 0u);
              }
            if (PAIR) umma_commit_2cta(&empty[stage]);
            else umma_commit(&empty[stage]);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (PAIR) umma_commit_2cta(&tfull[as]);
        else umma_commit(&tfull[as]);
      }
    }
  } else {
    const int q = warp & 3;
    int t = 0;
    for (int tile = worker; tile < num_tiles; tile += num_workers, ++t) {
      const int ks = tile / num_mn, mn = tile % num_mn;
      const int m_blk = PAIR ? 2 * (mn % num_m) + static_cast<int>(rank) : mn % num_m, n_blk = mn / num_m;
      const int iw = m_blk % g.nw, ih = (m_blk / g.nw) % g.nh, it = m_blk / (g.nw * g.nh);
      const int as = t & 1;
      const uint32_t aphase = (t >> 1) & 1;
      const int m = q * 32 + lane;  // row in tile -> voxel inside the box (w fastest)
      const int vw = iw * g.bw + m % g.bw;
      const int vh = ih * g.bh + (m / g.bw) % g.bh;
      const int vt = it * g.bt + m / (g.bw * g.bh);
      const bool valid = vw < g.W && vh < g.H && vt < g.T;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * BN;
      if (MODE != 0 && MODE != 4) {
        mbar_wait(&tfull[as], aphase);
        tc_fence_after();
      }
      if (MODE == 0 || MODE == 4) {
        // plain conv (+bias, +residual): the accumulator chunk is transposed through a warp-private smem tile (see
        // gemm_epilogue.cuh) so that 8 lanes cover 128 contiguous bytes of one voxel's channels; the lane's 8 voxel
        // offsets are computed once per tile, the residual values are fetched before the first store
        float* stage = epi_stage + (warp - 2) * (EPI_STAGE_BYTES / 4);
        const int cg = lane & 7, rsub = lane >> 3;
        float* outp = ep.out + static_cast<int64_t>(ks) * g.T * g.H * g.W * g.Cout;   // split-K: this group's partial slab
        int64_t voff[8];
        int64_t poff[8];     // MODE 4: the voxel's place in the next conv's padded volume
        float ssv[8];        // MODE 4: running sum of squares of x_new over this lane's channels
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int mm = q * 32 + rsub + 4 * i;
          const int w2 = iw * g.bw + mm % g.bw, h2 = ih * g.bh + (mm / g.bw) % g.bh, t2 = it * g.bt + mm / (g.bw * g.bh);
          voff[i] = (w2 < g.W && h2 < g.H && t2 < g.T) ? ((static_cast<int64_t>(t2) * g.H + h2) * g.W + w2) * g.Cout : -1;
          poff[i] = ((static_cast<int64_t>(t2 + ep.next_tshift) * (g.H + 2) + (h2 + 1)) * (g.W + 2) + (w2 + 1)) * g.Cout;
          ssv[i] = 0.f;
        }
        // the residual values of a chunk are requested one chunk ahead -- the first before the accumulator is even waited
        // for: fetched at the point of use, their latency (x 4 chunks) made this epilogue longer than the main loop of a
        // 128-channel tile (ncu: the issuing thread spent 80 % of its time waiting for a free accumulator)
        float4 xnext[8];
        auto fetch_resid = [&](int c) {
          const int col = n_blk * BN + c * 32 + cg * 4;
#pragma unroll
          for (int i = 0; i < 8; ++i)
            xnext[i] = (ep.resid && voff[i] >= 0 && col < g.Cout) ? *reinterpret_cast<const float4*>(ep.resid + voff[i] + col)
                                                                  : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        fetch_resid(0);
        mbar_wait(&tfull[as], aphase);
        tc_fence_after();
        uint32_t r[32];
        tmem_ld32(taddr, r);
#pragma unroll 1
        for (int c = 0; c < BN / 32; ++c) {
          tmem_ld_wait();
          epi_stage_write(stage, lane, r);
          __syncwarp();
          if (c + 1 < BN / 32) tmem_ld32(taddr + (c + 1) * 32, r);
          const int col = n_blk * BN + c * 32 + cg * 4;
          float4 xin[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) xin[i] = xnext[i];
          if (c + 1 < BN / 32) fetch_resid(c + 1);
          if (col < g.Cout) {
            const float4 bv = ep.bias ? *reinterpret_cast<const float4*>(ep.bias + col) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              if (voff[i] < 0) continue;
              const int rr = rsub + 4 * i;
              const float4 a = reinterpret_cast<const float4*>(stage)[rr * 8 + (cg ^ (rr & 7))];
              const float4 v = make_float4(a.x + bv.x + xin[i].x, a.y + bv.y + xin[i].y, a.z + bv.z + xin[i].z, a.w + bv.w + xin[i].w);
              *reinterpret_cast<float4*>(outp + voff[i] + col) = v;
              if (MODE == 4) ssv[i] += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
            }
          }
          __syncwarp();
        }
        if (MODE == 4) {
          // conv2 of a res block handing over to the next block's conv1: x_new (just stored as fp32, the residual stream)
          // also goes, pixel-normalised / modulated with the NEXT block's (scale1, shift1) / SiLU'd, as bf16 into the
          // interior of the next conv's padded volume.  The 8 lanes that share a voxel combine their partial sums; each lane
          // then re-reads exactly the float4 it stored above (same thread: program order) and writes 8 bytes, 64 contiguous
          // bytes per voxel and chunk.
          auto fetch_x = [&](int c) {   // (xnext is free again: one chunk ahead, as above)
            const int col = c * 32 + cg * 4;
#pragma unroll
            for (int i = 0; i < 8; ++i)
              xnext[i] = (voff[i] >= 0 && col < g.Cout) ? *reinterpret_cast<const float4*>(outp + voff[i] + col) : make_float4(0.f, 0.f, 0.f, 0.f);
          };
          fetch_x(0);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float t = ssv[i];
            t += __shfl_xor_sync(0xffffffffu, t, 1);
            t += __shfl_xor_sync(0xffffffffu, t, 2);
            t += __shfl_xor_sync(0xffffffffu, t, 4);
            ssv[i] = rsqrtf(t / g.Cout + 1e-8f);
          }
#pragma unroll 1
          for (int c = 0; c < BN / 32; ++c) {
            const int col = c * 32 + cg * 4;
            if (col >= g.Cout) break;
            float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ep.next_scale) {
              const float4 t = *reinterpret_cast<const float4*>(ep.next_scale + col);
              sc = make_float4(1.f + t.x, 1.f + t.y, 1.f + t.z, 1.f + t.w);
              sh = *reinterpret_cast<const float4*>(ep.next_shift + col);
            }
            float4 xv[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) xv[i] = xnext[i];
            if (c + 1 < BN / 32) fetch_x(c + 1);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              if (voff[i] < 0) continue;
              const float r0 = ssv[i];
              *reinterpret_cast<uint2*>(ep.next_pad + poff[i] + col) =
                  make_uint2(pack_bf16(silu(xv[i].x * r0 * sc.x + sh.x), silu(xv[i].y * r0 * sc.y + sh.y)),
                             pack_bf16(silu(xv[i].z * r0 * sc.z + sh.z), silu(xv[i].w * r0 * sc.w + sh.w)));
            }
          }
        }
      } else if (MODE == 3) {
        // fused prologue of the next conv (one tile holds all Cout channels of a voxel; thread = voxel): pass 1 sums the
        // squares of (acc + bias) straight from TMEM, pass 2 re-reads TMEM, normalises, modulates, SiLU, packs to bf16 and
        // stores 64 B per 32 channels into the interior of the next padded volume
        const int nch = (g.Cout + 31) / 32;
        float ss = 0.f;
#pragma unroll 1
        for (int c = 0; c < nch; ++c) {
          uint32_t r[32];
          tmem_ld32(taddr + c * 32, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float v = __uint_as_float(r[j]) + ep.bias[c * 32 + j];
            ss += v * v;
          }
        }
        const float rstd = rsqrtf(ss / g.Cout + 1e-8f);
        bf16* dst = ep.next_pad + ((static_cast<int64_t>(vt + ep.next_tshift) * (g.H + 2) + (vh + 1)) * (g.W + 2) + (vw + 1)) * g.Cout;
#pragma unroll 1
        for (int c = 0; c < nch; ++c) {
          uint32_t r[32];
          tmem_ld32(taddr + c * 32, r);
          tmem_ld_wait();
          if (valid) {
            uint32_t pk[16];
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              const int col = c * 32 + j;
              const float sc0 = ep.next_scale ? 1.f + ep.next_scale[col] : 1.f, sc1 = ep.next_scale ? 1.f + ep.next_scale[col + 1] : 1.f;
              const float sh0 = ep.next_shift ? ep.next_shift[col] : 0.f, sh1 = ep.next_shift ? ep.next_shift[col + 1] : 0.f;
              const float a = silu((__uint_as_float(r[j]) + ep.bias[col]) * rstd * sc0 + sh0);
              const float b = silu((__uint_as_float(r[j + 1]) + ep.bias[col + 1]) * rstd * sc1 + sh1);
              pk[j >> 1] = pack_bf16(a, b);
            }
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4)
              *reinterpret_cast<uint4*>(dst + c * 32 + q4 * 8) = make_uint4(pk[4 * q4], pk[4 * q4 + 1], pk[4 * q4 + 2], pk[4 * q4 + 3]);
          }
        }
      } else if (MODE == CONV_EPI_RGB8 || MODE == CONV_EPI_I420) {
        // the first column chunk stays in registers until the second (channels 32-47) is in: one voxel = one whole pixel block
        uint32_t r0[32], r1[32];
        tmem_ld32(taddr, r0);
        tmem_ld32(taddr + 32, r1);
        tmem_ld_wait();
        if (valid) conv_store_frames_u8<MODE>(r0, r1, vt, vh, vw, g, ep);
      } else {
#pragma unroll 1
        for (int c = 0; c < BN / 32; ++c) {
          uint32_t r[32];
          tmem_ld32(taddr + c * 32, r);
          tmem_ld_wait();
          if (valid) conv_epilogue_chunk<MODE>(r, vt, vh, vw, n_blk * BN + c * 32, g, ep);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_remote(&tempty[as], 0);
        else mbar_arrive(&tempty[as]);
      }
    }
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all();
  else __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    if (PAIR) tmem_dealloc_2cta<Cfg::TMEM_COLS>(tmem_base);
    else tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

template <int BN, int MODE, int KS>
__global__ void __launch_bounds__(CONV_THREADS, 1)
conv3d_tcgen05(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW, const ConvGeom g,
               const ConvEpi ep) {
  conv3d_body<BN, MODE, KS, false>(tmX, tmW, g, ep);
}

template <int BN, int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(CONV_THREADS, 1)
conv3d_slab_tcgen05(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW, const ConvGeom g,
                    const ConvEpi ep) {
  conv3d_body<BN, MODE, 1, true, true>(tmX, tmW, g, ep);
}

template <int BN, int MODE, int KS>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(CONV_THREADS, 1)
conv3d_pair_tcgen05(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW, const ConvGeom g,
                    const ConvEpi ep) {
  conv3d_body<BN, MODE, KS, true>(tmX, tmW, g, ep);
}

// ---------------------------------------------------------------------------------------------
// Padding prologue: one warp per padded voxel.
// mode 0: copy ; 1: x*a[c] + b[c] ; 2: silu(x / sqrt(mean_c x^2 + 1e-8) * (1 + a[c]) + b[c]) (a, b nullable: plain
// pixel-norm + SiLU, the encoder's res block) ; 3: silu(x*a[c] + b[c]) (GroupNorm folded into a per-channel affine + SiLU)
// pad: bit 0 causal (two leading frame copies instead of one leading + one trailing), bit 1 zero spatial padding instead
// of reflect (the encoder, V/VideoEncoder.swift:226-227), bit 2 zero temporal padding (MLX Conv3d padding: 1, the upscaler)
// ---------------------------------------------------------------------------------------------
// (x, a, b are produced by preceding kernels: no const __restrict__, see griddep_wait in ptx.cuh)
// VPL = float4 per lane per voxel (C <= 128 * VPL); a warp keeps U = 8 / VPL voxels in flight so that 8 independent 16-byte
// loads per lane are outstanding (one voxel per warp iteration was latency-bound at 1.8 TB/s), reads each voxel once
// (registers between the channel reduction and the output) and reduces the U sums of squares together.
template <int VPL>
__global__ void __launch_bounds__(256) vae_prep_kernel(const float* x, bf16* out, int T, int H, int W, int C, int mode,
                                                        const float* a, const float* b, int pad) {
  griddep_launch();
  griddep_wait();
  constexpr int U = VPL >= 8 ? 1 : 8 / VPL;
  const int tshift = (pad & 1) ? 2 : 1;
  const bool zero_hw = (pad & 2) != 0, zero_t = (pad & 4) != 0;
  const int lane = threadIdx.x & 31;
  const int64_t nvox = static_cast<int64_t>(T + 2) * (H + 2) * (W + 2);
  const int64_t wid0 = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int nv = C >> 2;
  float4 av[VPL], bv[VPL];   // per-channel scale / shift: the same for every voxel
#pragma unroll
  for (int k = 0; k < VPL; ++k) {
    const int i = lane + 32 * k;
    av[k] = bv[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (mode != 0 && a != nullptr && i < nv) { av[k] = reinterpret_cast<const float4*>(a)[i]; bv[k] = reinterpret_cast<const float4*>(b)[i]; }
  }
  for (int64_t pv0 = wid0 * U; pv0 < nvox; pv0 += nwarps * U) {
    float4 v[U][VPL];
    bool zero[U];   // padding voxel of a zero-padded axis: written as 0 (after the activation, like the conv's own padding)
    // coordinates of the first voxel by 32-bit division (the launcher checks nvox < 2^31; 64-bit divisions -- three per voxel,
    // ~100 instructions each, redundantly on every lane -- made the 128-channel prologue issue-bound at 1.85 TB/s), the
    // following U - 1 by stepping
    const uint32_t p0 = static_cast<uint32_t>(pv0), Wp = static_cast<uint32_t>(W + 2), Hp = static_cast<uint32_t>(H + 2);
    int pw = static_cast<int>(p0 % Wp), ph = static_cast<int>((p0 / Wp) % Hp), pt = static_cast<int>(p0 / (Wp * Hp));
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t pv = pv0 + u;
      if (u > 0 && ++pw == W + 2) {
        pw = 0;
        if (++ph == H + 2) { ph = 0; ++pt; }
      }
      int ws = pw - 1, hs = ph - 1, ts = pt - (zero_t ? 1 : tshift);
      zero[u] = (zero_hw && (ws < 0 || ws >= W || hs < 0 || hs >= H)) || (zero_t && (ts < 0 || ts >= T));
      ws = ws < 0 ? -ws : (ws >= W ? 2 * W - 2 - ws : ws);   // reflect (VideoConvolution.swift:257-266)
      hs = hs < 0 ? -hs : (hs >= H ? 2 * H - 2 - hs : hs);
      ts = ts < 0 ? 0 : (ts >= T ? T - 1 : ts);              // frame replication (:281-294)
      if (zero[u]) { ws = 0; hs = 0; ts = 0; }
      const float4* src = reinterpret_cast<const float4*>(x + ((static_cast<int64_t>(ts) * H + hs) * W + ws) * C);
#pragma unroll
      for (int k = 0; k < VPL; ++k) {
        const int i = lane + 32 * k;
        v[u][k] = (pv < nvox && i < nv && !zero[u]) ? src[i] : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    float rs[U];
#pragma unroll
    for (int u = 0; u < U; ++u) rs[u] = 1.0f;
    if (mode == 2) {
      float ss[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        ss[u] = 0.f;
#pragma unroll
        for (int k = 0; k < VPL; ++k) ss[u] += v[u][k].x * v[u][k].x + v[u][k].y * v[u][k].y + v[u][k].z * v[u][k].z + v[u][k].w * v[u][k].w;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int u = 0; u < U; ++u) ss[u] += __shfl_xor_sync(0xffffffffu, ss[u], o);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) rs[u] = rsqrtf(ss[u] / C + 1e-8f);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t pv = pv0 + u;
      if (pv >= nvox) break;
      uint2* dst = reinterpret_cast<uint2*>(out + pv * C);
#pragma unroll
      for (int k = 0; k < VPL; ++k) {
        const int i = lane + 32 * k;
        if (i >= nv) break;
        float4 o = v[u][k];
        if (mode == 1) {
          o.x = o.x * av[k].x + bv[k].x; o.y = o.y * av[k].y + bv[k].y; o.z = o.z * av[k].z + bv[k].z; o.w = o.w * av[k].w + bv[k].w;
        } else if (mode == 2) {
          o.x = silu(o.x * rs[u] * (1.f + av[k].x) + bv[k].x);
          o.y = silu(o.y * rs[u] * (1.f + av[k].y) + bv[k].y);
          o.z = silu(o.z * rs[u] * (1.f + av[k].z) + bv[k].z);
          o.w = silu(o.w * rs[u] * (1.f + av[k].w) + bv[k].w);
        } else if (mode == 3) {
          o.x = silu(o.x * av[k].x + bv[k].x); o.y = silu(o.y * av[k].y + bv[k].y);
          o.z = silu(o.z * av[k].z + bv[k].z); o.w = silu(o.w * av[k].w + bv[k].w);
        }
        if (zero[u]) o = make_float4(0.f, 0.f, 0.f, 0.f);
        dst[i] = make_uint2(pack_bf16(o.x, o.y), pack_bf16(o.z, o.w));
      }
    }
  }
}

// out = sum_ks partial[ks] + bias (+ resid), fixed summation order (deterministic); float4 over [V, Cout]
__global__ void conv_splitk_reduce_kernel(const float* part, int ksplit, int64_t slab4, int C4, const float* bias, const float* resid,
                                          float* out) {
  griddep_launch();
  griddep_wait();
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < slab4;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float4 a = reinterpret_cast<const float4*>(part)[i];
    for (int k = 1; k < ksplit; ++k) {
      const float4 b = reinterpret_cast<const float4*>(part)[k * slab4 + i];
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    const float4 bv = reinterpret_cast<const float4*>(bias)[i % C4];
    a.x += bv.x; a.y += bv.y; a.z += bv.z; a.w += bv.w;
    if (resid) {
      const float4 r = reinterpret_cast<const float4*>(resid)[i];
      a.x += r.x; a.y += r.y; a.z += r.z; a.w += r.w;
    }
    reinterpret_cast<float4*>(out)[i] = a;
  }
}

// Padding voxels of a bf16 padded volume from its interior (see launch_vae_halo_fill); one warp per padding voxel.
// Only the padding voxels are enumerated (a scan over the whole padded volume with an interior test spent ~50 us per call at
// the 128-channel stage, 10 x the bytes it moves): first the whole time-padding frames, then, per interior frame, the top and
// bottom rows and the two end columns.  t0 = index of the first interior frame.
__global__ void __launch_bounds__(256) vae_halo_fill_kernel(bf16* vol, int T, int H, int W, int C, int pad) {
  griddep_launch();
  griddep_wait();
  const int tshift = (pad & 1) ? 2 : 1;
  const bool zero_hw = (pad & 2) != 0, zero_t = (pad & 4) != 0;
  const int lane = threadIdx.x & 31;
  const int Hp = H + 2, Wp = W + 2, t0 = zero_t ? 1 : tshift;
  const int frame = Hp * Wp, n_a = 2 * frame, n_border = 2 * Wp + 2 * H;
  const int n_halo = n_a + T * n_border;
  const int wid0 = static_cast<int>((blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5);
  const int nwarps = static_cast<int>((static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5);
  const int nv = C >> 3;   // uint4 = 8 bf16
  for (int idx = wid0; idx < n_halo; idx += nwarps) {
    int pt, ph, pw;
    if (idx < n_a) {
      const int f = idx / frame, r = idx - f * frame;
      pt = f < t0 ? f : f + T;
      ph = r / Wp;
      pw = r - ph * Wp;
    } else {
      const int j = idx - n_a, f = j / n_border, e = j - f * n_border;
      pt = t0 + f;
      if (e < Wp) { ph = 0; pw = e; }
      else if (e < 2 * Wp) { ph = Hp - 1; pw = e - Wp; }
      else { const int e2 = e - 2 * Wp; ph = 1 + (e2 >> 1); pw = (e2 & 1) ? Wp - 1 : 0; }
    }
    int ws = pw - 1, hs = ph - 1, ts = pt - t0;
    const bool zero = (zero_hw && (ws < 0 || ws >= W || hs < 0 || hs >= H)) || (zero_t && (ts < 0 || ts >= T));
    ws = ws < 0 ? -ws : (ws >= W ? 2 * W - 2 - ws : ws);
    hs = hs < 0 ? -hs : (hs >= H ? 2 * H - 2 - hs : hs);
    ts = ts < 0 ? 0 : (ts >= T ? T - 1 : ts);
    const int tpad = ts + t0;
    const uint4* src = reinterpret_cast<const uint4*>(vol + ((static_cast<int64_t>(tpad) * Hp + hs + 1) * Wp + ws + 1) * C);
    uint4* dst = reinterpret_cast<uint4*>(vol + ((static_cast<int64_t>(pt) * Hp + ph) * Wp + pw) * C);
    for (int i = lane; i < nv; i += 32) dst[i] = zero ? make_uint4(0u, 0u, 0u, 0u) : src[i];
  }
}

int best_pow2(int extent, int budget) {
  // power of two <= budget that wastes the least of `extent` when tiling; ties -> larger
  int best = 1;
  double best_u = 0.0;
  for (int b = 1; b <= budget; b <<= 1) {
    const int tiles = (extent + b - 1) / b;
    const double u = static_cast<double>(extent) / (static_cast<double>(tiles) * b);
    if (u >= best_u - 1e-9) { best_u = u; best = b; }
  }
  return best;
}

template <int BN, int MODE, int KS>
void conv_launch_ks(const CUtensorMap& tmX, const CUtensorMap& tmW, const ConvGeom& g, const ConvEpi& ep, cudaStream_t s) {
  using Cfg = ConvCfg<BN, KS>;
  auto kern = conv3d_tcgen05<BN, MODE, KS>;
  ensure_dyn_smem(kern, Cfg::SMEM);
  const int tiles = g.nt * g.nh * g.nw * ((g.Cout + BN - 1) / BN) * g.ksplit;
  const int grid = tiles < device_sm_count() ? tiles : device_sm_count();
  launch_pdl(PDL_VAE, kern, dim3(grid), dim3(CONV_THREADS), Cfg::SMEM, s, tmX, tmW, g, ep);
  LTX_CUDA(cudaGetLastError());
}

// CTA pairs: one work item = two adjacent voxel tiles x one channel tile (x one tap group); a cluster per SM pair
template <int BN, int MODE>
void conv_launch_pair(const CUtensorMap& tmX, const CUtensorMap& tmW, const ConvGeom& g, const ConvEpi& ep, cudaStream_t s) {
  using Cfg = ConvCfg<BN, 2, true>;
  auto kern = conv3d_pair_tcgen05<BN, MODE, 2>;
  ensure_dyn_smem(kern, Cfg::SMEM);
  const int items = ((g.nt * g.nh * g.nw + 1) / 2) * ((g.Cout + BN - 1) / BN) * g.ksplit;
  const int clusters = device_sm_count() / 2;
  const int grid = 2 * (items < clusters ? items : clusters);
  launch_pdl(PDL_VAE, kern, dim3(grid), dim3(CONV_THREADS), Cfg::SMEM, s, tmX, tmW, g, ep);
  LTX_CUDA(cudaGetLastError());
}

template <int BN, int MODE>
void conv_launch_slab(const CUtensorMap& tmX, const CUtensorMap& tmW, const ConvGeom& g, const ConvEpi& ep, cudaStream_t s) {
  if constexpr (BN <= 128) {
    using Cfg = ConvCfg<BN, 1, true, true>;
    auto kern = conv3d_slab_tcgen05<BN, MODE>;
    ensure_dyn_smem(kern, Cfg::SMEM);
    const int items = ((g.nt * g.nh * g.nw + 1) / 2) * ((g.Cout + BN - 1) / BN) * g.ksplit;
    const int clusters = device_sm_count() / 2;
    const int grid = 2 * (items < clusters ? items : clusters);
    launch_pdl(PDL_VAE, kern, dim3(grid), dim3(CONV_THREADS), Cfg::SMEM, s, tmX, tmW, g, ep);
    LTX_CUDA(cudaGetLastError());
  } else {
    LTX_CHECK(false, 2, "conv3d: slab stages are for tiles up to 128 columns");
  }
}

template <int BN, int MODE>
void conv_launch(const CUtensorMap& tmX, const CUtensorMap& tmW, const ConvGeom& g, const ConvEpi& ep, cudaStream_t s, bool pair) {
  if (g.slab) { conv_launch_slab<BN, MODE>(tmX, tmW, g, ep, s); return; }
  // 128-channel stages where they fit: tiles up to 128 columns (3 / 4 stages of 64 / 48 KB stay in flight) and whole pairs of chunks
  if (pair) conv_launch_pair<BN, MODE>(tmX, tmW, g, ep, s);
  else if (BN <= 128 && g.Cin % (2 * CBK) == 0) conv_launch_ks<BN, MODE, (BN <= 128 ? 2 : 1)>(tmX, tmW, g, ep, s);
  else conv_launch_ks<BN, MODE, 1>(tmX, tmW, g, ep, s);
}

template <int BN>
void conv_launch_mode(const CUtensorMap& tmX, const CUtensorMap& tmW, const ConvGeom& g, const ConvEpi& ep, cudaStream_t s, bool pair) {
  switch (ep.mode) {
    case 0: conv_launch<BN, 0>(tmX, tmW, g, ep, s, pair); break;
    case 1: conv_launch<BN, 1>(tmX, tmW, g, ep, s, pair); break;
    case 2: conv_launch<BN, 2>(tmX, tmW, g, ep, s, pair); break;
    case 3: conv_launch<BN, 3>(tmX, tmW, g, ep, s, pair); break;
    case 4: conv_launch<BN, 4>(tmX, tmW, g, ep, s, pair); break;
    case CONV_EPI_RGB8:
    case CONV_EPI_I420:
      // Cout = 48 always plans 64-wide tiles: the 8-bit stores are only instantiated there
      if constexpr (BN == 64) {
        if (ep.mode == CONV_EPI_RGB8) conv_launch<BN, CONV_EPI_RGB8>(tmX, tmW, g, ep, s, pair);
        else conv_launch<BN, CONV_EPI_I420>(tmX, tmW, g, ep, s, pair);
      } else {
        LTX_CHECK(false, 2, "conv3d: 8-bit frame stores need 64-wide tiles");
      }
      break;
    default: LTX_CHECK(false, 2, "bad conv epilogue mode");
  }
}

// LTX_CONV_SLAB=0: per-tap A boxes also for tiles up to 128 columns (read per call, as LTX_CONV_PAIR)
bool conv_slab_enabled() {
  const char* e = getenv("LTX_CONV_SLAB");
  return e ? atoi(e) != 0 : true;
}

// LTX_CONV_PAIR (read per call: the parity tests run both forms): 0 = one CTA per voxel tile, default = CTA pairs whenever the
// input channels come in 128-channel stages
bool conv_pair_enabled() {
  const char* e = getenv("LTX_CONV_PAIR");
  return e ? atoi(e) != 0 : true;
}

}  // namespace

bool conv3d_wants_tap_split(int H, int W, int Cin, int Cout) {
  return H * W <= 1024 && Cout >= 256 && Cout % 4 == 0 && static_cast<int64_t>(27) * Cin >= 8192;
}

// Everything launch_conv3d decides from the shape, as a pure function (also behind ltx_conv3d_plan for the host-side tests).
// Two of the decisions change the ORDER in which the taps are added up -- slab stages and the tap split -- and so must never
// depend on T: a temporal shard of a clip has to round exactly like the whole clip (tests/test_host.py holds the rule to that).
ConvPlan conv3d_plan(int T, int H, int W, int Cin, int Cout, int mode, int ntaps, bool scratch_ok, int sm_count, bool pair_on,
                     bool slab_on) {
  ConvPlan p;
  p.bw = best_pow2(W, 128);
  p.bh = best_pow2(H, 128 / p.bw);
  p.bt = 128 / (p.bw * p.bh);
  p.ksplit = 1;
  p.slab = 0;
  // tile width: 256 when that still gives every SM a tile, else 128 (the 1024-channel stage of a 25-frame decode has only
  // 12 voxel tiles: 48 tiles of 256 channels leave two thirds of the SMs idle); 64 for the narrow output conv (128 -> 48)
  const int m_tiles = ((T + p.bt - 1) / p.bt) * ((H + p.bh - 1) / p.bh) * ((W + p.bw - 1) / p.bw);
  p.bn = Cout >= 256 ? 256 : (Cout > 64 ? 128 : 64);
  // Tile-starved convs (the 1024-channel stage of a 25-frame decode has 12 voxel tiles x 4 channel tiles for 148 SMs, each
  // 27 x 1024 deep): split the taps into 3 groups (one per dt) -> 3x the work items at full tile width; the partial sums go to
  // a scratch slab each and are added in a fixed order by a small reduction pass (+ bias, + residual).
  // The rule looks at the frame geometry and the channel counts only -- never at T.
  const bool can_split = mode == 0 && ntaps == 27 && scratch_ok && conv3d_wants_tap_split(H, W, Cin, Cout);
  if (can_split) p.ksplit = 3;
  else if (mode != 3 && mode != 4 && p.bn == 256 && m_tiles * ((Cout + 255) / 256) < sm_count * 2 / 3) p.bn = 128;   // (measured: 128-wide tiles
  // cost ~0.7 of a 256-wide one, so they only pay when 256 leaves most SMs without a tile; same summation order either way)
  p.pair = (pair_on && Cin % (2 * CBK) == 0 && sm_count >= 2) ? 1 : 0;
  if (p.pair && Cout < 256 && slab_on) {
    // slab stages: one frame per tile (bt = 1), [bh, bw] voxels with bw a multiple of the 8-row swizzle atom; fewest tiles
    // first, then fewest slab rows.  Slab stages add the taps up in another order than the per-tap stages, so the choice
    // between them must not look at T: Cout < 256 -- NOT the tile width, which the tile-starved rule above narrows for short
    // shards -- and H, W only.
    int bbh = 0, bbw = 0;
    int64_t btiles = 0, brows = 0;
    for (int bw = 32; bw >= 8; bw >>= 1) {
      const int bh = 128 / bw;
      const int64_t tiles = static_cast<int64_t>((W + bw - 1) / bw) * ((H + bh - 1) / bh), rows = static_cast<int64_t>(bh + 2) * bw;
      if (bbw == 0 || tiles < btiles || (tiles == btiles && rows < brows)) { bbh = bh; bbw = bw; btiles = tiles; brows = rows; }
    }
    p.slab = 1; p.bt = 1; p.bh = bbh; p.bw = bbw;
  }
  return p;
}

bool conv3d_pair_default() { return conv_pair_enabled(); }
bool conv3d_slab_default() { return conv_slab_enabled(); }

void launch_conv3d(const bf16* x_pad, const bf16* w, int T, int H, int W, int Cin, int Cout, const ConvEpi& epi_in,
                   cudaStream_t s, int ntaps, float* splitk_scratch, size_t splitk_scratch_bytes) {
  ConvEpi epi = epi_in;
  LTX_CHECK(T > 0 && H > 1 && W > 1, 2, "conv3d: bad volume (reflect padding needs H, W >= 2)");
  LTX_CHECK(ntaps == 27 || ntaps == 9, 2, "conv3d: 27 taps (3x3x3) or 9 taps (per-frame 3x3)");
  LTX_CHECK(Cin > 0 && Cin % 64 == 0 && Cout > 0, 2, "conv3d: Cin must be a positive multiple of 64");
  LTX_CHECK(epi.mode >= 0 && epi.mode <= CONV_EPI_I420, 2, "bad conv epilogue mode");
  const bool u8 = epi.mode == CONV_EPI_RGB8 || epi.mode == CONV_EPI_I420;
  LTX_CHECK(epi.mode == 3 || (u8 ? epi.out_u8 != nullptr : epi.out != nullptr), 2, "conv3d: no output buffer");
  LTX_CHECK(!u8 || (Cout == 48 && ntaps == 27 && reinterpret_cast<uintptr_t>(epi.out_u8) % 4 == 0), 2,
            "conv3d: 8-bit frame stores need Cout = 48 and a 4-byte aligned output");
  LTX_CHECK(epi.mode != 0 || Cout % 4 == 0, 2, "conv3d: Cout must be a multiple of 4");
  LTX_CHECK(epi.mode != 1 || (Cout % 32 == 0 && Cin % 8 == 0 && epi.resid != nullptr && (epi.t_shift == 0 || epi.t_shift == 1)), 2,
            "conv3d: bad d2s configuration");
  // the unpatchify store writes frame channel co >> 4 of a 3-channel frame
  LTX_CHECK(epi.mode != 2 || Cout == 48, 2, "conv3d: the unpatchify epilogue needs Cout = 48 (3 channels x 4 x 4)");
  LTX_CHECK(epi.mode != 4 || (epi.resid != nullptr && epi.out != nullptr), 2, "conv3d: mode 4 needs the residual stream");
  LTX_CHECK((epi.mode != 3 && epi.mode != 4) || (Cout % 32 == 0 && Cout <= 256 && Cout > 64 && epi.next_pad != nullptr && ntaps == 27), 2,
            "conv3d: the fused-prologue epilogue needs 64 < Cout <= 256 (one tile = all channels of a voxel)");
  LTX_CHECK((epi.mode != 3 && epi.mode != 4) ||
                ((epi.next_tshift == 1 || epi.next_tshift == 2) && (epi.next_scale == nullptr) == (epi.next_shift == nullptr)),
            2, "conv3d: fused-prologue epilogue needs next_tshift 1 or 2 and both or neither of next_scale / next_shift");
  const size_t slab = static_cast<size_t>(T) * H * W * Cout * 4;
  const bool scratch_ok = splitk_scratch != nullptr && 3 * slab <= splitk_scratch_bytes;
  const ConvPlan pl = conv3d_plan(T, H, W, Cin, Cout, epi.mode, ntaps, scratch_ok, device_sm_count(), conv_pair_enabled(), conv_slab_enabled());
  // only the mode-0 / mode-4 store of an unsplit conv can do without a bias
  LTX_CHECK(epi.bias != nullptr || ((epi.mode == 0 || epi.mode == 4) && pl.ksplit == 1), 2, "conv3d: no bias");
  ConvGeom g;
  g.T = T; g.H = H; g.W = W; g.Cin = Cin; g.Cout = Cout;
  g.bt = pl.bt; g.bh = pl.bh; g.bw = pl.bw;
  g.nt = (T + g.bt - 1) / g.bt; g.nh = (H + g.bh - 1) / g.bh; g.nw = (W + g.bw - 1) / g.bw;
  g.ntaps = ntaps; g.tap0 = ntaps == 9 ? 9 : 0;
  g.ksplit = pl.ksplit;
  g.slab = pl.slab;
  const int bn = pl.bn;
  const bool pair = pl.pair != 0;
  const float* final_bias = epi.bias;
  const float* final_resid = epi.resid;
  float* final_out = epi.out;
  if (g.ksplit > 1) { epi.out = splitk_scratch; epi.bias = nullptr; epi.resid = nullptr; }
  LTX_CHECK((epi.mode != 3 && epi.mode != 4) || bn >= Cout, 2, "conv3d: fused-prologue epilogue needs the whole channel range in one tile");
  CUtensorMap tmX = make_tmap_thwc(x_pad, T + 2, H + 2, W + 2, Cin, g.bt, g.slab ? g.bh + 2 : g.bh, g.bw);
  CUtensorMap tmW = make_tmap_2d(w, static_cast<uint64_t>(ntaps) * Cout, Cin, Cin, pair ? bn / 2 : bn);   // pair: each CTA stages half a weight tile
  if (bn == 256)
    conv_launch_mode<256>(tmX, tmW, g, epi, s, pair);
  else if (bn == 128)
    conv_launch_mode<128>(tmX, tmW, g, epi, s, pair);
  else
    conv_launch_mode<64>(tmX, tmW, g, epi, s, pair);
  if (g.ksplit > 1) {
    const int64_t slab4 = static_cast<int64_t>(slab / 16);
    int64_t blocks = (slab4 + 255) / 256;
    if (blocks > device_sm_count() * 8) blocks = device_sm_count() * 8;
    launch_pdl(PDL_VAE, conv_splitk_reduce_kernel, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, s, splitk_scratch, g.ksplit, slab4,
               Cout / 4, final_bias, final_resid, final_out);
    LTX_CUDA(cudaGetLastError());
  }
}

void launch_vae_halo_fill(bf16* vol, int T, int H, int W, int C, int pad, cudaStream_t s) {
  LTX_CHECK(C % 8 == 0 && T > 0 && H > 1 && W > 1, 2, "vae_halo_fill: bad shape");
  LTX_CHECK(pad >= 0 && pad <= 7, 2, "vae_halo_fill: pad takes the VAE_PAD_* bits only");
  // work = the padding voxels only; a warp per voxel
  const int64_t nvox = 2 * static_cast<int64_t>(H + 2) * (W + 2) + static_cast<int64_t>(T) * (2 * (W + 2) + 2 * H);
  LTX_CHECK(nvox < (1ll << 30), 2, "vae_halo_fill: volume too large");
  int64_t blocks = (nvox + 7) / 8;
  const int64_t cap = static_cast<int64_t>(device_sm_count()) * 16;
  if (blocks > cap) blocks = cap;
  launch_pdl(PDL_VAE, vae_halo_fill_kernel, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, s, vol, T, H, W, C, pad);
  LTX_CUDA(cudaGetLastError());
}

void launch_vae_prep(const float* x, bf16* out, int T, int H, int W, int C, int mode, const float* a, const float* b,
                     int pad, cudaStream_t s) {
  LTX_CHECK(C % 4 == 0 && C <= 2048 && T > 0 && H > 1 && W > 1, 2, "vae_prep: bad shape (C must be a multiple of 4, at most 2048)");
  LTX_CHECK(mode >= 0 && mode <= 3 && pad >= 0 && pad <= 7, 2, "vae_prep: bad mode or pad bits");
  // modes 1 / 3 read both tables; mode 2 reads both or neither (a != NULL selects the modulation)
  LTX_CHECK(mode == 0 || (a != nullptr && b != nullptr) || (mode == 2 && a == nullptr && b == nullptr), 2, "vae_prep: bad scale / shift tables");
  const int64_t nvox = static_cast<int64_t>(T + 2) * (H + 2) * (W + 2);
  LTX_CHECK(nvox < (1ll << 31), 2, "vae_prep: volume too large");
  int64_t blocks = (nvox + 7) / 8;
  const int64_t cap = static_cast<int64_t>(device_sm_count()) * 16;
  if (blocks > cap) blocks = cap;
  const dim3 gr(static_cast<int>(blocks)), bl(256);
  const int ts = pad;
  if (C <= 128) launch_pdl(PDL_VAE, vae_prep_kernel<1>, gr, bl, 0, s, x, out, T, H, W, C, mode, a, b, ts);
  else if (C <= 256) launch_pdl(PDL_VAE, vae_prep_kernel<2>, gr, bl, 0, s, x, out, T, H, W, C, mode, a, b, ts);
  else if (C <= 512) launch_pdl(PDL_VAE, vae_prep_kernel<4>, gr, bl, 0, s, x, out, T, H, W, C, mode, a, b, ts);
  else if (C <= 1024) launch_pdl(PDL_VAE, vae_prep_kernel<8>, gr, bl, 0, s, x, out, T, H, W, C, mode, a, b, ts);
  else launch_pdl(PDL_VAE, vae_prep_kernel<16>, gr, bl, 0, s, x, out, T, H, W, C, mode, a, b, ts);
  LTX_CUDA(cudaGetLastError());
}

}  // namespace ltx
