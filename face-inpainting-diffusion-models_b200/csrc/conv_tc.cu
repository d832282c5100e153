// K1: 3x3 / 1x1 convolution as implicit GEMM on the 5th-generation tensor cores (tcgen05).
//
//   D[M = B*H*W pixels, N = Cout] = sum over taps (r,s) and 64-channel slices of
//                                   A_{r,s}[M, 64] * W[N, (r,s), 64]^T         (bf16 x bf16 -> fp32)
//
// Replaces cuDNN's implicit-GEMM behind every conv_nd of the reference (nn.py:102,153,176,182,184,
// 252,254; unet.py:55,151).  Design:
//   * An M tile is a TW x TH x TN box of output pixels (TW*TH*TN = 128).  For tap (r,s) the A operand
//     is the same box of the NHWC input shifted by (r-1, s-1); one 4-D TMA box load fetches it, the
//     hardware zero-fills the out-of-image halo (= the conv's zero padding) and writes 128 rows of
//     64 bf16 with the 128-byte swizzle -- exactly the canonical K-major UMMA operand.  No im2col
//     buffer ever exists.
//   * The weight slice [BLOCK_N][64] for (tap, channel slice) is a 2-D TMA box of the KRSC matrix.
//   * 320 threads: warps 0-7 = epilogue (two warpgroups), warp 8 = TMA producer, warp 9 = MMA issuer (one thread issues
//     tcgen05.mma, accumulators live in TMEM, double-buffered so the epilogue of tile i overlaps the MMAs of tile i+1).
//     Epilogue: tcgen05.ld (one pixel row per thread) -> + bias[c] + emb[n][c] + residual -> bf16 -> swizzled smem ->
//     TMA store (zero-copy into channel slices of concat buffers through the tensor map strides), or fp32 NCHW stores
//     for the 6-channel head.
//   * The producer and the MMA issuer are single threads: their loops carry the tap / channel-slice position
//     incrementally and divide by launch constants with FastDiv (a runtime `/` in the producer loop paced every K loop
//     at 330-430 ns per 64-deep block against 270 ns of MMAs; tools/lowres_timeline.py).
//   * An optional second (activation, weight) pair is accumulated as extra K iterations: the 1x1
//     skip_connection of channel-changing ResBlocks (nn.py:184,212) costs no extra pass.
//   * Persistent CTAs (one per SM), static tile striding; tiles that share an M box are adjacent
//     so their A boxes hit L2.
//   * Low-resolution layers (few pixel tiles, deep K) split the K loop of a tile over the 2 / 4 / 8 CTAs of a
//     thread-block cluster: partials parked in an L2-resident workspace, one cluster barrier, every CTA folds (split
//     order: bit-reproducible) and finishes 128 / S rows -- cluster_fold_store below.
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"
#include "conv_epilogue.cuh"
#include "conv_host.cuh"
#include "sm100_primitives.cuh"

namespace fidm {
using namespace sm100;

struct ConvTcParams {
  int B, H, W;             // OUTPUT spatial size
  int stride;              // 1, or 2: input is 2H x 2W and tap (r,s) of output pixel (h,w) reads input (2h + r - 1, 2w + s - 1)
  int TW, TH, TN;          // pixel box of one M tile
  int tiles_w, tiles_h, tiles_n;
  int n_blocks;            // Cout / BLOCK_N
  int ksize, kc1, cin1;    // taps = ksize^2, kc1 = Cin/64
  int kc2;                 // Cin2/64 (0: no second source)
  int ab_f16;              // primary A/B operands are fp16 (normalized activations), else bf16
  const float* bias;
  const float* row_add; int ld_row_add;
  const __nv_bfloat16* residual; int ld_res;
  float* y_nchw; int cout_valid;   // non-null: fp32 NCHW output of the first cout_valid channels
  float* colsum; int colsum_slots; int cout;   // optional fused GroupNorm column sums
  int split_k;             // >1: the K loop of every tile is split over split_k CTAs (low-resolution layers)
  float* sk_ws; int* sk_cnt;   // fp32 partial tiles [tile][split][BLOCK_N][128], per-tile arrival counters
  int cluster_split;           // 1: the split_k CTAs of a tile form a thread-block cluster (split_k in {2, 4, 8}, grid ==
                               // units) and share the fold behind a cluster barrier; 0: arrival counter, last CTA folds
  __nv_bfloat16* y_out; int ld_y;   // cluster_split: NHWC output written with plain 16-byte stores
  int tw_sh, th_sh;            // log2 of TW, TH
  FastDiv fd_split, fd_nblocks, fd_tw, fd_th, fd_kc1, fd_ks;   // divisors: split_k, n_blocks, tiles_w, tiles_h, kc1, ksize
  unsigned long long* prof;    // probe only (tools/lowres_timeline.py): [CTA][32] globaltimer stamps of the first work unit
};

__device__ __forceinline__ unsigned long long gtime_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// L1 prefetch of an epilogue operand (bias / emb / residual): the epilogues consume them group by group, each group a
// dependent L2 round trip (~0.4 us) on the tail of a launch; prefetched while the accumulator / the partial tiles are
// still in flight, the later loads hit L1.
__device__ __forceinline__ void prefetch_l1(const void* ptr) { asm volatile("prefetch.global.L1 [%0];" ::"l"(ptr)); }
#define TL(i) do { if (p.prof) p.prof[32 * blockIdx.x + (i)] = gtime_ns(); } while (0)
#define TL1(i) do { if (p.prof && wu == unit) p.prof[32 * blockIdx.x + (i)] = gtime_ns(); } while (0)

constexpr int kEpiWarps = 8;            // two warpgroups: chunk ch of a tile is drained by warpgroup (ch & 1)
constexpr long long kSplitCounterBytes = 65536;
constexpr int kThreads = 320;            // 8 epilogue warps, warp 8 = TMA producer, warp 9 = MMA issuer
constexpr int kABytes = 128 * 128;                 // 128 rows x 64 bf16
constexpr int kStagingBytes = 128 * 128;           // one 128 x 64 bf16 output chunk

// CG = 1: one CTA per 128 x BLOCK_N tile.  CG = 2: a CTA pair (cta_group::2) owns a 256 x BLOCK_N tile; each
// CTA stages its own 128 pixel rows of A and HALF of the weight tile, which cuts the shared-memory traffic
// per MMA from 48 KB to 32 KB per 64-deep K block -- the 1-CTA kernel is shared-memory-bandwidth bound
// (48 KB written by TMA + 48 KB read by the tensor core every 512 cycles = 192 B/clk/SM).
template <int BLOCK_N, int CG> struct ConvCfg {
  static constexpr int kBRows = BLOCK_N / CG;
  static constexpr int kBBytes = kBRows * 128;
  static constexpr int kStageBytes = kABytes + (kBBytes < 1024 ? 1024 : kBBytes);
  static constexpr int kStages = (192 * 1024) / kStageBytes > 8 ? 8 : (192 * 1024) / kStageBytes;
  static constexpr int kTmemCols = 2 * BLOCK_N < 32 ? 32 : 2 * BLOCK_N;
  static constexpr int kSmemBytes = kStages * kStageBytes + 2 * kStagingBytes + 256 + 1024;
};

// Cluster split-K, second half: CTA `rank` of the cluster folds rows [rank * 128 / S, (rank + 1) * 128 / S) of the S
// partial tiles (fp32 [BLOCK_N][128] column-major in the L2-resident workspace, made visible by the cluster barrier)
// in split order -- the same fixed summation order whichever CTA does it -- and finishes them: + bias + emb + residual
// -> bf16 -> 16-byte stores.  A thread owns 4 consecutive rows (pixels of one image row: TW >= 8) x 8 consecutive
// channels: 8 float4 loads per split, up to 4 splits (32 loads) in flight, so the fold is one or two L2 round trips.
// (The partials do NOT travel through distributed shared memory: measured, 28 KB per CTA took 3-4 us that way,
// 5 B/clk -- tools/lowres_timeline.py.  Also measured and rejected: a [column quad][row][4] workspace layout with
// 16-byte park stores and L1-cached fold loads -- the stores are issued 4x faster, but the cluster barrier then waits
// that much longer for them to land and the fold's 16-byte cells at a 64-byte stride read slower: +0.5-0.9 us per launch.)
template <int BLOCK_N, int S>
__device__ __forceinline__ void cluster_fold_store(const ConvTcParams& p, const float* part, int rank, int tid, int co0,
                                                   int w0, int h0, int n0) {
  constexpr int kQuads = 128 / S / 4;               // row quads of this CTA's slice
  constexpr int kGroups = BLOCK_N / 8;              // 8-channel groups per row
  constexpr int SB = S < 4 ? S : 4;                 // splits loaded together
#pragma unroll 1
  for (int g = tid; g < kQuads * kGroups; g += kEpiWarps * 32) {
    const int row = rank * (128 / S) + (g % kQuads) * 4, c8 = g / kQuads;
    const int wl = row & (p.TW - 1), hl = (row >> p.tw_sh) & (p.TH - 1), nl = row >> (p.tw_sh + p.th_sh);
    const int n = n0 + nl;
    if (n >= p.B) continue;                          // phantom rows of a tile that runs past the batch
    const long long pix = ((long long)n * p.H + h0 + hl) * p.W + w0 + wl;     // the quad's pixels are pix .. pix + 3
    const int c = co0 + c8 * 8;
    if (p.bias) prefetch_l1(p.bias + c);
    if (p.row_add) prefetch_l1(p.row_add + (long long)n * p.ld_row_add + c);
    if (p.residual) {
#pragma unroll
      for (int q = 0; q < 4; ++q) prefetch_l1(p.residual + (pix + q) * p.ld_res + c);
    }
    const float* rp = part + (c8 * 8) * 128 + row;
    float f[4][8];
#pragma unroll
    for (int sb = 0; sb < S; sb += SB) {
      float4 v[SB][8];
#pragma unroll
      for (int s = 0; s < SB; ++s)
#pragma unroll
        for (int j = 0; j < 8; ++j) v[s][j] = __ldcg(reinterpret_cast<const float4*>(rp + (sb + s) * (BLOCK_N * 128) + j * 128));
#pragma unroll
      for (int s = 0; s < SB; ++s)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (sb == 0 && s == 0) { f[0][j] = v[s][j].x; f[1][j] = v[s][j].y; f[2][j] = v[s][j].z; f[3][j] = v[s][j].w; }
          else { f[0][j] += v[s][j].x; f[1][j] += v[s][j].y; f[2][j] += v[s][j].z; f[3][j] += v[s][j].w; }
        }
    }
    float add[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (p.bias) {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + c));
      const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + c) + 1);
      add[0] += b0.x; add[1] += b0.y; add[2] += b0.z; add[3] += b0.w; add[4] += b1.x; add[5] += b1.y; add[6] += b1.z; add[7] += b1.w;
    }
    if (p.row_add) {
      const float4* r4 = reinterpret_cast<const float4*>(p.row_add + (long long)n * p.ld_row_add + c);
      const float4 b0 = __ldg(r4), b1 = __ldg(r4 + 1);
      // (acc + bias) + emb, as the other epilogues add them
      if (p.bias) {
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
          for (int j = 0; j < 8; ++j) f[q][j] += add[j];
      }
      add[0] = b0.x; add[1] = b0.y; add[2] = b0.z; add[3] = b0.w; add[4] = b1.x; add[5] = b1.y; add[6] = b1.z; add[7] = b1.w;
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
#pragma unroll
      for (int j = 0; j < 8; ++j) f[q][j] += add[j];
      if (p.residual) epi::add_bf16x8(f[q], __ldg(reinterpret_cast<const uint4*>(p.residual + (pix + q) * p.ld_res + c)));
      *reinterpret_cast<uint4*>(p.y_out + (pix + q) * p.ld_y + c) = epi::pack_bf16x8(f[q]);
    }
  }
}

template <int BLOCK_N, int CG>
__global__ void __launch_bounds__(kThreads, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2,
               const __grid_constant__ CUtensorMap tmY, const ConvTcParams p) {
  using Cfg = ConvCfg<BLOCK_N, CG>;
  constexpr int kStages = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* staging = smem + kStages * Cfg::kStageBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(staging + 2 * kStagingBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full = empty_bar + kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  volatile uint32_t* sk_flag = tmem_slot + 1;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    TL(0);
    if (p.prof) p.prof[32 * blockIdx.x + 14] = ((unsigned long long)gridDim.x << 32) | (BLOCK_N << 8) | p.split_k;
  }
  const uint32_t cta_rank = CG == 2 ? cluster_ctarank() : 0u;      // rank 0 = leader (issues the MMAs)
  const bool csplit = CG == 1 && BLOCK_N >= 64 && p.cluster_split;  // cluster of split_k CTAs per tile, one unit per CTA
  const int unit = CG == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;   // tile (CG=1) / tile-pair (CG=2) slot
  const int n_units = CG == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int taps = p.ksize * p.ksize;
  const int k_iters = taps * p.kc1 + p.kc2;
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  // CG = 2: work items are PAIRS of consecutive M tiles (a phantom tile past the end is zero-filled by
  // TMA and clipped on store)
  const int S = p.split_k;
  const int total_tiles = ((m_tiles + CG - 1) / CG) * p.n_blocks * S;     // work units = (tile, K split)
  const int pad = p.ksize >> 1;

  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (p.kc2) { tma_prefetch_desc(&tmA2); tma_prefetch_desc(&tmB2); }
    if (!p.y_nchw) tma_prefetch_desc(&tmY);
  }
  if (warp == 9) {
    if (lane == 0) {
      for (int i = 0; i < kStages; ++i) { mbar_init(&full_bar[i], CG); mbar_init(&empty_bar[i], 1); }
      for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], CG * kEpiWarps); }
      fence_barrier_init();
    }
    __syncwarp();
    if (CG == 2) { tmem_alloc_2sm(tmem_slot, Cfg::kTmemCols); tmem_relinquish_2sm(); }
    else { tmem_alloc(tmem_slot, Cfg::kTmemCols); tmem_relinquish(); }
  }
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) TL(1);

  if (warp == 8) {
    // ===================================================================== TMA producer
    if (lane == 0) {
      TL(16);
      int stage = 0; uint32_t phase = 0;
      const int main_iters = taps * p.kc1;
      for (int wu = unit; wu < total_tiles; wu += n_units) {
        const int tile = fdiv(wu, p.fd_split), split = wu - tile * S;
        const int it0 = fdiv(split * k_iters, p.fd_split), it1 = fdiv((split + 1) * k_iters, p.fd_split);
        const int tq = fdiv(tile, p.fd_nblocks);
        const int n_blk = tile - tq * p.n_blocks, m_blk = tq * CG + (int)cta_rank;
        const int mq = fdiv(m_blk, p.fd_tw), mq2 = fdiv(mq, p.fd_th);
        const int w0 = (m_blk - mq * p.tiles_w) * p.TW;
        const int h0 = (mq - mq2 * p.tiles_h) * p.TH;
        const int n0 = mq2 * p.TN;
        const int co0 = n_blk * BLOCK_N + (int)cta_rank * Cfg::kBRows;   // this CTA's share of the weight tile
        // The loop below is ONE thread's dependent instruction stream and paces the whole K loop when it is long (it was:
        // two runtime divisions per iteration, ~630 cycles against 200-512 cycles of MMAs): the tap / channel-slice
        // position is carried incrementally.
        int kc64, cw, ch, wcol;                    // channel offset, input column / row of the box, weight-matrix column
        {
          const int itc = it0 < main_iters ? it0 : 0;
          const int tap = fdiv(itc, p.fd_kc1), r = fdiv(tap, p.fd_ks);
          kc64 = (itc - tap * p.kc1) * 64;
          cw = w0 * p.stride + (tap - r * p.ksize) - pad;
          ch = h0 * p.stride + r - pad;
          wcol = itc * 64;                         // == tap * cin1 + kc * 64
        }
        const int cw_wrap = w0 * p.stride + p.ksize - pad;
        TL1(17);
        for (int it = it0; it < it1; ++it) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * Cfg::kStageBytes;
          uint8_t* sb = sa + kABytes;
          if (CG == 1) {
            mbar_expect_tx(&full_bar[stage], kABytes + Cfg::kBBytes);
          } else if (cta_rank == 0) {
            mbar_expect_tx(&full_bar[stage], 2 * (kABytes + Cfg::kBBytes));   // both CTAs' bytes land on the leader
          } else {
            mbar_arrive_cluster(&full_bar[stage], 0);
          }
          if (it < main_iters) {
            if (CG == 1) {
              tma_load_4d(&tmA, &full_bar[stage], sa, kc64, cw, ch, n0);
              tma_load_2d(&tmB, &full_bar[stage], sb, wcol, co0);
            } else {
              tma_load_4d_2sm(&tmA, &full_bar[stage], sa, kc64, cw, ch, n0);
              tma_load_2d_2sm(&tmB, &full_bar[stage], sb, wcol, co0);
            }
            kc64 += 64; wcol += 64;
            if (kc64 == p.cin1) {                  // next tap
              kc64 = 0;
              if (++cw == cw_wrap) { cw -= p.ksize; ++ch; }
            }
          } else {
            const int kc = it - main_iters;
            if (CG == 1) {
              tma_load_4d(&tmA2, &full_bar[stage], sa, kc * 64, w0, h0, n0);
              tma_load_2d(&tmB2, &full_bar[stage], sb, kc * 64, co0);
            } else {
              tma_load_4d_2sm(&tmA2, &full_bar[stage], sa, kc * 64, w0, h0, n0);
              tma_load_2d_2sm(&tmB2, &full_bar[stage], sb, kc * 64, co0);
            }
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        TL1(3);
      }
    }
  } else if (warp == 9) {
    // ===================================================================== MMA issuer
    if (lane == 0 && cta_rank == 0) {
      // second-source (raw residual stream) operands are always bf16
      constexpr uint32_t idesc_bf16 = umma_idesc_bf16(128 * CG, BLOCK_N);
      const uint32_t idesc_main = p.ab_f16 ? umma_idesc_f16(128 * CG, BLOCK_N) : idesc_bf16;
      const int main_iters = p.ksize * p.ksize * p.kc1;
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int wu = unit; wu < total_tiles; wu += n_units) {
        const int split = wu - fdiv(wu, p.fd_split) * S;
        const int it0 = fdiv(split * k_iters, p.fd_split), it1 = fdiv((split + 1) * k_iters, p.fd_split);
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BLOCK_N);
        for (int it = it0; it < it1; ++it) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * Cfg::kStageBytes);
          const uint64_t da = umma_desc_sw128(sa);
          const uint64_t db = umma_desc_sw128(sa + kABytes);
          const uint32_t idesc = it < main_iters ? idesc_main : idesc_bf16;
#pragma unroll
          for (int k = 0; k < 4; ++k) { // 4 x (K = 16 elements = 32 B) inside the 128-byte swizzle atom
            const uint32_t accum = (it > it0 || k > 0) ? 1u : 0u;
            if (CG == 1) umma_bf16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, accum);
            else umma_f16_2sm(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, accum);
          }
          // frees the smem stage (in both CTAs of a pair) once these MMAs have read it
          if (CG == 1) umma_commit(&empty_bar[stage]); else umma_commit_2sm(&empty_bar[stage], 3);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        TL1(5);
        // accumulator complete -> epilogue warps (of both CTAs)
        if (CG == 1) umma_commit(&tmem_full[acc]); else umma_commit_2sm(&tmem_full[acc], 3);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ===================================================================== epilogue (warps 0-7)
    // The epilogue paces the kernel when it is slower than the MMAs of one tile (18.4k cycles for K = 2304), so
    // two warpgroups drain the accumulator concurrently: warpgroup wg owns the 64-column chunks with (ch & 1) == wg,
    // its own staging tile, its own named barriers and its own TMA-store issuer.
    const int wg = warp >> 2, qw = warp & 3;          // warp (qw) may only touch TMEM lanes [32 qw, 32 qw + 32)
    const int row = qw * 32 + lane;                   // TMEM lane == pixel row of the tile
    const int etid = row;                             // thread index within the warpgroup
    const uint32_t lane_sel = (uint32_t)(qw * 32) << 16;
    const int wl = row % p.TW, hl = (row / p.TW) % p.TH, nl = row / (p.TW * p.TH);
    const bool issuer = (etid == 0);
    const uint32_t bar_a = 1 + 2 * wg, bar_b = 2 + 2 * wg;
    uint8_t* const stage_out = staging + wg * kStagingBytes;
    int acc = 0; uint32_t acc_phase = 0;
    if constexpr (CG == 1 && BLOCK_N >= 64) {
      if (csplit) {
        // ---- cluster split-K, first half: this CTA's fp32 partial tile -> the workspace ([column][row]: coalesced).
        // Warpgroup wg drains the column half wg.  The fold comes after the role switch, behind the cluster barrier.
        mbar_wait(&tmem_full[0], 0);
        tc_fence_after();
        if (threadIdx.x == 0) TL(6);
        float* wsp = p.sk_ws + (long long)unit * (BLOCK_N * 128) + row;       // unit == tile * S + split
#pragma unroll 1
        for (int c = wg * (BLOCK_N / 2); c < (wg + 1) * (BLOCK_N / 2); c += 32) {
          uint32_t v[32];
          tmem_ld_32x32(tmem_base + lane_sel + (uint32_t)c, v);
          tc_wait_ld();
#pragma unroll
          for (int j = 0; j < 32; ++j) __stcg(wsp + (c + j) * 128, __uint_as_float(v[j]));
        }
        tc_fence_before();
        if (threadIdx.x == 0) TL(7);
      }
    }
    for (int wu = unit; wu < total_tiles && !csplit; wu += n_units) {
      const int tile = fdiv(wu, p.fd_split), split = wu - tile * S;
      const int tq = fdiv(tile, p.fd_nblocks);
      const int n_blk = tile - tq * p.n_blocks, m_blk = tq * CG + (int)cta_rank;
      const int mq = fdiv(m_blk, p.fd_tw), mq2 = fdiv(mq, p.fd_th);
      const int w0 = (m_blk - mq * p.tiles_w) * p.TW;
      const int h0 = (mq - mq2 * p.tiles_h) * p.TH;
      const int n0 = mq2 * p.TN;
      const int co0 = n_blk * BLOCK_N;
      const int n = n0 + nl, h = h0 + hl, w = w0 + wl;
      const bool valid = n < p.B;
      const long long pix = ((long long)n * p.H + h) * p.W + w;

      if constexpr (BLOCK_N >= 64) {
        if (valid) {
#pragma unroll 1
          for (int ch = wg; ch < BLOCK_N / 64; ch += 2) {
            const int cbase = co0 + ch * 64;
            if (p.bias) { prefetch_l1(p.bias + cbase); prefetch_l1(p.bias + cbase + 32); }
            if (p.row_add) {
              prefetch_l1(p.row_add + (long long)n * p.ld_row_add + cbase);
              prefetch_l1(p.row_add + (long long)n * p.ld_row_add + cbase + 32);
            }
            if (p.residual) prefetch_l1(p.residual + pix * p.ld_res + cbase);
          }
        }
      }
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      if (threadIdx.x == 0) TL1(6);
      const uint32_t t_acc = tmem_base + lane_sel + (uint32_t)(acc * BLOCK_N);

      if constexpr (BLOCK_N >= 64) {
        bool finish = true;
        if (S > 1) {
          // ---- split-K: park this CTA's fp32 partial tile ([column][row]: coalesced), then the LAST CTA of the
          // tile to arrive folds the S partials in split order (deterministic) and runs the epilogue.
          float* wsp = p.sk_ws + ((long long)tile * S + split) * (BLOCK_N * 128) + row;
#pragma unroll 1
          for (int ch = wg; ch < BLOCK_N / 64; ch += 2) {
            uint32_t v0[32], v1[32];
            tmem_ld_32x32(t_acc + ch * 64, v0);
            tmem_ld_32x32(t_acc + ch * 64 + 32, v1);
            tc_wait_ld();
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              __stcg(wsp + (ch * 64 + j) * 128, __uint_as_float(v0[j]));
              __stcg(wsp + (ch * 64 + 32 + j) * 128, __uint_as_float(v1[j]));
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty[acc]);
          __threadfence();
          named_bar_sync(5, kEpiWarps * 32);
          if (threadIdx.x == 0) TL1(7);
          if (threadIdx.x == 0) {
            const int prev = atomicAdd(p.sk_cnt + tile, 1);
            const bool last = (prev == S - 1);
            if (last) p.sk_cnt[tile] = 0;            // re-arm for the next launch
            *sk_flag = last ? 1u : 0u;
          }
          named_bar_sync(6, kEpiWarps * 32);
          finish = (*sk_flag != 0u);
          if (finish) __threadfence();
          if (threadIdx.x == 0) { TL1(8); if (p.prof && wu == unit) p.prof[32 * blockIdx.x + 13] = finish ? 1 : 0; }
        }
        if (finish) {
        if (S == 1 && wg >= BLOCK_N / 64) {           // narrow tile: this warpgroup has no chunk, only releases TMEM
          __syncwarp();
          if (lane == 0) { if (CG == 1) mbar_arrive(&tmem_empty[acc]); else mbar_arrive_cluster(&tmem_empty[acc], 0); }
        }
#pragma unroll 1
        for (int ch = wg; ch < BLOCK_N / 64; ch += 2) {
          const int cbase = co0 + ch * 64;
          float f[64];
          if (S > 1) {
            const float* rp = p.sk_ws + (long long)tile * S * (BLOCK_N * 128) + (ch * 64) * 128 + row;
#pragma unroll
            for (int j = 0; j < 64; ++j) f[j] = __ldcg(rp + j * 128);
            for (int sp = 1; sp < S; ++sp) {
              rp += BLOCK_N * 128;
#pragma unroll
              for (int j = 0; j < 64; ++j) f[j] += __ldcg(rp + j * 128);
            }
            if (threadIdx.x == 0 && ch == 0) TL1(9);
          } else {
          uint32_t v0[32], v1[32];
          tmem_ld_32x32(t_acc + ch * 64, v0);
          tmem_ld_32x32(t_acc + ch * 64 + 32, v1);
          tc_wait_ld();
          if (ch + 2 >= BLOCK_N / 64) {       // this warp's last TMEM read of the accumulator
            tc_fence_before();
            __syncwarp();
            if (lane == 0) { if (CG == 1) mbar_arrive(&tmem_empty[acc]); else mbar_arrive_cluster(&tmem_empty[acc], 0); }
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) { f[j] = __uint_as_float(v0[j]); f[32 + j] = __uint_as_float(v1[j]); }
          }
          if (p.bias) epi::add_f32_row(f, p.bias + cbase);
          if (p.row_add && valid) epi::add_f32_row(f, p.row_add + (long long)n * p.ld_row_add + cbase);
          if (p.residual && valid) epi::add_bf16_row(f, p.residual + pix * p.ld_res + cbase);
          if (p.y_nchw) {
            if (valid) {
              const long long hw = (long long)p.H * p.W;
              float* o = p.y_nchw + ((long long)n * p.cout_valid) * hw + (long long)h * p.W + w;
#pragma unroll
              for (int j = 0; j < 64; ++j)
                if (cbase + j < p.cout_valid) o[(long long)(cbase + j) * hw] = f[j];
            }
          } else {
            // this warpgroup's staging tile was last read by the TMA store of its previous chunk
            if (issuer) bulk_wait_group_read<0>();
            named_bar_sync(bar_a, 128);
            epi::stage_bf16_row(stage_out + row * 128, row, f);
            fence_proxy_async_smem();
            named_bar_sync(bar_b, 128);
            if (issuer) {
              tma_store_4d(&tmY, stage_out, cbase, w0, h0, n0);
              bulk_commit_group();
              if (threadIdx.x == 0) TL1(10);
            }
            if (p.colsum) {
              // Fused GroupNorm statistics of the bf16 tile just staged.  Rows 0-63 / 64-127 are separate partial
              // rows (with TN == 2 they are two different images).
              const int col = etid & 63, half = etid >> 6;
              const float2 st = epi::staged_col_stats(smem_u32(stage_out), col, half);
              const int img = n0 + (p.TN == 2 ? half : 0);
              if (img < p.B && m_blk < m_tiles) {
                const int slot = (p.TN == 1) ? ((m_blk % (p.tiles_w * p.tiles_h)) * 2 + half) : 0;
                float2* dst = reinterpret_cast<float2*>(p.colsum) +
                              ((long long)img * p.colsum_slots + slot) * p.cout + cbase + col;
                *dst = st;
              }
            }
          }
        }
        }  // if (finish)
      } else {
        // BLOCK_N == 16: narrow head (out.2, 6 of 16 channels), fp32 NCHW output only
        uint32_t v[16];
        tmem_ld_32x16(t_acc, v);
        tc_wait_ld();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tmem_empty[acc]);
        if (valid && p.y_nchw && wg == 0) epi::store_head16(p, v, co0, n, h, w);
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (issuer) bulk_wait_group_read<0>();
    if (threadIdx.x == 0) TL(11);
  }

  if constexpr (CG == 1 && BLOCK_N >= 64) {
    if (csplit) {
      cluster_sync_all();                 // release / acquire at cluster scope: every partial of the tile is visible
      if (threadIdx.x == 0) TL(8);
      if (warp < kEpiWarps) {
        const int rank = (int)cluster_ctarank();
        const int tile = fdiv(unit, p.fd_split);
        const int tq = fdiv(tile, p.fd_nblocks);
        const int n_blk = tile - tq * p.n_blocks, m_blk = tq;
        const int mq = fdiv(m_blk, p.fd_tw), mq2 = fdiv(mq, p.fd_th);
        const int w0 = (m_blk - mq * p.tiles_w) * p.TW, h0 = (mq - mq2 * p.tiles_h) * p.TH, n0 = mq2 * p.TN;
        const float* part = p.sk_ws + (long long)tile * S * (BLOCK_N * 128);
        if (S == 2) cluster_fold_store<BLOCK_N, 2>(p, part, rank, (int)threadIdx.x, n_blk * BLOCK_N, w0, h0, n0);
        else if (S == 4) cluster_fold_store<BLOCK_N, 4>(p, part, rank, (int)threadIdx.x, n_blk * BLOCK_N, w0, h0, n0);
        else cluster_fold_store<BLOCK_N, 8>(p, part, rank, (int)threadIdx.x, n_blk * BLOCK_N, w0, h0, n0);
      }
      if (threadIdx.x == 0) TL(11);
    }
  }
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  if (threadIdx.x == 0) TL(12);
  if (warp == 9) {
    tc_fence_after();
    if (CG == 2) tmem_dealloc_2sm(tmem_base, Cfg::kTmemCols); else tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------ host
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// NHWC bf16 tensor [N][H][W][C] (pixel stride ld elements) as a 4-D map, box = {64, bw, bh, bn}.
int make_nhwc_map(CUtensorMap* m, const void* base, int C, int W, int H, int N, int ld, int bw, int bh, int bn,
                  int f16, int pixel_stride) {
  EncodeTiledFn enc = get_encode_tiled();
  FIDM_REQUIRE(enc != nullptr, FIDM_E_DRIVER, "cuTensorMapEncodeTiled is not available from the driver");
  FIDM_REQUIRE(((uintptr_t)base % 16) == 0 && ld % 8 == 0, FIDM_E_ALIGN, "tensor map: base/stride must be 16-byte aligned");
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)ld * 2, (cuuint64_t)W * ld * 2, (cuuint64_t)H * W * ld * 2};
  // pixel_stride 2 (stride-2 convolution, nn.py:126): the box TRAVERSES 2 bw x 2 bh pixels and loads every other one
  // (ceil(boxDim / elementStride) = bw x bh pixels land in shared memory)
  const cuuint32_t ps = (cuuint32_t)pixel_stride;
  cuuint32_t box[4] = {64, (cuuint32_t)bw * ps, (cuuint32_t)bh * ps, (cuuint32_t)bn};
  cuuint32_t es[4] = {1, ps, ps, 1};
  FIDM_REQUIRE(box[1] <= 256 && box[2] <= 256, FIDM_E_SHAPE, "tensor map: strided box %ux%u exceeds 256", box[1], box[2]);
  CUresult r = enc(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FIDM_REQUIRE(r == CUDA_SUCCESS, FIDM_E_DRIVER, "cuTensorMapEncodeTiled(NHWC C=%d W=%d H=%d N=%d ld=%d box=%d,%d,%d) failed: %d",
               C, W, H, N, ld, bw, bh, bn, (int)r);
  return 0;
}

// Row-major bf16 matrix [rows][cols] (row stride ld elements) as a 2-D map, box = {64, box_rows}.
int make_matrix_map(CUtensorMap* m, const void* base, int cols, int rows, int ld, int box_rows, int f16) {
  EncodeTiledFn enc = get_encode_tiled();
  FIDM_REQUIRE(enc != nullptr, FIDM_E_DRIVER, "cuTensorMapEncodeTiled is not available from the driver");
  FIDM_REQUIRE(((uintptr_t)base % 16) == 0 && ld % 16 == 0, FIDM_E_ALIGN, "tensor map: base/stride must be 16-byte aligned");
  // f16: 0 = bf16, 1 = fp16, 2 = 8-bit elements (e4m3 weights): a 128-byte box row is then 128 elements
  const int esz = f16 == 2 ? 1 : 2;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * esz};
  cuuint32_t box[2] = {(cuuint32_t)(128 / esz), (cuuint32_t)box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, f16 == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                   const_cast<void*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FIDM_REQUIRE(r == CUDA_SUCCESS, FIDM_E_DRIVER, "cuTensorMapEncodeTiled(matrix cols=%d rows=%d ld=%d box=%d) failed: %d",
               cols, rows, ld, box_rows, (int)r);
  return 0;
}

static int pow2_floor(int v) { int p = 1; while (p * 2 <= v) p *= 2; return p; }
static int pow2_div(int v, int cap) { int p = 1; while (p * 2 <= cap && v % (p * 2) == 0) p *= 2; return p; }

// Pixel box of an M tile: TW * TH * TN == 128, TW | W, TH | H.
int pick_pixel_box(int W, int H, int* tw, int* th, int* tn) {
  const int w = pow2_div(W, 128);
  const int h = pow2_div(H, 128 / w);
  *tw = w; *th = h; *tn = 128 / (w * h);
  (void)pow2_floor;
  return 0;
}

// CTAs of conv_tc_kernel<BLOCK_N, 1> that can be co-resident when launched as clusters of S (a cluster needs S free
// SMs inside one GPC), per device; 0 if the query fails.
template <int BLOCK_N>
static int cluster_capacity(int S) {
  static int cache[kMaxDevices][9] = {};
  const int dev = current_device();
  if (dev < 0 || dev >= kMaxDevices || S < 1 || S > 8) return 0;
  if (cache[dev][S] == 0) {
    using Cfg = ConvCfg<BLOCK_N, 1>;
    static bool attr_set[kMaxDevices] = {};
    if (ensure_dynamic_smem(conv_tc_kernel<BLOCK_N, 1>, Cfg::kSmemBytes, attr_set) != cudaSuccess) return 0;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(S * 64); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = S; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, conv_tc_kernel<BLOCK_N, 1>, &cfg) != cudaSuccess) { cudaGetLastError(); n = 0; }
    cache[dev][S] = n > 0 ? n * S : -1;
  }
  return cache[dev][S] > 0 ? cache[dev][S] : 0;
}

static int log2_exact(int v) { int s = 0; while ((1 << s) < v) ++s; return s; }

// split_k > 1: the K loop of a tile is shared by split_k CTAs.  cluster_split: they are one thread-block cluster and
// fold through distributed shared memory (split_k in {2, 4, 8}); otherwise through the global workspace.
template <int BLOCK_N, int CG>
static int launch_conv_tc(const fidm_conv_args& a, cudaStream_t st, int split_k = 1, bool cluster_split = false) {
  using Cfg = ConvCfg<BLOCK_N, CG>;
  ConvTcParams p;
  p.split_k = split_k; p.sk_ws = nullptr; p.sk_cnt = nullptr;
  p.cluster_split = cluster_split && split_k > 1 ? 1 : 0;
  p.prof = conv_profile_buffer();
  p.fd_split = make_fastdiv(split_k);
  const int Ho = a.height / a.stride, Wo = a.width / a.stride;          // a.height / a.width are the INPUT size
  p.B = a.batch; p.H = Ho; p.W = Wo; p.stride = a.stride;
  pick_pixel_box(Wo, Ho, &p.TW, &p.TH, &p.TN);
  FIDM_REQUIRE(p.TN <= 256, FIDM_E_SHAPE, "conv_tc: image %dx%d too small for a 128-pixel tile", Ho, Wo);
  p.tiles_w = Wo / p.TW; p.tiles_h = Ho / p.TH; p.tiles_n = (a.batch + p.TN - 1) / p.TN;
  p.n_blocks = a.cout / BLOCK_N;
  p.ksize = a.ksize; p.kc1 = a.cin / 64; p.cin1 = a.cin;
  p.fd_nblocks = make_fastdiv(p.n_blocks); p.fd_tw = make_fastdiv(p.tiles_w); p.fd_th = make_fastdiv(p.tiles_h);
  p.fd_kc1 = make_fastdiv(p.kc1); p.fd_ks = make_fastdiv(p.ksize);
  p.kc2 = a.x2 ? a.cin2 / 64 : 0;
  p.ab_f16 = a.dtype == FIDM_F16;
  const int f16 = p.ab_f16;
  set_epilogue_params(p, a);
  p.colsum_slots = (p.TN == 1) ? p.tiles_w * p.tiles_h * 2 : 1;
  p.y_out = reinterpret_cast<__nv_bfloat16*>(a.y); p.ld_y = a.ld_y;
  p.tw_sh = log2_exact(p.TW); p.th_sh = log2_exact(p.TH);
  if (p.cluster_split)
    FIDM_REQUIRE(CG == 1 && BLOCK_N >= 64 && (split_k == 2 || split_k == 4 || split_k == 8) && !a.colsum && !a.y_nchw_f32 &&
                     (uintptr_t)a.y % 16 == 0 && a.ld_y % 8 == 0 && p.TW >= 4,
                 FIDM_E_BADARG, "conv_tc: cluster split-K needs a 64+ wide NHWC tile, split 2|4|8 and no fused statistics");
  if (a.colsum) FIDM_REQUIRE(!a.y_nchw_f32 && p.TN <= 2 && BLOCK_N >= 64, FIDM_E_SHAPE, "conv_tc: colsum not supported for this shape");

  CUtensorMap tmA, tmB, tmA2, tmB2, tmY;
  int rc;
  if ((rc = make_nhwc_map(&tmA, a.x, a.cin, a.width, a.height, a.batch, a.ld_x, p.TW, p.TH, p.TN, f16, a.stride))) return rc;
  if ((rc = make_matrix_map(&tmB, a.w, a.ksize * a.ksize * a.cin, a.cout, a.ksize * a.ksize * a.cin, Cfg::kBRows, f16))) return rc;
  if (a.x2) {
    if ((rc = make_nhwc_map(&tmA2, a.x2, a.cin2, Wo, Ho, a.batch, a.ld_x2, p.TW, p.TH, p.TN, 0))) return rc;
    if ((rc = make_matrix_map(&tmB2, a.w2, a.cin2, a.cout, a.cin2, Cfg::kBRows, 0))) return rc;
  } else {
    tmA2 = tmA; tmB2 = tmB;
  }
  if (!a.y_nchw_f32) {
    if ((rc = make_nhwc_map(&tmY, a.y, a.cout, Wo, Ho, a.batch, a.ld_y, p.TW, p.TH, p.TN, 0))) return rc;
  } else {
    tmY = tmA;
  }
  static bool attr_set[kMaxDevices] = {};      // per (instantiation, device)
  FIDM_CUDA(ensure_dynamic_smem(conv_tc_kernel<BLOCK_N, CG>, Cfg::kSmemBytes, attr_set));
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  if (split_k > 1) {
    // workspace: the first kSplitCounterBytes hold one int arrival counter per tile (zero on entry and on exit --
    // a FIXED region, so that partial tiles of one launch can never be read as counters by the next), then
    // [tiles * split_k] fp32 partial tiles.
    const long long tiles = (long long)m_tiles * p.n_blocks;
    const long long need = kSplitCounterBytes + tiles * split_k * BLOCK_N * 128 * 4;
    FIDM_REQUIRE(CG == 1 && BLOCK_N >= 64 && a.splitk_ws && a.splitk_ws_bytes >= need &&
                     (p.cluster_split || tiles * 4 <= kSplitCounterBytes),
                 FIDM_E_BADARG, "conv_tc: split-K workspace too small (%lld needed)", need);
    p.sk_cnt = reinterpret_cast<int*>(a.splitk_ws);
    p.sk_ws = reinterpret_cast<float*>(reinterpret_cast<char*>(a.splitk_ws) + kSplitCounterBytes);
  }
  const int units = ((m_tiles + CG - 1) / CG) * p.n_blocks * split_k;  // (tile | tile pair) x K split
  const int slots = num_sms() / CG;
  // cluster split: one unit per CTA (clusters beyond the machine's capacity queue behind the first wave)
  const int grid = p.cluster_split ? units : (units < slots ? units : slots) * CG;
  FIDM_CUDA(launch_kernel(conv_tc_kernel<BLOCK_N, CG>, dim3(grid), dim3(kThreads), Cfg::kSmemBytes, st,
                          p.cluster_split ? split_k : CG, tmA, tmB, tmA2, tmB2, tmY, p));
  FIDM_CHECK_LAUNCH("conv_tc");
  return 0;
}

}  // namespace fidm

extern "C" int fidm_conv_colsum_slots(int32_t height, int32_t width) {
  int tw, th, tn;
  fidm::pick_pixel_box(width, height, &tw, &th, &tn);
  if (tn == 1) return (width / tw) * (height / th) * 2;
  if (tn == 2) return 1;
  return 0;
}

extern "C" int fidm_conv_gn_fusable(int32_t batch, int32_t height, int32_t width, int32_t cin, int32_t cout,
                                    int32_t ksize, int32_t stride) {
  fidm_conv_args a = {};
  a.dtype = FIDM_F16; a.batch = batch; a.height = height; a.width = width;
  a.cin = cin; a.cout = cout; a.ksize = ksize; a.stride = stride;
  a.y_nchw_f32 = cout == 16;        // the 16-wide variant is the fp32-NCHW head
  constexpr int min_fill = 75;      // percent of the CTA pairs (K1s: of the SMs) that must have a unit
  if (fidm::conv_halo_swap_preferred(a)) {
    // K1s: one 16 x 16 pixel box x 128 output channels per SM
    const long long units = (long long)batch * (height / 16) * (width / 16) * (cout == 16 ? 1 : cout / 128);
    return units * 100 >= (long long)fidm::num_sms() * min_fill ? 1 : 0;
  }
  if (!fidm::conv_halo_supported(a)) return 0;
  // worth it only when the CTA pairs of the machine are (nearly) all busy: 8 x 16 pixel boxes, two per pair
  const long long units = (long long)batch * (height / 16) * (width / 16) *
                          (cout == 16 ? 1 : cout / (cout % 256 == 0 ? 256 : 128));
  return units * 100 >= (long long)(fidm::num_sms() / 2) * min_fill ? 1 : 0;
}

extern "C" int fidm_conv2d_nhwc_bf16(const fidm_conv_args* a, fidm_stream_t stream) {
  using namespace fidm;
  FIDM_REQUIRE(a && a->x && a->w && a->y, FIDM_E_BADARG, "conv_tc: null x/w/y");
  FIDM_REQUIRE(a->dtype == FIDM_BF16 || a->dtype == FIDM_F16 || (a->dtype == FIDM_E4M3 && a->gn_coef), FIDM_E_BADARG,
               "conv_tc: dtype must be bf16 or f16 (e4m3 only with the fused GroupNorm operand path)");
  FIDM_REQUIRE((a->stride == 1 && (a->ksize == 1 || a->ksize == 3)) ||
               (a->stride == 2 && a->ksize == 3 && a->height % 2 == 0 && a->width % 2 == 0 && !a->gn_coef && !a->x2),
               FIDM_E_SHAPE, "conv_tc: stride 1 with ksize 1|3, or stride 2 with ksize 3 on an even-sized input");
  FIDM_REQUIRE(a->cin % 64 == 0 && a->cin > 0, FIDM_E_SHAPE, "conv_tc: cin %d must be a multiple of 64", a->cin);
  FIDM_REQUIRE(a->cout % 16 == 0, FIDM_E_SHAPE, "conv_tc: cout %d must be a multiple of 16", a->cout);
  if (a->x2) FIDM_REQUIRE(a->w2 && a->cin2 % 64 == 0 && a->cin2 > 0, FIDM_E_SHAPE, "conv_tc: bad second source");
  FIDM_REQUIRE(a->cout_valid > 0 && a->cout_valid <= a->cout, FIDM_E_BADARG, "conv_tc: cout_valid");
  if (a->bias) FIDM_REQUIRE((uintptr_t)a->bias % 16 == 0, FIDM_E_ALIGN, "conv_tc: bias must be 16-byte aligned");
  if (a->row_add)
    FIDM_REQUIRE((uintptr_t)a->row_add % 16 == 0 && a->ld_row_add % 4 == 0, FIDM_E_ALIGN, "conv_tc: row_add alignment");
  if (a->residual)
    FIDM_REQUIRE((uintptr_t)a->residual % 16 == 0 && a->ld_res % 8 == 0, FIDM_E_ALIGN, "conv_tc: residual alignment");
  cudaStream_t st = (cudaStream_t)stream;
  if (a->gn_coef || a->halo_copy) return launch_conv_halo(*a, st);      // GroupNorm + SiLU of the raw input applied in the operand path
  if (a->cout % 64 != 0 || a->y_nchw_f32) {
    FIDM_REQUIRE(a->y_nchw_f32 && a->cout == 16 && !a->residual, FIDM_E_SHAPE,
                 "conv_tc: cout %d is only supported as the 16-wide fp32-NCHW head", a->cout);
    return launch_conv_tc<16, 1>(*a, st);
  }
  // Widest N tile that still yields about one tile per SM; narrow tiles for the small low-resolution layers.
  int tw, th, tn;
  const int Ho = a->height / a->stride, Wo = a->width / a->stride;
  pick_pixel_box(Wo, Ho, &tw, &th, &tn);
  const long long m_tiles = (long long)(Wo / tw) * (Ho / th) * ((a->batch + tn - 1) / tn);
  const int want = (num_sms() * 3) / 4;
  if (a->cout % 256 == 0 && m_tiles * (a->cout / 256) >= want) return launch_conv_tc<256, 2>(*a, st);
  // Low-resolution layers (few pixel tiles, deep K).  Candidate (N tile, K split) pairs are scored with a small
  // cost model in SM cycles: tensor time of one CTA's share of the K loop, L2->SM operand traffic of the whole grid
  // against the ~12 KB/clk the L2 delivers (measured: 442 MB in 62 us on the 16x16 layers; these layers re-read the
  // weights once per pixel tile), and the fold of the split partials (shared by the cluster, or by the last CTA of a
  // tile on the workspace path).  tools/conv_tune.py checks the pick against every forced candidate.
  const int k_iters = a->ksize * a->ksize * (a->cin / 64) + (a->x2 ? a->cin2 / 64 : 0);
  // FIDM_CONV_SPLIT_CLUSTER=0: fold split partials through the global workspace (the round-1 path) instead of a cluster
  static const bool cluster_ok = getenv("FIDM_CONV_SPLIT_CLUSTER") == nullptr || atoi(getenv("FIDM_CONV_SPLIT_CLUSTER")) != 0;
  // (the shared fold hands a thread 4 consecutive pixels of one box row: TW >= 4)
  const bool use_cluster = cluster_ok && !a->colsum && (uintptr_t)a->y % 16 == 0 && a->ld_y % 8 == 0 && tw >= 4;
  int best_n = 0, best_s = 1;
  double best = 1e30;
  const int ns[3] = {256, 128, 64};
  const int sms = num_sms();
  for (int i = 0; i < 3; ++i) {
    const int N = ns[i];
    if (a->cout % N) continue;
    const long long tiles = m_tiles * (a->cout / N);
    for (int S = 1; S <= 8; ++S) {
      if (S > 1 && k_iters / S < 4) break;
      if (use_cluster && S != 1 && S != 2 && S != 4 && S != 8) continue;
      if (S > 1 && (!a->splitk_ws || a->splitk_ws_bytes < kSplitCounterBytes + tiles * S * N * 128 * 4 ||
                    (!use_cluster && tiles * 4 > kSplitCounterBytes)))
        break;
      // an SS-mode MMA with M = 128 streams its 128 A rows at one row per cycle whatever N is: a 64-deep K block costs
      // 4 x 128 cycles on every tile width (tools/lowres_timeline.py: 270 ns per block for N = 64 ... 256)
      int cap = sms;                                 // co-resident CTAs
      if (use_cluster && S > 1) {
        cap = N == 256 ? cluster_capacity<256>(S) : N == 128 ? cluster_capacity<128>(S) : cluster_capacity<64>(S);
        if (cap <= 0) continue;
      }
      const double waves = (double)((tiles * S + cap - 1) / cap);
      const double compute = waves * (double)((k_iters + S - 1) / S) * 512.0;
      const double traffic = (double)tiles * k_iters * (16384.0 + N * 128.0) / 12000.0;
      const double fold = S == 1 ? 0.0 : use_cluster ? 2000.0 + 35.0 * N :      // park + barrier + shared fold, measured
                          (double)S * (N / 64) * 900.0 + 4000.0;
      const double epi = use_cluster && S > 1 ? 0.0 : (N / 64) * 600.0 * waves;
      const double cost = (compute > traffic ? compute : traffic) + fold + epi + 3000.0;
      if (cost < best) { best = cost; best_n = N; best_s = S; }
    }
  }
  // FIDM_CONV_FORCE="N,S": tuning override (tools/conv_tune.py times every candidate against the model's pick)
  if (const char* force = getenv("FIDM_CONV_FORCE")) {
    int fn = 0, fs = 0;
    if (sscanf(force, "%d,%d", &fn, &fs) == 2 && (fn == 64 || fn == 128 || fn == 256) && a->cout % fn == 0 && fs >= 1 && fs <= 8 &&
        (fs == 1 || (k_iters / fs >= 1 && (!use_cluster || fs == 2 || fs == 4 || fs == 8) && a->splitk_ws &&
                     a->splitk_ws_bytes >= kSplitCounterBytes + m_tiles * (a->cout / fn) * fs * fn * 128 * 4))) {
      best_n = fn; best_s = fs;
    }
  }
  if (getenv("FIDM_CONV_TRACE"))
    fprintf(stderr, "conv_tc: %dx%d B%d cin %d cout %d k%d -> N tile %d split %d %s (model %.0f cycles)\n", Ho, Wo, a->batch,
            a->cin, a->cout, a->ksize, best_n, best_s, use_cluster && best_s > 1 ? "cluster" : "workspace", best);
  if (use_cluster && best_s > 1) {
    if (best_n == 256) return launch_conv_tc<256, 1>(*a, st, best_s, true);
    if (best_n == 128) return launch_conv_tc<128, 1>(*a, st, best_s, true);
    return launch_conv_tc<64, 1>(*a, st, best_s, true);
  }
  if (best_n == 256) return launch_conv_tc<256, 1>(*a, st, best_s);
  if (best_n == 128) return launch_conv_tc<128, 1>(*a, st, best_s);
  return launch_conv_tc<64, 1>(*a, st, best_s);
}
