// K1h: 3x3 convolution with the producer's GroupNorm(32) [* (1+scale) + shift] + SiLU applied in the operand path.
//
//   D[M = B*H*W pixels, N = Cout] = sum over taps (r,s) and 64-channel slices of
//                                   act(X)_{r,s}[M, 64] * W[N, (r,s), 64]^T ,   act(x) = silu(x * A[n][c] + B[n][c])
//
// Replaces, for the convolutions that follow a GroupNorm, BOTH the normalisation pass and the conv
// (nn.py:151-153, 173-176, 203-207: in_layers / out_layers of ResBlock).  The separate GroupNorm "apply" pass
// (2 B read + 2 B written per element, 13 % of a UNet evaluation) disappears, and the activation tensor is
// fetched once per 64-channel slice instead of once per tap:
//
//   * An M tile is an 8 x 16 box of output pixels of one image.  For every 64-channel slice ONE TMA box load
//     fetches the 10 x 18 halo tile of the RAW bf16 stream (out-of-image pixels are zero-filled by the hardware).
//   * Five transform warps read the halo tile once, apply h = x*A' + B' ; y = h + h*tanh(h)  (= silu(x*A + B) with
//     A' = A/2, B' = B/2: one MUFU op), force the conv's zero padding (out-of-image pixels are 0 AFTER the
//     activation), and write three column-shifted copies (s = 0,1,2) of [18 rows][8 pixels][64 ch] 16-bit in the
//     canonical K-major 128-byte-swizzled UMMA layout.  A row of a copy is exactly one 1024-byte swizzle atom, so
//     tap (r,s) is the descriptor  copy_s + r * 1024  -- always atom-aligned: nine MMAs per halo tile.
//   * Weights stream through a TMA ring as in K1; the optional 1x1 skip source (nn.py:184,212) rides the same
//     ring (one stage for its A box, one for its weights) as extra K iterations.
//   * CTA pair (cta_group::2): each CTA transforms its own 128 pixel rows and stages half of the weight tile.
//   * Epilogue as K1's, from the same pieces (conv_epilogue.cuh): bias, timestep row, residual, bf16 TMA store into
//     concat slices, fused GroupNorm statistics of the output.
//   * UP: `up` ResBlocks (nn.py:190-195) -- the halo tile is the 6 x 10 box of the HALF-resolution stream it covers
//     after a nearest 2x upsample; every source pixel is activated once and stored to its 2 x 2 halo positions.  The
//     second conv of the block reads its identity skip at (h/2, w/2) (res_half).  BLOCK_N = 16: the 6-channel head
//     (unet.py:148-152) with fp32 NCHW stores.  BLOCK_N = 128: Cout % 256 != 0 (runs at half the tensor rate: a
//     tcgen05.mma with the A operand in shared memory takes as long for N = 128 as for N = 256).
//
// Warp roles (512 threads): warps 0-7 epilogue (two warpgroups), 8-12 transform, 13 weight-ring TMA producer,
// 14 MMA issuer (+ TMEM owner), 15 halo TMA producer.  128 registers per thread suit every role.
#include <cuda.h>
#include <stdlib.h>

#include "common.cuh"
#include "conv_act.cuh"
#include "conv_epilogue.cuh"
#include "conv_host.cuh"
#include "sm100_primitives.cuh"

namespace fidm {
using namespace sm100;

struct ConvHaloParams {
  int B, H, W;
  int tiles_w, tiles_h;     // 8 x 16 pixel boxes per image
  int n_blocks;             // Cout / BLOCK_N
  int kc1, cin1;            // Cin / 64, Cin
  int kc2;                  // Cin2 / 64 of the optional 1x1 second source
  const float2* coef; int ld_coef;   // [B][ld_coef] (A/2, B/2) per (image, input channel)
  const float* w_scale;     // optional per-output-channel scale of the accumulator (e4m3 weights)
  const float* bias;
  const float* row_add; int ld_row_add;
  const __nv_bfloat16* residual; int ld_res;
  int res_tma;              // residual tile fetched by TMA into the staging buffer (full-resolution residual)
  int res_half;             // residual is stored at HALF resolution (x_upd of an up ResBlock, nn.py:194): read (h/2, w/2)
  float* colsum; int colsum_slots; int cout;
  float* y_nchw; int cout_valid;     // BLOCK_N == 16 (the 6-channel head, unet.py:151): fp32 NCHW output of cout_valid channels
  unsigned long long* prof;   // profiling buffer (fidm_conv_set_profile_buffer): [CTA][role][4] cycle counters; only the
                              // PROF = true instantiations read clock64() around their waits (tools/halo_probe.py) -- the
                              // product instantiations carry no timing code at all
};

namespace halo {
constexpr int kThreads = 512;
constexpr int kEpiWarps = 8;
constexpr int kXfWarps = 5;                            // transform warps (8-12)
constexpr int kTW = 8, kTH = 16;                       // output pixel box of one CTA
constexpr int kHW = kTW + 2, kHH = kTH + 2;            // halo tile
constexpr int kHaloPix = kHW * kHH;                    // 180
constexpr int kRawBytes = kHaloPix * 128;              // 23040: TMA transaction of one halo tile (64-channel slice)
constexpr int kUpW = 6, kUpH = 10;                     // source box of the halo under a nearest 2x upsample
constexpr int kRawBytesUp = kUpW * kUpH * 128;         // 7680
constexpr int kRawStride = 23 * 1024;                  // buffers stay 1024-byte aligned (swizzle atom)
constexpr int kCopyBytes = kHH * 1024;                 // [18 rows][8 pixels][128 B]
constexpr int kRingStageBytes = 16384;                 // one weight half-tile (<= 128 rows x 128 B) or one A2 box
constexpr int kRingStages = 5;
constexpr int kStagingBytes = 128 * 128;
constexpr int kOffRaw = 0;
constexpr int kOffCopy = kOffRaw + 2 * kRawStride;
constexpr int kOffRing = kOffCopy + 3 * kCopyBytes;
constexpr int kOffStaging = kOffRing + kRingStages * kRingStageBytes;
constexpr int kOffBars = kOffStaging + 2 * kStagingBytes;
constexpr int kSmemBytes = kOffBars + 256 + 1024;
static_assert(kOffCopy % 1024 == 0 && kOffRing % 1024 == 0 && kOffStaging % 1024 == 0, "swizzle-atom alignment");
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");
}  // namespace halo

// OPK: operand kind staged by the transform and multiplied with the weights: 0 = bf16, 1 = fp16 (kind::f16),
// 2 = fp8 e4m3 (kind::f8f6f4: a 128-byte operand row holds 128 channels, so a K slice is TWO 64-channel halo tiles;
// BLOCK_N = 256, no UP).
template <int BLOCK_N, int OPK, bool UP, bool PROF>
__global__ void __launch_bounds__(halo::kThreads, 1)
conv_halo_kernel(const __grid_constant__ CUtensorMap tmRaw, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2,
                 const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmRes,
                 const ConvHaloParams p) {
  using namespace halo;
  constexpr bool OUT_F16 = OPK == 1;
  constexpr bool FP8 = OPK == 2;
  static_assert(!FP8 || (BLOCK_N == 256 && !UP), "fp8 operands: 256-wide tiles, no upsampling transform");
  constexpr int kKW = FP8 ? 128 : 64;                    // channels per K slice (= per 128-byte operand row)
  constexpr int kBBytes = (BLOCK_N / 2) * 128;           // this CTA's half of one weight tile
  constexpr int kTmemCols = 2 * BLOCK_N < 32 ? 32 : 2 * BLOCK_N;
  static_assert(BLOCK_N == 16 || BLOCK_N == 128 || BLOCK_N == 256, "BLOCK_N");
  static_assert(kBBytes <= kRingStageBytes, "ring stage too small");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* const raw_buf = smem + kOffRaw;
  uint8_t* const copy_buf = smem + kOffCopy;
  uint8_t* const ring = smem + kOffRing;
  uint8_t* const staging = smem + kOffStaging;
  uint64_t* const bars = reinterpret_cast<uint64_t*>(smem + kOffBars);
  uint64_t* const raw_full = bars;              // [2]  TMA -> transform
  uint64_t* const raw_empty = bars + 2;         // [2]  transform -> halo producer
  uint64_t* const a_full = bars + 4;            // [3]  transform (both CTAs) -> MMA issuer   (leader's copy is used)
  uint64_t* const a_empty = bars + 7;           // [3]  MMA commit -> transform (multicast to both CTAs)
  uint64_t* const ring_full = bars + 10;        // [kRingStages]
  uint64_t* const ring_empty = bars + 10 + kRingStages;
  uint64_t* const tmem_full = bars + 10 + 2 * kRingStages;    // [2]
  uint64_t* const tmem_empty = tmem_full + 2;                 // [2]
  uint64_t* const res_bar = tmem_empty + 2;                   // [2]  residual tile landed in a warpgroup's staging buffer
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(res_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();          // rank 0 = leader (issues the MMAs)
  const int unit = (int)(blockIdx.x >> 1);
  const int n_units = (int)(gridDim.x >> 1);
  const int tiles_img = p.tiles_w * p.tiles_h;
  const int m_tiles = tiles_img * p.B;                   // even (tiles_w is even)
  const int total_units = (m_tiles >> 1) * p.n_blocks;   // (pair of horizontally adjacent boxes) x N block

  if (warp == 13 && lane == 0) {
    tma_prefetch_desc(&tmRaw);
    tma_prefetch_desc(&tmB);
    if (p.kc2) { tma_prefetch_desc(&tmA2); tma_prefetch_desc(&tmB2); }
    if (BLOCK_N >= 64) tma_prefetch_desc(&tmY);
    if (BLOCK_N >= 64 && p.res_tma) tma_prefetch_desc(&tmRes);
  }
  if (warp == 14) {
    if (lane == 0) {
      // the five transform warps never synchronise with each other: each arrives on the mbarriers itself
      for (int i = 0; i < 2; ++i) { mbar_init(&raw_full[i], 1); mbar_init(&raw_empty[i], kXfWarps); }
      for (int i = 0; i < 3; ++i) { mbar_init(&a_full[i], 2 * kXfWarps); mbar_init(&a_empty[i], 1); }
      for (int i = 0; i < kRingStages; ++i) { mbar_init(&ring_full[i], 2); mbar_init(&ring_empty[i], 1); }
      for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 2 * kEpiWarps); }
      for (int i = 0; i < 2; ++i) mbar_init(&res_bar[i], 1);
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc_2sm(tmem_slot, kTmemCols);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp >= 13) {
    if (warp == 13 && lane == 0) {
      // ================================================================ weight / second-source ring producer
      int stage = 0; uint32_t phase = 0;
      auto acquire = [&](uint32_t bytes_per_cta) {
        mbar_wait(&ring_empty[stage], phase ^ 1);
        if (cta_rank == 0) mbar_expect_tx(&ring_full[stage], 2 * bytes_per_cta);   // both CTAs' bytes land on the leader
        else mbar_arrive_cluster(&ring_full[stage], 0);
      };
      auto advance = [&]() { if (++stage == kRingStages) { stage = 0; phase ^= 1; } };
      for (int wu = unit; wu < total_units; wu += n_units) {
        const int n_blk = wu % p.n_blocks, m_blk = (wu / p.n_blocks) * 2 + (int)cta_rank;
        const int w0 = (m_blk % p.tiles_w) * kTW;
        const int h0 = ((m_blk / p.tiles_w) % p.tiles_h) * kTH;
        const int n0 = m_blk / tiles_img;
        const int co0 = n_blk * BLOCK_N + (int)cta_rank * (BLOCK_N / 2);
        for (int kc = 0; kc < p.cin1 / kKW; ++kc)
          for (int s = 0; s < 3; ++s)
            for (int r = 0; r < 3; ++r) {
              acquire(kBBytes);
              tma_load_2d_2sm(&tmB, &ring_full[stage], ring + stage * kRingStageBytes, (r * 3 + s) * p.cin1 + kc * kKW, co0);
              advance();
            }
        for (int kc = 0; kc < p.kc2; ++kc) {
          acquire(kTW * kTH * 128);
          tma_load_4d_2sm(&tmA2, &ring_full[stage], ring + stage * kRingStageBytes, kc * 64, w0, h0, n0);
          advance();
          acquire(kBBytes);
          tma_load_2d_2sm(&tmB2, &ring_full[stage], ring + stage * kRingStageBytes, kc * 64, co0);
          advance();
        }
      }
    } else if (warp == 15 && lane == 0) {
      // ================================================================ halo producer: this CTA's own 10 x 18 boxes of the
      // raw stream (6 x 10 boxes of the half-resolution stream under UP); out-of-image pixels are zero-filled
      uint32_t g = 0;
      for (int wu = unit; wu < total_units; wu += n_units) {
        const int m_blk = (wu / p.n_blocks) * 2 + (int)cta_rank;
        const int w0 = (m_blk % p.tiles_w) * kTW;
        const int h0 = ((m_blk / p.tiles_w) % p.tiles_h) * kTH;
        const int n0 = m_blk / tiles_img;
        for (int kc = 0; kc < p.kc1; ++kc, ++g) {
          const uint32_t rb = g & 1u;
          mbar_wait(&raw_empty[rb], ((g >> 1) & 1u) ^ 1u);
          mbar_expect_tx(&raw_full[rb], UP ? kRawBytesUp : kRawBytes);
          if (UP) tma_load_4d(&tmRaw, &raw_full[rb], raw_buf + rb * kRawStride, kc * 64, (w0 >> 1) - 1, (h0 >> 1) - 1, n0);
          else tma_load_4d(&tmRaw, &raw_full[rb], raw_buf + rb * kRawStride, kc * 64, w0 - 1, h0 - 1, n0);
        }
      }
    } else if (warp == 14 && lane == 0 && cta_rank == 0) {
      // ================================================================ MMA issuer (leader CTA)
      constexpr uint32_t idesc_bf16 = umma_idesc_bf16(256, BLOCK_N);
      // kind::f8f6f4 with e4m3 x e4m3 -> f32 has the same descriptor bits as kind::f16 with f16 x f16 (format code 0)
      constexpr uint32_t idesc_main = (OUT_F16 || FP8) ? umma_idesc_f16(256, BLOCK_N) : idesc_bf16;
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      uint32_t g = 0;
      const uint32_t copy_addr = smem_u32(copy_buf), ring_addr = smem_u32(ring);
      long long pf_tmem = 0, pf_a = 0, pf_ring = 0, pf_t = 0;
      const long long pf_start = PROF ? clock64() : 0;
      for (int wu = unit; wu < total_units; wu += n_units) {
        if constexpr (PROF) pf_t = clock64();
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        if constexpr (PROF) pf_tmem += clock64() - pf_t;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BLOCK_N);
        uint32_t accum = 0;
        for (int kc = 0; kc < p.cin1 / kKW; ++kc, ++g) {
          for (int s = 0; s < 3; ++s) {
            if constexpr (PROF) pf_t = clock64();
            mbar_wait(&a_full[s], g & 1u);
            if constexpr (PROF) pf_a += clock64() - pf_t;
            tc_fence_after();
            for (int r = 0; r < 3; ++r) {
              if constexpr (PROF) pf_t = clock64();
              mbar_wait(&ring_full[stage], phase);
              if constexpr (PROF) pf_ring += clock64() - pf_t;
              tc_fence_after();
              const uint64_t da = umma_desc_sw128(copy_addr + s * kCopyBytes + r * 1024);
              const uint64_t db = umma_desc_sw128(ring_addr + stage * kRingStageBytes);
#pragma unroll
              for (int k = 0; k < 4; ++k) {      // 4 x 32 bytes of K inside the 128-byte swizzle atom (16 x 16-bit | 32 x fp8)
                if constexpr (FP8) umma_f8_2sm(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc_main, accum);
                else umma_f16_2sm(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc_main, accum);
                accum = 1;
              }
              umma_commit_2sm(&ring_empty[stage], 3);
              if (++stage == kRingStages) { stage = 0; phase ^= 1; }
            }
            umma_commit_2sm(&a_empty[s], 3);      // copy s may be overwritten (in both CTAs) once these MMAs have read it
          }
        }
        for (int kc = 0; kc < p.kc2; ++kc) {
          const int st_a = stage;
          mbar_wait(&ring_full[stage], phase);
          if (++stage == kRingStages) { stage = 0; phase ^= 1; }
          mbar_wait(&ring_full[stage], phase);
          tc_fence_after();
          const uint64_t da = umma_desc_sw128(ring_addr + st_a * kRingStageBytes);
          const uint64_t db = umma_desc_sw128(ring_addr + stage * kRingStageBytes);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            umma_f16_2sm(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc_bf16, accum);
            accum = 1;
          }
          umma_commit_2sm(&ring_empty[st_a], 3);
          umma_commit_2sm(&ring_empty[stage], 3);
          if (++stage == kRingStages) { stage = 0; phase ^= 1; }
        }
        umma_commit_2sm(&tmem_full[acc], 3);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      if (PROF && p.prof) {
        unsigned long long* o = p.prof + 16 * blockIdx.x;
        o[0] = (unsigned long long)(clock64() - pf_start); o[1] = pf_tmem; o[2] = pf_a; o[3] = pf_ring;
      }
    }
  } else if (warp >= 8) {
    // ==================================================================== transform warps (8-12, 160 threads)
    const int tt = (int)threadIdx.x - 256;
    const int j = tt & 7;                      // 16-byte channel chunk (8 channels) of the 64-channel slice
    const int l20 = tt >> 3;
    const uint32_t raw_addr = smem_u32(raw_buf), copy_addr = smem_u32(copy_buf);
    uint32_t g = 0;
    long long pf_raw = 0, pf_ae = 0, pf_work = 0, pf_t = 0;
    const long long pf_start = PROF ? clock64() : 0;
    if constexpr (UP) {
      // Up ResBlock (nn.py:190-195): the operand is nearest-2x-upsample(silu(GN(x))) of the HALF-resolution raw stream.
      // The 10 x 18 halo of the upsampled image covers a 6 x 10 box of source pixels; thread = (chunk j, source column
      // lx, row phase lyq) owns the source pixels (lx, lyq + 3i), i = 0..3, activates each ONCE and stores it to the
      // up to 2 x 2 halo positions it covers (x in {2lx-1, 2lx}, y in {2ly-1, 2ly}) of each shifted copy.
      const int lx = l20 % kUpW, lyq = l20 / kUpW;
      const bool lane_on = l20 < 3 * kUpW;
      const int Hs = p.H >> 1, Ws = p.W >> 1;
      // source pixel q = ly * 6 + lx of the TMA box sits at q * 128, 16-byte chunks XOR-swizzled by (q & 7)
      uint32_t ro[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int q = (lyq + 3 * i) * kUpW + lx;
        ro[i] = raw_addr + q * 128 + ((j ^ (q & 7)) << 4);
      }
      // store bases for (halo column x in {2lx-1, 2lx}) x (copy s), halo row 2*lyq (row 2*lyq - 1 is 1024 B below)
      uint32_t sb[2][3];
      bool sv[2][3];
#pragma unroll
      for (int xk = 0; xk < 2; ++xk) {
        const int x = 2 * lx - 1 + xk;
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          const int xx = x - s;
          sv[xk][s] = lane_on && (unsigned)x < (unsigned)kHW && (unsigned)xx < 8u;
          sb[xk][s] = copy_addr + s * kCopyBytes + (2 * lyq) * 1024 + (xx & 7) * 128 + ((j ^ (xx & 7)) << 4);
        }
      }
      for (int wu = unit; wu < total_units; wu += n_units) {
        const int m_blk = (wu / p.n_blocks) * 2 + (int)cta_rank;
        const int w0 = (m_blk % p.tiles_w) * kTW;
        const int h0 = ((m_blk / p.tiles_w) % p.tiles_h) * kTH;
        const int n0 = m_blk / tiles_img;
        const float4* cf = reinterpret_cast<const float4*>(p.coef + (long long)n0 * p.ld_coef + j * 8);
        // zero padding applies AFTER the activation: source pixels outside the image stay 0
        const int lw = (w0 >> 1) - 1 + lx, lh = (h0 >> 1) - 1 + lyq;
        const bool col_ok = lane_on && (unsigned)lw < (unsigned)Ws;
        for (int kc = 0; kc < p.kc1; ++kc, ++g) {
          float4 c[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) c[q] = __ldg(cf + kc * 32 + q);
          const uint32_t rb = g & 1u;
          if constexpr (PROF) pf_t = clock64();
          mbar_wait(&raw_full[rb], (g >> 1) & 1u);
          if constexpr (PROF) pf_raw += clock64() - pf_t;
          if constexpr (PROF) pf_t = clock64();
          const uint32_t roff = rb * kRawStride;
          uint4 v[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            v[i] = make_uint4(0u, 0u, 0u, 0u);
            if (col_ok && lyq + 3 * i < kUpH && (unsigned)(lh + 3 * i) < (unsigned)Hs) {
              const uint4 r = ld_shared_u32x4(ro[i] + roff);
              v[i].x = act_pair<OUT_F16>(r.x, c[0].x, c[0].y, c[0].z, c[0].w);
              v[i].y = act_pair<OUT_F16>(r.y, c[1].x, c[1].y, c[1].z, c[1].w);
              v[i].z = act_pair<OUT_F16>(r.z, c[2].x, c[2].y, c[2].z, c[2].w);
              v[i].w = act_pair<OUT_F16>(r.w, c[3].x, c[3].y, c[3].z, c[3].w);
            }
          }
          if constexpr (PROF) pf_work += clock64() - pf_t;
#pragma unroll
          for (int s = 0; s < 3; ++s) {
            if constexpr (PROF) pf_t = clock64();
            mbar_wait(&a_empty[s], (g & 1u) ^ 1u);
            if constexpr (PROF) pf_ae += clock64() - pf_t;
#pragma unroll
            for (int xk = 0; xk < 2; ++xk) {
              if (sv[xk][s]) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  const int ly = lyq + 3 * i;                       // source row of the box, 0..9
                  if (ly < kUpH) {
                    if (ly >= 1) st_shared_u32x4(sb[xk][s] - 1024 + i * 6144, v[i]);    // halo row 2 ly - 1
                    if (ly <= 8) st_shared_u32x4(sb[xk][s] + i * 6144, v[i]);           // halo row 2 ly
                  }
                }
              }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              if (s == 0) mbar_arrive(&raw_empty[rb]);      // this warp has read its part of the source box
              mbar_arrive_cluster(&a_full[s], 0);
            }
          }
        }
      }
    } else {
      // Thread = (chunk j, halo column x, row parity yh); it owns the halo pixels (x, yh + 2i), i = 0..8.  Every
      // shared-memory offset below is a per-thread constant plus an immediate: no address arithmetic in the loop.
      const int x = l20 % kHW, yh = l20 / kHW;
      const int px0 = yh * kHW + x, px1 = px0 + 2 * kHW;
      // halo pixel px of the TMA box sits at px * 128 with its 16-byte chunks XOR-swizzled by (px & 7); px advances
      // by 20 per step of i, so the swizzle term alternates between two values (40 % 8 == 0)
      const uint32_t ro_even = raw_addr + px0 * 128 + ((j ^ (px0 & 7)) << 4);
      const uint32_t ro_odd = raw_addr + px1 * 128 + ((j ^ (px1 & 7)) << 4);
      // copy s: halo row y, pixel x - s  ->  row (y * 8 + x - s) of a K-major 128-byte-swizzled tile
      uint32_t so[3];
      bool in_copy[3];
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        const int xx = x - s;
        in_copy[s] = (unsigned)xx < 8u;
        so[s] = copy_addr + s * kCopyBytes + (yh * 8 + (xx & 7)) * 128 + ((j ^ (xx & 7)) << 4);
      }
      // fp8: the thread's 8 channels are 8 bytes: 16-byte chunk (4 half + j / 2) of the row, upper or lower half of it
      uint32_t so8a[3], so8b[3];
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        const int xx = x - s;
        const uint32_t row = copy_addr + s * kCopyBytes + (yh * 8 + (xx & 7)) * 128 + (j & 1) * 8;
        so8a[s] = row + (((j >> 1) ^ (xx & 7)) << 4);
        so8b[s] = row + (((4 + (j >> 1)) ^ (xx & 7)) << 4);
      }
      for (int wu = unit; wu < total_units; wu += n_units) {
        const int m_blk = (wu / p.n_blocks) * 2 + (int)cta_rank;
        const int w0 = (m_blk % p.tiles_w) * kTW;
        const int h0 = ((m_blk / p.tiles_w) % p.tiles_h) * kTH;
        const int n0 = m_blk / tiles_img;
        const float4* cf = reinterpret_cast<const float4*>(p.coef + (long long)n0 * p.ld_coef + j * 8);
        // The conv zero-pads the ACTIVATED tensor: halo pixels outside the image must be 0 after the activation.
        // Only the first / last halo row and column of a box can be outside (H % 16 == 0, W % 8 == 0).
        const bool col_out = (unsigned)(w0 - 1 + x) >= (unsigned)p.W;
        const bool first_out = col_out || (yh == 0 && h0 == 0);                 // i == 0  (halo row yh)
        const bool last_out = col_out || (yh == 1 && h0 + kTH == p.H);          // i == 8  (halo row 16 + yh)
        for (int kc = 0; kc < p.kc1; ++kc, ++g) {
          float4 c[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) c[q] = __ldg(cf + kc * 32 + q);      // (A/2, B/2) of channels 2q, 2q+1 of this chunk
          const uint32_t rb = g & 1u;
          if constexpr (PROF) pf_t = clock64();
          mbar_wait(&raw_full[rb], (g >> 1) & 1u);
          if constexpr (PROF) pf_raw += clock64() - pf_t;
          if constexpr (PROF) pf_t = clock64();
          const uint32_t roff = rb * kRawStride;
          if constexpr (FP8) {
            // Two 64-channel halo tiles make one K slice: tile `half` fills bytes [64 half, 64 half + 64) of every
            // 128-byte operand row (8 channels of a thread = 8 bytes); the copies are published after the second tile.
            const uint32_t half = (uint32_t)kc & 1u, G = g >> 1;
            uint2 v8[9];
#pragma unroll
            for (int i = 0; i < 9; ++i) {
              const uint4 r = ld_shared_u32x4(((i & 1) ? ro_odd : ro_even) + roff + (i >> 1) * (4 * kHW * 128));
              v8[i].x = act_pair_e4m3(r.x, c[0].x, c[0].y, c[0].z, c[0].w) | (act_pair_e4m3(r.y, c[1].x, c[1].y, c[1].z, c[1].w) << 16);
              v8[i].y = act_pair_e4m3(r.z, c[2].x, c[2].y, c[2].z, c[2].w) | (act_pair_e4m3(r.w, c[3].x, c[3].y, c[3].z, c[3].w) << 16);
              const bool out = (i == 0) ? first_out : (i == 8) ? last_out : col_out;
              if (out) v8[i] = make_uint2(0u, 0u);
            }
            if constexpr (PROF) pf_work += clock64() - pf_t;
            if (half == 0) {                         // first tile: nothing is published, but the raw buffer is free again
              __syncwarp();
              if (lane == 0) mbar_arrive(&raw_empty[rb]);
            }
#pragma unroll
            for (int s = 0; s < 3; ++s) {
              if (half == 0) {
                if constexpr (PROF) pf_t = clock64();
                mbar_wait(&a_empty[s], (G & 1u) ^ 1u);
                if constexpr (PROF) pf_ae += clock64() - pf_t;
              }
              if (in_copy[s]) {
                const uint32_t base = (half ? so8b[s] : so8a[s]);
#pragma unroll
                for (int i = 0; i < 9; ++i) st_shared_u32x2(base + i * 2048, v8[i].x, v8[i].y);
              }
              if (half == 1) {
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                  if (s == 0) mbar_arrive(&raw_empty[rb]);
                  mbar_arrive_cluster(&a_full[s], 0);
                }
              }
            }
          } else {
          uint4 v[9];
#pragma unroll
          for (int i = 0; i < 9; ++i) {
            const uint4 r = ld_shared_u32x4(((i & 1) ? ro_odd : ro_even) + roff + (i >> 1) * (4 * kHW * 128));
            v[i].x = act_pair<OUT_F16>(r.x, c[0].x, c[0].y, c[0].z, c[0].w);
            v[i].y = act_pair<OUT_F16>(r.y, c[1].x, c[1].y, c[1].z, c[1].w);
            v[i].z = act_pair<OUT_F16>(r.z, c[2].x, c[2].y, c[2].z, c[2].w);
            v[i].w = act_pair<OUT_F16>(r.w, c[3].x, c[3].y, c[3].z, c[3].w);
            const bool out = (i == 0) ? first_out : (i == 8) ? last_out : col_out;
            if (out) v[i] = make_uint4(0u, 0u, 0u, 0u);
          }
          if constexpr (PROF) pf_work += clock64() - pf_t;
#pragma unroll
          for (int s = 0; s < 3; ++s) {
            if constexpr (PROF) pf_t = clock64();
            mbar_wait(&a_empty[s], (g & 1u) ^ 1u);
            if constexpr (PROF) pf_ae += clock64() - pf_t;
            if (in_copy[s]) {
#pragma unroll
              for (int i = 0; i < 9; ++i) st_shared_u32x4(so[s] + i * 2048, v[i]);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              if (s == 0) mbar_arrive(&raw_empty[rb]);      // this warp has read its part of the halo tile
              mbar_arrive_cluster(&a_full[s], 0);
            }
          }
          }  // 16-bit operands
        }
      }
    }
    if (PROF && p.prof && tt == 0) {
      unsigned long long* o = p.prof + 16 * blockIdx.x + 4;
      o[0] = (unsigned long long)(clock64() - pf_start); o[1] = pf_raw; o[2] = pf_ae; o[3] = pf_work;
    }
  } else {
    // ==================================================================== epilogue (warps 0-7), as in K1 (conv_epilogue.cuh)
    const int wg = warp >> 2, qw = warp & 3;          // warp (qw) may only touch TMEM lanes [32 qw, 32 qw + 32)
    const int row = qw * 32 + lane;                   // TMEM lane == pixel row of this CTA's box
    const uint32_t lane_sel = (uint32_t)(qw * 32) << 16;
    const int wl = row & 7, hl = row >> 3;
    const bool issuer = (row == 0);
    const uint32_t bar_a = 1 + 2 * wg, bar_b = 2 + 2 * wg;
    uint8_t* const stage_out = staging + wg * kStagingBytes;
    int acc = 0; uint32_t acc_phase = 0;
    uint32_t res_phase = 0;
    long long pf_full = 0, pf_t = 0;
    const long long pf_start = PROF ? clock64() : 0;
    for (int wu = unit; wu < total_units; wu += n_units) {
      const int n_blk = wu % p.n_blocks, m_blk = (wu / p.n_blocks) * 2 + (int)cta_rank;
      const int w0 = (m_blk % p.tiles_w) * kTW;
      const int h0 = ((m_blk / p.tiles_w) % p.tiles_h) * kTH;
      const int n = m_blk / tiles_img;
      const int co0 = n_blk * BLOCK_N;
      const long long pix = p.res_half ? ((long long)n * (p.H >> 1) + ((h0 + hl) >> 1)) * (p.W >> 1) + ((w0 + wl) >> 1)
                                       : ((long long)n * p.H + (h0 + hl)) * p.W + (w0 + wl);      // residual pixel

      if constexpr (PROF) pf_t = clock64();
      mbar_wait(&tmem_full[acc], acc_phase);
      if constexpr (PROF) pf_full += clock64() - pf_t;
      tc_fence_after();
      const uint32_t t_acc = tmem_base + lane_sel + (uint32_t)(acc * BLOCK_N);
      if constexpr (BLOCK_N == 16) {
        // narrow head (out.2: 6 of 16 output channels): fp32 NCHW stores straight from the accumulator
        uint32_t v16[16];
        tmem_ld_32x16(t_acc, v16);
        tc_wait_ld();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(&tmem_empty[acc], 0);
        if (wg == 0) epi::store_head16(p, v16, 0, n, h0 + hl, w0 + wl);
      } else {
#pragma unroll 1
      for (int ch = wg; ch < BLOCK_N / 64; ch += 2) {
        const int cbase = co0 + ch * 64;
        if (p.res_tma) {
          // The residual tile of this chunk travels by TMA into the (idle) staging buffer while the accumulator is
          // drained: 268 MB exactly once through the L2 -> SM path, instead of per-thread 16-byte loads through an L1
          // that the 218 KB shared-memory carve-out leaves too small to keep a 128-byte row alive between them.
          named_bar_sync(bar_a, 128);                        // nobody still reads the buffer (statistics of the last chunk)
          if (issuer) {
            bulk_wait_group_read<0>();                       // the previous TMA store has finished reading it too
            mbar_expect_tx(&res_bar[wg], kStagingBytes);
            tma_load_4d(&tmRes, &res_bar[wg], stage_out, cbase, w0, h0, n);
          }
        }
        float f[64];
        {
          uint32_t v0[32], v1[32];
          tmem_ld_32x32(t_acc + ch * 64, v0);
          tmem_ld_32x32(t_acc + ch * 64 + 32, v1);
          tc_wait_ld();
          if (ch + 2 >= BLOCK_N / 64) {       // this warp's last TMEM read of the accumulator
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(&tmem_empty[acc], 0);
          }
#pragma unroll
          for (int q = 0; q < 32; ++q) { f[q] = __uint_as_float(v0[q]); f[32 + q] = __uint_as_float(v1[q]); }
        }
        if (p.w_scale) {      // dequantisation of e4m3 weights: per-output-channel scale on the accumulator, before the bias
          const float4* s4 = reinterpret_cast<const float4*>(p.w_scale + cbase);
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            const float4 t = __ldg(s4 + q);
            f[4 * q] *= t.x; f[4 * q + 1] *= t.y; f[4 * q + 2] *= t.z; f[4 * q + 3] *= t.w;
          }
        }
        if (p.bias) epi::add_f32_row(f, p.bias + cbase);
        if (p.row_add) epi::add_f32_row(f, p.row_add + (long long)n * p.ld_row_add + cbase);
        if (p.res_tma) {
          mbar_wait(&res_bar[wg], res_phase);
          res_phase ^= 1u;
          epi::add_bf16_row_smem(f, smem_u32(stage_out) + row * 128, row);
        } else if (p.residual) {
          epi::add_bf16_row(f, p.residual + pix * p.ld_res + cbase);
        }
        // this warpgroup's staging tile was last read by the TMA store of its previous chunk
        if (issuer) bulk_wait_group_read<0>();
        named_bar_sync(bar_a, 128);
        epi::stage_bf16_row(stage_out + row * 128, row, f);
        fence_proxy_async_smem();
        named_bar_sync(bar_b, 128);
        if (issuer) {
          tma_store_4d(&tmY, stage_out, cbase, w0, h0, n);
          bulk_commit_group();
        }
        if (p.colsum) {
          // Fused GroupNorm statistics of the OUTPUT (for its consumer), of the bf16 tile just staged; rows 0-63 /
          // 64-127 are separate partial rows (fixed-order fold later).
          const int col = row & 63, half = row >> 6;
          const float2 st = epi::staged_col_stats(smem_u32(stage_out), col, half);
          const int slot = (m_blk % tiles_img) * 2 + half;
          float2* dst = reinterpret_cast<float2*>(p.colsum) + ((long long)n * p.colsum_slots + slot) * p.cout + cbase + col;
          *dst = st;
        }
      }
      }  // BLOCK_N >= 64
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (BLOCK_N >= 64 && issuer) bulk_wait_group_read<0>();
    if (PROF && p.prof && threadIdx.x == 0) {
      unsigned long long* o = p.prof + 16 * blockIdx.x + 8;
      o[0] = (unsigned long long)(clock64() - pf_start); o[1] = pf_full;
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 14) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------ host
static unsigned long long* g_prof = nullptr;
unsigned long long* conv_profile_buffer() { return g_prof; }

bool conv_halo_supported(const fidm_conv_args& a) {
  return a.ksize == 3 && a.stride == 1 && a.height % halo::kTH == 0 && a.width % (2 * halo::kTW) == 0 &&
         a.cin % 64 == 0 && a.cin > 0 &&
         ((a.cout % 128 == 0 && !a.y_nchw_f32) || (a.cout == 16 && a.y_nchw_f32 && !a.x2 && !a.residual && !a.colsum)) &&
         (a.dtype == FIDM_F16 || a.dtype == FIDM_BF16 ||
          (a.dtype == FIDM_E4M3 && a.cin % 128 == 0 && a.cout % 256 == 0 && !a.x_half_res && !a.y_nchw_f32 && a.w_scale));
}

template <int BLOCK_N, int OPK, bool UP, bool PROF = false>
static int launch_conv_halo_t(const fidm_conv_args& a, cudaStream_t st) {
  using namespace halo;
  ConvHaloParams p;
  p.B = a.batch; p.H = a.height; p.W = a.width;
  p.tiles_w = a.width / kTW; p.tiles_h = a.height / kTH;
  p.n_blocks = a.cout / BLOCK_N;
  p.kc1 = a.cin / 64; p.cin1 = a.cin;
  p.kc2 = a.x2 ? a.cin2 / 64 : 0;
  p.coef = reinterpret_cast<const float2*>(a.gn_coef); p.ld_coef = a.ld_gn_coef;
  p.w_scale = OPK == 2 ? a.w_scale : nullptr;
  set_epilogue_params(p, a);
  p.res_half = a.residual_half_res;
  p.res_tma = (BLOCK_N >= 64 && a.residual && !a.residual_half_res) ? 1 : 0;
  p.colsum_slots = p.tiles_w * p.tiles_h * 2;
  p.prof = PROF ? g_prof : nullptr;

  CUtensorMap tmRaw, tmB, tmA2, tmB2, tmY, tmRes;
  int rc;
  // the raw stream is bf16; only the element SIZE matters to the copy engine
  if (UP) {
    if ((rc = make_nhwc_map(&tmRaw, a.x, a.cin, a.width / 2, a.height / 2, a.batch, a.ld_x, kUpW, kUpH, 1, 0))) return rc;
  } else {
    if ((rc = make_nhwc_map(&tmRaw, a.x, a.cin, a.width, a.height, a.batch, a.ld_x, kHW, kHH, 1, 0))) return rc;
  }
  if (OPK == 2) {      // e4m3 weights: [cout][9 * cin] bytes, box = 128 channels x BLOCK_N / 2 rows
    if ((rc = make_matrix_map(&tmB, a.w, 9 * a.cin, a.cout, 9 * a.cin, BLOCK_N / 2, 2))) return rc;
  } else {
    if ((rc = make_matrix_map(&tmB, a.w, 9 * a.cin, a.cout, 9 * a.cin, BLOCK_N / 2, OPK == 1 ? 1 : 0))) return rc;
  }
  if (a.x2) {
    if ((rc = make_nhwc_map(&tmA2, a.x2, a.cin2, a.width, a.height, a.batch, a.ld_x2, kTW, kTH, 1, 0))) return rc;
    if ((rc = make_matrix_map(&tmB2, a.w2, a.cin2, a.cout, a.cin2, BLOCK_N / 2, 0))) return rc;
  } else {
    tmA2 = tmB; tmB2 = tmB;
  }
  if (BLOCK_N >= 64) {
    if ((rc = make_nhwc_map(&tmY, a.y, a.cout, a.width, a.height, a.batch, a.ld_y, kTW, kTH, 1, 0))) return rc;
  } else {
    tmY = tmB;
  }
  tmRes = tmB;
  if (p.res_tma) {
    if ((rc = make_nhwc_map(&tmRes, a.residual, a.cout, a.width, a.height, a.batch, a.ld_res, kTW, kTH, 1, 0))) return rc;
  }
  static bool attr_set[kMaxDevices] = {};      // per (instantiation, device)
  FIDM_CUDA(ensure_dynamic_smem(conv_halo_kernel<BLOCK_N, OPK, UP, PROF>, kSmemBytes, attr_set));
  const int units = (p.tiles_w * p.tiles_h * p.B / 2) * p.n_blocks;
  const int slots = num_sms() / 2;
  const int grid = (units < slots ? units : slots) * 2;
  FIDM_CUDA(launch_kernel(conv_halo_kernel<BLOCK_N, OPK, UP, PROF>, dim3(grid), dim3(kThreads), kSmemBytes, st, 2, tmRaw, tmB, tmA2,
                          tmB2, tmY, tmRes, p));
  FIDM_CHECK_LAUNCH("conv_halo");
  return 0;
}

int launch_conv_halo(const fidm_conv_args& a, cudaStream_t st) {
  if (a.halo_copy) return launch_conv_halo_swap(a, st, nullptr);      // un-normalized operand through the halo path (stem)
  FIDM_REQUIRE(a.gn_coef && a.ld_gn_coef >= a.cin && (uintptr_t)a.gn_coef % 16 == 0 && a.ld_gn_coef % 2 == 0, FIDM_E_BADARG,
               "conv (fused GroupNorm operand): gn_coef must be 16-byte aligned [batch][ld >= cin] float2");
  if (a.dtype != FIDM_E4M3 && conv_halo_swap_preferred(a)) return launch_conv_halo_swap(a, st, g_prof);
  FIDM_REQUIRE(conv_halo_supported(a), FIDM_E_SHAPE,
               "conv (fused GroupNorm operand): needs 3x3 stride 1, H %% 16 == 0, W %% 16 == 0, cin %% 64 == 0, cout %% 128 == 0 "
               "(or the 16-wide fp32-NCHW head); e4m3 operands: cin %% 128 == 0, cout %% 256 == 0, w_scale, no upsampling");
  const bool f16 = a.dtype == FIDM_F16;
  if (a.dtype == FIDM_E4M3) return launch_conv_halo_t<256, 2, false>(a, st);
  if (a.x_half_res) {
    FIDM_REQUIRE(a.cout != 16, FIDM_E_SHAPE, "conv (fused GroupNorm operand): the head variant does not upsample");
    if (a.cout % 256 == 0) return f16 ? launch_conv_halo_t<256, true, true>(a, st) : launch_conv_halo_t<256, false, true>(a, st);
    return f16 ? launch_conv_halo_t<128, true, true>(a, st) : launch_conv_halo_t<128, false, true>(a, st);
  }
  if (g_prof && f16 && a.cout != 16) {     // instrumented instantiations (probe tool only)
    if (a.cout % 256 == 0) return launch_conv_halo_t<256, true, false, true>(a, st);
    return launch_conv_halo_t<128, true, false, true>(a, st);
  }
  if (a.cout == 16) return f16 ? launch_conv_halo_t<16, true, false>(a, st) : launch_conv_halo_t<16, false, false>(a, st);
  if (a.cout % 256 == 0) return f16 ? launch_conv_halo_t<256, true, false>(a, st) : launch_conv_halo_t<256, false, false>(a, st);
  return f16 ? launch_conv_halo_t<128, true, false>(a, st) : launch_conv_halo_t<128, false, false>(a, st);
}

}  // namespace fidm

extern "C" int fidm_conv_set_profile_buffer(uint64_t* device_buffer) {
  fidm::g_prof = reinterpret_cast<unsigned long long*>(device_buffer);
  return 0;
}
