// K1s: K1h with the operand roles swapped -- for layers whose Cout is NOT a multiple of 256 (the 128-channel layers of
// REF-FFHQ256, train_inpainting.py:208-224) and for the 6-channel head (unet.py:148-152).
//
//   D^T[M = 128 output channels, N = 256 pixels] = sum over taps (r,s) and 64-channel slices of
//                                                  W[M, (r,s), 64] * act(X)_{r,s}[N, 64]^T
//
// Why: a tcgen05.mma with its A operand in shared memory streams the 128 A rows at a fixed pace, so an MMA with
// N = 128 takes as long as one with N = 256 -- K1h's 128-wide tiles (pixels as M, 128 output channels as N) run at half
// the tensor rate (profiles/r1c_halo_probe_ref128.txt: MMA issuer busy 78 %, 760-820 TFLOP/s).  Here the WEIGHTS are the
// A operand (128 rows) and the transformed pixels the B operand (N = 256): every instruction is a full 128 x 256 x 16.
//
//   * One CTA per SM (no CTA pair: M = 128 is one CTA's worth), tile = a 16 x 16 box of output pixels of one image.
//   * Per 64-channel slice ONE TMA box load fetches the 18 x 18 halo tile of the raw bf16 stream; nine transform warps
//     (thread = 16-byte chunk x halo column x upper/lower half, nine rows each) apply silu(x*A + B) once and write the
//     three column-shifted copies [18 rows][16 pixels][64 ch] in the K-major 128-byte-swizzled layout.  A halo row of a
//     copy is two swizzle atoms, so tap (r,s) is the descriptor  copy_s + r * 2048  -- 256 consecutive pixel rows.
//     The warps never synchronise with each other (each arrives on the mbarriers itself); the coefficients of the
//     current image sit in shared memory.
//   * Weights: 4-stage TMA ring of [128 rows][64 ch] tiles (half the L2->SM bytes per MMA cycle of K1h).
//   * Accumulator in TMEM: lane = output channel, column = pixel; double-buffered (2 x 256 columns = all of TMEM).
//   * Epilogue (2 x 4 warps, thread = output channel): tcgen05.ld gives a thread 16 consecutive pixels of its channel;
//     bias / timestep row are per-thread scalars; a warp's 32 channels of one pixel are 64 contiguous bytes of the NHWC
//     output, so results are stored (and the residual loaded) with 2-byte accesses straight from registers -- no
//     shared-memory transpose, no proxy fence.  The GroupNorm statistics of the output (per-channel sum / sum of squares
//     of the stored bf16 values) accumulate in registers.
//   * Head (kHead): 16 weight rows are loaded (6 valid), fp32 NCHW stores straight from the accumulator -- a thread's
//     16 pixels are one 64-byte row segment of its channel plane.
//   * The optional 1x1 skip source (nn.py:184,212) rides the weight ring: per 64-channel slice two 16 x 8 pixel boxes in
//     adjacent stages (one 256-row B operand) and its weights.
//
// Warp roles (640 threads, 96 registers): 0-7 epilogue (two warpgroups), 8-16 transform, 17 weight-ring producer,
// 18 MMA issuer + TMEM owner, 19 halo producer.
#include <cuda.h>

#include "common.cuh"
#include "conv_act.cuh"
#include "conv_host.cuh"
#include "sm100_primitives.cuh"

namespace fidm {
using namespace sm100;

struct ConvSwapParams {
  int B, H, W;
  int tiles_w, tiles_h;     // 16 x 16 pixel boxes per image
  int n_blocks;             // ceil(Cout / 128)
  int kc1, cin1;            // Cin / 64, Cin
  int kc2;                  // Cin2 / 64 of the optional 1x1 second source
  const float2* coef; int ld_coef;
  const float* bias;
  const float* row_add; int ld_row_add;
  const unsigned short* residual; int ld_res;   // optional bf16 NHWC at output resolution ...
  int res_half;                                 // ... or at HALF resolution (x_upd of an up ResBlock, nn.py:194): read (h/2, w/2)
  unsigned short* y; int ld_y;                  // bf16 NHWC output (a channel slice of a wider buffer when ld_y > cout)
  float* colsum; int colsum_slots; int cout;
  float* y_nchw; int cout_valid;
  unsigned long long* prof;   // PROF instantiation only (tools/halo_probe.py): [CTA][16] cycle counters, layout as K1h
};

#define PF_T0() do { if constexpr (PROF) pf_t = clock64(); } while (0)
#define PF_ADD(x) do { if constexpr (PROF) (x) += clock64() - pf_t; } while (0)

namespace halo_s {
constexpr int kThreads = 640;
constexpr int kEpiThreads = 128;                       // per epilogue warpgroup (warps 0-3, 4-7)
constexpr int kXfThreads = 288;                        // warps 8-16
constexpr int kT = 16, kHalo = 18;
constexpr int kRawBytes = kHalo * kHalo * 128;         // 41472: one halo tile of a 64-channel slice
constexpr int kUp = 10;                                // source box of the halo under a nearest 2x upsample: 10 x 10
constexpr int kRawBytesUp = kUp * kUp * 128;           // 12800
constexpr int kRawStride = 41 * 1024;
constexpr int kCopyBytes = kHalo * 2048;               // [18 rows][16 pixels][128 B]
constexpr int kRingStageBytes = 16384;                 // [128 rows][128 B] weights, or one 16 x 8 pixel box of the skip source
constexpr int kRingStages = 4;
constexpr int kOffRaw = 0;
constexpr int kOffCopy = kOffRaw + kRawStride;
constexpr int kOffRing = kOffCopy + 3 * kCopyBytes;
constexpr int kMaxCin = 1024;                          // the coefficient table of one image lives in shared memory
constexpr int kOffCoef = kOffRing + kRingStages * kRingStageBytes;
constexpr int kOffBars = kOffCoef + kMaxCin * 8;
constexpr int kSmemBytes = kOffBars + 256 + 1024;
static_assert(kOffCopy % 1024 == 0 && kOffRing % 1024 == 0, "swizzle-atom alignment");
static_assert(kRawBytes <= kRawStride, "raw buffer");
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");
static_assert(kRingStages >= 4, "a skip-source slice needs up to 4 stages: alignment skip, two pixel boxes, weights");
}  // namespace halo_s

// ACT = false: the operand is x itself (16-bit, already in the weights' dtype) -- the stem convolution, which has no
// GroupNorm in front of it (unet.py:55) but the same 3x3 structure; the transform is then a plain shifted copy.
// UP = true: `up` ResBlocks (nn.py:190-195) -- x is the HALF-resolution raw stream, the operand its activated nearest-2x
// upsample: the 18 x 18 halo covers a 10 x 10 box of source pixels, each activated once and stored to its 2 x 2 positions.
template <bool OUT_F16, bool kHead, bool PROF, bool ACT, bool UP>
__global__ void __launch_bounds__(halo_s::kThreads, 1)
conv_halo_swap_kernel(const __grid_constant__ CUtensorMap tmRaw, const __grid_constant__ CUtensorMap tmW,
                      const __grid_constant__ CUtensorMap tmX2, const __grid_constant__ CUtensorMap tmW2,
                      const ConvSwapParams p) {
  using namespace halo_s;
  constexpr int kWRows = kHead ? 16 : 128;               // weight rows actually loaded (the head has 16, 6 valid)
  constexpr uint32_t kWBytes = kWRows * 128;
  constexpr int kTmemCols = 512;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* const raw_buf = smem + kOffRaw;
  uint8_t* const copy_buf = smem + kOffCopy;
  uint8_t* const ring = smem + kOffRing;
  uint8_t* const coef_tab = smem + kOffCoef;
  uint64_t* const bars = reinterpret_cast<uint64_t*>(smem + kOffBars);
  uint64_t* const raw_full = bars;              // [1]  TMA -> transform
  uint64_t* const raw_empty = bars + 1;         // [1]  transform -> halo producer
  uint64_t* const a_full = bars + 2;            // [3]  transform -> MMA issuer
  uint64_t* const a_empty = bars + 5;           // [3]  MMA commit -> transform
  uint64_t* const ring_full = bars + 8;         // [kRingStages]
  uint64_t* const ring_empty = bars + 8 + kRingStages;
  uint64_t* const tmem_full = bars + 8 + 2 * kRingStages;     // [2]
  uint64_t* const tmem_empty = tmem_full + 2;                 // [2]
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_img = p.tiles_w * p.tiles_h;
  const int total_units = tiles_img * p.B * p.n_blocks;

  if (warp == 17 && lane == 0) {
    tma_prefetch_desc(&tmRaw);
    tma_prefetch_desc(&tmW);
    if (p.kc2) { tma_prefetch_desc(&tmX2); tma_prefetch_desc(&tmW2); }
  }
  if (warp == 18) {
    if (lane == 0) {
      mbar_init(&raw_full[0], 1); mbar_init(&raw_empty[0], kXfThreads / 32);
      for (int i = 0; i < 3; ++i) { mbar_init(&a_full[i], kXfThreads / 32); mbar_init(&a_empty[i], 1); }
      for (int i = 0; i < kRingStages; ++i) { mbar_init(&ring_full[i], 1); mbar_init(&ring_empty[i], 1); }
      for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 8); }
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp >= 17) {
    if (warp == 17 && lane == 0) {
      // ================================================================ weight / skip-source ring producer
      int stage = 0; uint32_t phase = 0;
      auto acquire = [&](uint32_t bytes) {
        mbar_wait(&ring_empty[stage], phase ^ 1);
        mbar_expect_tx(&ring_full[stage], bytes);
      };
      auto advance = [&]() { if (++stage == kRingStages) { stage = 0; phase ^= 1; } };
      for (int wu = blockIdx.x; wu < total_units; wu += gridDim.x) {
        const int n_blk = wu % p.n_blocks, tile = wu / p.n_blocks;
        const int w0 = (tile % p.tiles_w) * kT;
        const int h0 = ((tile / p.tiles_w) % p.tiles_h) * kT;
        const int n0 = tile / tiles_img;
        const int co0 = n_blk * 128;
        for (int kc = 0; kc < p.kc1; ++kc)
          for (int s = 0; s < 3; ++s)
            for (int r = 0; r < 3; ++r) {
              acquire(kWBytes);
              tma_load_2d(&tmW, &ring_full[stage], ring + stage * kRingStageBytes, (r * 3 + s) * p.cin1 + kc * 64, co0);
              advance();
            }
        for (int kc = 0; kc < p.kc2; ++kc) {
          // the two 16 x 8 pixel boxes of the skip source must sit in ADJACENT stages (one N = 256 operand of 32 KB):
          // a pair may not start in the last stage -- skip it (the consumer follows the same rule)
          if (stage == kRingStages - 1) {
            mbar_wait(&ring_empty[stage], phase ^ 1);
            mbar_arrive(&ring_full[stage]);
            advance();
          }
          for (int hb = 0; hb < 2; ++hb) {
            acquire(kRingStageBytes);
            tma_load_4d(&tmX2, &ring_full[stage], ring + stage * kRingStageBytes, kc * 64, w0, h0 + hb * 8, n0);
            advance();
          }
          acquire(kRingStageBytes);
          tma_load_2d(&tmW2, &ring_full[stage], ring + stage * kRingStageBytes, kc * 64, co0);
          advance();
        }
      }
    } else if (warp == 19 && lane == 0) {
      // ================================================================ halo producer: 18 x 18 boxes of the raw stream
      uint32_t g = 0;
      for (int wu = blockIdx.x; wu < total_units; wu += gridDim.x) {
        const int tile = wu / p.n_blocks;
        const int w0 = (tile % p.tiles_w) * kT;
        const int h0 = ((tile / p.tiles_w) % p.tiles_h) * kT;
        const int n0 = tile / tiles_img;
        for (int kc = 0; kc < p.kc1; ++kc, ++g) {
          mbar_wait(&raw_empty[0], (g & 1u) ^ 1u);
          mbar_expect_tx(&raw_full[0], UP ? kRawBytesUp : kRawBytes);
          if (UP) tma_load_4d(&tmRaw, &raw_full[0], raw_buf, kc * 64, (w0 >> 1) - 1, (h0 >> 1) - 1, n0);
          else tma_load_4d(&tmRaw, &raw_full[0], raw_buf, kc * 64, w0 - 1, h0 - 1, n0);
        }
      }
    } else if (warp == 18 && lane == 0) {
      // ================================================================ MMA issuer
      constexpr uint32_t idesc_main = OUT_F16 ? umma_idesc_f16(128, 256) : umma_idesc_bf16(128, 256);
      constexpr uint32_t idesc_skip = umma_idesc_bf16(128, 256);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      uint32_t g = 0;
      const uint32_t copy_addr = smem_u32(copy_buf), ring_addr = smem_u32(ring);
      long long pf_tmem = 0, pf_a = 0, pf_ring = 0, pf_t = 0;
      const long long pf_start = PROF ? clock64() : 0;
      for (int wu = blockIdx.x; wu < total_units; wu += gridDim.x) {
        PF_T0();
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        PF_ADD(pf_tmem);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * 256);
        uint32_t accum = 0;
        for (int kc = 0; kc < p.kc1; ++kc, ++g) {
          for (int s = 0; s < 3; ++s) {
            PF_T0();
            mbar_wait(&a_full[s], g & 1u);
            PF_ADD(pf_a);
            tc_fence_after();
            for (int r = 0; r < 3; ++r) {
              PF_T0();
              mbar_wait(&ring_full[stage], phase);
              PF_ADD(pf_ring);
              tc_fence_after();
              const uint64_t da = umma_desc_sw128(ring_addr + stage * kRingStageBytes);          // weights: 128 rows
              const uint64_t db = umma_desc_sw128(copy_addr + s * kCopyBytes + r * 2048);        // 256 pixel rows
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                umma_bf16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc_main, accum);
                accum = 1;
              }
              umma_commit(&ring_empty[stage]);
              if (++stage == kRingStages) { stage = 0; phase ^= 1; }
            }
            umma_commit(&a_empty[s]);      // copy s may be overwritten once these MMAs have read it
          }
        }
        for (int kc = 0; kc < p.kc2; ++kc) {
          auto next = [&]() { if (++stage == kRingStages) { stage = 0; phase ^= 1; } };
          if (stage == kRingStages - 1) {          // alignment skip, see the producer
            mbar_wait(&ring_full[stage], phase);
            umma_commit(&ring_empty[stage]);
            next();
          }
          const int st_x = stage;                  // pixels: stages st_x, st_x + 1 (256 rows), then the weights
          mbar_wait(&ring_full[stage], phase); next();
          mbar_wait(&ring_full[stage], phase); next();
          const int st_w = stage;
          mbar_wait(&ring_full[stage], phase); next();
          tc_fence_after();
          const uint64_t da = umma_desc_sw128(ring_addr + st_w * kRingStageBytes);
          const uint64_t db = umma_desc_sw128(ring_addr + st_x * kRingStageBytes);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc_skip, 1u);
          umma_commit(&ring_empty[st_x]);
          umma_commit(&ring_empty[st_x + 1]);
          umma_commit(&ring_empty[st_w]);
        }
        umma_commit(&tmem_full[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      if (PROF && p.prof) {
        unsigned long long* o = p.prof + 16 * blockIdx.x;
        o[0] = (unsigned long long)(clock64() - pf_start); o[1] = pf_tmem; o[2] = pf_a; o[3] = pf_ring;
      }
    }
  } else if (warp >= 8) {
    // ==================================================================== transform warps (8-16, 288 threads)
    // Thread = (16-byte chunk j, halo column x, half yh); it owns the halo pixels (x, 9 yh + i), i = 0..8.
    const int tt = (int)threadIdx.x - 2 * kEpiThreads;
    const int j = tt & 7;
    const int l36 = tt >> 3;
    const int x = l36 % kHalo, yh = l36 / kHalo;
    const uint32_t raw_addr = smem_u32(raw_buf), copy_addr = smem_u32(copy_buf);
    // halo pixel px = y * 18 + x of the TMA box sits at px * 128, its 16-byte chunks XOR-swizzled by (px & 7)
    const int px0 = yh * 9 * kHalo + x;
    const uint32_t raw0 = raw_addr + px0 * 128;
    const uint32_t j16 = (uint32_t)j << 4;
    // copy s: halo pixel (x, y) is pixel xx = x - s of row y: atom (xx >> 3), row (xx & 7) of the atom
    uint32_t so[3];
    bool in_copy[3];
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      const int xx = x - s;
      in_copy[s] = (unsigned)xx < 16u;
      so[s] = copy_addr + s * kCopyBytes + (yh * 9) * 2048 + ((xx >> 3) & 1) * 1024 + (xx & 7) * 128 + ((j ^ (xx & 7)) << 4);
    }
    const uint32_t coef_s = smem_u32(coef_tab) + (uint32_t)j * 64u;      // 8 channels x (A/2, B/2) per 16-byte chunk j
    uint32_t coef_q[4];                                                  // rotated quarters, see the table fill below
#pragma unroll
    for (int q = 0; q < 4; ++q) coef_q[q] = (uint32_t)((q + (j >> 1)) & 3) * 16u;
    int coef_n = -1;
    uint32_t g = 0;
    long long pf_raw = 0, pf_ae = 0, pf_work = 0, pf_t = 0;
    const long long pf_start = PROF ? clock64() : 0;
    if constexpr (UP) {
      // thread = (chunk j, source column lx, row phase lyq) owns the source pixels (lx, lyq + 3i), i < 4 (rows < 10); a source
      // pixel (lx, ly) covers halo columns {2lx - 1, 2lx} and rows {2ly - 1, 2ly} (those inside the 18 x 18 halo)
      const int lx = l36 % kUp, lyq = l36 / kUp;
      const bool lane_on = l36 < 3 * kUp;
      const int Hs = p.H >> 1, Ws = p.W >> 1;
      uint32_t ro[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int q = (lyq + 3 * i) * kUp + lx;               // source pixel q of the TMA box sits at q * 128, swizzled by (q & 7)
        ro[i] = raw_addr + q * 128 + ((j ^ (q & 7)) << 4);
      }
      uint32_t sb[2][3];
      bool sv[2][3];
#pragma unroll
      for (int xk = 0; xk < 2; ++xk) {
        const int xh = 2 * lx - 1 + xk;                       // halo column
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          const int xx = xh - s;
          sv[xk][s] = lane_on && (unsigned)xh < (unsigned)kHalo && (unsigned)xx < 16u;
          sb[xk][s] = copy_addr + s * kCopyBytes + (2 * lyq) * 2048 + ((xx >> 3) & 1) * 1024 + (xx & 7) * 128 + ((j ^ (xx & 7)) << 4);
        }
      }
      for (int wu = blockIdx.x; wu < total_units; wu += gridDim.x) {
        const int tile = wu / p.n_blocks;
        const int w0 = (tile % p.tiles_w) * kT;
        const int h0 = ((tile / p.tiles_w) % p.tiles_h) * kT;
        const int n0 = tile / tiles_img;
        if (n0 != coef_n) {
          named_bar_sync(7, kXfThreads);
          const float4* src = reinterpret_cast<const float4*>(p.coef + (long long)n0 * p.ld_coef);
          for (int i = tt; i < p.cin1 / 2; i += kXfThreads) {
            const float4 t = __ldg(src + i);
            const uint32_t ch = (uint32_t)i >> 2, off = ch * 64u + ((((uint32_t)i & 3u) + ((ch & 7u) >> 1)) & 3u) * 16u;
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(smem_u32(coef_tab) + off), "f"(t.x), "f"(t.y),
                         "f"(t.z), "f"(t.w) : "memory");
          }
          named_bar_sync(7, kXfThreads);
          coef_n = n0;
        }
        // zero padding applies AFTER the activation: source pixels outside the (half-resolution) image stay 0
        const int lw = (w0 >> 1) - 1 + lx, lh = (h0 >> 1) - 1 + lyq;
        const bool col_ok = lane_on && (unsigned)lw < (unsigned)Ws;
        for (int kc = 0; kc < p.kc1; ++kc, ++g) {
          PF_T0();
          mbar_wait(&raw_full[0], g & 1u);
          PF_ADD(pf_raw);
          PF_T0();
          float4 c[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(c[q].x), "=f"(c[q].y), "=f"(c[q].z), "=f"(c[q].w)
                         : "r"(coef_s + (uint32_t)(kc * 512) + coef_q[q]));
          }
          uint4 v[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            v[i] = make_uint4(0u, 0u, 0u, 0u);
            if (col_ok && lyq + 3 * i < kUp && (unsigned)(lh + 3 * i) < (unsigned)Hs) {
              const uint4 r = ld_shared_u32x4(ro[i]);
              v[i].x = act_pair<OUT_F16>(r.x, c[0].x, c[0].y, c[0].z, c[0].w);
              v[i].y = act_pair<OUT_F16>(r.y, c[1].x, c[1].y, c[1].z, c[1].w);
              v[i].z = act_pair<OUT_F16>(r.z, c[2].x, c[2].y, c[2].z, c[2].w);
              v[i].w = act_pair<OUT_F16>(r.w, c[3].x, c[3].y, c[3].z, c[3].w);
            }
          }
          PF_ADD(pf_work);
#pragma unroll
          for (int s = 0; s < 3; ++s) {
            PF_T0();
            mbar_wait(&a_empty[s], (g & 1u) ^ 1u);
            PF_ADD(pf_ae);
#pragma unroll
            for (int xk = 0; xk < 2; ++xk) {
              if (sv[xk][s]) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  const int ly = lyq + 3 * i;                         // source row of the box, 0..9
                  if (ly < kUp) {
                    if (ly >= 1) st_shared_u32x4(sb[xk][s] - 2048 + i * (6 * 2048), v[i]);     // halo row 2 ly - 1
                    if (ly <= 8) st_shared_u32x4(sb[xk][s] + i * (6 * 2048), v[i]);            // halo row 2 ly
                  }
                }
              }
            }
            if (s != 1) {
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) {
                if (s == 0) mbar_arrive(&raw_empty[0]);
                if (s == 2) mbar_arrive(&a_full[1]);
                mbar_arrive(&a_full[s]);
              }
            }
          }
        }
      }
    } else {
    for (int wu = blockIdx.x; wu < total_units; wu += gridDim.x) {
      const int tile = wu / p.n_blocks;
      const int w0 = (tile % p.tiles_w) * kT;
      const int h0 = ((tile / p.tiles_w) % p.tiles_h) * kT;
      const int n0 = tile / tiles_img;
      if (ACT && n0 != coef_n) {
        // per-(image, channel) coefficients of this image -> shared memory (once per image: tiles of an image are
        // consecutive); the barriers keep warps that still read the old table apart from the copy
        named_bar_sync(7, kXfThreads);
        const float4* src = reinterpret_cast<const float4*>(p.coef + (long long)n0 * p.ld_coef);
        for (int i = tt; i < p.cin1 / 2; i += kXfThreads) {
          // float4 i = channels 2i, 2i+1 = quarter (i & 3) of 16-byte chunk (i >> 2): the four quarters of a chunk are
          // rotated by (chunk >> 1) so that the eight chunks of a warp's load fall into eight different bank groups
          // (unrotated, chunks j and j + 2 collide: 4-way conflicts, a quarter of the kernel's shared wavefronts)
          const float4 t = __ldg(src + i);
          const uint32_t ch = (uint32_t)i >> 2, off = ch * 64u + ((((uint32_t)i & 3u) + ((ch & 7u) >> 1)) & 3u) * 16u;
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(smem_u32(coef_tab) + off), "f"(t.x), "f"(t.y),
                       "f"(t.z), "f"(t.w) : "memory");
        }
        named_bar_sync(7, kXfThreads);
        coef_n = n0;
      }
      // the conv zero-pads the ACTIVATED tensor: halo pixels outside the image are 0 after the activation
      const bool col_out = (unsigned)(w0 - 1 + x) >= (unsigned)p.W;
      const bool first_out = col_out || (yh == 0 && h0 == 0);                 // i == 0 of the upper half: halo row 0
      const bool last_out = col_out || (yh == 1 && h0 + kT == p.H);           // i == 8 of the lower half: halo row 17
      for (int kc = 0; kc < p.kc1; ++kc, ++g) {
        PF_T0();
        mbar_wait(&raw_full[0], g & 1u);
        PF_ADD(pf_raw);
        PF_T0();
        float4 c[4];
        if constexpr (ACT) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {    // (A/2, B/2) of channels 2q, 2q+1 of this chunk, from the shared-memory table
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(c[q].x), "=f"(c[q].y), "=f"(c[q].z), "=f"(c[q].w)
                         : "r"(coef_s + (uint32_t)(kc * 512) + coef_q[q]));
          }
        }
        uint4 v[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) {
          const uint32_t sw = (uint32_t)((px0 + i * kHalo) & 7) << 4;
          const uint4 r = ld_shared_u32x4(raw0 + i * (kHalo * 128) + (j16 ^ sw));
          if constexpr (ACT) {
            v[i].x = act_pair<OUT_F16>(r.x, c[0].x, c[0].y, c[0].z, c[0].w);
            v[i].y = act_pair<OUT_F16>(r.y, c[1].x, c[1].y, c[1].z, c[1].w);
            v[i].z = act_pair<OUT_F16>(r.z, c[2].x, c[2].y, c[2].z, c[2].w);
            v[i].w = act_pair<OUT_F16>(r.w, c[3].x, c[3].y, c[3].z, c[3].w);
            const bool out = (i == 0) ? first_out : (i == 8) ? last_out : col_out;
            if (out) v[i] = make_uint4(0u, 0u, 0u, 0u);
          } else {
            v[i] = r;                                // out-of-image pixels were zero-filled by the TMA load: that IS the padding
          }
        }
        PF_ADD(pf_work);
        // The transform warps never synchronise with each other: every warp arrives on the mbarriers itself (count 9).
        // The halo buffer is released only after the first copy's stores: they depend on the loaded registers, so every
        // ld.shared of this warp has completed by then (an arrive issued right behind the loads is NOT ordered after
        // them -- with the activation compiled out (stem) the TMA refill overtook loads still in flight).
        // copy 0 is published on its own (the MMAs of this slice start with it); copies 1 and 2 share one proxy fence:
        // copy 1 is not needed before the three taps of copy 0 have been issued
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          PF_T0();
          mbar_wait(&a_empty[s], (g & 1u) ^ 1u);
          PF_ADD(pf_ae);
          if (in_copy[s]) {
#pragma unroll
            for (int i = 0; i < 9; ++i) st_shared_u32x4(so[s] + i * 2048, v[i]);
          }
          if (s != 1) {
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              if (s == 0) mbar_arrive(&raw_empty[0]);       // this warp has read its part of the halo tile
              if (s == 2) mbar_arrive(&a_full[1]);
              mbar_arrive(&a_full[s]);
            }
          }
        }
      }
    }
    }  // !UP
    if (PROF && p.prof && tt == 0) {
      unsigned long long* o = p.prof + 16 * blockIdx.x + 4;
      o[0] = (unsigned long long)(clock64() - pf_start); o[1] = pf_raw; o[2] = pf_ae; o[3] = pf_work;
    }
  } else {
    // ==================================================================== epilogue (warps 0-7): thread = output channel
    // Two warpgroups; warpgroup wg drains pixel columns [128 wg, 128 wg + 128) of the accumulator (box rows 8 wg .. 8 wg + 7)
    // in eight chunks of one 16-pixel box row.  No shared-memory transpose is needed: a warp holds 32 CONSECUTIVE channels
    // of one pixel per register index, so a 2-byte store per thread is one fully used 64-byte segment of the NHWC output
    // (and the residual a 64-byte load).  No staging buffer, no proxy fence, no barrier on this path.
    // (The first version staged [pixel][channel] tiles in shared memory for TMA stores: its fence.proxy.async -- a
    // MEMBAR.ALL.CTA that drains every shared store in flight -- and two named barriers per 4 KB chunk made the epilogue
    // pace the kernel at 15k cycles per tile against 9.2k cycles of MMAs, profiles/r2_k1s_probe.txt.)
    const int wg = warp >> 2, qw = warp & 3;           // warp qw may only touch TMEM lanes [32 qw, 32 qw + 32)
    const int cl = qw * 32 + lane;                     // TMEM lane == channel within the 128-channel block
    const uint32_t lane_sel = (uint32_t)(qw * 32) << 16;
    int acc = 0; uint32_t acc_phase = 0;
    long long pf_full = 0, pf_buf = 0, pf_ld = 0, pf_t = 0;
    const long long pf_start = PROF ? clock64() : 0;
    for (int wu = blockIdx.x; wu < total_units; wu += gridDim.x) {
      const int n_blk = wu % p.n_blocks, tile = wu / p.n_blocks;
      const int w0 = (tile % p.tiles_w) * kT;
      const int h0 = ((tile / p.tiles_w) % p.tiles_h) * kT + wg * 8;       // this warpgroup's first box row
      const int n = tile / tiles_img;
      const int co0 = n_blk * 128;
      const int c = co0 + cl;
      const bool c_ok = kHead ? (cl < p.cout_valid) : true;
      float add = 0.0f;
      if (c < p.cout) {
        if (p.bias) add = __ldg(p.bias + c);
        if (p.row_add) add += __ldg(p.row_add + (long long)n * p.ld_row_add + c);
      }
      float s1a = 0.0f, s1b = 0.0f, s2a = 0.0f, s2b = 0.0f;
      const long long pix0 = ((long long)n * p.H + h0) * p.W + w0;          // first pixel of this warpgroup's first row
      const unsigned short* rp = p.residual ? p.residual + pix0 * p.ld_res + c : nullptr;
      if (p.residual && p.res_half)      // first source pixel of this warpgroup's first row (h0, w0 are even)
        rp = p.residual + (((long long)n * (p.H >> 1) + (h0 >> 1)) * (p.W >> 1) + (w0 >> 1)) * p.ld_res + c;
      unsigned short* yp = kHead ? nullptr : p.y + pix0 * p.ld_y + c;

      PF_T0();
      mbar_wait(&tmem_full[acc], acc_phase);
      PF_ADD(pf_full);
      tc_fence_after();
      const uint32_t t_acc = tmem_base + lane_sel + (uint32_t)(acc * 256 + wg * 128);
#pragma unroll 1
      for (int chunk = 0; chunk < 8; ++chunk) {
        PF_T0();
        unsigned short rv[16];
        if (!kHead && rp) {                    // issued before the accumulator read: the loads fly under tcgen05.ld
          if (p.res_half) {                    // nearest-2x upsampled residual: source pixel (row >> 1, col >> 1)
            const unsigned short* r0 = rp + (long long)(chunk >> 1) * (p.W >> 1) * p.ld_res;
#pragma unroll
            for (int q = 0; q < 16; q += 2) rv[q] = rv[q + 1] = __ldg(r0 + (long long)(q >> 1) * p.ld_res);
          } else {
            const unsigned short* r0 = rp + (long long)chunk * p.W * p.ld_res;
#pragma unroll
            for (int q = 0; q < 16; ++q) rv[q] = __ldg(r0 + (long long)q * p.ld_res);
          }
        }
        PF_ADD(pf_buf);
        PF_T0();
        uint32_t v[16];
        tmem_ld_32x16(t_acc + (uint32_t)(chunk * 16), v);
        tc_wait_ld();
        PF_ADD(pf_ld);
        if (chunk == 7) {                      // this warp's last TMEM read of the accumulator
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty[acc]);
        }
        if constexpr (kHead) {
          if (c_ok) {
            const long long hw = (long long)p.H * p.W;
            float* o = p.y_nchw + ((long long)n * p.cout_valid + cl) * hw + (long long)(h0 + chunk) * p.W + w0;
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              float4 t;
              t.x = __uint_as_float(v[q4 * 4 + 0]) + add;
              t.y = __uint_as_float(v[q4 * 4 + 1]) + add;
              t.z = __uint_as_float(v[q4 * 4 + 2]) + add;
              t.w = __uint_as_float(v[q4 * 4 + 3]) + add;
              *reinterpret_cast<float4*>(o + q4 * 4) = t;
            }
          }
        } else {
          unsigned short* y0 = yp + (long long)chunk * p.W * p.ld_y;
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            float val = __uint_as_float(v[q]) + add;
            if (rp) val += __uint_as_float((uint32_t)rv[q] << 16);
            const unsigned short bits = __bfloat16_as_ushort(__float2bfloat16_rn(val));
            y0[(long long)q * p.ld_y] = bits;
            const float rb = __uint_as_float((uint32_t)bits << 16);
            if (q & 1) { s1b += rb; s2b = fmaf(rb, rb, s2b); } else { s1a += rb; s2a = fmaf(rb, rb, s2a); }
          }
        }
      }
      if (!kHead && p.colsum) {
        // fused GroupNorm statistics of the OUTPUT: this warpgroup's 128 pixels are one partial row, the next slot of the
        // pair (the slot grid is per 64 pixels, fidm_conv_colsum_slots) is zero; fixed-order fold later
        const int slot = (tile % tiles_img) * 4 + wg * 2;
        float2* dst = reinterpret_cast<float2*>(p.colsum) + ((long long)n * p.colsum_slots + slot) * p.cout + c;
        dst[0] = make_float2(s1a + s1b, s2a + s2b);
        dst[(long long)p.cout] = make_float2(0.0f, 0.0f);
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (PROF && p.prof && threadIdx.x == 0) {
      unsigned long long* o = p.prof + 16 * blockIdx.x + 8;
      o[0] = (unsigned long long)(clock64() - pf_start); o[1] = pf_full; o[2] = pf_buf; o[3] = pf_ld;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 18) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------ host
bool conv_halo_swap_supported(const fidm_conv_args& a) {
  using namespace halo_s;
  if (!(a.ksize == 3 && a.stride == 1 && a.height % kT == 0 && a.width % kT == 0 && a.cin % 64 == 0 && a.cin > 0 &&
        a.cin <= kMaxCin)) return false;
  if (a.x_half_res && (a.y_nchw_f32 || a.halo_copy)) return false;       // up-sampling transform: plain 128-wide layers only
  if (!(a.dtype == FIDM_F16 || a.dtype == FIDM_BF16)) return false;
  if (a.y_nchw_f32) return a.cout == 16 && !a.x2 && !a.residual && !a.colsum;
  return a.cout % 128 == 0;
}

bool conv_halo_swap_preferred(const fidm_conv_args& a) {
  return conv_halo_swap_supported(a) && (a.y_nchw_f32 || a.cout % 256 != 0);
}

template <bool OUT_F16, bool kHead, bool PROF = false, bool ACT = true, bool UP = false>
static int launch_conv_halo_swap_t(const fidm_conv_args& a, cudaStream_t st, unsigned long long* prof = nullptr) {
  using namespace halo_s;
  ConvSwapParams p;
  p.B = a.batch; p.H = a.height; p.W = a.width;
  p.tiles_w = a.width / kT; p.tiles_h = a.height / kT;
  p.n_blocks = kHead ? 1 : a.cout / 128;
  p.kc1 = a.cin / 64; p.cin1 = a.cin;
  p.kc2 = a.x2 ? a.cin2 / 64 : 0;
  p.coef = reinterpret_cast<const float2*>(a.gn_coef); p.ld_coef = a.ld_gn_coef;
  set_epilogue_params(p, a);                             // (the head variant is only supported without a residual)
  p.res_half = a.residual_half_res;
  p.y = reinterpret_cast<unsigned short*>(a.y); p.ld_y = a.ld_y;
  p.colsum_slots = p.tiles_w * p.tiles_h * 4;            // == fidm_conv_colsum_slots(H, W): one slot per 64 pixels
  p.prof = PROF ? prof : nullptr;

  CUtensorMap tmRaw, tmW, tmX2, tmW2;
  int rc;
  if (UP) {
    if ((rc = make_nhwc_map(&tmRaw, a.x, a.cin, a.width / 2, a.height / 2, a.batch, a.ld_x, kUp, kUp, 1, 0))) return rc;
  } else {
    if ((rc = make_nhwc_map(&tmRaw, a.x, a.cin, a.width, a.height, a.batch, a.ld_x, kHalo, kHalo, 1, 0))) return rc;
  }
  if ((rc = make_matrix_map(&tmW, a.w, 9 * a.cin, a.cout, 9 * a.cin, kHead ? 16 : 128, OUT_F16 ? 1 : 0))) return rc;
  if (a.x2) {
    if ((rc = make_nhwc_map(&tmX2, a.x2, a.cin2, a.width, a.height, a.batch, a.ld_x2, kT, 8, 1, 0))) return rc;
    if ((rc = make_matrix_map(&tmW2, a.w2, a.cin2, a.cout, a.cin2, 128, 0))) return rc;
  } else {
    tmX2 = tmW; tmW2 = tmW;
  }
  static bool attr_set[kMaxDevices] = {};
  FIDM_CUDA(ensure_dynamic_smem(conv_halo_swap_kernel<OUT_F16, kHead, PROF, ACT, UP>, kSmemBytes, attr_set));
  const int units = p.tiles_w * p.tiles_h * p.B * p.n_blocks;
  const int sms = num_sms();
  const int grid = units < sms ? units : sms;
  FIDM_CUDA(launch_kernel(conv_halo_swap_kernel<OUT_F16, kHead, PROF, ACT, UP>, dim3(grid), dim3(kThreads), kSmemBytes, st, 1, tmRaw, tmW, tmX2,
                          tmW2, p));
  FIDM_CHECK_LAUNCH("conv_halo_swap");
  return 0;
}

int launch_conv_halo_swap(const fidm_conv_args& a, cudaStream_t st, unsigned long long* prof) {
  FIDM_REQUIRE(conv_halo_swap_supported(a), FIDM_E_SHAPE,
               "conv (fused GroupNorm operand, swapped roles): needs 3x3 stride 1, H %% 16 == 0, W %% 16 == 0, cin %% 64 == 0, "
               "cout %% 128 == 0 (or the 16-wide fp32-NCHW head), full-resolution input");
  const bool f16 = a.dtype == FIDM_F16;
  if (a.halo_copy) {        // no activation: x is the operand (stem)
    FIDM_REQUIRE(!a.y_nchw_f32 && !a.gn_coef, FIDM_E_BADARG, "conv (halo copy): no head variant, no gn_coef");
    return f16 ? launch_conv_halo_swap_t<true, false, false, false>(a, st) : launch_conv_halo_swap_t<false, false, false, false>(a, st);
  }
  if (a.x_half_res)
    return f16 ? launch_conv_halo_swap_t<true, false, false, true, true>(a, st) : launch_conv_halo_swap_t<false, false, false, true, true>(a, st);
  if (prof && f16 && !a.y_nchw_f32) return launch_conv_halo_swap_t<true, false, true>(a, st, prof);   // instrumented (probe only)
  if (a.y_nchw_f32) return f16 ? launch_conv_halo_swap_t<true, true>(a, st) : launch_conv_halo_swap_t<false, true>(a, st);
  return f16 ? launch_conv_halo_swap_t<true, false>(a, st) : launch_conv_halo_swap_t<false, false>(a, st);
}

}  // namespace fidm
