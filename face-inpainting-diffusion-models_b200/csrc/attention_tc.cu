// K3: flash-style QKV attention on tcgen05 tensor cores (bf16, head_dim 64, non-causal).
//
// Replaces QKVAttention.forward (nn.py:222-235): the reference materialises the [B*heads, T, T] fp32
// score tensor (268 MB at T=1024, B=8) with two cuBLAS bmm calls and a softmax kernel; here a CTA
// owns 128 queries of one (batch, head) and streams 128-key tiles:
//     S = Q K^T        tcgen05.mma, A = Q tile, B = K tile (both K-major, TMA-swizzled), S in TMEM
//     P = softmax tile one query row per thread (TMEM lane == row), fp32, online max / sum
//     O += P V         tcgen05.mma, A = P (bf16, written to swizzled smem by the softmax warps),
//                      B = V tile used MN-major straight from its TMA box (no transpose pass)
// Q/K/V are read directly from the [B][T][3C] NHWC qkv buffer produced by the qkv 1x1 conv: head h is
// the channel slice [h*64,(h+1)*64) of each third (nn.py:226-234), addressed by TMA coordinates.
// warp 4 = TMA producer, warp 5 = MMA issuer, warps 0-3 = softmax / correction / epilogue.
#include <cuda.h>

#include "common.cuh"
#include "conv_host.cuh"
#include "sm100_primitives.cuh"

namespace fidm {
using namespace sm100;

struct AttnTcParams {
  int B, T, heads, C;      // C = heads * 64
  float scale_log2;        // head_dim^-1/2 * log2(e)
};

constexpr int kAttnThreads = 192;
constexpr int BQ = 128, BK = 128;
constexpr int kSubBytes = 128 * 128;      // one sub-tile: 128 rows x 64 bf16, 128-byte swizzled
constexpr int kKvStages = 2;
// HD = 64 | 128 (round 2: heads of 128 channels -- num_heads-defined heads, nn.py:245-249 -- on the tensor cores too).
// A Q / K / V tile is HD / 64 sub-tiles of [128 rows][64 channels]; P is two sub-tiles of [128 queries][64 keys].
// smem: Q | K[2] | V[2] | P (reused as the output staging tile) | barriers.  HD = 64: 112.25 KB, TWO CTAs per SM
// (with 1 KB of system reserve each), so that one CTA's softmax overlaps the other's MMAs; HD = 128: 192.25 KB, one CTA.
// No alignment slack: the dynamic shared window of a kernel without static shared memory starts 1024-byte aligned
// (checked at run time).
template <int HD> struct AttnCfg {
  static constexpr int kSub = HD / 64;
  static constexpr int kTileBytes = kSub * kSubBytes;
  static constexpr int kSmem = kTileBytes * (1 + 2 * kKvStages) + 2 * kSubBytes + 256;
  static constexpr int kCtasPerSm = HD == 64 ? 2 : 1;
};
constexpr int kAttnTmemCols = 256;        // S: columns [0,128), O tile: [128,128 + HD)

template <int HD>
__global__ void __launch_bounds__(kAttnThreads, AttnCfg<HD>::kCtasPerSm)
attn_tc_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmO, const AttnTcParams p) {
  constexpr int kSub = AttnCfg<HD>::kSub;
  constexpr int kTileBytes = AttnCfg<HD>::kTileBytes;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw;
  if ((smem_u32(smem) & 1023u) != 0u) {       // the 128-byte swizzle atoms need a 1024-byte aligned base
    if (threadIdx.x == 0) printf("fidm: attention shared memory base is not 1024-byte aligned\n");
    __trap();
  }
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + kTileBytes;
  uint8_t* sV = sK + kKvStages * kTileBytes;
  uint8_t* sP = sV + kKvStages * kTileBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 2 * kSubBytes);
  uint64_t* q_full = bars;               // 1
  uint64_t* kv_full = bars + 1;          // kKvStages
  uint64_t* kv_empty = kv_full + kKvStages;
  uint64_t* s_full = kv_empty + kKvStages;
  uint64_t* p_ready = s_full + 1;
  uint64_t* o_full = p_ready + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * BQ, h = blockIdx.y, b = blockIdx.z;
  const int n_kv = (p.T + BK - 1) / BK;

  if (warp == 4 && lane == 0) { tma_prefetch_desc(&tmQKV); tma_prefetch_desc(&tmO); }
  if (warp == 5) {
    if (lane == 0) {
      mbar_init(q_full, 1);
      for (int i = 0; i < kKvStages; ++i) { mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], 1); }
      mbar_init(s_full, 1);
      mbar_init(p_ready, 128);
      mbar_init(o_full, 1);
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, kAttnTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_S = tmem_base, tmem_O = tmem_base + 128;

  if (warp == 4) {
    if (lane == 0) {
      mbar_expect_tx(q_full, kTileBytes);
#pragma unroll
      for (int u = 0; u < kSub; ++u) tma_load_4d(&tmQKV, q_full, sQ + u * kSubBytes, h * HD + u * 64, q0, 0, b);
      int stage = 0; uint32_t phase = 0;
      for (int j = 0; j < n_kv; ++j) {
        mbar_wait(&kv_empty[stage], phase ^ 1);
        mbar_expect_tx(&kv_full[stage], 2 * kTileBytes);
#pragma unroll
        for (int u = 0; u < kSub; ++u) {
          tma_load_4d(&tmQKV, &kv_full[stage], sK + stage * kTileBytes + u * kSubBytes, p.C + h * HD + u * 64, j * BK, 0, b);
          tma_load_4d(&tmQKV, &kv_full[stage], sV + stage * kTileBytes + u * kSubBytes, 2 * p.C + h * HD + u * 64, j * BK, 0, b);
        }
        if (++stage == kKvStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 5) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = umma_idesc_bf16(128, BK, 0, 0);
      constexpr uint32_t idesc_o = umma_idesc_bf16(128, HD, 0, 1);   // B = V, MN-major
      const uint32_t aQ = smem_u32(sQ), aP = smem_u32(sP);
      mbar_wait(q_full, 0);
      int stage = 0; uint32_t phase = 0;
      // S_0
      mbar_wait(&kv_full[0], 0);
      tc_fence_after();
      {
        const uint32_t aK = smem_u32(sK);
#pragma unroll
        for (int k = 0; k < HD / 16; ++k)       // 16 channels per instruction, 64 per sub-tile
          umma_bf16(tmem_S, umma_desc_sw128(aQ + (k >> 2) * kSubBytes) + 2 * (k & 3),
                    umma_desc_sw128(aK + (k >> 2) * kSubBytes) + 2 * (k & 3), idesc_s, k ? 1u : 0u);
        umma_commit(s_full);
      }
      for (int j = 0; j < n_kv; ++j) {
        // O_tile = P_j V_j
        mbar_wait(p_ready, j & 1);
        tc_fence_after();
        const uint32_t aV = smem_u32(sV + stage * kTileBytes);
#pragma unroll
        for (int kk = 0; kk < BK / 16; ++kk) {
          const uint64_t dp = umma_desc_sw128(aP + (kk >> 2) * kSubBytes) + (uint64_t)(2 * (kk & 3));
          // V as the MN-major B operand: N = HD channels, 64 per sub-tile (LBO = distance between the 64-channel blocks)
          const uint64_t dv = umma_desc_sw128_mn(aV + kk * 2048, kSubBytes);
          umma_bf16(tmem_O, dp, dv, idesc_o, kk ? 1u : 0u);
        }
        umma_commit(&kv_empty[stage]);
        umma_commit(o_full);
        if (++stage == kKvStages) { stage = 0; phase ^= 1; }
        // S_{j+1} = Q K_{j+1}^T   (the softmax warps have finished reading S_j: p_ready_j)
        if (j + 1 < n_kv) {
          mbar_wait(&kv_full[stage], phase);
          tc_fence_after();
          const uint32_t aK = smem_u32(sK + stage * kTileBytes);
#pragma unroll
          for (int k = 0; k < HD / 16; ++k)
            umma_bf16(tmem_S, umma_desc_sw128(aQ + (k >> 2) * kSubBytes) + 2 * (k & 3),
                      umma_desc_sw128(aK + (k >> 2) * kSubBytes) + 2 * (k & 3), idesc_s, k ? 1u : 0u);
          umma_commit(s_full);
        }
      }
    }
  } else {
    // ------------------------------------------------------------ softmax / correction / epilogue
    const int row = warp * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(warp * 32) << 16;
    float m_run = -INFINITY, l_run = 0.0f;
    float o[HD];
#pragma unroll
    for (int i = 0; i < HD; ++i) o[i] = 0.0f;
    uint8_t* prow = sP + row * 128;

    for (int j = 0; j < n_kv; ++j) {
      const int kv_valid = min(BK, p.T - j * BK);
      mbar_wait(s_full, j & 1);
      tc_fence_after();
      // pass 1: row max
      float mx = -INFINITY;
#pragma unroll 1
      for (int c = 0; c < BK / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(tmem_S + lane_sel + c * 32, v);
        tc_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (c * 32 + i < kv_valid) mx = fmaxf(mx, __uint_as_float(v[i]));
      }
      const float m_new = fmaxf(m_run, mx);
      const float alpha = exp2f((m_run - m_new) * p.scale_log2);
      const float mb = m_new * p.scale_log2;
      // pass 2: P = exp2(s * c - m * c) -> bf16 -> swizzled smem (A operand of the PV MMA)
      float rs = 0.0f;
#pragma unroll 1
      for (int c = 0; c < BK / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(tmem_S + lane_sel + c * 32, v);
        tc_wait_ld();
        float pv[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float e = exp2f(fmaf(__uint_as_float(v[i]), p.scale_log2, -mb));
          pv[i] = (c * 32 + i < kv_valid) ? e : 0.0f;
          rs += pv[i];
        }
        uint8_t* chunk = prow + (c >> 1) * kSubBytes;      // 64 keys per swizzled K-chunk
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          uint4 pk;
          __nv_bfloat162 b0 = __floats2bfloat162_rn(pv[8 * u + 0], pv[8 * u + 1]);
          __nv_bfloat162 b1 = __floats2bfloat162_rn(pv[8 * u + 2], pv[8 * u + 3]);
          __nv_bfloat162 b2 = __floats2bfloat162_rn(pv[8 * u + 4], pv[8 * u + 5]);
          __nv_bfloat162 b3 = __floats2bfloat162_rn(pv[8 * u + 6], pv[8 * u + 7]);
          pk.x = *reinterpret_cast<uint32_t*>(&b0);
          pk.y = *reinterpret_cast<uint32_t*>(&b1);
          pk.z = *reinterpret_cast<uint32_t*>(&b2);
          pk.w = *reinterpret_cast<uint32_t*>(&b3);
          const int unit = (c & 1) * 4 + u;
          *reinterpret_cast<uint4*>(chunk + ((unit ^ (row & 7)) << 4)) = pk;
        }
      }
      l_run = l_run * alpha + rs;
      m_run = m_new;
      fence_proxy_async_smem();      // P visible to the tensor core (async proxy)
      tc_fence_before();             // our TMEM reads of S are ordered before the next S MMA
      mbar_arrive(p_ready);

      // O = O * alpha + P V
      mbar_wait(o_full, j & 1);
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < HD / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(tmem_O + lane_sel + c * 32, v);
        tc_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; ++i) o[c * 32 + i] = fmaf(o[c * 32 + i], alpha, __uint_as_float(v[i]));
      }
      tc_fence_before();
    }
    // ---- epilogue: O / l -> bf16 -> swizzled staging (reuses P chunk 0; the last PV MMA completed: o_full)
    const float inv = 1.0f / l_run;
#pragma unroll
    for (int u = 0; u < HD / 8; ++u) {       // 8 channels per 16-byte unit, 8 units per 64-channel sub-tile
      uint4 pk;
      __nv_bfloat162 b0 = __floats2bfloat162_rn(o[8 * u + 0] * inv, o[8 * u + 1] * inv);
      __nv_bfloat162 b1 = __floats2bfloat162_rn(o[8 * u + 2] * inv, o[8 * u + 3] * inv);
      __nv_bfloat162 b2 = __floats2bfloat162_rn(o[8 * u + 4] * inv, o[8 * u + 5] * inv);
      __nv_bfloat162 b3 = __floats2bfloat162_rn(o[8 * u + 6] * inv, o[8 * u + 7] * inv);
      pk.x = *reinterpret_cast<uint32_t*>(&b0);
      pk.y = *reinterpret_cast<uint32_t*>(&b1);
      pk.z = *reinterpret_cast<uint32_t*>(&b2);
      pk.w = *reinterpret_cast<uint32_t*>(&b3);
      *reinterpret_cast<uint4*>(prow + (u >> 3) * kSubBytes + (((u & 7) ^ (row & 7)) << 4)) = pk;
    }
    fence_proxy_async_smem();
    named_bar_sync(1, 128);
    if (threadIdx.x == 0) {
#pragma unroll
      for (int u = 0; u < kSub; ++u) tma_store_4d(&tmO, sP + u * kSubBytes, h * HD + u * 64, q0, 0, b);
      bulk_commit_group();
      bulk_wait_group_read<0>();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kAttnTmemCols);
  }
}

}  // namespace fidm

extern "C" int fidm_attention_qkv_nhwc_bf16(const fidm_attn_args* a, fidm_stream_t stream) {
  using namespace fidm;
  FIDM_REQUIRE(a && a->qkv && a->out, FIDM_E_BADARG, "attention_tc: null qkv/out");
  FIDM_REQUIRE(a->dtype == FIDM_BF16, FIDM_E_BADARG, "attention_tc: dtype must be bf16");
  FIDM_REQUIRE(a->head_dim == 64 || a->head_dim == 128, FIDM_E_SHAPE, "attention_tc: head_dim %d (64 or 128)", a->head_dim);
  FIDM_REQUIRE(a->batch > 0 && a->tokens > 0 && a->heads > 0, FIDM_E_BADARG, "attention_tc: empty shape");
  const int Cn = a->heads * a->head_dim;
  FIDM_REQUIRE(a->ld_qkv >= 3 * Cn && a->ld_out >= Cn, FIDM_E_BADARG, "attention_tc: ld too small");
  AttnTcParams p;
  p.B = a->batch; p.T = a->tokens; p.heads = a->heads; p.C = Cn;
  p.scale_log2 = (1.0f / sqrtf((float)a->head_dim)) * 1.4426950408889634f;     // (d^-1/4)^2 * log2(e)
  CUtensorMap tmQKV, tmO;
  int rc;
  // [B][T][3C] viewed as NHWC with H = 1: box = 64 channels x 128 tokens
  if ((rc = make_nhwc_map(&tmQKV, a->qkv, 3 * Cn, a->tokens, 1, a->batch, a->ld_qkv, 128, 1, 1, 0))) return rc;
  if ((rc = make_nhwc_map(&tmO, a->out, Cn, a->tokens, 1, a->batch, a->ld_out, 128, 1, 1, 0))) return rc;
  dim3 grid((a->tokens + BQ - 1) / BQ, a->heads, a->batch);
  if (a->head_dim == 64) {
    static bool attr_set[kMaxDevices] = {};      // per (instantiation, device)
    FIDM_CUDA(ensure_dynamic_smem(attn_tc_kernel<64>, AttnCfg<64>::kSmem, attr_set));
    FIDM_CUDA(launch_kernel(attn_tc_kernel<64>, grid, dim3(kAttnThreads), AttnCfg<64>::kSmem, (cudaStream_t)stream, 1, tmQKV, tmO, p));
  } else {
    static bool attr_set[kMaxDevices] = {};
    FIDM_CUDA(ensure_dynamic_smem(attn_tc_kernel<128>, AttnCfg<128>::kSmem, attr_set));
    FIDM_CUDA(launch_kernel(attn_tc_kernel<128>, grid, dim3(kAttnThreads), AttnCfg<128>::kSmem, (cudaStream_t)stream, 1, tmQKV, tmO, p));
  }
  FIDM_CHECK_LAUNCH("attention_tc");
  return 0;
}
