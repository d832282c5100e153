// K2: GroupNorm(32) [* (1+scale) + shift] [SiLU] [2x avg-pool | 2x nearest-up] on NHWC tensors.
//
// Replaces nn.GroupNorm + nn.SiLU (nn.py:46-48,151-152,173-174; unet.py:149-150; nn.py:251), the
// scale/shift modulation (nn.py:203-206) and the h_upd / x_upd resampling of up/down ResBlocks
// (nn.py:190-195).  HBM-bound: 2 B read (stats pass, normally L2-resident for the second pass) +
// 2 B read + 2 B write per bf16 element.
//
// Thread mapping (both passes): a thread owns one VEC-wide channel vector and walks pixels, so a
// warp reads consecutive 16-byte vectors of one pixel (fully coalesced) and keeps its per-channel
// affine coefficients in registers.  Statistics are accumulated in fp32 per thread, then reduced in
// double precision in a fixed order (block partials, folded by the last block of each image to finish):
// no floating-point atomics, so the result is bit-reproducible.

#include "common.cuh"

namespace fidm {

struct GnParams {
  fidm_gn_args a;
  int cv;          // channel vectors per pixel
  int ppi;         // pixels processed per block iteration
  int pix_per_blk; // pixels (of the iteration space) per block
};

// Halved affine coefficients of GroupNorm [* (1+scale) + shift] followed by SiLU for channel c of image n
// (silu(x*A + B) = h + h*tanh(h), h = x*A/2 + B/2): what the K1h conv applies in its operand path.
__device__ __forceinline__ float2 gn_half_coeff(const fidm_gn_args& a, int n, int c, float meanf, float rstd) {
  const float ga = a.gamma ? a.gamma[c] : 1.0f;
  const float be = a.beta ? a.beta[c] : 0.0f;
  float Ai = rstd * ga;
  float Bi = be - meanf * Ai;
  if (a.scale_shift) {
    const float sc = 1.0f + a.scale_shift[(long long)n * a.ld_ss + c];
    const float sh = a.scale_shift[(long long)n * a.ld_ss + a.channels + c];
    Ai *= sc;
    Bi = Bi * sc + sh;
  }
  return make_float2(0.5f * Ai, 0.5f * Bi);
}

// Pass 1: per-block partial (sum, sum of squares) of every group, reduced in a FIXED order (no
// atomics) so that results are bit-reproducible run to run.  partials: [batch][chunks][groups][2].
template <typename T, int VEC>
__global__ void gn_stats_kernel(const GnParams p, double* __restrict__ partials, int* __restrict__ counters,
                                float2* __restrict__ coef, int ld_coef) {
  const fidm_gn_args& a = p.a;
  extern __shared__ float red[];           // [blockDim][2]
  const int n = blockIdx.y;
  const int hw = a.height * a.width;
  const int v = threadIdx.x % p.cv;
  const int pl = threadIdx.x / p.cv;
  const int cpg = a.channels / a.groups;
  const int p0 = blockIdx.x * p.pix_per_blk;
  const int p1 = min(hw, p0 + p.pix_per_blk);
  const T* base = reinterpret_cast<const T*>(a.x) + (long long)n * hw * a.ld_x + v * VEC;
  float s = 0.0f, ss = 0.0f;
  for (int px = p0 + pl; px < p1; px += p.ppi) {
    float f[VEC];
    load_vec<T, VEC>(base + (long long)px * a.ld_x, f);
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      s += f[i];
      ss = fmaf(f[i], f[i], ss);
    }
  }
  red[2 * threadIdx.x] = s;
  red[2 * threadIdx.x + 1] = ss;
  __syncthreads();
  // group g owns vectors [g*vpg, (g+1)*vpg) of every pixel lane
  const int vpg = cpg / VEC;
  for (int g = threadIdx.x; g < a.groups; g += blockDim.x) {
    double ds = 0.0, dss = 0.0;
    for (int l = 0; l < p.ppi; ++l)
      for (int k = 0; k < vpg; ++k) {
        const int t = l * p.cv + g * vpg + k;
        ds += (double)red[2 * t];
        dss += (double)red[2 * t + 1];
      }
    double* o = partials + (((long long)n * gridDim.x + blockIdx.x) * a.groups + g) * 2;
    o[0] = ds;
    o[1] = dss;
  }
  // The last block of image n to finish folds all partials of that image, in a fixed order, into
  // (mean, rstd): deterministic, and no separate finalize launch.
  __shared__ int is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const int done = atomicAdd(&counters[n], 1);
    is_last = (done == (int)gridDim.x - 1);
    if (is_last) counters[n] = 0;             // re-arm for the next launch
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  __syncthreads();
  // slice j of the block sums chunks j, j+S, ... of group g (4 independent loads in flight), then the
  // S slice totals of each group are added in slice order: a fixed summation tree.
  const int chunks = gridDim.x;
  const int G = a.groups;
  const int S = max(1, min((int)blockDim.x / G, 8));
  double* red2 = reinterpret_cast<double*>(red);      // [S][G][2] doubles; red[] holds >= 2*blockDim floats
  const int g = threadIdx.x % G, j = threadIdx.x / G;
  if (j < S) {
    double ds = 0.0, dss = 0.0;
    const double* q = partials + ((long long)n * chunks * G + g) * 2;
    int c = j;
    for (; c + 3 * S < chunks; c += 4 * S) {
      const double2 v0 = __ldcg(reinterpret_cast<const double2*>(q + (long long)c * G * 2));
      const double2 v1 = __ldcg(reinterpret_cast<const double2*>(q + (long long)(c + S) * G * 2));
      const double2 v2 = __ldcg(reinterpret_cast<const double2*>(q + (long long)(c + 2 * S) * G * 2));
      const double2 v3 = __ldcg(reinterpret_cast<const double2*>(q + (long long)(c + 3 * S) * G * 2));
      ds += v0.x; dss += v0.y; ds += v1.x; dss += v1.y; ds += v2.x; dss += v2.y; ds += v3.x; dss += v3.y;
    }
    for (; c < chunks; c += S) {
      const double2 v = __ldcg(reinterpret_cast<const double2*>(q + (long long)c * G * 2));
      ds += v.x; dss += v.y;
    }
    red2[(j * G + g) * 2] = ds;
    red2[(j * G + g) * 2 + 1] = dss;
  }
  __syncthreads();
  if (threadIdx.x < G) {
    double ds = 0.0, dss = 0.0;
    for (int k = 0; k < S; ++k) {
      ds += red2[(k * G + g) * 2];
      dss += red2[(k * G + g) * 2 + 1];
    }
    const double count = (double)cpg * hw;
    const double mean = ds / count;
    double var = dss / count - mean * mean;
    if (var < 0.0) var = 0.0;
    float* mr = reinterpret_cast<float*>(a.stats) + ((long long)n * G + g) * 2;
    mr[0] = (float)mean;
    mr[1] = (float)(1.0 / sqrt(var + (double)a.eps));
  }
  if (coef) {      // statistics-only call: the last block also writes the per-channel coefficients (no extra launch)
    __threadfence_block();
    __syncthreads();
    const float* mr = reinterpret_cast<const float*>(a.stats) + (long long)n * G * 2;
    for (int c = threadIdx.x; c < a.channels; c += blockDim.x)
      coef[(long long)n * ld_coef + c] = gn_half_coeff(a, n, c, mr[2 * (c / cpg)], mr[2 * (c / cpg) + 1]);
  }
}

// Small tensors (L2-resident): one block per (image, group) reads that group's channel slice of every pixel
// and reduces it in a fixed tree -- no workspace, no cross-block step, one short launch.
template <typename T, int VEC>
__global__ void __launch_bounds__(256) gn_stats_direct_kernel(const GnParams p, float2* __restrict__ coef, int ld_coef) {
  const fidm_gn_args& a = p.a;
  __shared__ double red[8][2];
  __shared__ float mr_s[2];
  const int g = blockIdx.x, n = blockIdx.y;
  const int hw = a.height * a.width;
  const int cpg = a.channels / a.groups;
  const int vpp = cpg / VEC;                          // vectors per pixel in this group
  const T* base = reinterpret_cast<const T*>(a.x) + (long long)n * hw * a.ld_x + g * cpg;
  float s = 0.0f, ss = 0.0f;
  const int total = hw * vpp;
  for (int i = threadIdx.x; i < total; i += 256) {
    const int px = i / vpp, j = i - px * vpp;
    float f[VEC];
    load_vec<T, VEC>(base + (long long)px * a.ld_x + j * VEC, f);
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      s += f[k];
      ss = fmaf(f[k], f[k], ss);
    }
  }
  double ds = (double)s, dss = (double)ss;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ds += __shfl_xor_sync(0xffffffffu, ds, o);
    dss += __shfl_xor_sync(0xffffffffu, dss, o);
  }
  if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5][0] = ds; red[threadIdx.x >> 5][1] = dss; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a0 = 0.0, a1 = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { a0 += red[k][0]; a1 += red[k][1]; }
    const double cnt = (double)cpg * hw;
    const double mean = a0 / cnt;
    double var = a1 / cnt - mean * mean;
    if (var < 0.0) var = 0.0;
    float* mr = reinterpret_cast<float*>(a.stats) + ((long long)n * a.groups + g) * 2;
    mr[0] = mr_s[0] = (float)mean;
    mr[1] = mr_s[1] = (float)(1.0 / sqrt(var + (double)a.eps));
  }
  if (coef) {      // statistics-only call: this block writes the coefficients of its group's channels (no extra launch)
    __syncthreads();
    for (int c = g * cpg + threadIdx.x; c < (g + 1) * cpg; c += 256)
      coef[(long long)n * ld_coef + c] = gn_half_coeff(a, n, c, mr_s[0], mr_s[1]);
  }
}

template <bool FAST>
__device__ __forceinline__ float silu_f(float v) {
  if (FAST) {  // x*sigmoid(x) = h + h*tanh(h), h = x/2: one MUFU op (tanh.approx) instead of ex2 + rcp
    const float h = 0.5f * v;
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    return fmaf(h, t, h);
  }
  return v / (1.0f + expf(-v));
}

// Small (L2-resident) tensors: ONE launch.  A block owns one (image, group): it reads the group's channel slice of every
// pixel once into registers, reduces (sum, sum of squares) in a fixed tree, and writes the normalized / activated
// values -- instead of a statistics launch plus an apply launch that reads the tensor twice.  Up to NV 16-byte vectors
// per thread (NV * blockDim vectors per (image, group)).
// CS = 4 | 2: the (image, group) is shared by a thread-block CLUSTER of CS blocks (block r owns vectors k = r*NV ..
// r*NV+NV-1 of every thread slot); the (sum, sum of squares) partials are exchanged through distributed shared memory
// (16 bytes per block: the one place on this path where DSMEM's ~20 B/clk is plenty) and folded in rank order by every
// block.  Used where batch x groups blocks cannot fill the machine (batch 1-2): CS x the blocks, CS x the reach (a 64x64
// image of a 512-channel tensor, 8192 vectors per group, in one launch).
template <typename TY, int NV, int CS = 1>
__global__ void __launch_bounds__(512, 1) gn_fused_small_kernel(const fidm_gn_args a, int vpp, int stride) {
  __shared__ double red[16][2];
  __shared__ __align__(16) double part[2];
  __shared__ float mr[2];
  constexpr bool FAST = true;
  const int rank = CS > 1 ? (int)(blockIdx.x % CS) : 0;          // == %cluster_ctarank (cluster dims (CS, 1, 1))
  const int g = blockIdx.x / CS, n = blockIdx.y;
  const int hw = a.height * a.width;
  const int cpg = a.channels / a.groups;
  const int total = hw * vpp;                           // 16-byte vectors of this (image, group)
  const int t = threadIdx.x;
  const bool active = t < stride;                       // stride = largest multiple of vpp <= blockDim: the channel
  const int jv = t % vpp;                               // chunk (t % vpp) of a thread is the same for all its vectors
  const __nv_bfloat16* xin = reinterpret_cast<const __nv_bfloat16*>(a.x) + (long long)n * hw * a.ld_x + g * cpg;
  uint4 v[NV];
  float s = 0.0f, ss = 0.0f;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int i = t + (rank * NV + k) * stride;
    v[k] = make_uint4(0u, 0u, 0u, 0u);
    if (active && i < total) v[k] = *reinterpret_cast<const uint4*>(xin + (long long)(i / vpp) * a.ld_x + jv * 8);
  }
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const uint32_t u[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float f0 = __uint_as_float(u[e] << 16), f1 = __uint_as_float(u[e] & 0xFFFF0000u);
      s += f0 + f1;
      ss = fmaf(f0, f0, ss);
      ss = fmaf(f1, f1, ss);
    }
  }
  // the affine parameters do not depend on the statistics: their loads are issued here, under the reduction (the
  // kernel is a chain of latencies -- tensor read, reduction, parameter read, write -- not a bandwidth problem)
  const int c0 = g * cpg + jv * 8;
  float ga[8], be[8], sc[8], sh[8];
  auto load_affine = [&]() {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      ga[i] = (active && a.gamma) ? __ldg(a.gamma + c0 + i) : 1.0f;
      be[i] = (active && a.beta) ? __ldg(a.beta + c0 + i) : 0.0f;
      sc[i] = (active && a.scale_shift) ? 1.0f + __ldg(a.scale_shift + (long long)n * a.ld_ss + c0 + i) : 1.0f;
      sh[i] = (active && a.scale_shift) ? __ldg(a.scale_shift + (long long)n * a.ld_ss + a.channels + c0 + i) : 0.0f;
    }
  };
  load_affine();
  double ds = (double)s, dss = (double)ss;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ds += __shfl_xor_sync(0xffffffffu, ds, o);
    dss += __shfl_xor_sync(0xffffffffu, dss, o);
  }
  if ((t & 31) == 0) { red[t >> 5][0] = ds; red[t >> 5][1] = dss; }
  __syncthreads();
  if (CS > 1) {
    if (t == 0) {
      double a0 = 0.0, a1 = 0.0;
      for (int k = 0; k < (int)(blockDim.x >> 5); ++k) { a0 += red[k][0]; a1 += red[k][1]; }
      part[0] = a0;
      part[1] = a1;
    }
    // release / acquire at cluster scope: every block's partial is visible to its peers
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
  }
  if (t == 0) {
    double a0 = 0.0, a1 = 0.0;
    if (CS > 1) {
      const uint32_t local = (uint32_t)__cvta_generic_to_shared(part);
#pragma unroll
      for (int r = 0; r < CS; ++r) {               // fixed order: identical statistics in all blocks of the cluster
        double p0, p1;
        asm volatile(
            "{\n\t.reg .b32 ra;\n\t"
            "mapa.shared::cluster.u32 ra, %2, %3;\n\t"
            "ld.shared::cluster.v2.f64 {%0, %1}, [ra];\n\t}"
            : "=d"(p0), "=d"(p1) : "r"(local), "r"(r) : "memory");
        a0 += p0;
        a1 += p1;
      }
    } else {
      for (int k = 0; k < (int)(blockDim.x >> 5); ++k) { a0 += red[k][0]; a1 += red[k][1]; }
    }
    const double cnt = (double)cpg * hw;
    const double mean = a0 / cnt;
    double var = a1 / cnt - mean * mean;
    if (var < 0.0) var = 0.0;
    mr[0] = (float)mean;
    mr[1] = (float)(1.0 / sqrt(var + (double)a.eps));
  }
  __syncthreads();
  if (active) {
    const float meanf = mr[0], rstd = mr[1];
    float A[8], B[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float Ai = rstd * ga[i];
      float Bi = be[i] - meanf * Ai;
      if (a.scale_shift) {
        Ai *= sc[i];
        Bi = Bi * sc[i] + sh[i];
      }
      A[i] = Ai;
      B[i] = Bi;
    }
    TY* yo = reinterpret_cast<TY*>(a.y) + (long long)n * hw * a.ld_y + c0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int i = t + (rank * NV + k) * stride;
      if (i < total) {
        const uint32_t u[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
        float f[8];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float y0 = fmaf(__uint_as_float(u[e] << 16), A[2 * e], B[2 * e]);
          const float y1 = fmaf(__uint_as_float(u[e] & 0xFFFF0000u), A[2 * e + 1], B[2 * e + 1]);
          f[2 * e] = a.silu ? silu_f<FAST>(y0) : y0;
          f[2 * e + 1] = a.silu ? silu_f<FAST>(y1) : y1;
        }
        store_vec<TY, 8>(yo + (long long)(i / vpp) * a.ld_y, f);
      }
    }
  }
  // no block of the cluster may exit while a peer can still read its partial
  if (CS > 1) asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// bf16 input, no resampling, no fused producer statistics, 16-byte aligned group slices, <= 8 * 512 vectors per
// (image, group): the one-launch path.  Returns -1 when it does not apply.
static bool gn_fused_small_plan(const fidm_gn_args& a, int* vpp_o, int* threads_o, int* stride_o, int* per_thread_o,
                                int* cluster_o = nullptr) {
  const int cpg = a.channels / a.groups;
  if (a.dtype != FIDM_BF16 || (a.y_dtype != FIDM_BF16 && a.y_dtype != FIDM_F16)) return false;
  if (a.skip_norm || a.chansum || a.resample != FIDM_RESAMPLE_NONE || cpg % 8 != 0) return false;
  if (a.ld_x % 8 || a.ld_y % 8 || (uintptr_t)a.x % 16 || (uintptr_t)a.y % 16) return false;
  const int vpp = cpg / 8;
  const long long total = (long long)a.height * a.width * vpp;
  const int threads = total >= 512 ? 512 : (int)((total + 31) / 32) * 32;
  if (threads < vpp) return false;
  const int stride = (threads / vpp) * vpp;
  long long per_thread = (total + stride - 1) / stride;
  // a 4- or 2-block cluster per (image, group) where the clustered grid is still one wave (one 512-thread block per SM)
  // and a thread would otherwise hold more than 4 vectors -- measured at batch 1: 8 vectors per thread 8.8 us alone,
  // 6.9 us as a cluster; <= 4 vectors 6.4 us alone, 6.9 us as a cluster; 8192 vectors per group 23 us in two launches,
  // 8.3 us as a cluster (profiles/r2_launches_adm256_b1_summary.txt)
  int cluster = 1;
  if (per_thread > 4) {
    const long long blocks = (long long)a.batch * a.groups;
    if (blocks * 4 <= num_sms()) cluster = 4;
    else if (blocks * 2 <= num_sms()) cluster = 2;
    per_thread = (per_thread + cluster - 1) / cluster;
  }
  if (per_thread > 8) return false;    // 8 vectors (64 values) per thread stay in registers
  *vpp_o = vpp; *threads_o = threads; *stride_o = stride; *per_thread_o = (int)per_thread;
  if (cluster_o) *cluster_o = cluster;
  return true;
}

template <typename TY>
static int try_gn_fused_small(const fidm_gn_args& a, cudaStream_t st) {
  int vpp, threads, stride, per_thread, cluster;
  if (!gn_fused_small_plan(a, &vpp, &threads, &stride, &per_thread, &cluster)) return -1;
  dim3 grid(a.groups * cluster, a.batch);
  if (cluster == 4) {
    if (per_thread <= 2) launch_kernel(gn_fused_small_kernel<TY, 2, 4>, grid, dim3(threads), 0, st, 4, a, vpp, stride);
    else if (per_thread <= 4) launch_kernel(gn_fused_small_kernel<TY, 4, 4>, grid, dim3(threads), 0, st, 4, a, vpp, stride);
    else launch_kernel(gn_fused_small_kernel<TY, 8, 4>, grid, dim3(threads), 0, st, 4, a, vpp, stride);
  } else if (cluster == 2) {
    if (per_thread <= 4) launch_kernel(gn_fused_small_kernel<TY, 4, 2>, grid, dim3(threads), 0, st, 2, a, vpp, stride);
    else launch_kernel(gn_fused_small_kernel<TY, 8, 2>, grid, dim3(threads), 0, st, 2, a, vpp, stride);
  }
  else if (per_thread <= 2) launch_kernel(gn_fused_small_kernel<TY, 2>, grid, dim3(threads), 0, st, 1, a, vpp, stride);
  else if (per_thread <= 4) launch_kernel(gn_fused_small_kernel<TY, 4>, grid, dim3(threads), 0, st, 1, a, vpp, stride);
  else launch_kernel(gn_fused_small_kernel<TY, 8>, grid, dim3(threads), 0, st, 1, a, vpp, stride);
  FIDM_CHECK_LAUNCH("groupnorm (fused small)");
  return 0;
}

template <typename T, typename TY, int VEC, int RESAMPLE>
__global__ void __launch_bounds__(1024, 1) gn_apply_kernel(const GnParams p) {
  const fidm_gn_args& a = p.a;
  constexpr bool FAST = (sizeof(T) == 2);
  const int n = blockIdx.y;
  const int H = a.height, W = a.width, hw = H * W;
  const int v = threadIdx.x % p.cv;
  const int pl = threadIdx.x / p.cv;
  const int cpg = a.channels / a.groups;
  const int c0 = v * VEC;
  const int g = c0 / cpg;

  // per-thread affine coefficients  y = x * A + B
  float A[VEC], B[VEC];
  if (a.skip_norm) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) { A[i] = 1.0f; B[i] = 0.0f; }
  } else {
    float meanf, rstd;
    if (a.chansum) {
      // statistics from the producer conv's fused column sums: the block stages the image's channel sums in
      // shared memory (one coalesced read), `groups` threads fold their channels in a fixed order.
      extern __shared__ float2 cs_s[];                   // [channels] then [groups] (mean, rstd)
      float2* mr_s = cs_s + a.channels;
      const float2* cs = reinterpret_cast<const float2*>(a.chansum) + (long long)n * a.ld_chansum;
      for (int c = threadIdx.x; c < a.channels; c += blockDim.x) cs_s[c] = cs[c];
      __syncthreads();
      if (threadIdx.x < a.groups) {
        double ds = 0.0, dss = 0.0;
        for (int k = 0; k < cpg; ++k) {
          const float2 v = cs_s[threadIdx.x * cpg + k];
          ds += (double)v.x;
          dss += (double)v.y;
        }
        const double cnt = (double)cpg * hw;
        const double mean = ds / cnt;
        double var = dss / cnt - mean * mean;
        if (var < 0.0) var = 0.0;
        mr_s[threadIdx.x] = make_float2((float)mean, (float)(1.0 / sqrt(var + (double)a.eps)));
      }
      __syncthreads();
      meanf = mr_s[g].x;
      rstd = mr_s[g].y;
    } else {
      const float* mr = reinterpret_cast<const float*>(a.stats) + ((long long)n * a.groups + g) * 2;
      meanf = mr[0];
      rstd = mr[1];
    }
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float ga = a.gamma ? a.gamma[c0 + i] : 1.0f;
      const float be = a.beta ? a.beta[c0 + i] : 0.0f;
      float Ai = rstd * ga;
      float Bi = be - meanf * Ai;
      if (a.scale_shift) {
        const float sc = 1.0f + a.scale_shift[(long long)n * a.ld_ss + c0 + i];
        const float sh = a.scale_shift[(long long)n * a.ld_ss + a.channels + c0 + i];
        Ai *= sc;
        Bi = Bi * sc + sh;
      }
      A[i] = Ai;
      B[i] = Bi;
    }
  }
  const T* xin = reinterpret_cast<const T*>(a.x) + (long long)n * hw * a.ld_x + c0;
  TY* yo = reinterpret_cast<TY*>(a.y);
  T* yr = reinterpret_cast<T*>(a.y_raw);

  if (RESAMPLE == FIDM_RESAMPLE_NONE) {
    const int p0 = blockIdx.x * p.pix_per_blk, p1 = min(hw, p0 + p.pix_per_blk);
    // 4 independent 16-byte loads in flight per thread (kept packed to stay within 64 registers): with one
    // load per thread the kernel is latency-bound at ~70 % of the HBM copy rate (Little's law).
    constexpr int U = 4;
    for (int px = p0 + pl; px < p1; px += p.ppi * U) {
      Vec<T, VEC> raw[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int q = px + u * p.ppi;
        if (q < p1) raw[u] = *reinterpret_cast<const Vec<T, VEC>*>(xin + (long long)q * a.ld_x);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int q = px + u * p.ppi;
        if (q < p1) {
          float f[VEC];
#pragma unroll
          for (int i = 0; i < VEC; ++i) {
            const float y = fmaf(to_f32<T>(raw[u].v[i]), A[i], B[i]);
            f[i] = a.silu ? silu_f<FAST>(y) : y;
          }
          store_vec<TY, VEC>(yo + ((long long)n * hw + q) * a.ld_y + c0, f);
        }
      }
    }
  } else if (RESAMPLE == FIDM_RESAMPLE_DOWN) {
    const int Ho = H / 2, Wo = W / 2, ohw = Ho * Wo;
    const int p0 = blockIdx.x * p.pix_per_blk, p1 = min(ohw, p0 + p.pix_per_blk);
    for (int px = p0 + pl; px < p1; px += p.ppi) {
      const int ho = px / Wo, wo = px % Wo;
      float acc[VEC], raw[VEC];
#pragma unroll
      for (int i = 0; i < VEC; ++i) acc[i] = raw[i] = 0.0f;
#pragma unroll
      for (int d = 0; d < 4; ++d) {
        const int ip = (2 * ho + (d >> 1)) * W + 2 * wo + (d & 1);
        float f[VEC];
        load_vec<T, VEC>(xin + (long long)ip * a.ld_x, f);
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
          raw[i] += f[i];
          float y = fmaf(f[i], A[i], B[i]);
          acc[i] += a.silu ? silu_f<FAST>(y) : y;
        }
      }
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        acc[i] *= 0.25f;
        raw[i] *= 0.25f;
      }
      store_vec<TY, VEC>(yo + ((long long)n * ohw + px) * a.ld_y + c0, acc);
      if (yr) store_vec<T, VEC>(yr + ((long long)n * ohw + px) * a.ld_raw + c0, raw);
    }
  } else {  // nearest 2x up: one input pixel feeds four outputs
    const int Wo = 2 * W, ohw = 4 * hw;
    const int p0 = blockIdx.x * p.pix_per_blk, p1 = min(hw, p0 + p.pix_per_blk);
    for (int px = p0 + pl; px < p1; px += p.ppi) {
      const int h = px / W, w = px % W;
      float f[VEC], y[VEC];
      load_vec<T, VEC>(xin + (long long)px * a.ld_x, f);
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        float t = fmaf(f[i], A[i], B[i]);
        y[i] = a.silu ? silu_f<FAST>(t) : t;
      }
#pragma unroll
      for (int d = 0; d < 4; ++d) {
        const long long op = (long long)n * ohw + (long long)(2 * h + (d >> 1)) * Wo + 2 * w + (d & 1);
        store_vec<TY, VEC>(yo + op * a.ld_y + c0, y);
        if (yr) store_vec<T, VEC>(yr + op * a.ld_raw + c0, f);
      }
    }
  }
}


// Statistics -> per-(image, channel) affine coefficients of GroupNorm [* (1+scale) + shift] + SiLU, halved
// (silu(x*A + B) = h + h*tanh(h), h = x*A/2 + B/2).  Same arithmetic as the head of gn_apply_kernel, so a conv that
// applies the activation in its operand path sees exactly the coefficients the apply pass would have used.
__global__ void __launch_bounds__(256) gn_coeff_kernel(const fidm_gn_args a, float2* __restrict__ coef, int ld_coef) {
  __shared__ float2 mr_s[64];
  const int n = blockIdx.x;
  const int hw = a.height * a.width;
  const int cpg = a.channels / a.groups;
  if (a.chansum) {
    const float2* cs = reinterpret_cast<const float2*>(a.chansum) + (long long)n * a.ld_chansum;
    if (threadIdx.x < a.groups) {
      double ds = 0.0, dss = 0.0;
      for (int k = 0; k < cpg; ++k) {
        const float2 v = cs[threadIdx.x * cpg + k];
        ds += (double)v.x;
        dss += (double)v.y;
      }
      const double cnt = (double)cpg * hw;
      const double mean = ds / cnt;
      double var = dss / cnt - mean * mean;
      if (var < 0.0) var = 0.0;
      mr_s[threadIdx.x] = make_float2((float)mean, (float)(1.0 / sqrt(var + (double)a.eps)));
    }
  } else if (threadIdx.x < a.groups) {
    const float* mr = reinterpret_cast<const float*>(a.stats) + ((long long)n * a.groups + threadIdx.x) * 2;
    mr_s[threadIdx.x] = make_float2(mr[0], mr[1]);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < a.channels; c += blockDim.x) {
    const float2 mr = mr_s[c / cpg];
    coef[(long long)n * ld_coef + c] = gn_half_coeff(a, n, c, mr.x, mr.y);
  }
}

template <typename T, typename TY, int VEC>
static int launch_gn(const fidm_gn_args& a, cudaStream_t st, float2* coef = nullptr, int ld_coef = 0) {
  GnParams p;
  p.a = a;
  p.cv = a.channels / VEC;
  FIDM_REQUIRE(p.cv <= 1024, FIDM_E_SHAPE, "groupnorm: %d channels not supported", a.channels);
  p.ppi = p.cv >= 256 ? 1 : 256 / p.cv;
  const int threads = p.cv * p.ppi;
  const int hw = a.height * a.width;
  // iteration space of the apply pass (output pixels for DOWN, input pixels otherwise)
  const int it_hw = (a.resample == FIDM_RESAMPLE_DOWN) ? hw / 4 : hw;
  auto plan = [&](int npix) {
    int chunks = (num_sms() * 8 + a.batch - 1) / a.batch;
    const int max_chunks = (npix + p.ppi - 1) / p.ppi;
    if (chunks > max_chunks) chunks = max_chunks;
    if (chunks < 1) chunks = 1;
    p.pix_per_blk = (npix + chunks - 1) / chunks;
    return (npix + p.pix_per_blk - 1) / p.pix_per_blk;
  };
  int chunks;
  if (!a.skip_norm && !a.chansum && (long long)hw * (a.channels / a.groups) <= 32768) {    // <= 64 KB per (image, group) block
    launch_kernel(gn_stats_direct_kernel<T, VEC>, dim3(a.groups, a.batch), dim3(256), 0, st, 1, p, coef, ld_coef);
    FIDM_CHECK_LAUNCH("groupnorm stats (direct)");
  } else if (!a.skip_norm && !a.chansum) {
    // workspace: [batch*groups*2] floats (mean, rstd) padded to doubles, then the per-block partials
    double* partials = a.stats + (long long)a.batch * a.groups;
    chunks = plan(hw);
    int cap = FIDM_GN_MAX_BLOCKS / a.batch > 0 ? FIDM_GN_MAX_BLOCKS / a.batch : 1;
    // At small batch `plan` cuts an image into ~1000 blocks of a few pixels each, and the last block's fixed-order fold
    // over all of them IS the kernel (29 us for a 4 MB tensor at batch 1): keep at least 64 KB of the image per block.
    const long long want = (long long)hw * a.channels * (long long)sizeof(T) / 65536;
    if (want < cap) cap = want < 1 ? 1 : (int)want;
    if (chunks > cap) {
      p.pix_per_blk = (hw + cap - 1) / cap;
      chunks = (hw + p.pix_per_blk - 1) / p.pix_per_blk;
    }
    const long long blocks_cap = (FIDM_GN_MAX_BLOCKS > a.batch ? FIDM_GN_MAX_BLOCKS : a.batch) + a.batch;
    int* counters = reinterpret_cast<int*>(partials + blocks_cap * a.groups * 2);
    launch_kernel(gn_stats_kernel<T, VEC>, dim3(chunks, a.batch), dim3(threads),
                  sizeof(float) * 2 * threads + 8 * 64 * 2 * sizeof(double), st, 1, p, partials, counters, coef, ld_coef);
    FIDM_CHECK_LAUNCH("groupnorm stats");
  }
  if (coef) {      // statistics only: the consumer conv applies the activation in its operand path
    if (a.chansum) {         // (the statistics kernels above wrote the coefficients themselves)
      launch_kernel(gn_coeff_kernel, dim3(a.batch), dim3(256), 0, st, 1, a, coef, ld_coef);
      FIDM_CHECK_LAUNCH("groupnorm coeff");
    }
    return 0;
  }
  chunks = plan(it_hw);
  dim3 grid(chunks, a.batch);
  const size_t sm = a.chansum ? sizeof(float2) * (a.channels + a.groups) : 0;
  if (a.resample == FIDM_RESAMPLE_NONE)
    launch_kernel(gn_apply_kernel<T, TY, VEC, FIDM_RESAMPLE_NONE>, grid, dim3(threads), sm, st, 1, p);
  else if (a.resample == FIDM_RESAMPLE_DOWN)
    launch_kernel(gn_apply_kernel<T, TY, VEC, FIDM_RESAMPLE_DOWN>, grid, dim3(threads), sm, st, 1, p);
  else
    launch_kernel(gn_apply_kernel<T, TY, VEC, FIDM_RESAMPLE_UP>, grid, dim3(threads), sm, st, 1, p);
  FIDM_CHECK_LAUNCH("groupnorm apply");
  return 0;
}

template <typename T, typename TY>
static int dispatch_vec(const fidm_gn_args& a, cudaStream_t st, float2* coef = nullptr, int ld_coef = 0) {
  const int cpg = a.channels / a.groups;
  constexpr int MAXV = 16 / sizeof(T);  // 16-byte vectors
  auto aligned = [&](int v) {
    const size_t bytes = sizeof(T) * v;
    bool ok = (cpg % v == 0) && (a.ld_x % v == 0) && ((uintptr_t)a.x % bytes == 0);
    if (!coef) ok = ok && (a.ld_y % v == 0) && ((uintptr_t)a.y % bytes == 0);
    if (a.y_raw) ok = ok && (a.ld_raw % v == 0) && ((uintptr_t)a.y_raw % bytes == 0);
    return ok;
  };
  if (MAXV >= 8 && aligned(8)) return launch_gn<T, TY, 8>(a, st, coef, ld_coef);
  if (aligned(4)) return launch_gn<T, TY, 4>(a, st, coef, ld_coef);
  if (aligned(2)) return launch_gn<T, TY, 2>(a, st, coef, ld_coef);
  return launch_gn<T, TY, 1>(a, st, coef, ld_coef);
}

}  // namespace fidm

extern "C" int fidm_groupnorm_silu_nhwc(const fidm_gn_args* a, fidm_stream_t stream) {
  using namespace fidm;
  FIDM_REQUIRE(a && a->x && a->y && (a->stats || a->skip_norm || a->chansum), FIDM_E_BADARG, "groupnorm: null x/y/stats");
  FIDM_REQUIRE(a->batch > 0 && a->height > 0 && a->width > 0 && a->channels > 0, FIDM_E_BADARG, "groupnorm: empty shape");
  FIDM_REQUIRE(a->groups > 0 && a->groups <= 64 && a->channels % a->groups == 0, FIDM_E_SHAPE,
               "groupnorm: channels %d not divisible into %d groups", a->channels, a->groups);
  FIDM_REQUIRE(a->ld_x >= a->channels && a->ld_y >= a->channels, FIDM_E_BADARG, "groupnorm: ld < channels");
  FIDM_REQUIRE(a->resample >= 0 && a->resample <= 2, FIDM_E_BADARG, "groupnorm: bad resample %d", a->resample);
  if (a->resample == FIDM_RESAMPLE_DOWN)
    FIDM_REQUIRE(a->height % 2 == 0 && a->width % 2 == 0, FIDM_E_SHAPE, "groupnorm: odd size for 2x pooling");
  if (a->scale_shift) FIDM_REQUIRE(a->ld_ss >= 2 * a->channels, FIDM_E_BADARG, "groupnorm: ld_ss < 2*channels");
  if (a->dtype == FIDM_BF16 && a->y_dtype == FIDM_F16) {
    { const int rc = try_gn_fused_small<__half>(*a, (cudaStream_t)stream); if (rc >= 0) return rc; }
    return dispatch_vec<__nv_bfloat16, __half>(*a, (cudaStream_t)stream);
  }
  FIDM_REQUIRE(a->y_dtype == a->dtype, FIDM_E_BADARG, "groupnorm: y_dtype %d not supported with dtype %d", a->y_dtype, a->dtype);
  if (a->dtype == FIDM_BF16) {
    { const int rc = try_gn_fused_small<__nv_bfloat16>(*a, (cudaStream_t)stream); if (rc >= 0) return rc; }
    return dispatch_vec<__nv_bfloat16, __nv_bfloat16>(*a, (cudaStream_t)stream);
  }
  if (a->dtype == FIDM_F32) return dispatch_vec<float, float>(*a, (cudaStream_t)stream);
  FIDM_REQUIRE(false, FIDM_E_BADARG, "groupnorm: bad dtype %d", a->dtype);
}

extern "C" int fidm_groupnorm_silu_coeff(const fidm_gn_args* a, float* coef, int32_t ld_coef, fidm_stream_t stream) {
  using namespace fidm;
  FIDM_REQUIRE(a && a->x && coef && (a->stats || a->chansum), FIDM_E_BADARG, "groupnorm coeff: null x/coef/stats");
  FIDM_REQUIRE(a->batch > 0 && a->height > 0 && a->width > 0 && a->channels > 0, FIDM_E_BADARG, "groupnorm coeff: empty shape");
  FIDM_REQUIRE(a->groups > 0 && a->groups <= 64 && a->channels % a->groups == 0, FIDM_E_SHAPE,
               "groupnorm coeff: channels %d not divisible into %d groups", a->channels, a->groups);
  FIDM_REQUIRE(a->ld_x >= a->channels && ld_coef >= a->channels && !a->skip_norm, FIDM_E_BADARG, "groupnorm coeff: bad ld / skip_norm");
  if (a->scale_shift) FIDM_REQUIRE(a->ld_ss >= 2 * a->channels, FIDM_E_BADARG, "groupnorm coeff: ld_ss < 2*channels");
  fidm_gn_args b = *a;
  b.resample = FIDM_RESAMPLE_NONE;
  float2* c2 = reinterpret_cast<float2*>(coef);
  if (a->dtype == FIDM_BF16) return dispatch_vec<__nv_bfloat16, __nv_bfloat16>(b, (cudaStream_t)stream, c2, ld_coef);
  if (a->dtype == FIDM_F32) return dispatch_vec<float, float>(b, (cudaStream_t)stream, c2, ld_coef);
  FIDM_REQUIRE(false, FIDM_E_BADARG, "groupnorm coeff: bad dtype %d", a->dtype);
}

namespace fidm {
// chansum[n][c0+c] = sum_{slot} colsum[n][slot][c]   (double accumulation, fixed order)
// A block owns CB channels of one image and cuts the slot range into RS = 1024 / CB slices (thread = channel x slice);
// the summation tree is fixed: slots of a slice in order, slices strided by 8 in order, then the 8 partials in order.
// CB = 8 gives a 256-channel batch-1 tensor 32 blocks instead of 8 (the kernel is a latency chain of L2 reads: more
// blocks and 8 loads in flight per thread took it from 8 us to under 4).
template <int CB>
__global__ void __launch_bounds__(1024) gn_reduce_colsum_kernel(const float2* __restrict__ colsum, int slots, int C,
                                                                float2* __restrict__ chansum, int ld, int c0,
                                                                const fidm_gn_args a, float2* __restrict__ coef, int ld_coef) {
  constexpr int RS = 1024 / CB;
  __shared__ double red[RS][CB][2];
  __shared__ double red8[8][CB][2];
  __shared__ double csum[CB][2];
  __shared__ float2 mr_s[CB];
  const int n = blockIdx.y;
  const int cl = threadIdx.x % CB;
  const int c = blockIdx.x * CB + cl;
  const int j = threadIdx.x / CB;
  double ds = 0.0, dss = 0.0;
  if (c < C) {
    const float2* q = colsum + (long long)n * slots * C + c;
    int s = j;
    for (; s + 7 * RS < slots; s += 8 * RS) {
      float2 v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = __ldcg(q + (long long)(s + k * RS) * C);
#pragma unroll
      for (int k = 0; k < 8; ++k) { ds += (double)v[k].x; dss += (double)v[k].y; }
    }
    for (; s < slots; s += RS) {
      const float2 v = __ldcg(q + (long long)s * C);
      ds += (double)v.x; dss += (double)v.y;
    }
  }
  red[j][cl][0] = ds;
  red[j][cl][1] = dss;
  __syncthreads();
  if (j < 8) {
    double sa = 0.0, sb = 0.0;
#pragma unroll 4
    for (int k = j; k < RS; k += 8) { sa += red[k][cl][0]; sb += red[k][cl][1]; }
    red8[j][cl][0] = sa;
    red8[j][cl][1] = sb;
  }
  __syncthreads();
  if (j == 0) {
    double sa = 0.0, sb = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { sa += red8[k][cl][0]; sb += red8[k][cl][1]; }
    // the consumer sees the sums rounded to fp32 (chansum): fold exactly those, as gn_coeff_kernel would
    csum[cl][0] = (double)(float)sa;
    csum[cl][1] = (double)(float)sb;
    if (c < C) chansum[(long long)n * ld + c0 + c] = make_float2((float)sa, (float)sb);
  }
  if (!coef) return;
  // Single-producer case: this tensor IS the GroupNorm input of the next conv (K1h), and every group lies inside one
  // block's CB channels: fold the groups here and write the coefficients -- no separate coefficient launch.
  __syncthreads();
  const int cpg = a.channels / a.groups;
  const int gpb = CB / cpg;                               // groups per block
  if (threadIdx.x < gpb) {
    double gs = 0.0, gss = 0.0;
    for (int k = 0; k < cpg; ++k) { gs += csum[threadIdx.x * cpg + k][0]; gss += csum[threadIdx.x * cpg + k][1]; }
    const double cnt = (double)cpg * a.height * a.width;
    const double mean = gs / cnt;
    double var = gss / cnt - mean * mean;
    if (var < 0.0) var = 0.0;
    mr_s[threadIdx.x] = make_float2((float)mean, (float)(1.0 / sqrt(var + (double)a.eps)));
  }
  __syncthreads();
  if (j == 0 && c < C) {
    const float2 mr = mr_s[cl / cpg];
    coef[(long long)n * ld_coef + c] = gn_half_coeff(a, n, c, mr.x, mr.y);
  }
}

// channels per block: as few as the groups allow (cpg | CB) while the grid stays a sensible size
static int reduce_colsum_cb(int channels, int batch, int cpg) {
  const int cbs[3] = {8, 16, 32};
  for (int i = 0; i < 3; ++i) {
    const int cb = cbs[i];
    if (cb < cpg || cb % cpg != 0) continue;
    if ((long long)((channels + cb - 1) / cb) * batch <= 1024 || cb == 32) return cb;
  }
  return 32;
}

static void launch_reduce_colsum(int cb, dim3 grid, cudaStream_t st, const float2* colsum, int slots, int C, float2* chansum,
                                 int ld, int c0, const fidm_gn_args& a, float2* coef, int ld_coef) {
  if (cb == 8) launch_kernel(gn_reduce_colsum_kernel<8>, grid, dim3(1024), 0, st, 1, colsum, slots, C, chansum, ld, c0, a, coef, ld_coef);
  else if (cb == 16) launch_kernel(gn_reduce_colsum_kernel<16>, grid, dim3(1024), 0, st, 1, colsum, slots, C, chansum, ld, c0, a, coef, ld_coef);
  else launch_kernel(gn_reduce_colsum_kernel<32>, grid, dim3(1024), 0, st, 1, colsum, slots, C, chansum, ld, c0, a, coef, ld_coef);
}
}  // namespace fidm

extern "C" int fidm_groupnorm_reduce_colsum(const float* colsum, int32_t batch, int32_t slots, int32_t channels,
                                            float* chansum, int32_t ld_chansum, int32_t c0, fidm_stream_t stream) {
  using namespace fidm;
  FIDM_REQUIRE(colsum && chansum && batch > 0 && slots > 0 && channels > 0 && c0 >= 0 && c0 + channels <= ld_chansum,
               FIDM_E_BADARG, "reduce_colsum: bad args");
  // the channel partition must not depend on who asks: the fused-coefficient entry below folds the same tensor and the
  // two are required to agree bit for bit, so both derive CB from (channels, batch) and the usual 32 groups
  const int cb = reduce_colsum_cb(channels, batch, channels % 32 == 0 && channels / 32 <= 32 ? channels / 32 : 32);
  dim3 grid((channels + cb - 1) / cb, batch);
  fidm_gn_args none = {};
  launch_reduce_colsum(cb, grid, (cudaStream_t)stream, reinterpret_cast<const float2*>(colsum), slots, channels,
                       reinterpret_cast<float2*>(chansum), ld_chansum, c0, none, (float2*)nullptr, 0);
  FIDM_CHECK_LAUNCH("reduce_colsum");
  return 0;
}

extern "C" int fidm_groupnorm_reduce_colsum_coeff(const float* colsum, int32_t slots, float* chansum, int32_t ld_chansum,
                                                  int32_t c0, const fidm_gn_args* a, float* coef, int32_t ld_coef,
                                                  fidm_stream_t stream) {
  using namespace fidm;
  FIDM_REQUIRE(colsum && chansum && a && coef && slots > 0 && c0 >= 0 && c0 + a->channels <= ld_chansum, FIDM_E_BADARG,
               "reduce_colsum_coeff: bad args");
  FIDM_REQUIRE(a->groups > 0 && a->channels % a->groups == 0 && a->channels % 32 == 0, FIDM_E_SHAPE,
               "reduce_colsum_coeff: channels %d / groups %d", a->channels, a->groups);
  const int cpg = a->channels / a->groups;
  FIDM_REQUIRE(cpg <= 32 && 32 % cpg == 0, FIDM_E_SHAPE, "reduce_colsum_coeff: %d channels per group do not tile 32", cpg);
  FIDM_REQUIRE(ld_coef >= a->channels, FIDM_E_BADARG, "reduce_colsum_coeff: ld_coef");
  if (a->scale_shift) FIDM_REQUIRE(a->ld_ss >= 2 * a->channels, FIDM_E_BADARG, "reduce_colsum_coeff: ld_ss < 2*channels");
  const int cb = reduce_colsum_cb(a->channels, a->batch, cpg);
  dim3 grid(a->channels / cb, a->batch);
  launch_reduce_colsum(cb, grid, (cudaStream_t)stream, reinterpret_cast<const float2*>(colsum), slots, a->channels,
                       reinterpret_cast<float2*>(chansum), ld_chansum, c0, *a, reinterpret_cast<float2*>(coef), ld_coef);
  FIDM_CHECK_LAUNCH("reduce_colsum_coeff");
  return 0;
}

extern "C" int fidm_groupnorm_num_launches(const fidm_gn_args* a) {
  int v, t, s, pt;
  if (!a) return 0;
  if (a->skip_norm || a->chansum) return 1;
  return fidm::gn_fused_small_plan(*a, &v, &t, &s, &pt) ? 1 : 2;
}

extern "C" int64_t fidm_groupnorm_workspace_bytes(int32_t batch, int32_t groups) {
  const long long blocks = (FIDM_GN_MAX_BLOCKS > batch ? FIDM_GN_MAX_BLOCKS : batch) + batch;
  // (mean, rstd) floats | per-block partial sums | per-image completion counters (must start at zero)
  return (int64_t)sizeof(double) * ((long long)batch * groups + blocks * groups * 2 + (batch + 1) / 2 + 1);
}
