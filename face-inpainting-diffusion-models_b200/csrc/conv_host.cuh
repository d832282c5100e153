// Host-side helpers shared by the tensor-core convolution kernels (defined in conv_tc.cu unless inline here).
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace fidm {

// NHWC 16-bit tensor [N][H][W][C] (pixel stride ld elements) as a 4-D tiled map with the 128-byte swizzle,
// box = {64 channels, bw, bh, bn}.
// pixel_stride 2: the box loads every other pixel in W and H (stride-2 convolution).
int make_nhwc_map(CUtensorMap* m, const void* base, int C, int W, int H, int N, int ld, int bw, int bh, int bn,
                  int f16, int pixel_stride = 1);
// Row-major 16-bit matrix [rows][cols] (row stride ld elements) as a 2-D map, box = {64, box_rows}.
int make_matrix_map(CUtensorMap* m, const void* base, int cols, int rows, int ld, int box_rows, int f16);

// The epilogue fields that the K1, K1h and K1s parameter structs share, from the C ABI arguments.
template <class Params>
void set_epilogue_params(Params& p, const fidm_conv_args& a) {
  p.bias = a.bias; p.row_add = a.row_add; p.ld_row_add = a.ld_row_add;
  p.residual = reinterpret_cast<decltype(p.residual)>(a.residual); p.ld_res = a.ld_res;
  p.y_nchw = a.y_nchw_f32 ? reinterpret_cast<float*>(a.y) : nullptr; p.cout_valid = a.cout_valid;
  p.colsum = a.colsum; p.cout = a.cout;
}

// K1h (conv_halo.cu): 3x3 convolution whose A operand is silu(x * A[n][c] + B[n][c]) of the RAW input, applied
// while the operand tiles are staged (GroupNorm + SiLU fused into the consumer convolution).
bool conv_halo_supported(const fidm_conv_args& a);
int launch_conv_halo(const fidm_conv_args& a, cudaStream_t st);

// K1s (conv_halo_swap.cu): the same fused operand path with the operand roles swapped (weights = A operand, 256 pixels
// = N) for Cout % 256 != 0 and the 6-channel head, where K1h's narrow-N tiles run at half the tensor rate.
bool conv_halo_swap_supported(const fidm_conv_args& a);
bool conv_halo_swap_preferred(const fidm_conv_args& a);     // supported AND the better kernel for this shape
int launch_conv_halo_swap(const fidm_conv_args& a, cudaStream_t st, unsigned long long* prof = nullptr);

// probe buffer set by fidm_conv_set_profile_buffer (null in production)
unsigned long long* conv_profile_buffer();

}  // namespace fidm
