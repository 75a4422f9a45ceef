// Integer export of a calibrated model (reference: utils/integer.py:8-129): the int8 / uint8 layouts an integer
// inference engine consumes.  One streaming pass per tensor: fp32 in, one byte per element out -- HBM bound (5 bytes per
// element), 16 elements per thread, 16-byte stores.
//   mode 0  plain symmetric      int8  = clamp(rne(x / delta), -q, q-1)                        (integer.py:15-17, :64-67, :27-42)
//   mode 1  post-GELU twin       uint8 = (clamp(rne(x / d_pos), 0, q-1) + 128) + |clamp(rne(x / d_neg), -q+1, 0)|   (:51-62)
//   mode 2  split-of-softmax twin uint8 = (clamp(rne(clamp(x, s, 1) * (q-1)), 0, q-1) + 128) + clamp(rne(clamp(x, 0, s) / d), 0, q-1) (:78-87)
// The additions are uint8 additions as in the reference (its "+ 128" marks every element, also the negative ones, and
// the sum wraps modulo 256); step sizes that the reference holds as tensors divide the IEEE way, the constant
// post-GELU negative step (a Python scalar) through the fp32 reciprocal, as torch does on the GPU (see prep.cu).
#include "prep.cuh"
#include "../../include/ptq4vit_b200.h"

namespace {

struct ExportArgs {
  const float* src; uint8_t* dst; long long rows, cols;
  const float* delta; int rows_per_block, n_row_blocks, cols_per_block, n_col_blocks;
  int mode; float qmax; float d_neg; const float* split; int ieee_div;
};

__device__ __forceinline__ uint8_t encode(const ExportArgs& a, float x, float delta, float split, float rcp_neg) {
  const float q = a.qmax;
  if (a.mode == 0) {
    const float v = fminf(fmaxf(rintf(__fdiv_rn(x, delta)), -q), q - 1.f);
    return (uint8_t)(int8_t)(int)v;
  }
  if (a.mode == 1) {
    const float p = fminf(fmaxf(rintf(__fdiv_rn(x, delta)), 0.f), q - 1.f);
    const float nq = a.ieee_div ? __fdiv_rn(x, a.d_neg) : x * rcp_neg;
    const float n = fabsf(fminf(fmaxf(rintf(nq), -q + 1.f), 0.f));
    return (uint8_t)((uint8_t)((uint8_t)(int)p + 128u) + (uint8_t)(int)n);
  }
  const float hi = fminf(fmaxf(rintf(fminf(fmaxf(x, split), 1.f) * (q - 1.f)), 0.f), q - 1.f);
  const float lo = fminf(fmaxf(rintf(__fdiv_rn(fminf(fmaxf(x, 0.f), split), delta)), 0.f), q - 1.f);
  return (uint8_t)((uint8_t)((uint8_t)(int)hi + 128u) + (uint8_t)(int)lo);
}

__global__ void export_kernel(const ExportArgs a) {
  const long long n = a.rows * a.cols;
  const float split = a.split ? a.split[0] : 0.f;
  const float rcp_neg = a.d_neg > 0.f ? __fdiv_rn(1.f, a.d_neg) : 0.f;
  for (long long i0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 16; i0 < n; i0 += (long long)gridDim.x * blockDim.x * 16) {
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    const bool vec = i0 + 16 <= n;            // i0 is a multiple of 16: the 16-byte store is aligned
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      const long long i = i0 + e;
      if (i >= n) break;
      const long long row = i / a.cols; const int col = (int)(i - row * a.cols);
      const int rb = a.rows_per_block > 0 ? (int)((row / a.rows_per_block) % a.n_row_blocks) : 0;
      const float delta = a.delta[(size_t)rb * a.n_col_blocks + col / a.cols_per_block];
      const uint8_t b = encode(a, a.src[i], delta, split, rcp_neg);
      if (vec) w[e >> 2] |= (uint32_t)b << ((e & 3) * 8);
      else a.dst[i] = b;
    }
    if (vec) *reinterpret_cast<uint4*>(a.dst + i0) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

}  // namespace

extern "C" int p4v_export_quantized(const float* src, long long rows, long long cols, const float* delta, int rows_per_block,
                                    int n_row_blocks, int cols_per_block, int n_col_blocks, int mode, int bit, float d_neg,
                                    const float* split, void* dst, void* stream) {
  P4V_REQUIRE(src && delta && dst, "export: null pointer");
  P4V_REQUIRE(rows >= 0 && cols > 0 && n_row_blocks >= 1 && n_col_blocks >= 1 && cols_per_block >= 1, "export: bad geometry");
  P4V_REQUIRE(mode >= 0 && mode <= 2, "export: mode must be 0 (int8), 1 (post-GELU twin) or 2 (split-of-softmax twin)");
  P4V_REQUIRE(bit >= 2 && bit <= 8, "export: bit width must be in [2,8]");
  P4V_REQUIRE(mode != 2 || split, "export: mode 2 needs the split point");
  P4V_REQUIRE((long long)(n_col_blocks - 1) * cols_per_block < cols, "export: column blocks exceed the row length");
  if (rows == 0) return 0;
  ExportArgs a{src, (uint8_t*)dst, rows, cols, delta, rows_per_block, n_row_blocks, cols_per_block, n_col_blocks,
               mode, (float)(1 << (bit - 1)), d_neg, split, p4v_scalar_div_ieee()};
  const long long n = rows * cols;
  long long blocks = (n / 16 + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  export_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(a); p4v_count_launch();
  P4V_CUDA_OK(cudaGetLastError());
  return 0;
}
