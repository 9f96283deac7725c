// Bandwidth kernels shared by the backward passes (LSTM BPTT, ResNet trunk, WaveNet encoder): operand transposes for
// the split-K weight-gradient GEMMs, the fixed-order sum of their partials, and deterministic column sums for bias
// gradients.  `static`: every translation unit that includes this header gets its own copy.
#pragma once
#include "common.cuh"

namespace avvad {

// bf16 [R][ld] (first C columns) -> [C][Rp] with zero fill for r >= R
// mode 0: plain transpose.  mode 1: H_prev transpose: out[c][b*T + t] = in[b*T + t - 1][c] for t > 0, else 0.
static __global__ void transpose_bf16_kernel(const __nv_bfloat16* __restrict__ in, int64_t R, int C, int64_t ld,
                                             int64_t Rp, int mode, int T, __nv_bfloat16* __restrict__ out) {
  __shared__ __nv_bfloat16 tile[32][33];
  const int64_t r0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int64_t r = r0 + i;
    const int c = c0 + threadIdx.x;
    __nv_bfloat16 v = __float2bfloat16_rn(0.f);
    if (r < R && c < C) {
      if (mode == 0) v = in[r * ld + c];
      else if ((r % T) != 0) v = in[(r - 1) * ld + c];
    }
    tile[i][threadIdx.x] = v;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int c = c0 + i;
    const int64_t r = r0 + threadIdx.x;
    if (c < C && r < Rp) out[(int64_t)c * Rp + r] = tile[threadIdx.x][i];
  }
}

// out[c] = sum_r x[r][c]  (fp32, 64 columns per block, fixed-order reduction over four row lanes)
static __global__ void __launch_bounds__(256) colsum_f32_kernel(const float* __restrict__ x, int64_t R, int Ccols,
                                                                float* __restrict__ out) {
  __shared__ float sm[4][64];
  const int col = blockIdx.x * 64 + (threadIdx.x & 63);
  const int part = threadIdx.x >> 6;
  float acc = 0.f;
  if (col < Ccols)
    for (int64_t r = part; r < R; r += 4) acc += x[r * Ccols + col];
  sm[part][threadIdx.x & 63] = acc;
  __syncthreads();
  if (threadIdx.x < 64 && col < Ccols)
    out[col] = sm[0][threadIdx.x] + sm[1][threadIdx.x] + sm[2][threadIdx.x] + sm[3][threadIdx.x];
}

// acc[j] (+)= sum_s part[s][j]
static __global__ void sum_partials_kernel(const float* __restrict__ part, int nparts, int64_t elems, int accumulate,
                                           float* __restrict__ acc) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= elems) return;
  float t = accumulate ? acc[j] : 0.f;
  for (int s = 0; s < nparts; ++s) t += part[(int64_t)s * elems + j];
  acc[j] = t;
}

}  // namespace avvad
