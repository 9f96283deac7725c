// ResNet-18 trunk on single-channel 67x67 mouth ROIs (eval-mode BatchNorm folded into the convolutions).
//
// Reference semantics: packages/models/AV_Net.py:78-94 (channel triple + torchvision resnet18 children[:-1]).
// Data layout: activations NHWC bf16 [frame][h][w][c]; weights bf16 [Cout][R][S][Cin] (K order = tap-major,
// channel-minor, the order the implicit-GEMM producer walks); folded bias fp32.
//   conv1 7x7/2 + BN + ReLU + maxpool 3x3/2 : stem_s2d.cuh (the padded frame in shared memory is the UMMA A operand;
//                                             the three identical input channels are folded into one by summing
//                                             the weights); optionally fed from the u8 source frames
//   layer1 (4 convs)                         : conv_slab.cuh (slab with halo, row-shifted descriptors)
//   layer2..4 (12 launches)                  : gemm_tma.cuh (TMA-box im2col); the three downsample 1x1 branches are
//                                             K-concatenated into the following conv_b
//   global average pool                      : small bandwidth kernel, emits fp32 features and/or the bf16
//                                              LSTM operand columns
//   training mode (batch-statistics BN)      : raw convs + statistics / apply kernels, two-pass stem
#include <stdlib.h>

#include <mutex>

#include "gemm_tma.cuh"
#include "stem_s2d.cuh"

namespace avvad {
namespace tc {
// conv_block.cuh (compiled in conv_slab.cu): fused BasicBlock of layer1
int launch_block17(const __nv_bfloat16* x, const __nv_bfloat16* wa, const float* bias_a, const __nv_bfloat16* wb,
                   const float* bias_b, __nv_bfloat16* z, int64_t n, cudaStream_t st);
bool block17_enabled();
}  // namespace tc
}  // namespace avvad

namespace avvad {

struct ConvSpec {
  int cin, cout, k, stride, pad, hin, hout;
};
// index order documented in include/avvad.h
static const ConvSpec kSpecs[20] = {
    {3, 64, 7, 2, 3, 67, 34},                                                            // 0 conv1 (+pool -> 17)
    {64, 64, 3, 1, 1, 17, 17},   {64, 64, 3, 1, 1, 17, 17},                              // 1,2  l1.0
    {64, 64, 3, 1, 1, 17, 17},   {64, 64, 3, 1, 1, 17, 17},                              // 3,4  l1.1
    {64, 128, 3, 2, 1, 17, 9},   {128, 128, 3, 1, 1, 9, 9},  {64, 128, 1, 2, 0, 17, 9},  // 5,6,7  l2.0 (+ds)
    {128, 128, 3, 1, 1, 9, 9},   {128, 128, 3, 1, 1, 9, 9},                              // 8,9  l2.1
    {128, 256, 3, 2, 1, 9, 5},   {256, 256, 3, 1, 1, 5, 5},  {128, 256, 1, 2, 0, 9, 5},  // 10,11,12 l3.0
    {256, 256, 3, 1, 1, 5, 5},   {256, 256, 3, 1, 1, 5, 5},                              // 13,14 l3.1
    {256, 512, 3, 2, 1, 5, 3},   {512, 512, 3, 1, 1, 3, 3},  {256, 512, 1, 2, 0, 5, 3},  // 15,16,17 l4.0
    {512, 512, 3, 1, 1, 3, 3},   {512, 512, 3, 1, 1, 3, 3},                              // 18,19 l4.1
};
constexpr int64_t kFrameHW = 67 * 67;
constexpr int64_t kActBytesPerFrame = 17 * 17 * 64 * 2;  // largest NHWC bf16 activation (after the pool)

// ---- weight folding / packing ----------------------------------------------------------------------
__global__ void pack_conv_kernel(const float* __restrict__ w, const float* __restrict__ gamma,
                                 const float* __restrict__ beta, const float* __restrict__ mean,
                                 const float* __restrict__ var, float eps, int cout, int cin, int k,
                                 __nv_bfloat16* __restrict__ wp, float* __restrict__ bias) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int total = cout * cin * k * k;
  if (idx < cout) {
    const float sc = gamma[idx] / sqrtf(var[idx] + eps);
    bias[idx] = beta[idx] - mean[idx] * sc;
  }
  if (idx >= total) return;
  // destination order [o][r][s][i]
  const int i = idx % cin;
  const int s = (idx / cin) % k;
  const int r = (idx / (cin * k)) % k;
  const int o = idx / (cin * k * k);
  const float sc = gamma[o] / sqrtf(var[o] + eps);
  wp[idx] = __float2bfloat16_rn(w[((o * cin + i) * k + r) * k + s] * sc);
}

// conv1 for the tensor-core stem: same folding, bf16 [64 out][64 k] with k = r*7+s (49..63 zero)
__global__ void pack_conv1_tc_kernel(const float* __restrict__ w, const float* __restrict__ gamma,
                                     const float* __restrict__ beta, const float* __restrict__ mean,
                                     const float* __restrict__ var, float eps, __nv_bfloat16* __restrict__ w1b,
                                     float* __restrict__ bias) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < 64) {
    const float sc = gamma[idx] / sqrtf(var[idx] + eps);
    bias[idx] = beta[idx] - mean[idx] * sc;
  }
  if (idx >= 64 * 64) return;
  const int o = idx / 64, k = idx % 64;
  float v = 0.f;
  if (k < 49) {
    const float sc = gamma[o] / sqrtf(var[o] + eps);
    v = (w[(o * 3 + 0) * 49 + k] + w[(o * 3 + 1) * 49 + k] + w[(o * 3 + 2) * 49 + k]) * sc;
  }
  w1b[idx] = __float2bfloat16_rn(v);
}

// Downsample blocks: out = relu(conv_b(y) + bn_b + conv_ds(x) + bn_ds).  Both folded convolutions share the output
// grid, so the 1x1/stride-2 branch is appended to conv_b's K dimension: wf[o] = [ w_b[o][9*C] | w_ds[o][Cin] ],
// bias = bias_b + bias_ds, and one implicit GEMM accumulates both (gemm_tma.cuh, "second operand").
__global__ void concat_ds_kernel(const __nv_bfloat16* __restrict__ wb, const __nv_bfloat16* __restrict__ wds,
                                 const float* __restrict__ bb, const float* __restrict__ bds, int cout, int kb, int kds,
                                 __nv_bfloat16* __restrict__ wf, float* __restrict__ bf) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int kt = kb + kds;
  if (idx < cout) bf[idx] = bb[idx] + bds[idx];
  if (idx >= cout * kt) return;
  const int o = idx / kt, k = idx - o * kt;
  wf[idx] = (k < kb) ? wb[o * kb + k] : wds[o * kds + (k - kb)];
}

// ---- global average pool over the 3x3x512 map -----------------------------------------------------------
__global__ void avgpool_kernel(const __nv_bfloat16* __restrict__ act, int64_t n_frames, int hw, int C,
                               float* __restrict__ feat, __nv_bfloat16* __restrict__ feat_bf16, int64_t ld_bf16,
                               int64_t col_off) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int chunks = C / 8;
  if (idx >= n_frames * chunks) return;
  const int64_t f = idx / chunks;
  const int ch = (int)(idx - f * chunks);
  float s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const __nv_bfloat16* p = act + f * hw * C + ch * 8;
  for (int i = 0; i < hw; ++i) {
    const uint4 v = *reinterpret_cast<const uint4*>(p + (int64_t)i * C);
    const float2 a = unpack_bf16x2(v.x), b = unpack_bf16x2(v.y), c = unpack_bf16x2(v.z), d = unpack_bf16x2(v.w);
    s[0] += a.x; s[1] += a.y; s[2] += b.x; s[3] += b.y; s[4] += c.x; s[5] += c.y; s[6] += d.x; s[7] += d.y;
  }
  const float inv = 1.0f / (float)hw;
#pragma unroll
  for (int q = 0; q < 8; ++q) s[q] *= inv;
  if (feat) {
    float4* o = reinterpret_cast<float4*>(feat + f * C + ch * 8);
    o[0] = make_float4(s[0], s[1], s[2], s[3]);
    o[1] = make_float4(s[4], s[5], s[6], s[7]);
  }
  if (feat_bf16) {
    __nv_bfloat16* o = feat_bf16 + f * ld_bf16 + col_off + ch * 8;
#pragma unroll
    for (int q = 0; q < 8; ++q) o[q] = __float2bfloat16_rn(s[q]);  // col_off may be odd (513): scalar stores
  }
}

// ---- training-mode BatchNorm (batch statistics) -------------------------------------------------------------
// raw bf16 [M][C] -> per-channel sum / sum of squares.  A block owns kStatRows consecutive rows; thread = (8-channel
// group, row lane): 16-byte loads, many rows in flight, fp32 partial sums per thread, shared-memory tree over the row
// lanes, one fp64 atomic per channel and block.
constexpr int kStatRows = 2048;
__global__ void __launch_bounds__(256) bn_stats_kernel(const __nv_bfloat16* __restrict__ raw, int64_t M, int C,
                                                       double* __restrict__ stats) {
  extern __shared__ float st_sm[];  // [lanes][2*C] partial sums
  const int groups = C / 8;                 // 8, 16, 32 or 64
  const int lanes = 256 / groups;           // row lanes: 32, 16, 8 or 4
  const int gidx = threadIdx.x % groups, ln = threadIdx.x / groups;
  const int64_t r0 = (int64_t)blockIdx.x * kStatRows;
  const int64_t r1 = (r0 + kStatRows < M) ? r0 + kStatRows : M;
  float s[8] = {0, 0, 0, 0, 0, 0, 0, 0}, q[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int64_t r = r0 + ln; r < r1; r += lanes) {
    const uint4 v = *reinterpret_cast<const uint4*>(raw + r * C + gidx * 8);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float a = __uint_as_float(w[e] << 16), b = __uint_as_float(w[e] & 0xFFFF0000u);
      s[2 * e] += a; q[2 * e] = fmaf(a, a, q[2 * e]);
      s[2 * e + 1] += b; q[2 * e + 1] = fmaf(b, b, q[2 * e + 1]);
    }
  }
  float* mine = st_sm + (size_t)ln * 2 * C + gidx * 8;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    mine[e] = s[e];
    mine[C + e] = q[e];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * C; c += 256) {
    double acc = 0.0;
    for (int l = 0; l < lanes; ++l) acc += (double)st_sm[(size_t)l * 2 * C + c];
    atomicAdd(stats + c, acc);
  }
}
// per-channel scale / shift for the apply pass: y = x*a + b with a = invstd*gamma, b = beta - mean*a; running statistics
// updated like nn.BatchNorm2d (momentum, unbiased variance)
__global__ void bn_finalize_kernel(const double* __restrict__ stats, int64_t M, int C, float eps, float momentum,
                                   const float* __restrict__ gamma, const float* __restrict__ beta,
                                   float* __restrict__ scale_shift, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, float* __restrict__ mean_invstd_out = nullptr) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double mean = stats[c] / (double)M;
  double var = stats[C + c] / (double)M - mean * mean;
  if (var < 0) var = 0;
  if (mean_invstd_out) {  // kept on the tape for the BatchNorm backward (resnet_bwd.cuh)
    mean_invstd_out[c] = (float)mean;
    mean_invstd_out[C + c] = (float)(1.0 / sqrt(var + (double)eps));
  }
  // same fp32 operation order as before the scale/shift refactoring is not required: (x-mean)*invstd*gamma+beta is
  // evaluated as x*a + b in fp32 from fp64-derived a, b
  const double a = (1.0 / sqrt(var + (double)eps)) * (double)gamma[c];
  scale_shift[c] = (float)a;
  scale_shift[C + c] = (float)((double)beta[c] - mean * a);
  if (running_mean) {
    const double unbiased = M > 1 ? var * (double)M / (double)(M - 1) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
}
// out = act(raw * a + b (+ residual)); 8 channels per thread, the block's scale/shift staged in shared memory,
// kApplyRows rows per thread so the per-channel constants are read once
constexpr int kApplyRows = 4;
__global__ void __launch_bounds__(256) bn_apply_kernel(const __nv_bfloat16* __restrict__ raw, int64_t M, int C,
                                                       const float* __restrict__ scale_shift,
                                                       const __nv_bfloat16* __restrict__ residual, int relu,
                                                       __nv_bfloat16* __restrict__ out) {
  extern __shared__ float ss_sm[];  // [2*C]
  for (int i = threadIdx.x; i < 2 * C; i += 256) ss_sm[i] = scale_shift[i];
  __syncthreads();
  const int groups = C / 8;
  const int rows_per_block = (256 / groups) * kApplyRows;
  const int gidx = threadIdx.x % groups, ln = threadIdx.x / groups;
  float a[8], b[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    a[e] = ss_sm[gidx * 8 + e];
    b[e] = ss_sm[C + gidx * 8 + e];
  }
  const int64_t base = (int64_t)blockIdx.x * rows_per_block + ln;
  uint4 v[kApplyRows], rv[kApplyRows];
#pragma unroll
  for (int k = 0; k < kApplyRows; ++k) {
    const int64_t r = base + (int64_t)k * (256 / groups);
    if (r < M) {
      v[k] = *reinterpret_cast<const uint4*>(raw + r * C + gidx * 8);
      if (residual) rv[k] = *reinterpret_cast<const uint4*>(residual + r * C + gidx * 8);
    }
  }
#pragma unroll
  for (int k = 0; k < kApplyRows; ++k) {
    const int64_t r = base + (int64_t)k * (256 / groups);
    if (r >= M) continue;
    const uint32_t w[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
    const uint32_t rw[4] = {rv[k].x, rv[k].y, rv[k].z, rv[k].w};
    uint32_t o[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float y0 = fmaf(__uint_as_float(w[e] << 16), a[2 * e], b[2 * e]);
      float y1 = fmaf(__uint_as_float(w[e] & 0xFFFF0000u), a[2 * e + 1], b[2 * e + 1]);
      if (residual) {
        y0 += __uint_as_float(rw[e] << 16);
        y1 += __uint_as_float(rw[e] & 0xFFFF0000u);
      }
      o[e] = relu ? pack_relu_bf16x2(y0, y1) : pack_bf16x2(y0, y1);
    }
    *reinterpret_cast<uint4*>(out + r * C + gidx * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}
// raw (un-folded) weights: bf16 [O][R][S][I]; conv1: 3 channels summed, [64][64] with k = r*7+s
__global__ void pack_conv_raw_kernel(const float* __restrict__ w, int cout, int cin, int k,
                                     __nv_bfloat16* __restrict__ wp) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= cout * cin * k * k) return;
  const int i = idx % cin;
  const int s = (idx / cin) % k;
  const int r = (idx / (cin * k)) % k;
  const int o = idx / (cin * k * k);
  wp[idx] = __float2bfloat16_rn(w[((o * cin + i) * k + r) * k + s]);
}
// conv1 for the training stem: three input channels summed, fp32 [64][49]; and the fold of the batch scale
__global__ void pack_conv1_raw32_kernel(const float* __restrict__ w, float* __restrict__ w32) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * 49) return;
  const int o = idx / 49, k = idx % 49;
  w32[idx] = w[(o * 3 + 0) * 49 + k] + w[(o * 3 + 1) * 49 + k] + w[(o * 3 + 2) * 49 + k];
}
__global__ void fold_conv1_kernel(const float* __restrict__ w32, const float* __restrict__ scale_shift,
                                  __nv_bfloat16* __restrict__ w1fold) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * 64) return;
  const int o = idx / 64, k = idx % 64;
  w1fold[idx] = __float2bfloat16_rn(k < 49 ? w32[o * 49 + k] * scale_shift[o] : 0.f);
}
__global__ void pack_conv1_raw_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ w1) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * 64) return;
  const int o = idx / 64, k = idx % 64;
  float v = 0.f;
  if (k < 49) v = w[(o * 3 + 0) * 49 + k] + w[(o * 3 + 1) * 49 + k] + w[(o * 3 + 2) * 49 + k];
  w1[idx] = __float2bfloat16_rn(v);
}

}  // namespace avvad

using namespace avvad;

struct avvad_resnet18 {
  __nv_bfloat16* w[20];
  float* bias[20];
  __nv_bfloat16* w1b;  // conv1 folded bf16 [64][64], k = r*7+s (3 input channels summed)
  bool set[20];
  // downsample blocks (stages 2-4): conv_b weights with the 1x1 branch appended along K, summed folded biases
  __nv_bfloat16* wf[3];
  float* bf[3];
  bool fused_ready;
  // training mode (batch-statistics BN): un-folded bf16 weights and BN affine parameters
  __nv_bfloat16* wraw[20];
  float* w1raw32;        // conv1 raw weights, three input channels summed, fp32 [64][49]
  __nv_bfloat16* w1fold;  // conv1 weights with the batch scale folded in (training stem, second pass)
  float* gamma[20];
  float* beta[20];
  bool set_train[20];
};

extern "C" int avvad_resnet18_create(avvad_resnet18** out) {
  AVVAD_CHECK_ARG(out, "null out");
  avvad_resnet18* h = new avvad_resnet18();
  for (int i = 0; i < 20; ++i) {
    h->w[i] = nullptr;
    h->bias[i] = nullptr;
    h->set[i] = false;
  }
  for (int i = 0; i < 20; ++i) {
    h->wraw[i] = nullptr;
    h->gamma[i] = h->beta[i] = nullptr;
    h->set_train[i] = false;
  }
  h->w1b = nullptr;
  for (int i = 0; i < 3; ++i) {
    h->wf[i] = nullptr;
    h->bf[i] = nullptr;
  }
  h->fused_ready = false;
  h->w1raw32 = nullptr;
  h->w1fold = nullptr;
  for (int i = 0; i < 20; ++i) {
    const ConvSpec& s = kSpecs[i];
    AVVAD_CUDA(cudaMalloc(&h->bias[i], sizeof(float) * s.cout));
    if (i == 0) {
      AVVAD_CUDA(cudaMalloc(&h->w1b, sizeof(__nv_bfloat16) * 64 * 64));
    } else {
      AVVAD_CUDA(cudaMalloc(&h->w[i], sizeof(__nv_bfloat16) * (size_t)s.cout * s.cin * s.k * s.k));
    }
  }
  *out = h;
  return AVVAD_OK;
}

extern "C" void avvad_resnet18_destroy(avvad_resnet18* h) {
  if (!h) return;
  for (int i = 0; i < 20; ++i) {
    cudaFree(h->w[i]);
    cudaFree(h->bias[i]);
  }
  for (int i = 0; i < 20; ++i) {
    cudaFree(h->wraw[i]);
    cudaFree(h->gamma[i]);
    cudaFree(h->beta[i]);
  }
  cudaFree(h->w1b);
  cudaFree(h->w1raw32);
  cudaFree(h->w1fold);
  for (int i = 0; i < 3; ++i) {
    cudaFree(h->wf[i]);
    cudaFree(h->bf[i]);
  }
  delete h;
}

extern "C" int avvad_resnet18_set_conv(avvad_resnet18* h, int layer, const float* w, const float* gamma,
                                       const float* beta, const float* mean, const float* var, float bn_eps,
                                       void* stream) {
  AVVAD_CHECK_ARG(h && layer >= 0 && layer < 20, "bad handle/layer");
  AVVAD_CHECK_ARG(w && gamma && beta && mean && var, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const ConvSpec& s = kSpecs[layer];
  if (layer == 0) {
    pack_conv1_tc_kernel<<<(64 * 64 + 255) / 256, 256, 0, st>>>(w, gamma, beta, mean, var, bn_eps, h->w1b, h->bias[0]);
  } else {
    const int total = s.cout * s.cin * s.k * s.k;
    pack_conv_kernel<<<(total + 255) / 256, 256, 0, st>>>(w, gamma, beta, mean, var, bn_eps, s.cout, s.cin, s.k,
                                                          h->w[layer], h->bias[layer]);
  }
  AVVAD_LAUNCHED();
  h->set[layer] = true;
  h->fused_ready = false;
  return AVVAD_OK;
}

static const int kDsBlocks[3][2] = {{6, 7}, {11, 12}, {16, 17}};  // (conv_b, downsample) layer indices of stages 2-4

static int build_fused(avvad_resnet18* h, cudaStream_t st) {
  if (h->fused_ready) return AVVAD_OK;
  for (int i = 0; i < 3; ++i) {
    const int lb = kDsBlocks[i][0], lds = kDsBlocks[i][1];
    const ConvSpec& sb = kSpecs[lb];
    const ConvSpec& sd = kSpecs[lds];
    const int kb = sb.k * sb.k * sb.cin, kds = sd.cin;
    const size_t total = (size_t)sb.cout * (kb + kds);
    if (!h->wf[i]) {
      AVVAD_CUDA(cudaMalloc(&h->wf[i], total * sizeof(__nv_bfloat16)));
      AVVAD_CUDA(cudaMalloc(&h->bf[i], sb.cout * sizeof(float)));
    }
    concat_ds_kernel<<<(unsigned)ceil_div((int64_t)total, 256), 256, 0, st>>>(h->w[lb], h->w[lds], h->bias[lb],
                                                                             h->bias[lds], sb.cout, kb, kds, h->wf[i],
                                                                             h->bf[i]);
    AVVAD_LAUNCHED();
  }
  h->fused_ready = true;
  return AVVAD_OK;
}

static int64_t chunk_of(int64_t n_frames, int64_t chunk) {
  if (chunk <= 0) chunk = 2048;
  return n_frames < chunk ? n_frames : chunk;
}

extern "C" size_t avvad_resnet18_workspace_bytes(int64_t n_frames, int64_t chunk_frames) {
  if (n_frames <= 0) return 0;
  const int64_t mc = chunk_of(n_frames, chunk_frames);
  return (size_t)(4 * align_up((size_t)mc * kActBytesPerFrame, 1024));  // four rotating NHWC activation buffers
}

static int run_conv(avvad_resnet18* h, int layer, const __nv_bfloat16* in, const __nv_bfloat16* residual,
                    __nv_bfloat16* out, int64_t n, int relu, cudaStream_t st) {
  const ConvSpec& s = kSpecs[layer];
  return avvad_conv2d_nhwc_bf16(in, h->w[layer], h->bias[layer], residual, out, n, s.hin, s.hin, s.cin, s.cout, s.k,
                                s.k, s.stride, s.pad, relu, st);
}

// Runs conv layers in execution order on one chunk; stops after layer `upto` (20 = run everything).
// Returns the buffer index holding the last produced activation in *last.
// Video source of one trunk call: fp32 frames (already standardised) or u8 frames at the source rate + the gather
struct StemInput {
  const float* frames = nullptr;  // [n][67*67]
  const uint8_t* src = nullptr;   // [B][f_max][67*67]
  const int32_t* n_src = nullptr;
  const int32_t* n_out = nullptr;
  int f_max = 0, t_max = 0, num = 0, den = 0, standardise = 0;
  int64_t src_bytes = 0;  // size of `src`
  float mean = 0.f, denom = 1.f;
  StemInput advance(int64_t f0) const {  // the same source seen from frame f0 on (chunking)
    StemInput r = *this;
    r.first = first + f0;
    return r;
  }
  int64_t first = 0;  // global index of the first frame of this (sub-)call
};

// w / bias: the conv1 operands of this launch (folded eval-mode weights by default); stats != NULL selects the
// statistics-only first pass of the training stem (fp32 frames)
static int launch_stem_s2d(avvad_resnet18* h, const StemInput& in, int64_t n, __nv_bfloat16* out, cudaStream_t st,
                           const __nv_bfloat16* w = nullptr, const float* bias = nullptr, double* stats = nullptr) {
  static PerDeviceOnce once;
  AVVAD_CUDA(once.run([] {
    cudaError_t e = cudaFuncSetAttribute(tc::stem_s2d_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::kS2Smem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(tc::stem_s2d_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::kS2Smem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(tc::stem_s2d_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::kS2Smem);
    return e;
  }));
  static int num_sms = [] {
    int dev = 0, v = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v > 0 ? v : 148;
  }();
  tc::StemS2Params p{};
  p.n_frames = n;
  p.w1b = w ? w : h->w1b;
  p.bias = w ? bias : h->bias[0];
  p.out = out;
  p.stats = stats;
  const int64_t batches = (n + tc::kS2FramesPerBatch - 1) / tc::kS2FramesPerBatch;
  const unsigned grid = (unsigned)(batches < num_sms ? batches : num_sms);
  void* tok = nullptr;
  tc::prof_begin(st, &tok);
  if (in.src) {
    // frame n of this launch is global frame in.first + n = (b, k); shift the per-utterance arrays so that the kernel's
    // n / t_max arithmetic stays local: only whole-utterance offsets are representable, so pass `first` through
    p.src = in.src; p.n_src = in.n_src; p.n_out = in.n_out; p.src_bytes = in.src_bytes;
    p.f_max = in.f_max; p.t_max = in.t_max; p.num = in.num; p.den = in.den;
    p.mean = in.mean; p.denom = in.denom; p.standardise = in.standardise;
    p.first = in.first;
    tc::stem_s2d_kernel<1><<<grid, tc::kS2Threads, tc::kS2Smem, st>>>(p);
  } else if (stats) {
    p.frames = in.frames + in.first * kFrameHW;
    tc::stem_s2d_kernel<0, true><<<grid, tc::kS2Threads, tc::kS2Smem, st>>>(p);
  } else {
    p.frames = in.frames + in.first * kFrameHW;
    tc::stem_s2d_kernel<0><<<grid, tc::kS2Threads, tc::kS2Smem, st>>>(p);
  }
  AVVAD_LAUNCHED();
  tc::prof_end(st, tok, 3, 2.0 * (double)n * 1156 * 64 * 49);
  return AVVAD_OK;
}

static int launch_stem(avvad_resnet18* h, const StemInput& in, int64_t n, __nv_bfloat16* out, cudaStream_t st) {
  return launch_stem_s2d(h, in, n, out, st);
}

// per-frame elements of a stage's input / output activation and its tensor-core MACs per frame
static const int64_t kStageIn[4] = {17 * 17 * 64, 17 * 17 * 64, 9 * 9 * 128, 5 * 5 * 256};
static const int64_t kStageOut[4] = {17 * 17 * 64, 9 * 9 * 128, 5 * 5 * 256, 3 * 3 * 512};
static const double kStageMac[4] = {42614784.0, 42467328.0, 52428800.0, 75497472.0};

// Runs the trunk on one chunk; stops after layer `upto` (20 = run everything).  Returns the buffer index holding the
// last produced activation in *last.  Stage s = torchvision layer(s+1): two BasicBlocks, the first of stages 1-3 with
// a stride-2 conv_a and a 1x1 downsample branch, K-concatenated into conv_b (the layer-by-layer hook, upto == the
// downsample layer, runs it as a separate 1x1 convolution added as the residual).
static int run_trunk_chunk(avvad_resnet18* h, const StemInput& in, int64_t n, __nv_bfloat16* const buf[4], int upto,
                           int* last, cudaStream_t st) {
  int frc = build_fused(h, st);
  if (frc) return frc;
  // Note: running layer1/layer2 depth-first over L2-sized slices of the chunk was measured SLOWER (each persistent
  // launch pays a prologue and a tail; 512-frame slices cost +15 % on the convolutions), larger chunks are faster:
  // chunk 2048 -> 20288 frames = 36.3 -> 33.3 ms of convolutions per 81,152 frames.
  const bool whole = upto < 20;  // layer-by-layer test hook: per-launch profiling records
  int cur = 0;
  *last = cur;
  int layer = 1;
  for (int stage = 0; stage < 4; ++stage) {
    {
      const int64_t f0 = 0, nn = n;
      if (stage == 0) {
        int rc = launch_stem(h, in.advance(f0), nn, buf[0] + f0 * kStageIn[0], st);
        if (rc) return rc;
        if (upto == 0) return AVVAD_OK;
      }
      // one profiling record per stage: its convolution launches and their algorithmic FLOPs
      void* gtok = nullptr;
      if (!whole) tc::prof_group_begin(st, &gtok);
      struct GroupEnd {
        cudaStream_t st; void* tok; double flops;
        ~GroupEnd() { tc::prof_group_end(st, tok, 0, flops); }
      } group_end{st, gtok, 2.0 * (double)nn * kStageMac[stage]};
      for (int blk = 0; blk < 2; ++blk) {
        int o[3], k = 0;
        for (int i = 0; i < 4; ++i)
          if (i != cur) o[k++] = i;
        const bool ds = (stage > 0 && blk == 0);
        const int la = layer, lb = layer + 1, lds = layer + 2;
        // the block input has the stage-input geometry only for the first block of the stage
        const __nv_bfloat16* xin = buf[cur] + f0 * (blk == 0 ? kStageIn[stage] : kStageOut[stage]);
        __nv_bfloat16* y0 = buf[o[0]] + f0 * kStageOut[stage];
        __nv_bfloat16* y1 = buf[o[1]] + f0 * kStageOut[stage];
        __nv_bfloat16* y2 = buf[o[2]] + f0 * kStageOut[stage];
        if (stage == 0 && !whole && tc::block17_enabled() &&
            ((reinterpret_cast<uintptr_t>(xin) | reinterpret_cast<uintptr_t>(y2)) & 31) == 0) {
          // layer1: the whole BasicBlock in one kernel, conv_a's output stays in shared memory (conv_block.cuh)
          int rcb = tc::launch_block17(xin, h->w[la], h->bias[la], h->w[lb], h->bias[lb], y2, nn, st);
          if (rcb) return rcb;
          cur = o[2];
          *last = cur;
          layer += 2;
          continue;
        }
        int rc = run_conv(h, la, xin, nullptr, y0, nn, 1, st);
        if (rc) return rc;
        if (upto == la) { *last = o[0]; return AVVAD_OK; }
        const __nv_bfloat16* res = xin;
        if (ds && upto != lds) {
          // conv_b with the downsample branch appended along K: no 1x1 launch, no residual round trip
          const ConvSpec& sb = kSpecs[lb];
          const ConvSpec& sd = kSpecs[lds];
          tc::EpiParams ep{};
          ep.bias = h->bf[stage - 1];
          ep.C = y2;
          ep.ldc = sb.cout;
          ep.relu = 1;
          tc::SecondOperand so;
          so.in2 = xin;
          so.H2 = sd.hin; so.W2 = sd.hin; so.Cin2 = sd.cin; so.stride2 = sd.stride;
          rc = tc::launch_tma_conv(y0, h->wf[stage - 1], ep, nn, sb.hin, sb.hin, sb.cin, sb.cout, sb.k, sb.k, sb.stride,
                                   sb.pad, 0, st, 0, 0.0, &so);
          if (rc) return rc;
          cur = o[2];
          *last = cur;
          if (upto == lb) return AVVAD_OK;
          layer += 3;
          continue;
        }
        if (ds) {
          rc = run_conv(h, lds, xin, nullptr, y1, nn, 0, st);
          if (rc) return rc;
          if (upto == lds) { *last = o[1]; return AVVAD_OK; }
          res = y1;
        }
        rc = run_conv(h, lb, y0, res, y2, nn, 1, st);
        if (rc) return rc;
        cur = o[2];
        *last = cur;
        if (upto == lb) return AVVAD_OK;
        layer += ds ? 3 : 2;
      }
    }
  }
  return AVVAD_OK;
}

static int check_loaded(avvad_resnet18* h) {
  for (int i = 0; i < 20; ++i)
    if (!h->set[i]) {
      set_error("resnet18: conv layer " + std::to_string(i) + " not loaded");
      return AVVAD_ERR_STATE;
    }
  return AVVAD_OK;
}

static int forward_common(avvad_resnet18* h, const StemInput& in, int64_t n_frames, int64_t chunk_frames,
                          void* workspace, size_t workspace_bytes, float* feat, void* feat_bf16, int64_t ld_bf16,
                          int64_t col_off, cudaStream_t st) {
  AVVAD_CHECK_ARG(feat || feat_bf16, "at least one output required");
  int rc = check_loaded(h);
  if (rc) return rc;
  if (workspace_bytes < avvad_resnet18_workspace_bytes(n_frames, chunk_frames)) {
    set_error("resnet18: workspace too small");
    return AVVAD_ERR_WORKSPACE;
  }
  const int64_t mc = chunk_of(n_frames, chunk_frames);
  const size_t bsz = align_up((size_t)mc * kActBytesPerFrame, 1024);
  __nv_bfloat16* buf[4];
  for (int i = 0; i < 4; ++i) buf[i] = reinterpret_cast<__nv_bfloat16*>((uint8_t*)workspace + i * bsz);
  for (int64_t f0 = 0; f0 < n_frames; f0 += mc) {
    const int64_t n = (n_frames - f0 < mc) ? (n_frames - f0) : mc;
    int last = 0;
    rc = run_trunk_chunk(h, in.advance(f0), n, buf, 20, &last, st);
    if (rc) return rc;
    const int64_t total = n * (512 / 8);
    avgpool_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(
        buf[last], n, 9, 512, feat ? feat + f0 * 512 : nullptr,
        feat_bf16 ? (__nv_bfloat16*)feat_bf16 + f0 * ld_bf16 : nullptr, ld_bf16, col_off);
    AVVAD_LAUNCHED();
  }
  return AVVAD_OK;
}

extern "C" int avvad_resnet18_forward(avvad_resnet18* h, const float* frames, int64_t n_frames, int64_t chunk_frames,
                                      void* workspace, size_t workspace_bytes, float* feat, void* feat_bf16,
                                      int64_t ld_bf16, int64_t col_off, void* stream) {
  AVVAD_CHECK_ARG(h && frames && workspace && n_frames > 0, "bad argument");
  StemInput in;
  in.frames = frames;
  return forward_common(h, in, n_frames, chunk_frames, workspace, workspace_bytes, feat, feat_bf16, ld_bf16, col_off,
                        (cudaStream_t)stream);
}

// Same trunk fed straight from the 30 fps u8 source frames: output frame (b, k), k < t_max, is source frame
// upsample_src_index(k, n_src[b]) standardised as (v - mean) / (std + eps) when k < n_out[b], else the collate zero
// frame -- exactly what avvad_upsample_gather writes, without the fp32 (B, t_max, 67, 67) round trip through HBM.
extern "C" int avvad_resnet18_forward_u8(avvad_resnet18* h, const uint8_t* src, const int32_t* n_src,
                                         const int32_t* n_out, int32_t B, int32_t f_max, int32_t t_max, int32_t num,
                                         int32_t den, float mean, float stdv, float eps, int standardise,
                                         int64_t chunk_frames, void* workspace, size_t workspace_bytes, float* feat,
                                         void* feat_bf16, int64_t ld_bf16, int64_t col_off, void* stream) {
  AVVAD_CHECK_ARG(h && src && n_src && n_out && workspace, "null pointer");
  AVVAD_CHECK_ARG(B > 0 && f_max > 0 && t_max > 0 && num > 0 && den > 0, "non-positive size");
  StemInput in;
  in.src = src; in.n_src = n_src; in.n_out = n_out;
  in.f_max = f_max; in.t_max = t_max; in.num = num; in.den = den;
  in.mean = mean; in.denom = stdv + eps; in.standardise = standardise;
  in.src_bytes = (int64_t)B * f_max * kFrameHW;
  return forward_common(h, in, (int64_t)B * t_max, chunk_frames, workspace, workspace_bytes, feat, feat_bf16, ld_bf16,
                        col_off, (cudaStream_t)stream);
}

extern "C" int avvad_resnet18_forward_upto(avvad_resnet18* h, const float* frames, int64_t n_frames, int upto,
                                           void* workspace, size_t workspace_bytes, void* out_act, void* stream) {
  AVVAD_CHECK_ARG(h && frames && workspace && out_act && n_frames > 0 && upto >= 0 && upto < 20, "bad argument");
  int rc = check_loaded(h);
  if (rc) return rc;
  if (workspace_bytes < avvad_resnet18_workspace_bytes(n_frames, n_frames)) {
    set_error("resnet18: workspace too small (forward_upto runs a single chunk)");
    return AVVAD_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const size_t bsz = align_up((size_t)n_frames * kActBytesPerFrame, 1024);
  __nv_bfloat16* buf[4];
  for (int i = 0; i < 4; ++i) buf[i] = reinterpret_cast<__nv_bfloat16*>((uint8_t*)workspace + i * bsz);
  int last = 0;
  StemInput in;
  in.frames = frames;
  rc = run_trunk_chunk(h, in, n_frames, buf, upto, &last, st);
  if (rc) return rc;
  const ConvSpec& s = kSpecs[upto];
  const int ho = (upto == 0) ? 17 : s.hout;
  const size_t bytes = (size_t)n_frames * ho * ho * s.cout * sizeof(__nv_bfloat16);
  AVVAD_CUDA(cudaMemcpyAsync(out_act, buf[last], bytes, cudaMemcpyDeviceToDevice, st));
  return AVVAD_OK;
}

// =====================================================================================================================
// Training-mode forward: BatchNorm uses batch statistics over ALL frames of the call (scripts/train_AV_net.py:253 puts
// the frozen trunk's BN layers into train mode) and updates the running statistics in place.  Layer-major over the
// whole batch: conv (raw, un-folded weights) -> per-channel statistics -> normalise + affine (+ residual) + ReLU.
// =====================================================================================================================
extern "C" int avvad_resnet18_set_conv_train(avvad_resnet18* h, int layer, const float* w, const float* gamma,
                                             const float* beta, void* stream) {
  AVVAD_CHECK_ARG(h && layer >= 0 && layer < 20 && w && gamma && beta, "bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const ConvSpec& s = kSpecs[layer];
  const size_t wn = (layer == 0) ? 64 * 64 : (size_t)s.cout * s.cin * s.k * s.k;
  if (!h->wraw[layer]) {
    AVVAD_CUDA(cudaMalloc(&h->wraw[layer], wn * sizeof(__nv_bfloat16)));
    AVVAD_CUDA(cudaMalloc(&h->gamma[layer], s.cout * sizeof(float)));
    AVVAD_CUDA(cudaMalloc(&h->beta[layer], s.cout * sizeof(float)));
  }
  if (layer == 0) {
    if (!h->w1raw32) {
      AVVAD_CUDA(cudaMalloc(&h->w1raw32, 64 * 49 * sizeof(float)));
      AVVAD_CUDA(cudaMalloc(&h->w1fold, 64 * 64 * sizeof(__nv_bfloat16)));
    }
    pack_conv1_raw32_kernel<<<13, 256, 0, st>>>(w, h->w1raw32);
    AVVAD_LAUNCHED();
    pack_conv1_raw_kernel<<<16, 256, 0, st>>>(w, h->wraw[0]);
  } else
    pack_conv_raw_kernel<<<(unsigned)ceil_div((int64_t)wn, 256), 256, 0, st>>>(w, s.cout, s.cin, s.k, h->wraw[layer]);
  AVVAD_LAUNCHED();
  AVVAD_CUDA(cudaMemcpyAsync(h->gamma[layer], gamma, s.cout * sizeof(float), cudaMemcpyDeviceToDevice, st));
  AVVAD_CUDA(cudaMemcpyAsync(h->beta[layer], beta, s.cout * sizeof(float), cudaMemcpyDeviceToDevice, st));
  h->set_train[layer] = true;
  return AVVAD_OK;
}

extern "C" size_t avvad_resnet18_train_workspace_bytes(int64_t n_frames) {
  if (n_frames <= 0) return 0;
  const size_t act = align_up((size_t)n_frames * kActBytesPerFrame, 1024);
  return 5 * act + 64 * 1024;  // four rotating activations, one raw conv output, statistics
}

namespace {
struct TrainCtx {
  avvad_resnet18* h;
  int64_t n;
  double* stats;        // [2*512]
  float* mean_invstd;   // [2*512]
  float bn_eps, momentum;
  float* const* running_mean;
  float* const* running_var;
  cudaStream_t st;
};

// raw [M][C] -> out = act(bn(raw) (+res)); updates the running statistics of `layer`
int bn_train(const TrainCtx& c, int layer, const __nv_bfloat16* raw, int64_t M, int C, const __nv_bfloat16* residual,
             int relu, __nv_bfloat16* out, float* mean_invstd_out = nullptr) {
  AVVAD_CUDA(cudaMemsetAsync(c.stats, 0, sizeof(double) * 2 * C, c.st));
  const int lanes = 256 / (C / 8);
  bn_stats_kernel<<<(unsigned)ceil_div(M, kStatRows), 256, (size_t)lanes * 2 * C * sizeof(float), c.st>>>(raw, M, C,
                                                                                                        c.stats);
  AVVAD_LAUNCHED();
  bn_finalize_kernel<<<(unsigned)ceil_div(C, 128), 128, 0, c.st>>>(
      c.stats, M, C, c.bn_eps, c.momentum, c.h->gamma[layer], c.h->beta[layer], c.mean_invstd,
      c.running_mean ? c.running_mean[layer] : nullptr, c.running_var ? c.running_var[layer] : nullptr, mean_invstd_out);
  AVVAD_LAUNCHED();
  const int rows_per_block = lanes * kApplyRows;
  bn_apply_kernel<<<(unsigned)ceil_div(M, rows_per_block), 256, 2 * C * sizeof(float), c.st>>>(
      raw, M, C, c.mean_invstd, residual, relu, out);
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}

int conv_raw(const TrainCtx& c, int layer, const __nv_bfloat16* in, __nv_bfloat16* raw) {
  const ConvSpec& s = kSpecs[layer];
  return avvad_conv2d_nhwc_bf16(in, c.h->wraw[layer], nullptr, nullptr, raw, c.n, s.hin, s.hin, s.cin, s.cout, s.k, s.k,
                                s.stride, s.pad, 0, c.st);
}
}  // namespace

// running_mean / running_var: arrays of 20 device pointers (the module's BatchNorm buffers, updated in place with
// `momentum`), or NULL to leave running statistics untouched.
extern "C" int avvad_resnet18_forward_train(avvad_resnet18* h, const float* frames, int64_t n_frames, void* workspace,
                                            size_t workspace_bytes, float bn_eps, float momentum,
                                            float* const* running_mean, float* const* running_var, float* feat,
                                            void* feat_bf16, int64_t ld_bf16, int64_t col_off, void* stream) {
  AVVAD_CHECK_ARG(h && frames && workspace && n_frames > 0 && (feat || feat_bf16), "bad argument");
  for (int i = 0; i < 20; ++i)
    if (!h->set_train[i]) {
      set_error("resnet18: training weights of conv layer " + std::to_string(i) + " not loaded");
      return AVVAD_ERR_STATE;
    }
  if (workspace_bytes < avvad_resnet18_train_workspace_bytes(n_frames)) {
    set_error("resnet18: training workspace too small");
    return AVVAD_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n = n_frames;
  const size_t act = align_up((size_t)n * kActBytesPerFrame, 1024);
  uint8_t* p = (uint8_t*)workspace;
  __nv_bfloat16* buf[4];
  for (int i = 0; i < 4; ++i) buf[i] = reinterpret_cast<__nv_bfloat16*>(p + i * act);
  __nv_bfloat16* raw = reinterpret_cast<__nv_bfloat16*>(p + 4 * act);  // raw conv output (largest: layer1)
  double* stats = reinterpret_cast<double*>(p + 5 * act);
  float* mean_invstd = reinterpret_cast<float*>(p + 5 * act + 16 * 1024);  // scale [C] | shift [C]
  TrainCtx c{h, n, stats, mean_invstd, bn_eps, momentum, running_mean, running_var, st};

  // stem, two passes of the image-as-operand kernel (no 34x34x64 tensor in HBM):
  //   1. raw conv1 (un-folded weights, no bias) -> per-channel batch statistics only
  //   2. batch scale folded into the weights, batch shift as bias -> conv + BN + ReLU + max-pool as in eval mode
  {
    StemInput sin;
    sin.frames = frames;
    AVVAD_CUDA(cudaMemsetAsync(stats, 0, sizeof(double) * 2 * 64, st));
    int rc = launch_stem_s2d(h, sin, n, nullptr, st, h->wraw[0], nullptr, stats);
    if (rc) return rc;
    bn_finalize_kernel<<<1, 128, 0, st>>>(stats, n * 1156, 64, bn_eps, momentum, h->gamma[0], h->beta[0], mean_invstd,
                                          running_mean ? running_mean[0] : nullptr,
                                          running_var ? running_var[0] : nullptr);
    AVVAD_LAUNCHED();
    fold_conv1_kernel<<<16, 256, 0, st>>>(h->w1raw32, mean_invstd, h->w1fold);
    AVVAD_LAUNCHED();
    rc = launch_stem_s2d(h, sin, n, buf[0], st, h->w1fold, mean_invstd + 64);
    if (rc) return rc;
  }
  int cur = 0, layer = 1;
  for (int stage = 0; stage < 4; ++stage) {
    for (int blk = 0; blk < 2; ++blk) {
      int o[3], k = 0;
      for (int i = 0; i < 4; ++i)
        if (i != cur) o[k++] = i;
      const bool ds = (stage > 0 && blk == 0);
      const int la = layer, lb = layer + 1, lds = layer + 2;
      const ConvSpec& sa = kSpecs[la];
      const int64_t Mo = n * sa.hout * sa.hout;
      int rc = conv_raw(c, la, buf[cur], raw);
      if (rc) return rc;
      rc = bn_train(c, la, raw, Mo, sa.cout, nullptr, 1, buf[o[0]]);
      if (rc) return rc;
      const __nv_bfloat16* res = buf[cur];
      if (ds) {
        rc = conv_raw(c, lds, buf[cur], raw);
        if (rc) return rc;
        rc = bn_train(c, lds, raw, Mo, sa.cout, nullptr, 0, buf[o[1]]);
        if (rc) return rc;
        res = buf[o[1]];
      }
      rc = conv_raw(c, lb, buf[o[0]], raw);
      if (rc) return rc;
      rc = bn_train(c, lb, raw, Mo, sa.cout, res, 1, buf[o[2]]);
      if (rc) return rc;
      cur = o[2];
      layer += ds ? 3 : 2;
    }
  }
  const int64_t total = n * (512 / 8);
  avgpool_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(buf[cur], n, 9, 512, feat,
                                                                 (__nv_bfloat16*)feat_bf16, ld_bf16, col_off);
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}

#include "resnet_bwd.cuh"
