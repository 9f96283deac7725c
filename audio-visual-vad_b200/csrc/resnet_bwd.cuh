// Back-propagation through the ResNet-18 trunk (included at the end of resnet.cu: same translation unit, it uses the
// trunk handle, kSpecs and the BatchNorm kernels defined there).
//
// Reference semantics: autograd of packages/models/Video_Net.py:60-99 with the trunk TRAINABLE -- what
// scripts/train_video_net.py:145-173 does (all parameters handed to Adam, model.train(): batch-statistics BatchNorm).
//
// Forward with a tape (avvad_resnet18_forward_tape): the training-mode forward of resnet.cu, layer-major over the whole
// call, but every tensor the backward needs is kept -- raw convolution outputs (the BatchNorm inputs), the
// post-activation tensors (the convolution inputs and ReLU masks), per-layer batch mean / inverse std.  The stem runs
// un-fused here (direct conv1 -> BN -> ReLU -> max-pool as separate kernels) because the max-pool backward needs the
// 34x34x64 map the fused inference stem never writes.
//
// Backward (avvad_resnet18_backward), per BasicBlock in reverse:
//   ReLU mask + BatchNorm backward : two passes over (raw, upstream gradient): per-channel sums in fp64, then
//                                    dRaw = gamma*invstd*(g - mean(g) - xhat*mean(g*xhat)); dgamma, dbeta on the way
//   dgrad (data gradient)          : the forward implicit-GEMM engine (tcgen05, TMA-box im2col) run on the gradient with
//                                    the weights flipped and transposed ([Cin][R][S][Cout]); stride-2 layers first
//                                    zero-insert the gradient to the input resolution
//   wgrad (weight gradient)        : dW[o][tap][i] = sum_pixels dRaw[pixel][o] * X[pixel + tap][i] as a tcgen05 GEMM with
//                                    K = pixels: transposed copies of dRaw ([Cout][P]) and of the im2col matrix
//                                    ([taps*Cin][P], gather + transpose in one kernel), split-K over the SMs, fp32
//   max-pool / average-pool        : index-exact (first maximum in scan order, as PyTorch's kernels pick)
// Gradient activations travel in bf16 (fp32 accumulation inside every kernel), parameters' gradients come back fp32 in
// PyTorch's layout.

namespace avvad {
namespace bwd {

// ---- tape geometry ----------------------------------------------------------------------------------------------
// tensor ids: 0 raw0 (n,34,34,64) | 1 act0 (n,34,34,64) | 2 pool (n,17,17,64) | 3+l-1: raw of conv l (1..19) |
// 22+2*bk: y1 of block bk | 23+2*bk: out of block bk | then per-layer float [20][1024] (mean | invstd)
constexpr int kNumTensors = 3 + 19 + 16;
struct BlockDef {
  int la, lb, lds;  // conv layer indices (lds = -1: identity shortcut)
};
static const BlockDef kBlocks[8] = {{1, 2, -1}, {3, 4, -1}, {5, 6, 7}, {8, 9, -1}, {10, 11, 12}, {13, 14, -1},
                                    {15, 16, 17}, {18, 19, -1}};

static size_t tensor_elems_per_frame(int id) {
  if (id == 0 || id == 1) return 34 * 34 * 64;
  if (id == 2) return 17 * 17 * 64;
  if (id < 22) {
    const ConvSpec& s = kSpecs[id - 2];
    return (size_t)s.hout * s.hout * s.cout;
  }
  const int bk = (id - 22) / 2;
  const ConvSpec& s = kSpecs[kBlocks[bk].lb];
  return (size_t)s.hout * s.hout * s.cout;
}
struct Tape {
  uint8_t* base;
  size_t off[kNumTensors + 1];
  size_t stats_off, total;
  __nv_bfloat16* t(int id) const { return reinterpret_cast<__nv_bfloat16*>(base + off[id]); }
  __nv_bfloat16* raw(int l) const { return l == 0 ? t(0) : t(2 + l); }
  __nv_bfloat16* y1(int bk) const { return t(22 + 2 * bk); }
  __nv_bfloat16* out(int bk) const { return t(23 + 2 * bk); }
  float* stats(int l) const { return reinterpret_cast<float*>(base + stats_off) + (size_t)l * 1024; }
};
static Tape make_tape(void* base, int64_t n) {
  Tape tp;
  tp.base = (uint8_t*)base;
  size_t o = 0;
  for (int i = 0; i < kNumTensors; ++i) {
    tp.off[i] = o;
    o += align_up(tensor_elems_per_frame(i) * (size_t)n * 2, 1024);
  }
  tp.off[kNumTensors] = o;
  tp.stats_off = o;
  tp.total = o + 20 * 1024 * sizeof(float);
  return tp;
}

// ---- stem, un-fused (tape path) -------------------------------------------------------------------------------
// conv1 7x7/2 pad 3 on the single-channel frame with the three input channels' weights summed (fp32 [64][49]).
// One block per frame; the padded frame and the filter bank live in shared memory; a thread owns an output pixel.
__global__ void __launch_bounds__(256) conv1_direct_kernel(const float* __restrict__ frames, int64_t n,
                                                           const float* __restrict__ w32,
                                                           __nv_bfloat16* __restrict__ raw) {
  __shared__ float img[73 * 73];
  __shared__ float w[64 * 49];
  for (int i = threadIdx.x; i < 64 * 49; i += 256) w[i] = w32[i];
  for (int64_t f = blockIdx.x; f < n; f += gridDim.x) {
    __syncthreads();
    for (int i = threadIdx.x; i < 73 * 73; i += 256) {
      const int y = i / 73 - 3, x = i % 73 - 3;
      img[i] = (y >= 0 && y < 67 && x >= 0 && x < 67) ? frames[f * 67 * 67 + y * 67 + x] : 0.f;
    }
    __syncthreads();
    for (int p = threadIdx.x; p < 34 * 34; p += 256) {
      const int oh = p / 34, ow = p % 34;
      float px[49];
#pragma unroll
      for (int r = 0; r < 7; ++r)
#pragma unroll
        for (int s = 0; s < 7; ++s) px[r * 7 + s] = img[(2 * oh + r) * 73 + 2 * ow + s];
      __nv_bfloat16* dst = raw + (f * 1156 + p) * 64;
      for (int o = 0; o < 64; o += 2) {
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int k = 0; k < 49; ++k) {
          a0 = fmaf(px[k], w[o * 49 + k], a0);
          a1 = fmaf(px[k], w[(o + 1) * 49 + k], a1);
        }
        *reinterpret_cast<uint32_t*>(dst + o) = pack_bf16x2(a0, a1);
      }
    }
  }
}

// max-pool 3x3 / stride 2 / pad 1 on NHWC bf16 (34x34 -> 17x17), 8 channels per thread
__global__ void maxpool_fwd_kernel(const __nv_bfloat16* __restrict__ in, int64_t n, int Hin, int Hout, int C,
                                   __nv_bfloat16* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int groups = C / 8;
  if (idx >= n * Hout * Hout * groups) return;
  const int gq = (int)(idx % groups);
  const int64_t pix = idx / groups;
  const int ow = (int)(pix % Hout), oh = (int)((pix / Hout) % Hout);
  const int64_t f = pix / ((int64_t)Hout * Hout);
  float m[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) m[e] = -INFINITY;
  for (int r = 0; r < 3; ++r) {
    const int ih = 2 * oh - 1 + r;
    if (ih < 0 || ih >= Hin) continue;
    for (int s = 0; s < 3; ++s) {
      const int iw = 2 * ow - 1 + s;
      if (iw < 0 || iw >= Hin) continue;
      const uint4 v = *reinterpret_cast<const uint4*>(in + ((f * Hin + ih) * Hin + iw) * C + gq * 8);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        m[2 * e] = fmaxf(m[2 * e], __uint_as_float(w[e] << 16));
        m[2 * e + 1] = fmaxf(m[2 * e + 1], __uint_as_float(w[e] & 0xFFFF0000u));
      }
    }
  }
  uint4 o;
  o.x = pack_bf16x2(m[0], m[1]); o.y = pack_bf16x2(m[2], m[3]); o.z = pack_bf16x2(m[4], m[5]); o.w = pack_bf16x2(m[6], m[7]);
  *reinterpret_cast<uint4*>(out + pix * C + gq * 8) = o;
}

// Gradient of the max-pool, two small kernels (no atomics, no recomputation per input pixel):
//   1. per pooled output and channel: which of the 9 window positions holds the FIRST maximum (scan order rows, then
//      columns, strict '>' as in PyTorch's kernels) -> one byte (0..8);
//   2. per input pixel and 8 channels: sum the gradients of the (at most four) windows that selected it.
__global__ void maxpool_argmax_kernel(const __nv_bfloat16* __restrict__ act, int64_t n, int Hin, int Hout, int C,
                                      uint8_t* __restrict__ which) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int groups = C / 8;
  if (idx >= n * Hout * Hout * groups) return;
  const int gq = (int)(idx % groups);
  const int64_t pix = idx / groups;
  const int ow = (int)(pix % Hout), oh = (int)((pix / Hout) % Hout);
  const int64_t f = pix / ((int64_t)Hout * Hout);
  float best[8];
  uint32_t sel[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { best[e] = -INFINITY; sel[e] = 0; }
  for (int r = 0; r < 3; ++r) {
    const int y = 2 * oh - 1 + r;
    if (y < 0 || y >= Hin) continue;
    for (int s = 0; s < 3; ++s) {
      const int x = 2 * ow - 1 + s;
      if (x < 0 || x >= Hin) continue;
      const uint4 v = *reinterpret_cast<const uint4*>(act + ((f * Hin + y) * Hin + x) * C + gq * 8);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float a = __uint_as_float(w[e] << 16), b = __uint_as_float(w[e] & 0xFFFF0000u);
        if (a > best[2 * e]) { best[2 * e] = a; sel[2 * e] = r * 3 + s; }
        if (b > best[2 * e + 1]) { best[2 * e + 1] = b; sel[2 * e + 1] = r * 3 + s; }
      }
    }
  }
  uint2 o;
  o.x = sel[0] | (sel[1] << 8) | (sel[2] << 16) | (sel[3] << 24);
  o.y = sel[4] | (sel[5] << 8) | (sel[6] << 16) | (sel[7] << 24);
  *reinterpret_cast<uint2*>(which + pix * C + gq * 8) = o;
}
__global__ void maxpool_bwd_kernel(const uint8_t* __restrict__ which, const __nv_bfloat16* __restrict__ gpool, int64_t n,
                                   int Hin, int Hout, int C, __nv_bfloat16* __restrict__ gact) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int groups = C / 8;
  if (idx >= n * Hin * Hin * groups) return;
  const int gq = (int)(idx % groups);
  const int64_t pix = idx / groups;
  const int iw = (int)(pix % Hin), ih = (int)((pix / Hin) % Hin);
  const int64_t f = pix / ((int64_t)Hin * Hin);
  float acc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] = 0.f;
  // windows covering (ih, iw): oh with 2*oh-1 <= ih <= 2*oh+1, i.e. ih even: {ih/2}; ih odd: {(ih-1)/2, (ih+1)/2}
  for (int oh = ih / 2; oh <= (ih + 1) / 2; ++oh) {
    if (oh >= Hout) continue;
    for (int ow = iw / 2; ow <= (iw + 1) / 2; ++ow) {
      if (ow >= Hout) continue;
      const uint32_t me = (uint32_t)((ih - (2 * oh - 1)) * 3 + (iw - (2 * ow - 1)));   // my position inside that window
      const int64_t o = ((f * Hout + oh) * Hout + ow) * C + gq * 8;
      const uint2 w = *reinterpret_cast<const uint2*>(which + o);
      const uint4 gv = *reinterpret_cast<const uint4*>(gpool + o);
      const uint32_t gw[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const uint32_t s0 = ((e < 2 ? w.x : w.y) >> (16 * (e & 1))) & 0xFFu, s1 = ((e < 2 ? w.x : w.y) >> (16 * (e & 1) + 8)) & 0xFFu;
        if (s0 == me) acc[2 * e] += __uint_as_float(gw[e] << 16);
        if (s1 == me) acc[2 * e + 1] += __uint_as_float(gw[e] & 0xFFFF0000u);
      }
    }
  }
  uint4 o;
  o.x = pack_bf16x2(acc[0], acc[1]); o.y = pack_bf16x2(acc[2], acc[3]);
  o.z = pack_bf16x2(acc[4], acc[5]); o.w = pack_bf16x2(acc[6], acc[7]);
  *reinterpret_cast<uint4*>(gact + pix * C + gq * 8) = o;
}

// global average pool backward: g[f][p][c] = dfeat[f][c] / hw
__global__ void avgpool_bwd_kernel(const float* __restrict__ dfeat, int64_t n, int hw, int C, __nv_bfloat16* __restrict__ g) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int groups = C / 8;
  if (idx >= n * hw * groups) return;
  const int gq = (int)(idx % groups);
  const int64_t fp = idx / groups;
  const int64_t f = fp / hw;
  const float inv = 1.0f / (float)hw;
  const float4 a = *reinterpret_cast<const float4*>(dfeat + f * C + gq * 8);
  const float4 b = *reinterpret_cast<const float4*>(dfeat + f * C + gq * 8 + 4);
  uint4 o;
  o.x = pack_bf16x2(a.x * inv, a.y * inv); o.y = pack_bf16x2(a.z * inv, a.w * inv);
  o.z = pack_bf16x2(b.x * inv, b.y * inv); o.w = pack_bf16x2(b.z * inv, b.w * inv);
  *reinterpret_cast<uint4*>(g + fp * C + gq * 8) = o;
}

// ---- BatchNorm backward (batch statistics) with the ReLU mask of the layer's output folded in -------------------
// gm = g * (mask > 0) (mask == nullptr: gm = g);  xhat = (raw - mean) * invstd
// pass 1: sums[c] = sum gm, sums[C + c] = sum gm * xhat   (fp32 per thread, fp64 atomics per block -- as bn_stats_kernel)
__global__ void __launch_bounds__(256) bn_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ raw,
                                                            const __nv_bfloat16* __restrict__ g,
                                                            const __nv_bfloat16* __restrict__ mask, int64_t M, int C,
                                                            const float* __restrict__ mean_invstd,
                                                            double* __restrict__ sums) {
  extern __shared__ float rb_sm[];  // [lanes][2*C]
  const int groups = C / 8;
  const int lanes = 256 / groups;
  const int gidx = threadIdx.x % groups, ln = threadIdx.x / groups;
  float mu[8], is[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    mu[e] = mean_invstd[gidx * 8 + e];
    is[e] = mean_invstd[C + gidx * 8 + e];
  }
  const int64_t r0 = (int64_t)blockIdx.x * kStatRows;
  const int64_t r1 = (r0 + kStatRows < M) ? r0 + kStatRows : M;
  float s1[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s2[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int64_t r = r0 + ln; r < r1; r += lanes) {
    const uint4 xv = *reinterpret_cast<const uint4*>(raw + r * C + gidx * 8);
    const uint4 gv = *reinterpret_cast<const uint4*>(g + r * C + gidx * 8);
    uint4 mv = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
    if (mask) mv = *reinterpret_cast<const uint4*>(mask + r * C + gidx * 8);
    const uint32_t xw[4] = {xv.x, xv.y, xv.z, xv.w}, gw[4] = {gv.x, gv.y, gv.z, gv.w}, mw[4] = {mv.x, mv.y, mv.z, mv.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float g0 = (__uint_as_float(mw[e] << 16) > 0.f) ? __uint_as_float(gw[e] << 16) : 0.f;
      const float g1 = (__uint_as_float(mw[e] & 0xFFFF0000u) > 0.f) ? __uint_as_float(gw[e] & 0xFFFF0000u) : 0.f;
      const float x0 = (__uint_as_float(xw[e] << 16) - mu[2 * e]) * is[2 * e];
      const float x1 = (__uint_as_float(xw[e] & 0xFFFF0000u) - mu[2 * e + 1]) * is[2 * e + 1];
      s1[2 * e] += g0; s2[2 * e] = fmaf(g0, x0, s2[2 * e]);
      s1[2 * e + 1] += g1; s2[2 * e + 1] = fmaf(g1, x1, s2[2 * e + 1]);
    }
  }
  float* mine = rb_sm + (size_t)ln * 2 * C + gidx * 8;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    mine[e] = s1[e];
    mine[C + e] = s2[e];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * C; c += 256) {
    double acc = 0.0;
    for (int l = 0; l < lanes; ++l) acc += (double)rb_sm[(size_t)l * 2 * C + c];
    atomicAdd(sums + c, acc);
  }
}
// dbeta = S1, dgamma = S2; coef[c] = S1/M, coef[C+c] = S2/M for the apply pass
__global__ void bn_bwd_finalize_kernel(const double* __restrict__ sums, int64_t M, int C, float* __restrict__ dgamma,
                                       float* __restrict__ dbeta, float* __restrict__ coef) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  dbeta[c] = (float)sums[c];
  dgamma[c] = (float)sums[C + c];
  coef[c] = (float)(sums[c] / (double)M);
  coef[C + c] = (float)(sums[C + c] / (double)M);
}
// pass 2: dRaw = gamma*invstd*(gm - S1/M - xhat*S2/M); optionally also writes gm (the masked gradient, which the
// identity shortcut carries on)
__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ raw,
                                                           const __nv_bfloat16* __restrict__ g,
                                                           const __nv_bfloat16* __restrict__ mask, int64_t M, int C,
                                                           const float* __restrict__ mean_invstd,
                                                           const float* __restrict__ gamma, const float* __restrict__ coef,
                                                           __nv_bfloat16* __restrict__ draw,
                                                           __nv_bfloat16* __restrict__ gm_out) {
  const int groups = C / 8;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * groups) return;
  const int gidx = (int)(idx % groups);
  const int64_t r = idx / groups;
  const uint4 xv = *reinterpret_cast<const uint4*>(raw + r * C + gidx * 8);
  const uint4 gv = *reinterpret_cast<const uint4*>(g + r * C + gidx * 8);
  uint4 mv = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
  if (mask) mv = *reinterpret_cast<const uint4*>(mask + r * C + gidx * 8);
  const uint32_t xw[4] = {xv.x, xv.y, xv.z, xv.w}, gw[4] = {gv.x, gv.y, gv.z, gv.w}, mw[4] = {mv.x, mv.y, mv.z, mv.w};
  uint32_t o[4], om[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int c0 = gidx * 8 + 2 * e, c1 = c0 + 1;
    const float g0 = (__uint_as_float(mw[e] << 16) > 0.f) ? __uint_as_float(gw[e] << 16) : 0.f;
    const float g1 = (__uint_as_float(mw[e] & 0xFFFF0000u) > 0.f) ? __uint_as_float(gw[e] & 0xFFFF0000u) : 0.f;
    const float is0 = mean_invstd[C + c0], is1 = mean_invstd[C + c1];
    const float x0 = (__uint_as_float(xw[e] << 16) - mean_invstd[c0]) * is0;
    const float x1 = (__uint_as_float(xw[e] & 0xFFFF0000u) - mean_invstd[c1]) * is1;
    const float d0 = gamma[c0] * is0 * (g0 - coef[c0] - x0 * coef[C + c0]);
    const float d1 = gamma[c1] * is1 * (g1 - coef[c1] - x1 * coef[C + c1]);
    o[e] = pack_bf16x2(d0, d1);
    om[e] = pack_bf16x2(g0, g1);
  }
  *reinterpret_cast<uint4*>(draw + r * C + gidx * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  if (gm_out) *reinterpret_cast<uint4*>(gm_out + r * C + gidx * 8) = make_uint4(om[0], om[1], om[2], om[3]);
}

// ---- convolution gradients ---------------------------------------------------------------------------------------
// dgrad weights: Wd[i][r][s][o] = W[o][k-1-r][k-1-s][i]  (W packed [O][R][S][I] bf16)
__global__ void flip_weights_kernel(const __nv_bfloat16* __restrict__ w, int O, int I, int k, __nv_bfloat16* __restrict__ wd) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)O * I * k * k) return;
  const int o = (int)(idx % O);
  const int s = (int)((idx / O) % k);
  const int r = (int)((idx / ((int64_t)O * k)) % k);
  const int i = (int)(idx / ((int64_t)O * k * k));
  wd[idx] = w[(((int64_t)o * k + (k - 1 - r)) * k + (k - 1 - s)) * I + i];
}
// zero-insertion for stride-2 layers: up[f][2*oh][2*ow][c] = g[f][oh][ow][c], everything else 0 (Hup = 2*Hout - 1)
__global__ void zero_insert_kernel(const __nv_bfloat16* __restrict__ g, int64_t n, int Hout, int C, __nv_bfloat16* __restrict__ up) {
  const int Hup = 2 * Hout - 1;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int groups = C / 8;
  if (idx >= n * Hup * Hup * groups) return;
  const int gq = (int)(idx % groups);
  const int64_t pix = idx / groups;
  const int x = (int)(pix % Hup), y = (int)((pix / Hup) % Hup);
  const int64_t f = pix / ((int64_t)Hup * Hup);
  uint4 v = make_uint4(0u, 0u, 0u, 0u);
  if (!(x & 1) && !(y & 1)) v = *reinterpret_cast<const uint4*>(g + ((f * Hout + y / 2) * Hout + x / 2) * C + gq * 8);
  *reinterpret_cast<uint4*>(up + pix * C + gq * 8) = v;
}
// bf16 [P][C] -> [C][Pp] (zero fill for p >= P)
__global__ void transpose_pc_kernel(const __nv_bfloat16* __restrict__ in, int64_t P, int C, int64_t Pp,
                                    __nv_bfloat16* __restrict__ out) {
  __shared__ __nv_bfloat16 tile[32][33];
  const int64_t p0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int64_t p = p0 + i;
    tile[i][threadIdx.x] = (p < P) ? in[p * C + c0 + threadIdx.x] : __float2bfloat16_rn(0.f);
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int64_t p = p0 + threadIdx.x;
    if (p < Pp) out[(int64_t)(c0 + i) * Pp + p] = tile[threadIdx.x][i];
  }
}
// transposed im2col: col[(tap*Cin + c)][p] = X[f][oh*stride + r - pad][ow*stride + s - pad][c] (0 outside the frame or for
// p >= P), p = (f*OH + oh)*OW + ow over the frames of the chunk.  One block moves a 64-pixel x 64-channel tile of one tap
// through shared memory: 16-byte loads along the channels of a pixel (whole 128-byte pixel rows per 8 lanes), 16-byte
// stores along the pixels of a channel (whole 128-byte rows of the K-major GEMM operand per 8 lanes).  Tile rows are
// pitched 33 words so both phases are (nearly) bank-conflict free.  (The first version moved 32x32 tiles element by
// element: 33.6 ms of an 82 ms video-net training step, 8x off the HBM time of the 12 GB it writes.)
__global__ void __launch_bounds__(256) im2col_t_kernel(const __nv_bfloat16* __restrict__ x, int H, int Cin, int OH, int k,
                                                       int stride, int pad, int64_t P, int64_t Pp,
                                                       __nv_bfloat16* __restrict__ col) {
  __shared__ uint32_t tile[64 * 33];
  const int64_t p0 = (int64_t)blockIdx.x * 64;
  const int c0 = blockIdx.y * 64;
  const int tap = blockIdx.z;
  const int r = tap / k, s = tap % k;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int i = threadIdx.x + q * 256;
    const int pix = i >> 3, ch = i & 7;
    const int64_t p = p0 + pix;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (p < P) {
      const int ow = (int)(p % OH), oh = (int)((p / OH) % OH);
      const int64_t f = p / ((int64_t)OH * OH);
      const int ih = oh * stride + r - pad, iw = ow * stride + s - pad;
      if (ih >= 0 && ih < H && iw >= 0 && iw < H)
        v = *reinterpret_cast<const uint4*>(x + ((f * H + ih) * H + iw) * Cin + c0 + ch * 8);
    }
    uint32_t* dst = tile + pix * 33 + ch * 4;
    dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
  }
  __syncthreads();
  const uint16_t* t16 = reinterpret_cast<const uint16_t*>(tile);
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int i = threadIdx.x + q * 256;
    const int c = i >> 3, pc = i & 7;
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t lo = t16[(pc * 8 + 2 * j) * 66 + c], hi = t16[(pc * 8 + 2 * j + 1) * 66 + c];
      w[j] = lo | (hi << 16);
    }
    *reinterpret_cast<uint4*>(col + ((int64_t)tap * Cin + c0 + c) * Pp + p0 + pc * 8) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}
// acc[j] (+)= sum_s part[s][j]
__global__ void sum_partials_kernel(const float* __restrict__ part, int nparts, int64_t elems, int accumulate,
                                    float* __restrict__ acc) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= elems) return;
  float t = accumulate ? acc[j] : 0.f;
  for (int s = 0; s < nparts; ++s) t += part[(int64_t)s * elems + j];
  acc[j] = t;
}
// [O][tap][I] fp32 -> PyTorch layout [O][I][k][k]
__global__ void wgrad_layout_kernel(const float* __restrict__ acc, int O, int I, int k, float* __restrict__ dw) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)O * I * k * k) return;
  const int tap = (int)(idx % (k * k));
  const int i = (int)((idx / (k * k)) % I);
  const int o = (int)(idx / ((int64_t)k * k * I));
  dw[idx] = acc[((int64_t)o * k * k + tap) * I + i];
}
// conv1 weight gradient: dW0[o][tap] = sum_{f,p} dRaw0[f][p][o] * frame[f][2*oh + r - 3][2*ow + s - 3]; thread = (o, tap
// quarter); block loops over frames, one fp32 atomic per output and block at the end
__global__ void __launch_bounds__(256) conv1_wgrad_kernel(const float* __restrict__ frames, int64_t n,
                                                          const __nv_bfloat16* __restrict__ draw, float* __restrict__ dw0) {
  __shared__ float img[73 * 73];
  const int o = threadIdx.x & 63, q = threadIdx.x >> 6;  // taps q, q+4, q+8, ...
  float acc[13];
  int off[13];   // image offset of tap q + 4j relative to the window origin (hoisted: q is a run-time value)
#pragma unroll
  for (int j = 0; j < 13; ++j) {
    acc[j] = 0.f;
    const int tap = q + 4 * j;
    off[j] = tap < 49 ? (tap / 7) * 73 + tap % 7 : 0;
  }
  for (int64_t f = blockIdx.x; f < n; f += gridDim.x) {
    __syncthreads();
    for (int i = threadIdx.x; i < 73 * 73; i += 256) {
      const int y = i / 73 - 3, x = i % 73 - 3;
      img[i] = (y >= 0 && y < 67 && x >= 0 && x < 67) ? frames[f * 67 * 67 + y * 67 + x] : 0.f;
    }
    __syncthreads();
    const __nv_bfloat16* d = draw + f * 1156 * 64 + o;
    for (int p = 0; p < 1156; ++p) {
      const float dv = __bfloat162float(d[(int64_t)p * 64]);
      const int oh = p / 34, ow = p % 34;
      const float* base = img + (2 * oh) * 73 + 2 * ow;
#pragma unroll
      for (int j = 0; j < 13; ++j) acc[j] = fmaf(dv, base[off[j]], acc[j]);   // tap >= 49: accumulates garbage, never stored
    }
  }
#pragma unroll
  for (int j = 0; j < 13; ++j) {
    const int tap = q + 4 * j;
    if (tap < 49) atomicAdd(dw0 + o * 49 + tap, acc[j]);
  }
}
// [64][49] -> [64][3][7][7]: the three input channels see the same image, so their gradients are identical
__global__ void conv1_expand_kernel(const float* __restrict__ dw0, float* __restrict__ dw) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * 3 * 49) return;
  const int o = idx / (3 * 49), k = idx % 49;
  dw[idx] = dw0[o * 49 + k];
}

struct BwdCtx {
  avvad_resnet18* h;
  int64_t n;
  float bn_eps;
  cudaStream_t st;
  double* sums;    // [2*512]
  float* coef;     // [2*512]
  __nv_bfloat16* wd;       // flipped weights, largest layer
  __nv_bfloat16* drawT;    // [Cout][Pp]
  __nv_bfloat16* colT;     // [taps*Cin][Pp]
  float* part;             // split-K partials
  float* acc;              // [Cout][taps][Cin]
  int64_t chunk_pixels;    // pixels per wgrad chunk
};

// workspace sizing shared by the query and the implementation
constexpr int64_t kWgradPixels = 1 << 19;  // pixels per weight-gradient chunk (K of the GEMM): sizes the workspace
// AVVAD_WGRAD_PIXELS (<= 2^19) shrinks the chunk: the tests use it to drive the multi-chunk accumulation on small inputs
static int64_t wgrad_pixels() {
  static int64_t v = [] {
    const char* e = getenv("AVVAD_WGRAD_PIXELS");
    const int64_t x = e ? atoll(e) : kWgradPixels;
    return (x >= 64 && x <= kWgradPixels) ? x / 64 * 64 : kWgradPixels;
  }();
  return v;
}
static size_t wgrad_part_bytes() { return (size_t)64 * 1024 * 1024; }

static int bn_backward(const BwdCtx& c, int layer, const __nv_bfloat16* raw, const __nv_bfloat16* g,
                       const __nv_bfloat16* mask, const float* stats, int64_t M, int C, __nv_bfloat16* draw,
                       __nv_bfloat16* gm_out, float* dgamma, float* dbeta) {
  AVVAD_CUDA(cudaMemsetAsync(c.sums, 0, sizeof(double) * 2 * C, c.st));
  const int lanes = 256 / (C / 8);
  bn_bwd_reduce_kernel<<<(unsigned)ceil_div(M, kStatRows), 256, (size_t)lanes * 2 * C * sizeof(float), c.st>>>(
      raw, g, mask, M, C, stats, c.sums);
  AVVAD_LAUNCHED();
  bn_bwd_finalize_kernel<<<(unsigned)ceil_div(C, 128), 128, 0, c.st>>>(c.sums, M, C, dgamma, dbeta, c.coef);
  AVVAD_LAUNCHED();
  bn_bwd_apply_kernel<<<(unsigned)ceil_div(M * (C / 8), 256), 256, 0, c.st>>>(raw, g, mask, M, C, stats,
                                                                            c.h->gamma[layer], c.coef, draw, gm_out);
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}

// data gradient of conv `layer`: gin (n, hin, hin, cin) = conv_transpose(draw (n, hout, hout, cout)); `up` is scratch for
// the zero-inserted gradient of stride-2 layers; `residual` (optional, gin's shape) is added in the epilogue
static int conv_dgrad(const BwdCtx& c, int layer, const __nv_bfloat16* draw, __nv_bfloat16* up,
                      const __nv_bfloat16* residual, __nv_bfloat16* gin) {
  const ConvSpec& s = kSpecs[layer];
  const int64_t wn = (int64_t)s.cout * s.cin * s.k * s.k;
  flip_weights_kernel<<<(unsigned)ceil_div(wn, 256), 256, 0, c.st>>>(c.h->wraw[layer], s.cout, s.cin, s.k, c.wd);
  AVVAD_LAUNCHED();
  const __nv_bfloat16* src = draw;
  if (s.stride == 2) {
    const int64_t total = c.n * s.hin * s.hin * (s.cout / 8);
    zero_insert_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, c.st>>>(draw, c.n, s.hout, s.cout, up);
    AVVAD_LAUNCHED();
    src = up;
  }
  return avvad_conv2d_nhwc_bf16(src, c.wd, nullptr, residual, gin, c.n, s.hin, s.hin, s.cout, s.cin, s.k, s.k, 1,
                                s.k - 1 - s.pad, 0, c.st);
}

// weight gradient of conv `layer` from its input x (n, hin, hin, cin) and dRaw (n, hout, hout, cout) -> dw (torch layout)
static int conv_wgrad(const BwdCtx& c, int layer, const __nv_bfloat16* x, const __nv_bfloat16* draw, float* dw) {
  const ConvSpec& s = kSpecs[layer];
  const int taps = s.k * s.k;
  const int N = taps * s.cin, M = s.cout;
  const int64_t pix_per_frame = (int64_t)s.hout * s.hout;
  int64_t fc = c.chunk_pixels / pix_per_frame;
  if (fc < 1) fc = 1;
  // 64-column tiles (the split-K configuration the LSTM BPTT exercises) unless the GEMM is wide and tall enough for
  // 256-column tiles
  const int bn = (N % 256 == 0 && M >= 128) ? 256 : 64;
  const int tiles = (int)(ceil_div(M, 128) * ceil_div(N, bn));
  bool first = true;
  for (int64_t f0 = 0; f0 < c.n; f0 += fc) {
    const int64_t nf = (c.n - f0 < fc) ? c.n - f0 : fc;
    const int64_t P = nf * pix_per_frame, Pp = (P + 63) / 64 * 64;
    const __nv_bfloat16* dr = draw + f0 * pix_per_frame * s.cout;
    const __nv_bfloat16* xi = x + f0 * (int64_t)s.hin * s.hin * s.cin;
    dim3 g1((unsigned)ceil_div(Pp, 32), (unsigned)(s.cout / 32));
    transpose_pc_kernel<<<g1, dim3(32, 8), 0, c.st>>>(dr, P, s.cout, Pp, c.drawT);
    AVVAD_LAUNCHED();
    dim3 g2((unsigned)(Pp / 64), (unsigned)(s.cin / 64), (unsigned)taps);
    im2col_t_kernel<<<g2, 256, 0, c.st>>>(xi, s.hin, s.cin, s.hout, s.k, s.stride, s.pad, P, Pp, c.colT);
    AVVAD_LAUNCHED();
    // split K = pixels over the SMs
    const int64_t kblocks = Pp / 64;
    int ksplit = (int)std::min<int64_t>(std::max<int64_t>(1, 296 / tiles), kblocks);
    const size_t per = (size_t)M * N * sizeof(float);
    if ((size_t)ksplit * per > wgrad_part_bytes()) ksplit = (int)std::max<size_t>(1, wgrad_part_bytes() / per);
    {  // every split must own at least one K block (an empty split would leave its partial unwritten)
      const int64_t per_split = ceil_div(kblocks, ksplit);
      ksplit = (int)ceil_div(kblocks, per_split);
    }
    tc::EpiParams ep{};
    ep.C = c.part;
    ep.ldc = N;
    int rc = tc::launch_tma_gemm(c.drawT, Pp, c.colT, Pp, M, N, (int)Pp, ep, tc::EPI_F32, bn, c.st, ksplit, (int64_t)M * N);
    if (rc) return rc;
    const int64_t elems = (int64_t)M * N;
    sum_partials_kernel<<<(unsigned)ceil_div(elems, 256), 256, 0, c.st>>>(c.part, ksplit, elems, first ? 0 : 1, c.acc);
    AVVAD_LAUNCHED();
    first = false;
  }
  const int64_t total = (int64_t)s.cout * s.cin * taps;
  wgrad_layout_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, c.st>>>(c.acc, s.cout, s.cin, s.k, dw);
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}

}  // namespace bwd
}  // namespace avvad

using namespace avvad;

extern "C" size_t avvad_resnet18_tape_bytes(int64_t n_frames) {
  if (n_frames <= 0) return 0;
  return bwd::make_tape(nullptr, n_frames).total;
}

// Byte offsets of the tape's tensors (test / inspection hook): offsets[0..37] = raw0, act0, pool, raw of conv 1..19,
// then (y1, out) of blocks 0..7 -- all NHWC bf16 --, offsets[38] = per-layer statistics, float [20][1024] (mean | invstd).
extern "C" int avvad_resnet18_tape_layout(int64_t n_frames, int64_t* offsets, int count) {
  AVVAD_CHECK_ARG(n_frames > 0 && offsets && count == bwd::kNumTensors + 1, "offsets must hold 39 entries");
  const bwd::Tape tp = bwd::make_tape(nullptr, n_frames);
  for (int i = 0; i < bwd::kNumTensors; ++i) offsets[i] = (int64_t)tp.off[i];
  offsets[bwd::kNumTensors] = (int64_t)tp.stats_off;
  return AVVAD_OK;
}

extern "C" size_t avvad_resnet18_tape_workspace_bytes(int64_t n_frames) {
  if (n_frames <= 0) return 0;
  // one activation-sized scratch (the downsample branch's BN output) + statistics
  return align_up((size_t)n_frames * kActBytesPerFrame, 1024) + 64 * 1024;
}

// Training-mode forward that keeps everything avvad_resnet18_backward needs in `tape`.
extern "C" int avvad_resnet18_forward_tape(avvad_resnet18* h, const float* frames, int64_t n_frames, void* workspace,
                                           size_t workspace_bytes, void* tape, size_t tape_bytes, float bn_eps,
                                           float momentum, float* const* running_mean, float* const* running_var,
                                           float* feat, void* feat_bf16, int64_t ld_bf16, int64_t col_off, void* stream) {
  AVVAD_CHECK_ARG(h && frames && workspace && tape && n_frames > 0 && (feat || feat_bf16), "bad argument");
  for (int i = 0; i < 20; ++i)
    if (!h->set_train[i]) {
      set_error("resnet18: training weights of conv layer " + std::to_string(i) + " not loaded");
      return AVVAD_ERR_STATE;
    }
  if (workspace_bytes < avvad_resnet18_tape_workspace_bytes(n_frames) || tape_bytes < avvad_resnet18_tape_bytes(n_frames)) {
    set_error("resnet18: tape / workspace too small");
    return AVVAD_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n = n_frames;
  bwd::Tape tp = bwd::make_tape(tape, n);
  const size_t act = align_up((size_t)n * kActBytesPerFrame, 1024);
  __nv_bfloat16* tmp = reinterpret_cast<__nv_bfloat16*>(workspace);
  double* stats = reinterpret_cast<double*>((uint8_t*)workspace + act);
  float* scale_shift = reinterpret_cast<float*>((uint8_t*)workspace + act + 16 * 1024);
  TrainCtx c{h, n, stats, scale_shift, bn_eps, momentum, running_mean, running_var, st};

  auto bn = [&](int layer, const __nv_bfloat16* raw, int64_t M, int C, const __nv_bfloat16* res, int relu,
                __nv_bfloat16* out) -> int { return bn_train(c, layer, raw, M, C, res, relu, out, tp.stats(layer)); };

  // stem, un-fused: conv1 -> BN(batch statistics) -> ReLU -> max-pool
  bwd::conv1_direct_kernel<<<(unsigned)std::min<int64_t>(n, 148 * 8), 256, 0, st>>>(frames, n, h->w1raw32, tp.raw(0));
  AVVAD_LAUNCHED();
  int rc = bn(0, tp.raw(0), n * 1156, 64, nullptr, 1, tp.t(1));
  if (rc) return rc;
  {
    const int64_t total = n * 17 * 17 * (64 / 8);
    bwd::maxpool_fwd_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(tp.t(1), n, 34, 17, 64, tp.t(2));
    AVVAD_LAUNCHED();
  }
  const __nv_bfloat16* x = tp.t(2);
  for (int bk = 0; bk < 8; ++bk) {
    const bwd::BlockDef& b = bwd::kBlocks[bk];
    const ConvSpec& sa = kSpecs[b.la];
    const int64_t Mo = n * sa.hout * sa.hout;
    rc = conv_raw(c, b.la, x, tp.raw(b.la));
    if (rc) return rc;
    rc = bn(b.la, tp.raw(b.la), Mo, sa.cout, nullptr, 1, tp.y1(bk));
    if (rc) return rc;
    const __nv_bfloat16* res = x;
    if (b.lds >= 0) {
      rc = conv_raw(c, b.lds, x, tp.raw(b.lds));
      if (rc) return rc;
      rc = bn(b.lds, tp.raw(b.lds), Mo, sa.cout, nullptr, 0, tmp);
      if (rc) return rc;
      res = tmp;
    }
    rc = conv_raw(c, b.lb, tp.y1(bk), tp.raw(b.lb));
    if (rc) return rc;
    rc = bn(b.lb, tp.raw(b.lb), Mo, sa.cout, res, 1, tp.out(bk));
    if (rc) return rc;
    x = tp.out(bk);
  }
  const int64_t total = n * (512 / 8);
  avgpool_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(x, n, 9, 512, feat, (__nv_bfloat16*)feat_bf16, ld_bf16,
                                                                 col_off);
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}

extern "C" size_t avvad_resnet18_backward_workspace_bytes(int64_t n_frames) {
  if (n_frames <= 0) return 0;
  const size_t act = align_up((size_t)n_frames * kActBytesPerFrame, 1024);        // (n,17,17,64) bf16
  const size_t big = align_up((size_t)n_frames * 34 * 34 * 64 * 2, 1024);         // stem resolution
  size_t s = 6 * act + 2 * act /* zero-inserted (n,17,17,128) */ + 2 * big;
  s += align_up((size_t)512 * 512 * 9 * 2, 1024);                                 // flipped weights
  s += align_up((size_t)512 * (bwd::kWgradPixels + 64) * 2, 1024);                // dRaw^T
  s += align_up((size_t)9 * 64 * (bwd::kWgradPixels + 64) * 2, 1024) * 1;         // im2col^T: taps*Cin*pixels is constant
  s += bwd::wgrad_part_bytes() + align_up((size_t)512 * 4608 * 4, 1024);
  return s + 64 * 1024;
}

// dfeat f32 [n][512] -> dW[l] (torch layout [O][I][k][k]; conv1: [64][3][7][7]), dgamma[l], dbeta[l] for the 20 layers.
extern "C" int avvad_resnet18_backward(avvad_resnet18* h, const float* frames, int64_t n_frames, void* tape,
                                       const float* dfeat, void* workspace, size_t workspace_bytes, float bn_eps,
                                       float* const* dW, float* const* dgamma, float* const* dbeta, void* stream) {
  AVVAD_CHECK_ARG(h && frames && tape && dfeat && workspace && dW && dgamma && dbeta && n_frames > 0, "bad argument");
  if (workspace_bytes < avvad_resnet18_backward_workspace_bytes(n_frames)) {
    set_error("resnet18 backward: workspace too small");
    return AVVAD_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n = n_frames;
  bwd::Tape tp = bwd::make_tape(tape, n);
  const size_t act = align_up((size_t)n * kActBytesPerFrame, 1024);
  const size_t big = align_up((size_t)n * 34 * 34 * 64 * 2, 1024);
  uint8_t* p = (uint8_t*)workspace;
  auto take = [&](size_t bytes) { void* q = p; p += align_up(bytes, 1024); return q; };
  __nv_bfloat16* G[2] = {(__nv_bfloat16*)take(act), (__nv_bfloat16*)take(act)};  // upstream gradient, ping-pong
  __nv_bfloat16* draw_b = (__nv_bfloat16*)take(act);
  __nv_bfloat16* gm = (__nv_bfloat16*)take(act);
  __nv_bfloat16* gy1 = (__nv_bfloat16*)take(act);
  __nv_bfloat16* draw_a = (__nv_bfloat16*)take(act);
  __nv_bfloat16* up = (__nv_bfloat16*)take(2 * act);
  __nv_bfloat16* gbig0 = (__nv_bfloat16*)take(big);
  __nv_bfloat16* gbig1 = (__nv_bfloat16*)take(big);
  bwd::BwdCtx c{};
  c.h = h; c.n = n; c.bn_eps = bn_eps; c.st = st;
  c.wd = (__nv_bfloat16*)take((size_t)512 * 512 * 9 * 2);
  c.drawT = (__nv_bfloat16*)take((size_t)512 * (bwd::kWgradPixels + 64) * 2);
  c.colT = (__nv_bfloat16*)take((size_t)9 * 64 * (bwd::kWgradPixels + 64) * 2);
  c.part = (float*)take(bwd::wgrad_part_bytes());
  c.acc = (float*)take((size_t)512 * 4608 * 4);
  c.sums = (double*)take(16 * 1024);
  c.coef = (float*)take(16 * 1024);

  // gradient w.r.t. the last block's output
  int cur = 0;
  __nv_bfloat16* g_out = G[cur];
  {
    const int64_t total = n * 9 * (512 / 8);
    bwd::avgpool_bwd_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(dfeat, n, 9, 512, g_out);
    AVVAD_LAUNCHED();
  }
  for (int bk = 7; bk >= 0; --bk) {
    const bwd::BlockDef& b = bwd::kBlocks[bk];
    const ConvSpec& sa = kSpecs[b.la];
    const ConvSpec& sb = kSpecs[b.lb];
    const int64_t Mo = n * sb.hout * sb.hout;
    const __nv_bfloat16* x = (bk == 0) ? tp.t(2) : tp.out(bk - 1);
    // pixels per wgrad chunk such that taps*Cin*pixels stays within the im2col^T buffer (9*64*kWgradPixels elements)
    auto chunk_for = [&](const ConvSpec& s) {
      const int64_t cap = (int64_t)9 * 64 * bwd::kWgradPixels / ((int64_t)s.k * s.k * s.cin);
      return std::min<int64_t>(bwd::wgrad_pixels(), cap / 64 * 64);
    };
    __nv_bfloat16* gx = G[cur ^ 1];
    // out = relu(bn_b(conv_b(y1)) + shortcut): mask with out, BatchNorm backward of layer lb
    int rc = bwd::bn_backward(c, b.lb, tp.raw(b.lb), g_out, tp.out(bk), tp.stats(b.lb), Mo, sb.cout, draw_b, gm,
                              dgamma[b.lb], dbeta[b.lb]);
    if (rc) return rc;
    c.chunk_pixels = chunk_for(sb);
    rc = bwd::conv_wgrad(c, b.lb, tp.y1(bk), draw_b, dW[b.lb]);
    if (rc) return rc;
    rc = bwd::conv_dgrad(c, b.lb, draw_b, up, nullptr, gy1);
    if (rc) return rc;
    // y1 = relu(bn_a(conv_a(x)))
    rc = bwd::bn_backward(c, b.la, tp.raw(b.la), gy1, tp.y1(bk), tp.stats(b.la), Mo, sa.cout, draw_a, nullptr,
                          dgamma[b.la], dbeta[b.la]);
    if (rc) return rc;
    c.chunk_pixels = chunk_for(sa);
    rc = bwd::conv_wgrad(c, b.la, x, draw_a, dW[b.la]);
    if (rc) return rc;
    const __nv_bfloat16* shortcut_grad = gm;  // identity shortcut: the masked gradient itself
    if (b.lds >= 0) {
      const ConvSpec& sd = kSpecs[b.lds];
      __nv_bfloat16* draw_d = draw_b;  // draw_b is dead by now
      rc = bwd::bn_backward(c, b.lds, tp.raw(b.lds), gm, nullptr, tp.stats(b.lds), Mo, sd.cout, draw_d, nullptr,
                            dgamma[b.lds], dbeta[b.lds]);
      if (rc) return rc;
      c.chunk_pixels = chunk_for(sd);
      rc = bwd::conv_wgrad(c, b.lds, x, draw_d, dW[b.lds]);
      if (rc) return rc;
      rc = bwd::conv_dgrad(c, b.lds, draw_d, up, nullptr, gy1);  // gy1 is free: (n, hin, hin, cin)
      if (rc) return rc;
      shortcut_grad = gy1;
    }
    rc = bwd::conv_dgrad(c, b.la, draw_a, up, shortcut_grad, gx);
    if (rc) return rc;
    cur ^= 1;  // gx becomes the next block's upstream gradient
    g_out = G[cur];
  }
  // stem: max-pool backward -> ReLU mask + BatchNorm backward -> conv1 weight gradient
  {
    uint8_t* which = reinterpret_cast<uint8_t*>(gbig1);   // (n,17,17,64) bytes; gbig1 is free until the BatchNorm backward
    const int64_t total_o = n * 17 * 17 * (64 / 8);
    bwd::maxpool_argmax_kernel<<<(unsigned)ceil_div(total_o, 256), 256, 0, st>>>(tp.t(1), n, 34, 17, 64, which);
    AVVAD_LAUNCHED();
    const int64_t total = n * 34 * 34 * (64 / 8);
    bwd::maxpool_bwd_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(which, g_out, n, 34, 17, 64, gbig0);
    AVVAD_LAUNCHED();
    int rc = bwd::bn_backward(c, 0, tp.raw(0), gbig0, tp.t(1), tp.stats(0), n * 1156, 64, gbig1, nullptr, dgamma[0],
                              dbeta[0]);
    if (rc) return rc;
    AVVAD_CUDA(cudaMemsetAsync(c.acc, 0, 64 * 49 * sizeof(float), st));
    bwd::conv1_wgrad_kernel<<<(unsigned)std::min<int64_t>(n, 148 * 4), 256, 0, st>>>(frames, n, gbig1, c.acc);
    AVVAD_LAUNCHED();
    bwd::conv1_expand_kernel<<<(unsigned)ceil_div(64 * 3 * 49, 256), 256, 0, st>>>(c.acc, dW[0]);
    AVVAD_LAUNCHED();
  }
  return AVVAD_OK;
}
