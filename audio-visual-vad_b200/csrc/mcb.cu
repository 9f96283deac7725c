// Multimodal Compact Bilinear fusion: count sketches -> circular convolution (in-SMEM FFT) -> signed sqrt
// -> whole-tensor L2 normalisation -> BatchNorm1d (eval) -> bf16 LSTM operand.
//
// Reference semantics: packages/models/compact_bilinear_pooling.py:7-27,140-173 and
// packages/models/AV_Net.py:111-121.  The two real sketches are packed into one complex 1024-point FFT
// (Z = px + i*py); X and Y are separated by Hermitian symmetry, multiplied, and transformed back with a second
// forward FFT of the conjugate.  The scatter-add of the reference is replaced by a deterministic inverse
// (CSR) gather that sums colliding inputs in index order, which is the order the reference's CPU
// scatter_add_ visits them.
#include <vector>

#include "fft.cuh"
#include "fft_reg.cuh"

namespace avvad {
namespace tc {
int prof_begin(cudaStream_t st, void** tok);
void prof_end(cudaStream_t st, void* tok, int cat, double flops);
}  // namespace tc
}  // namespace avvad

namespace avvad {

constexpr int kMcbOut = 1024;
constexpr int kNA = 513, kNV = 512;

struct McbTables {
  const int32_t* off1;  // [1025]
  const int32_t* idx1;  // [513]
  const float* s1;      // [513]
  const int32_t* off2;  // [1025]
  const int32_t* idx2;  // [512]
  const float* s2;      // [512]
};

__global__ void __launch_bounds__(kFftThreads)
mcb_row_kernel(const float* __restrict__ audio, const float* __restrict__ video, McbTables tb,
               const float2* __restrict__ tw_g, float eps, float* __restrict__ y_out, float* __restrict__ rowsq,
               const int32_t* __restrict__ lengths = nullptr, int t_max = 0) {
  __shared__ float2 sa[kFftN];
  __shared__ float2 sb[kFftN];
  __shared__ float2 stw[kFftTwStage];
  __shared__ float xa[kNA];
  __shared__ float xv[kNV];
  __shared__ float red[8];

  const int tid = threadIdx.x;
  const int64_t row = blockIdx.x;
  // grouped calls (avvad_mcb_forward_grouped): rows behind an utterance's length belong to no call of the reference
  if (lengths && (int)(row % t_max) >= lengths[row / t_max]) return;
#pragma unroll
  for (int q = 0; q < kFftTwStage / kFftThreads; ++q)
    stw[tid + q * kFftThreads] = tw_g[kFftTwHann + tid + q * kFftThreads];
  for (int i = tid; i < kNA; i += kFftThreads) xa[i] = audio[row * kNA + i];
  for (int i = tid; i < kNV; i += kFftThreads) xv[i] = video[row * kNV + i];
  __syncthreads();

  // count sketches: out[j] = sum_{i : h_i = j} s_i * x_i
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int j = tid + q * kFftThreads;
    float px = 0.f, py = 0.f;
    for (int e = tb.off1[j]; e < tb.off1[j + 1]; ++e) {
      const int i = tb.idx1[e];
      px += xa[i] * tb.s1[i];
    }
    for (int e = tb.off2[j]; e < tb.off2[j + 1]; ++e) {
      const int i = tb.idx2[e];
      py += xv[i] * tb.s2[i];
    }
    sa[j] = make_float2(px, py);
  }
  __syncthreads();
  float2* z1 = fft1024_smem(sa, sb, stw, tid);  // result buffer (the other one is free scratch)
  float2* z2 = (z1 == sa) ? sb : sa;

  // P[k] = X[k]*Y[k]; store conj(P) so that a second forward FFT yields N * ifft(P)
  for (int k = tid; k <= 512; k += kFftThreads) {
    if (k == 0 || k == 512) {
      const float2 z = z1[k];
      z1[k] = make_float2(z.x * z.y, 0.f);
    } else {
      const float2 zk = z1[k];
      const float2 zn = z1[kFftN - k];
      const float2 X = make_float2(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));
      const float2 Y = make_float2(0.5f * (zk.y + zn.y), 0.5f * (zn.x - zk.x));
      const float2 P = cmul(X, Y);
      z1[k] = make_float2(P.x, -P.y);        // conj(P[k])
      z1[kFftN - k] = make_float2(P.x, P.y);  // conj(P[N-k]) = P[k]
    }
  }
  __syncthreads();
  const float2* res = fft1024_smem(z1, z2, stw, tid);

  float ss = 0.f;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int j = tid + q * kFftThreads;
    const float p = res[j].x * (1.0f / kFftN);
    // torch.sign(p) * sqrt(|p| + eps)   (sign(0) = 0)
    const float r = sqrtf(fabsf(p) + eps);
    const float y = (p > 0.f) ? r : ((p < 0.f) ? -r : 0.f);
    y_out[row * kMcbOut + j] = y;
    ss += y * y;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((tid & 31) == 0) red[tid >> 5] = ss;
  __syncthreads();
  if (tid == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w];
    rowsq[row] = t;
  }
}

// ---- the same row function on the register FFT (fft_reg.cuh) ----------------------------------------------------
// Persistent CTAs of four 64-thread groups; a group owns one row at a time and never synchronises with the other
// groups (named barriers).  Staged ONCE per CTA: the two twiddle tables and the CSR count-sketch tables (offsets as
// u16, (input index, sign) pairs), which mcb_row_kernel re-read from L2 for every row (~20 KB per row of 4 KB input).
// A thread computes its 16 sketch outputs j = t + 64 m straight into the registers the first transform starts from
// (same summation order as mcb_row_kernel: ascending input index inside a bucket), the spectrum product needs one
// exchange through the group's buffer (partner of k is N - k: thread 64 - t), and the second transform leaves the
// thread with the 16 outputs it writes.  Shared-memory traffic per row: ~107 KB instead of ~225 KB.
constexpr int kRowGroups = 4;
constexpr int kRowXin = 1040;  // 513 + 512 inputs of a row, padded
constexpr int kMaxRounds = 32;
// Count sketch as conflict-free scatter ROUNDS: round r holds the inputs that are the r-th member (ascending input
// index) of their bucket, so inside a round no two inputs share a bucket and out[h] += s*x needs no atomics; a group
// barrier separates the rounds.  Every bucket therefore accumulates its members in ascending input order starting from
// zero -- exactly the sums of mcb_row_kernel's CSR gather, bit for bit -- but the work is one straight pass over the
// 513 + 512 inputs (8 per thread) instead of 2 x 1024 data-dependent gather loops (ncu: the gather form was 43 % of
// the kernel's shared-memory wavefronts and put branch_resolving among the top stalls).
struct McbRounds {
  const int32_t* ent1;   // [513] input index | bucket << 16, sorted by (round, input index)
  const int32_t* ent2;   // [512]
  const int32_t* roff1;  // [kMaxRounds + 1] first entry of every round
  const int32_t* roff2;
  int n_rounds;          // max over both sketches
};
struct RowSmem {
  float2 buf[kRowGroups][kRfBufEntries];
  float xin[kRowGroups][kRowXin];
  float2 twB[kFftTwB];
  float2 twC[kFftTwC];
  int2 ent1[kNA + 1];  // (input index | physical float offset of the bucket << 16, sign as float bits), round order
  int2 ent2[kNV];
  int roff1[kMaxRounds + 1];
  int roff2[kMaxRounds + 1];
  float red[kRowGroups];
};

__global__ void __launch_bounds__(kRowGroups * kRfThreads, 3)
mcb_row_reg_kernel(const float* __restrict__ audio, const float* __restrict__ video, McbTables tb, McbRounds rd,
                   const float2* __restrict__ tw_g, float eps, float* __restrict__ y_out, float* __restrict__ rowsq,
                   int64_t rows, const int32_t* __restrict__ lengths, int t_max) {
  extern __shared__ __align__(16) uint8_t row_smem_raw[];
  RowSmem& sm = *reinterpret_cast<RowSmem*>(row_smem_raw);
  const int tid = threadIdx.x;
  const int g = tid >> 6, t = tid & 63;
  const int bar_id = 1 + g;

  for (int i = tid; i < kFftTwB; i += blockDim.x) sm.twB[i] = tw_g[kFftTwHann + kFftTwStage + i];
  for (int i = tid; i < kFftTwC; i += blockDim.x) sm.twC[i] = tw_g[kFftTwHann + fft_tw_off(4) + i];
  for (int i = tid; i <= kMaxRounds; i += blockDim.x) {
    sm.roff1[i] = rd.roff1[i];
    sm.roff2[i] = rd.roff2[i];
  }
  // bucket j of the sketch pair lives at float offset 2 * phys(j) (+1 for the video sketch) of the exchange buffer
  for (int e = tid; e < kNA; e += blockDim.x) {
    const int p = rd.ent1[e], i = p & 0xFFFF, j = p >> 16;
    sm.ent1[e] = make_int2(i | ((2 * ((j >> 4) * kRfPitch + (j & 15))) << 16), __float_as_int(tb.s1[i]));
  }
  for (int e = tid; e < kNV; e += blockDim.x) {
    const int p = rd.ent2[e], i = p & 0xFFFF, j = p >> 16;
    sm.ent2[e] = make_int2(i | ((2 * ((j >> 4) * kRfPitch + (j & 15)) + 1) << 16), __float_as_int(tb.s2[i]));
  }
  __syncthreads();
  const int n_rounds = rd.n_rounds;

  float2* buf = sm.buf[g];
  float* xa = sm.xin[g];
  float* xv = xa + 528;  // 16-byte aligned behind the 513 audio values
  for (int64_t row = (int64_t)blockIdx.x * kRowGroups + g; row < rows; row += (int64_t)gridDim.x * kRowGroups) {
    if (lengths && (int)(row % t_max) >= lengths[row / t_max]) continue;  // group-uniform
    for (int i = t; i < kNA; i += kRfThreads) xa[i] = audio[row * kNA + i];
    for (int i = t; i < kNV; i += kRfThreads) xv[i] = video[row * kNV + i];
    // count sketches into the exchange buffer (.x audio, .y video), round by round (McbRounds)
    float2* mine = buf + (t >> 4) * kRfPitch + (t & 15);  // logical index t + 64 m lives at mine[4 m * kRfPitch]
#pragma unroll
    for (int m = 0; m < 16; ++m) mine[4 * m * kRfPitch] = make_float2(0.f, 0.f);
    rf_group_bar(bar_id);  // zeros and inputs visible to the group
    {
      float* sk = reinterpret_cast<float*>(buf);
#pragma unroll 1
      for (int r = 0; r < n_rounds; ++r) {
        for (int e = sm.roff1[r] + t, e1 = sm.roff1[r + 1]; e < e1; e += kRfThreads) {
          const int2 en = sm.ent1[e];
          sk[en.x >> 16] += xa[en.x & 0xFFFF] * __int_as_float(en.y);
        }
        for (int e = sm.roff2[r] + t, e1 = sm.roff2[r + 1]; e < e1; e += kRfThreads) {
          const int2 en = sm.ent2[e];
          sk[en.x >> 16] += xv[en.x & 0xFFFF] * __int_as_float(en.y);
        }
        rf_group_bar(bar_id);
      }
    }
    float2 v[16];
    // pass 0: Z = FFT(px + i py).  pass 1: FFT(conj(X Y)) = N * ifft(X Y) with X[k] = (Z[k] + conj(Z[N-k])) / 2,
    // Y[k] = (Z[k] - conj(Z[N-k])) / (2i); the partner of k = t + 64 m is held by thread 64 - t, hence the exchange.
    // One rolled loop so that the transform's code exists once.
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
      if (pass == 0) {
#pragma unroll
        for (int m = 0; m < 16; ++m) v[m] = mine[4 * m * kRfPitch];  // behind the last round's barrier
      } else {
#pragma unroll
        for (int m = 0; m < 16; ++m) mine[4 * m * kRfPitch] = v[m];
        rf_group_bar(bar_id);
#pragma unroll
        for (int m = 0; m < 16; ++m) {
          const int kn = (kFftN - (t + 64 * m)) & (kFftN - 1);
          const float2 zn = buf[(kn >> 4) * kRfPitch + (kn & 15)];
          const float2 zk = v[m];
          const float2 X = make_float2(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));
          const float2 Y = make_float2(0.5f * (zk.y + zn.y), 0.5f * (zn.x - zk.x));
          const float2 P = cmul(X, Y);
          v[m] = make_float2(P.x, -P.y);
        }
      }
      rf_group_bar(bar_id);  // the buffer is free (pass 0: sketches fetched; pass 1: all partners fetched)
      fft1024_reg(v, buf, sm.twB, sm.twC, t, bar_id);
    }

    float ss = 0.f;
#pragma unroll
    for (int m = 0; m < 16; ++m) {
      const float p = v[m].x * (1.0f / kFftN);
      const float r = sqrtf(fabsf(p) + eps);  // torch.sign(p) * sqrt(|p| + eps)   (sign(0) = 0)
      const float y = (p > 0.f) ? r : ((p < 0.f) ? -r : 0.f);
      y_out[row * kMcbOut + t + 64 * m] = y;
      ss += y * y;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    if (t == 32) sm.red[g] = ss;
    rf_group_bar(bar_id);
    if (t == 0) rowsq[row] = ss + sm.red[g];
  }
}

// MCB row pass: the register-FFT kernel (default) or the radix-4 shared-memory kernel (AVVAD_MCB_REG=0)
static int launch_mcb_rows(const float* audio, const float* video, const McbTables& tb, const McbRounds& rd,
                           const float2* tw, float eps, float* y, float* rowsq, int64_t rows, const int32_t* lengths,
                           int t_max, cudaStream_t st) {
  static int mode = -1;
  if (mode < 0) {
    const char* e = getenv("AVVAD_MCB_REG");
    mode = (e && e[0] == '0') ? 0 : 1;
  }
  if (mode == 0 || rd.n_rounds > kMaxRounds) {  // > 32 inputs in one bucket: not a hash any more, gather kernel
    mcb_row_kernel<<<(unsigned)rows, kFftThreads, 0, st>>>(audio, video, tb, tw, eps, y, rowsq, lengths, t_max);
    AVVAD_LAUNCHED();
    return AVVAD_OK;
  }
  static PerDeviceOnce attr_once;
  int sms = 0, dev = 0;
  AVVAD_CUDA(cudaGetDevice(&dev));
  AVVAD_CUDA(attr_once.run([] {
    return cudaFuncSetAttribute(mcb_row_reg_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RowSmem));
  }));
  AVVAD_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int64_t want = ceil_div(rows, (int64_t)kRowGroups);
  const unsigned grid = (unsigned)std::min<int64_t>(want, (int64_t)sms * 3);
  mcb_row_reg_kernel<<<grid, kRowGroups * kRfThreads, sizeof(RowSmem), st>>>(audio, video, tb, rd, tw, eps, y, rowsq,
                                                                            rows, lengths, t_max);
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}

// whole-tensor L2 norm: deterministic two-level reduction in double
__global__ void __launch_bounds__(1024) mcb_norm_kernel(const float* __restrict__ rowsq, int64_t rows,
                                                        float* __restrict__ norm_out) {
  __shared__ double sm[1024];
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < rows; i += 1024) acc += (double)rowsq[i];
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 512; s > 0; s >>= 1) {
    if (threadIdx.x < s) sm[threadIdx.x] += sm[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) norm_out[0] = (float)sqrt(sm[0]);
}

// y / norm -> BatchNorm1d (eval) -> bf16 (and / or fp32).  Eight consecutive channels per thread: two 128-bit loads of y,
// one 128-bit bf16 store (the scalar form ran at 1.8 TB/s: one 2-byte store and five loads per element).  `norms` holds
// one value (whole-call norm) or, with `lengths`, one per utterance of t_max rows (rows behind the length: zeros).
__global__ void __launch_bounds__(256)
mcb_apply_kernel(const float* __restrict__ y, const float* __restrict__ norms, const int32_t* __restrict__ lengths,
                 int t_max, const float* __restrict__ bn_mean, const float* __restrict__ bn_invstd,
                 const float* __restrict__ bn_gamma, const float* __restrict__ bn_beta, int64_t rows,
                 __nv_bfloat16* __restrict__ out_bf16, int64_t ld_out, float* __restrict__ out_f32) {
  const int64_t idx8 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // group of 8 channels
  if (idx8 >= rows * (kMcbOut / 8)) return;
  const int64_t r = idx8 / (kMcbOut / 8);
  const int j = (int)(idx8 - r * (kMcbOut / 8)) * 8;
  float o[8];
  bool live = true;
  float nrm;
  if (lengths) {
    const int64_t b = r / t_max;
    live = (int)(r - b * t_max) < lengths[b];
    nrm = norms[b];
  } else {
    nrm = norms[0];
  }
  if (live) {
    const float4 y0 = *reinterpret_cast<const float4*>(y + r * kMcbOut + j);
    const float4 y1 = *reinterpret_cast<const float4*>(y + r * kMcbOut + j + 4);
    const float yy[8] = {y0.x, y0.y, y0.z, y0.w, y1.x, y1.y, y1.z, y1.w};
    // 128-bit loads of the per-channel constants (32 scalar loads per thread throttled the load queue: ncu lg_throttle 40)
    float pm[8], pi[8], pg[8], pb[8];
    const bool vec = ((reinterpret_cast<uintptr_t>(bn_mean) | reinterpret_cast<uintptr_t>(bn_invstd) |
                       reinterpret_cast<uintptr_t>(bn_gamma) | reinterpret_cast<uintptr_t>(bn_beta)) & 15) == 0;
    if (!vec) {  // caller-owned gamma / beta (training) at an unaligned address
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        pm[e] = bn_mean[j + e]; pi[e] = bn_invstd[j + e]; pg[e] = bn_gamma[j + e]; pb[e] = bn_beta[j + e];
      }
    } else
#pragma unroll
    for (int hlf = 0; hlf < 2; ++hlf) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(bn_mean + j) + hlf);
      const float4 b = __ldg(reinterpret_cast<const float4*>(bn_invstd + j) + hlf);
      const float4 c = __ldg(reinterpret_cast<const float4*>(bn_gamma + j) + hlf);
      const float4 d = __ldg(reinterpret_cast<const float4*>(bn_beta + j) + hlf);
      pm[4 * hlf] = a.x; pm[4 * hlf + 1] = a.y; pm[4 * hlf + 2] = a.z; pm[4 * hlf + 3] = a.w;
      pi[4 * hlf] = b.x; pi[4 * hlf + 1] = b.y; pi[4 * hlf + 2] = b.z; pi[4 * hlf + 3] = b.w;
      pg[4 * hlf] = c.x; pg[4 * hlf + 1] = c.y; pg[4 * hlf + 2] = c.z; pg[4 * hlf + 3] = c.w;
      pb[4 * hlf] = d.x; pb[4 * hlf + 1] = d.y; pb[4 * hlf + 2] = d.z; pb[4 * hlf + 3] = d.w;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float v = yy[e] / nrm;
      o[e] = (v - pm[e]) * pi[e] * pg[e] + pb[e];
    }
  } else {
#pragma unroll
    for (int e = 0; e < 8; ++e) o[e] = 0.f;
  }
  if (out_bf16) {
    __nv_bfloat16* op = out_bf16 + r * ld_out + j;
    if ((reinterpret_cast<uintptr_t>(op) & 15) == 0) {
      uint4 pk;
      pk.x = pack_bf16x2(o[0], o[1]);
      pk.y = pack_bf16x2(o[2], o[3]);
      pk.z = pack_bf16x2(o[4], o[5]);
      pk.w = pack_bf16x2(o[6], o[7]);
      *reinterpret_cast<uint4*>(op) = pk;
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) op[e] = __float2bfloat16_rn(o[e]);
    }
  }
  if (out_f32) {
    float4* of = reinterpret_cast<float4*>(out_f32 + r * kMcbOut + j);
    of[0] = make_float4(o[0], o[1], o[2], o[3]);
    of[1] = make_float4(o[4], o[5], o[6], o[7]);
  }
}

// ---- grouped calls: one L2 norm per utterance (= per forward call of the reference's evaluation loop) ----
// norms[b] = sqrt(sum_{t < len_b} rowsq[b*t_max + t]); one block per utterance, fixed-order fp64 tree
__global__ void __launch_bounds__(256) mcb_norm_grouped_kernel(const float* __restrict__ rowsq,
                                                               const int32_t* __restrict__ lengths, int t_max,
                                                               float* __restrict__ norms) {
  __shared__ double sm[256];
  const int64_t b = blockIdx.x;
  int n = lengths[b];
  n = n < 0 ? 0 : (n > t_max ? t_max : n);
  double acc = 0.0;
  for (int t = threadIdx.x; t < n; t += 256) acc += (double)rowsq[b * t_max + t];
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) sm[threadIdx.x] += sm[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) norms[b] = (float)sqrt(sm[0]);
}

// ---- training mode: BatchNorm1d with batch statistics over all rows, and the gradients of its affine parameters ----
// v = y / norm;  stats over rows per channel (fp64 accumulation, one block per channel, fixed order)
__global__ void __launch_bounds__(256) mcb_bn_stats_kernel(const float* __restrict__ y, const float* __restrict__ norm,
                                                           int64_t rows, float eps, float momentum,
                                                           float* __restrict__ mean_invstd,
                                                           float* __restrict__ running_mean,
                                                           float* __restrict__ running_var) {
  __shared__ double s1[256], s2[256];
  const int j = blockIdx.x;
  const double inv = 1.0 / (double)norm[0];
  double a = 0.0, b = 0.0;
  for (int64_t r = threadIdx.x; r < rows; r += 256) {
    const double v = (double)y[r * kMcbOut + j] * inv;
    a += v;
    b += v * v;
  }
  s1[threadIdx.x] = a;
  s2[threadIdx.x] = b;
  __syncthreads();
  for (int st = 128; st > 0; st >>= 1) {
    if (threadIdx.x < st) {
      s1[threadIdx.x] += s1[threadIdx.x + st];
      s2[threadIdx.x] += s2[threadIdx.x + st];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double mean = s1[0] / (double)rows;
    double var = s2[0] / (double)rows - mean * mean;
    if (var < 0) var = 0;
    mean_invstd[j] = (float)mean;
    mean_invstd[kMcbOut + j] = (float)(1.0 / sqrt(var + (double)eps));
    if (running_mean) {
      const double unbiased = rows > 1 ? var * (double)rows / (double)(rows - 1) : var;
      running_mean[j] = (1.f - momentum) * running_mean[j] + momentum * (float)mean;
      running_var[j] = (1.f - momentum) * running_var[j] + momentum * (float)unbiased;
    }
  }
}
// dgamma[j] = sum_r dx[r][j] * xhat[r][j], dbeta[j] = sum_r dx[r][j]
__global__ void __launch_bounds__(256) mcb_bn_grad_kernel(const float* __restrict__ y, const float* __restrict__ norm,
                                                          const float* __restrict__ mean_invstd,
                                                          const float* __restrict__ dx, int64_t ld_dx, int64_t rows,
                                                          float* __restrict__ dgamma, float* __restrict__ dbeta) {
  __shared__ double s1[256], s2[256];
  const int j = blockIdx.x;
  const float inv = 1.0f / norm[0];
  const float mean = mean_invstd[j], istd = mean_invstd[kMcbOut + j];
  double a = 0.0, b = 0.0;
  for (int64_t r = threadIdx.x; r < rows; r += 256) {
    const float g = dx[r * ld_dx + j];
    const float xh = (y[r * kMcbOut + j] * inv - mean) * istd;
    a += (double)g * xh;
    b += (double)g;
  }
  s1[threadIdx.x] = a;
  s2[threadIdx.x] = b;
  __syncthreads();
  for (int st = 128; st > 0; st >>= 1) {
    if (threadIdx.x < st) {
      s1[threadIdx.x] += s1[threadIdx.x + st];
      s2[threadIdx.x] += s2[threadIdx.x + st];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    dgamma[j] = (float)s1[0];
    dbeta[j] = (float)s2[0];
  }
}

// ---- stand-alone count sketch / compact bilinear pooling (compact_bilinear_pooling.py:59-113,140-263) ----
// Generic sizes: out[row][j] = sum_{i: h_i = j} s_i x[row][i], collisions summed in ascending i (CSR built by the host).
__global__ void count_sketch_fwd_kernel(const float* __restrict__ x, int64_t rows, int in_size, int out_size,
                                        const int32_t* __restrict__ off, const int32_t* __restrict__ idx,
                                        const float* __restrict__ s, float* __restrict__ out) {
  const int64_t row = blockIdx.x;
  const float* xr = x + row * in_size;
  for (int j = threadIdx.x; j < out_size; j += blockDim.x) {
    float acc = 0.f;
    for (int e = off[j]; e < off[j + 1]; ++e) {
      const int i = idx[e];
      acc += xr[i] * s[i];
    }
    out[row * out_size + j] = acc;
  }
}
// grad_x[row][i] = s_i * grad_out[row][h_i]   (CountSketchFn_backward, compact_bilinear_pooling.py:29-41)
__global__ void count_sketch_bwd_kernel(const float* __restrict__ go, int64_t rows, int in_size, int out_size,
                                        const int32_t* __restrict__ h, const float* __restrict__ s,
                                        float* __restrict__ gx) {
  const int64_t row = blockIdx.x;
  for (int i = threadIdx.x; i < in_size; i += blockDim.x) gx[row * in_size + i] = s[i] * go[row * out_size + h[i]];
}

// One row of irfft(rfft(u) * rfft(v)) (MODE 0: circular convolution) or irfft(rfft(u) * conj(rfft(v))) (MODE 1:
// circular correlation, the adjoint the reference's backward applies: compact_bilinear_pooling.py:186-215), u and v real
// length-1024 sequences already in `z` as (u, v) pairs.  Returns the buffer whose .x holds 1024 * result.
template <int MODE>
__device__ __forceinline__ const float2* circ_product_1024(float2* z, float2* scratch, const float2* stw, int tid) {
  float2* z1 = fft1024_smem(z, scratch, stw, tid);
  float2* z2 = (z1 == z) ? scratch : z;
  for (int k = tid; k <= 512; k += kFftThreads) {
    if (k == 0 || k == 512) {
      const float2 q = z1[k];
      z1[k] = make_float2(q.x * q.y, 0.f);
    } else {
      const float2 zk = z1[k];
      const float2 zn = z1[kFftN - k];
      const float2 X = make_float2(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));
      float2 Y = make_float2(0.5f * (zk.y + zn.y), 0.5f * (zn.x - zk.x));
      if (MODE == 1) Y.y = -Y.y;
      const float2 P = cmul(X, Y);
      z1[k] = make_float2(P.x, -P.y);
      z1[kFftN - k] = make_float2(P.x, P.y);
    }
  }
  __syncthreads();
  return fft1024_smem(z1, z2, stw, tid);
}

// MODE 0: out[1024] = sketch1(x) (*) sketch2(y)                       (forward)
// MODE 1: gx[513]  = sketch1^T( go (corr) sketch2(y) )                 (gradient w.r.t. x)
// MODE 2: gy[512]  = sketch2^T( go (corr) sketch1(x) )                 (gradient w.r.t. y)
template <int MODE>
__global__ void __launch_bounds__(kFftThreads)
mcb_raw_kernel(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ go, McbTables tb,
               const int32_t* __restrict__ hsel, const float2* __restrict__ tw_g, float* __restrict__ out) {
  __shared__ float2 sa[kFftN];
  __shared__ float2 sb[kFftN];
  __shared__ float2 stw[kFftTwStage];
  __shared__ float xin[kNA];
  const int tid = threadIdx.x;
  const int64_t row = blockIdx.x;
#pragma unroll
  for (int q = 0; q < kFftTwStage / kFftThreads; ++q)
    stw[tid + q * kFftThreads] = tw_g[kFftTwHann + tid + q * kFftThreads];
  if (MODE == 0) {
    __shared__ float yin[kNV];
    for (int i = tid; i < kNA; i += kFftThreads) xin[i] = x[row * kNA + i];
    for (int i = tid; i < kNV; i += kFftThreads) yin[i] = y[row * kNV + i];
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int j = tid + q * kFftThreads;
      float px = 0.f, py = 0.f;
      for (int e = tb.off1[j]; e < tb.off1[j + 1]; ++e) px += xin[tb.idx1[e]] * tb.s1[tb.idx1[e]];
      for (int e = tb.off2[j]; e < tb.off2[j + 1]; ++e) py += yin[tb.idx2[e]] * tb.s2[tb.idx2[e]];
      sa[j] = make_float2(px, py);
    }
  } else {
    // the sketch of the OTHER input is the correlation kernel
    const int n_other = (MODE == 1) ? kNV : kNA;
    const float* other = (MODE == 1) ? y : x;
    const int32_t* off = (MODE == 1) ? tb.off2 : tb.off1;
    const int32_t* idx = (MODE == 1) ? tb.idx2 : tb.idx1;
    const float* sg = (MODE == 1) ? tb.s2 : tb.s1;
    for (int i = tid; i < n_other; i += kFftThreads) xin[i] = other[row * n_other + i];
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int j = tid + q * kFftThreads;
      float p = 0.f;
      for (int e = off[j]; e < off[j + 1]; ++e) p += xin[idx[e]] * sg[idx[e]];
      sa[j] = make_float2(go[row * kMcbOut + j], p);
    }
  }
  __syncthreads();
  const float2* res = circ_product_1024<(MODE == 0) ? 0 : 1>(sa, sb, stw, tid);
  if (MODE == 0) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int j = tid + q * kFftThreads;
      out[row * kMcbOut + j] = res[j].x * (1.0f / kFftN);
    }
  } else {
    const int n_self = (MODE == 1) ? kNA : kNV;
    const float* ss = (MODE == 1) ? tb.s1 : tb.s2;
    for (int i = tid; i < n_self; i += kFftThreads) out[row * n_self + i] = ss[i] * res[hsel[i]].x * (1.0f / kFftN);
  }
}

__global__ void bn_invstd_kernel(const float* __restrict__ var, float eps, float* __restrict__ invstd, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) invstd[i] = 1.0f / sqrtf(var[i] + eps);
}

}  // namespace avvad

using namespace avvad;

struct avvad_mcb {
  int32_t *off1, *idx1, *off2, *idx2;
  int32_t *rnd;  // scatter rounds (McbRounds): ent1 [513] | ent2 [512] | roff1 [33] | roff2 [33]
  int n_rounds;
  float *s1, *s2;
  float *bn_gamma, *bn_beta, *bn_mean, *bn_invstd;
  float eps;
  bool loaded;
};

static McbRounds rounds_of(const avvad_mcb* h) {
  return McbRounds{h->rnd, h->rnd + kNA, h->rnd + kNA + kNV, h->rnd + kNA + kNV + kMaxRounds + 1, h->n_rounds};
}

extern "C" int avvad_mcb_create(avvad_mcb** out) {
  AVVAD_CHECK_ARG(out, "null out");
  avvad_mcb* h = new avvad_mcb();
  h->loaded = false;
  AVVAD_CUDA(cudaMalloc(&h->off1, sizeof(int32_t) * 1025));
  AVVAD_CUDA(cudaMalloc(&h->off2, sizeof(int32_t) * 1025));
  AVVAD_CUDA(cudaMalloc(&h->idx1, sizeof(int32_t) * kNA));
  AVVAD_CUDA(cudaMalloc(&h->idx2, sizeof(int32_t) * kNV));
  AVVAD_CUDA(cudaMalloc(&h->rnd, sizeof(int32_t) * (kNA + kNV + 2 * (kMaxRounds + 1))));
  h->n_rounds = 0;
  AVVAD_CUDA(cudaMalloc(&h->s1, sizeof(float) * kNA));
  AVVAD_CUDA(cudaMalloc(&h->s2, sizeof(float) * kNV));
  AVVAD_CUDA(cudaMalloc(&h->bn_gamma, sizeof(float) * kMcbOut));
  AVVAD_CUDA(cudaMalloc(&h->bn_beta, sizeof(float) * kMcbOut));
  AVVAD_CUDA(cudaMalloc(&h->bn_mean, sizeof(float) * kMcbOut));
  AVVAD_CUDA(cudaMalloc(&h->bn_invstd, sizeof(float) * kMcbOut));
  *out = h;
  return AVVAD_OK;
}

extern "C" void avvad_mcb_destroy(avvad_mcb* h) {
  if (!h) return;
  cudaFree(h->off1); cudaFree(h->off2); cudaFree(h->idx1); cudaFree(h->idx2); cudaFree(h->rnd);
  cudaFree(h->s1); cudaFree(h->s2);
  cudaFree(h->bn_gamma); cudaFree(h->bn_beta); cudaFree(h->bn_mean); cudaFree(h->bn_invstd);
  delete h;
}

static int build_csr(const int64_t* h_dev, int n, int32_t* off_dev, int32_t* idx_dev, cudaStream_t st,
                     int32_t* ent_dev = nullptr, int32_t* roff_dev = nullptr, int* n_rounds = nullptr) {
  std::vector<int64_t> hh(n);
  AVVAD_CUDA(cudaMemcpyAsync(hh.data(), h_dev, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, st));
  AVVAD_CUDA(cudaStreamSynchronize(st));
  std::vector<int32_t> off(kMcbOut + 1, 0), idx(n);
  for (int i = 0; i < n; ++i) {
    if (hh[i] < 0 || hh[i] >= kMcbOut) {
      set_error("mcb: sketch index out of range [0,1024)");
      return AVVAD_ERR_ARG;
    }
    off[hh[i] + 1]++;
  }
  for (int j = 0; j < kMcbOut; ++j) off[j + 1] += off[j];
  std::vector<int32_t> cur(off.begin(), off.end() - 1);
  for (int i = 0; i < n; ++i) idx[cur[hh[i]]++] = i;  // ascending i inside each bucket
  AVVAD_CUDA(cudaMemcpyAsync(off_dev, off.data(), sizeof(int32_t) * (kMcbOut + 1), cudaMemcpyHostToDevice, st));
  AVVAD_CUDA(cudaMemcpyAsync(idx_dev, idx.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, st));
  std::vector<int32_t> ent, roff(kMaxRounds + 1, n);
  if (ent_dev) {
    // scatter rounds: round r = the r-th member (ascending input index) of every bucket, each round in ascending
    // input order (coalesced input reads)
    std::vector<int32_t> rank(n);
    int rounds = 0;
    for (int j = 0; j < kMcbOut; ++j)
      for (int e = off[j]; e < off[j + 1]; ++e) {
        rank[idx[e]] = e - off[j];
        rounds = std::max(rounds, e - off[j] + 1);
      }
    ent.reserve(n);
    // (ordering a round's entries so that every 32 consecutive ones hit 32 distinct banks for both the input gather and
    // the bucket update was measured: no change, 0.7159 vs 0.7158 ms -- left in ascending input order)
    for (int r = 0; r < rounds; ++r) {
      if (r <= kMaxRounds) roff[r] = (int32_t)ent.size();
      for (int i = 0; i < n; ++i)
        if (rank[i] == r) ent.push_back(i | ((int32_t)hh[i] << 16));
    }
    *n_rounds = rounds;
    AVVAD_CUDA(cudaMemcpyAsync(ent_dev, ent.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, st));
    AVVAD_CUDA(cudaMemcpyAsync(roff_dev, roff.data(), sizeof(int32_t) * (kMaxRounds + 1), cudaMemcpyHostToDevice, st));
  }
  AVVAD_CUDA(cudaStreamSynchronize(st));
  return AVVAD_OK;
}

extern "C" int avvad_mcb_load(avvad_mcb* h, const int64_t* h1, const float* s1, const int64_t* h2, const float* s2,
                              const float* bn_gamma, const float* bn_beta, const float* bn_mean, const float* bn_var,
                              float eps, void* stream) {
  AVVAD_CHECK_ARG(h && h1 && s1 && h2 && s2 && bn_gamma && bn_beta && bn_mean && bn_var, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  int r1 = 0, r2 = 0;
  int rc = build_csr(h1, kNA, h->off1, h->idx1, st, h->rnd, h->rnd + kNA + kNV, &r1);
  if (rc) return rc;
  rc = build_csr(h2, kNV, h->off2, h->idx2, st, h->rnd + kNA, h->rnd + kNA + kNV + kMaxRounds + 1, &r2);
  if (rc) return rc;
  h->n_rounds = std::max(r1, r2);
  AVVAD_CUDA(cudaMemcpyAsync(h->s1, s1, sizeof(float) * kNA, cudaMemcpyDeviceToDevice, st));
  AVVAD_CUDA(cudaMemcpyAsync(h->s2, s2, sizeof(float) * kNV, cudaMemcpyDeviceToDevice, st));
  AVVAD_CUDA(cudaMemcpyAsync(h->bn_gamma, bn_gamma, sizeof(float) * kMcbOut, cudaMemcpyDeviceToDevice, st));
  AVVAD_CUDA(cudaMemcpyAsync(h->bn_beta, bn_beta, sizeof(float) * kMcbOut, cudaMemcpyDeviceToDevice, st));
  AVVAD_CUDA(cudaMemcpyAsync(h->bn_mean, bn_mean, sizeof(float) * kMcbOut, cudaMemcpyDeviceToDevice, st));
  bn_invstd_kernel<<<4, 256, 0, st>>>(bn_var, eps, h->bn_invstd, kMcbOut);
  AVVAD_LAUNCHED();
  h->eps = eps;
  h->loaded = true;
  return AVVAD_OK;
}

extern "C" size_t avvad_mcb_workspace_bytes(int64_t rows) {
  if (rows <= 0) return 0;
  // y (f32), per-row sums of squares, norm, [training] mean/invstd
  return align_up((size_t)rows * kMcbOut * sizeof(float), 256) + align_up((size_t)rows * sizeof(float), 256) + 256 +
         2 * kMcbOut * sizeof(float);
}

extern "C" int avvad_mcb_forward(avvad_mcb* h, const float* audio, const float* video, int64_t rows, void* workspace,
                                 size_t workspace_bytes, void* out_bf16, int64_t ld_out, float* out_f32,
                                 void* stream) {
  AVVAD_CHECK_ARG(h && audio && video && workspace && rows > 0, "bad argument");
  AVVAD_CHECK_ARG(out_bf16 || out_f32, "at least one output required");
  AVVAD_CHECK_ARG(!out_bf16 || ld_out >= kMcbOut, "ld_out must be >= 1024");
  if (!h->loaded) {
    set_error("mcb: not loaded");
    return AVVAD_ERR_STATE;
  }
  if (workspace_bytes < avvad_mcb_workspace_bytes(rows)) {
    set_error("mcb: workspace too small");
    return AVVAD_ERR_WORKSPACE;
  }
  AVVAD_CHECK_ARG(rows < (1ll << 31), "too many rows");
  const float2* tw = fft_twiddles_device();
  if (!tw) {
    set_error("twiddle table allocation failed");
    return AVVAD_ERR_CUDA;
  }
  cudaStream_t st = (cudaStream_t)stream;
  float* y = reinterpret_cast<float*>(workspace);
  float* rowsq = reinterpret_cast<float*>((uint8_t*)workspace + align_up((size_t)rows * kMcbOut * sizeof(float), 256));
  float* norm = reinterpret_cast<float*>((uint8_t*)rowsq + align_up((size_t)rows * sizeof(float), 256));
  McbTables tb{h->off1, h->idx1, h->s1, h->off2, h->idx2, h->s2};
  // profiling category 5: "flops" carries the algorithmic bytes (513 + 512 floats in, 1024 bf16 or fp32 out per row)
  void* ptok = nullptr;
  tc::prof_begin(st, &ptok);
  if (int rc = launch_mcb_rows(audio, video, tb, rounds_of(h), tw, h->eps, y, rowsq, rows, nullptr, 0, st)) return rc;
  mcb_norm_kernel<<<1, 1024, 0, st>>>(rowsq, rows, norm);
  AVVAD_LAUNCHED();
  const int64_t total = rows * kMcbOut;
  mcb_apply_kernel<<<(unsigned)ceil_div(total / 8, 256), 256, 0, st>>>(y, norm, nullptr, 0, h->bn_mean, h->bn_invstd,
                                                                       h->bn_gamma, h->bn_beta, rows,
                                                                       (__nv_bfloat16*)out_bf16, ld_out, out_f32);
  AVVAD_LAUNCHED();
  tc::prof_end(st, ptok, 5, (double)rows * (4100.0 + (out_f32 ? 4096.0 : 2048.0)));
  return AVVAD_OK;
}


// Grouped forward: the rows are n_groups utterances of t_max rows each ([b][t] layout, lengths[b] valid rows) and every
// utterance is normalised by its OWN L2 norm over its valid rows -- what the reference computes when its evaluation
// loop calls the model once per utterance (scripts/evaluate_AV_net.py:186-236: x[None], v[None], lengths = [T]), so a
// batched call reproduces n_groups stand-alone forward calls.  Rows behind an utterance's length are skipped (no
// sketch / FFT work) and written as zeros.
extern "C" size_t avvad_mcb_grouped_workspace_bytes(int64_t n_groups, int64_t t_max) {
  if (n_groups <= 0 || t_max <= 0) return 0;
  return avvad_mcb_workspace_bytes(n_groups * t_max) + align_up((size_t)n_groups * sizeof(float), 256);
}

// norms_in (optional, f32 [n_groups]): use these norms instead of computing them -- a streaming caller normalises
// every block of an utterance by one constant.  norms_out (optional): the norms the call used.
extern "C" int avvad_mcb_forward_grouped_norms(avvad_mcb* h, const float* audio, const float* video, int64_t n_groups,
                                               int64_t t_max, const int32_t* lengths, const float* norms_in,
                                               float* norms_out, void* workspace, size_t workspace_bytes,
                                               void* out_bf16, int64_t ld_out, float* out_f32, void* stream) {
  AVVAD_CHECK_ARG(h && audio && video && workspace && lengths && n_groups > 0 && t_max > 0, "bad argument");
  AVVAD_CHECK_ARG(out_bf16 || out_f32, "at least one output required");
  AVVAD_CHECK_ARG(!out_bf16 || ld_out >= kMcbOut, "ld_out must be >= 1024");
  AVVAD_CHECK_ARG(t_max < (1ll << 31) && n_groups < (1ll << 31) && n_groups * t_max < (1ll << 31), "too many rows");
  if (!h->loaded) {
    set_error("mcb: not loaded");
    return AVVAD_ERR_STATE;
  }
  if (workspace_bytes < avvad_mcb_grouped_workspace_bytes(n_groups, t_max)) {
    set_error("mcb: workspace too small");
    return AVVAD_ERR_WORKSPACE;
  }
  const float2* tw = fft_twiddles_device();
  if (!tw) {
    set_error("twiddle table allocation failed");
    return AVVAD_ERR_CUDA;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t rows = n_groups * t_max;
  float* y = reinterpret_cast<float*>(workspace);
  float* rowsq = reinterpret_cast<float*>((uint8_t*)workspace + align_up((size_t)rows * kMcbOut * sizeof(float), 256));
  float* norms = reinterpret_cast<float*>((uint8_t*)workspace + avvad_mcb_workspace_bytes(rows));
  McbTables tb{h->off1, h->idx1, h->s1, h->off2, h->idx2, h->s2};
  void* ptok = nullptr;
  tc::prof_begin(st, &ptok);
  if (int rc = launch_mcb_rows(audio, video, tb, rounds_of(h), tw, h->eps, y, rowsq, rows, lengths, (int)t_max, st)) return rc;
  const float* nrm = norms_in;
  if (!norms_in) {
    mcb_norm_grouped_kernel<<<(unsigned)n_groups, 256, 0, st>>>(rowsq, lengths, (int)t_max, norms);
    AVVAD_LAUNCHED();
    nrm = norms;
  }
  if (norms_out && norms_out != nrm)
    AVVAD_CUDA(cudaMemcpyAsync(norms_out, nrm, (size_t)n_groups * sizeof(float), cudaMemcpyDeviceToDevice, st));
  const int64_t total = rows * kMcbOut;
  mcb_apply_kernel<<<(unsigned)ceil_div(total / 8, 256), 256, 0, st>>>(
      y, nrm, lengths, (int)t_max, h->bn_mean, h->bn_invstd, h->bn_gamma, h->bn_beta, rows,
      (__nv_bfloat16*)out_bf16, ld_out, out_f32);
  AVVAD_LAUNCHED();
  tc::prof_end(st, ptok, 5, (double)rows * (4100.0 + (out_f32 ? 4096.0 : 2048.0)));
  return AVVAD_OK;
}

extern "C" int avvad_mcb_forward_grouped(avvad_mcb* h, const float* audio, const float* video, int64_t n_groups,
                                         int64_t t_max, const int32_t* lengths, void* workspace,
                                         size_t workspace_bytes, void* out_bf16, int64_t ld_out, float* out_f32,
                                         void* stream) {
  return avvad_mcb_forward_grouped_norms(h, audio, video, n_groups, t_max, lengths, nullptr, nullptr, workspace,
                                         workspace_bytes, out_bf16, ld_out, out_f32, stream);
}


// Training-mode forward (AV_Net.py:119 with the module in train()): BatchNorm1d uses the batch statistics of this call
// and the module's CURRENT affine parameters (gamma, beta: trainable, passed per call), and updates running_mean /
// running_var in place (NULL = leave).  The workspace keeps y, the norm and the batch statistics for
// avvad_mcb_backward_bn.
extern "C" int avvad_mcb_forward_train(avvad_mcb* h, const float* audio, const float* video, int64_t rows,
                                       void* workspace, size_t workspace_bytes, const float* gamma, const float* beta,
                                       float momentum, float* running_mean, float* running_var, void* out_bf16,
                                       int64_t ld_out, float* out_f32, void* stream) {
  AVVAD_CHECK_ARG(h && audio && video && workspace && gamma && beta && rows > 0, "bad argument");
  AVVAD_CHECK_ARG(out_bf16 || out_f32, "at least one output required");
  if (!h->loaded) { set_error("mcb: not loaded"); return AVVAD_ERR_STATE; }
  if (workspace_bytes < avvad_mcb_workspace_bytes(rows)) { set_error("mcb: workspace too small"); return AVVAD_ERR_WORKSPACE; }
  const float2* tw = fft_twiddles_device();
  if (!tw) { set_error("twiddle table allocation failed"); return AVVAD_ERR_CUDA; }
  cudaStream_t st = (cudaStream_t)stream;
  float* y = reinterpret_cast<float*>(workspace);
  float* rowsq = reinterpret_cast<float*>((uint8_t*)workspace + align_up((size_t)rows * kMcbOut * sizeof(float), 256));
  float* norm = reinterpret_cast<float*>((uint8_t*)rowsq + align_up((size_t)rows * sizeof(float), 256));
  float* mean_invstd = norm + 64;
  McbTables tb{h->off1, h->idx1, h->s1, h->off2, h->idx2, h->s2};
  if (int rc = launch_mcb_rows(audio, video, tb, rounds_of(h), tw, h->eps, y, rowsq, rows, nullptr, 0, st)) return rc;
  mcb_norm_kernel<<<1, 1024, 0, st>>>(rowsq, rows, norm);
  AVVAD_LAUNCHED();
  mcb_bn_stats_kernel<<<kMcbOut, 256, 0, st>>>(y, norm, rows, h->eps, momentum, mean_invstd, running_mean, running_var);
  AVVAD_LAUNCHED();
  const int64_t total = rows * kMcbOut;
  mcb_apply_kernel<<<(unsigned)ceil_div(total / 8, 256), 256, 0, st>>>(y, norm, nullptr, 0, mean_invstd,
                                                                       mean_invstd + kMcbOut, gamma, beta, rows,
                                                                       (__nv_bfloat16*)out_bf16, ld_out, out_f32);
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}

// dx: f32 [rows][ld_dx] gradient w.r.t. the BatchNorm output (first 1024 columns) -> dgamma, dbeta [1024].
// `workspace` must be the one the matching avvad_mcb_forward_train call filled.
extern "C" int avvad_mcb_backward_bn(avvad_mcb* h, void* workspace, const float* dx, int64_t ld_dx, int64_t rows,
                                     float* dgamma, float* dbeta, void* stream) {
  AVVAD_CHECK_ARG(h && workspace && dx && dgamma && dbeta && rows > 0 && ld_dx >= kMcbOut, "bad argument");
  float* y = reinterpret_cast<float*>(workspace);
  float* rowsq = reinterpret_cast<float*>((uint8_t*)workspace + align_up((size_t)rows * kMcbOut * sizeof(float), 256));
  float* norm = reinterpret_cast<float*>((uint8_t*)rowsq + align_up((size_t)rows * sizeof(float), 256));
  float* mean_invstd = norm + 64;
  mcb_bn_grad_kernel<<<kMcbOut, 256, 0, (cudaStream_t)stream>>>(y, norm, mean_invstd, dx, ld_dx, rows, dgamma, dbeta);
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}

// ---- stand-alone modules (CountSketch / CompactBilinearPooling used outside DeepVAD_AV) ----
extern "C" int avvad_count_sketch_forward(const float* x, int64_t rows, int in_size, int out_size, const int32_t* off,
                                          const int32_t* idx, const float* s, float* out, void* stream) {
  AVVAD_CHECK_ARG(x && off && idx && s && out && rows > 0 && in_size > 0 && out_size > 0, "bad argument");
  AVVAD_CHECK_ARG(rows < (1ll << 31), "too many rows");
  count_sketch_fwd_kernel<<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>(x, rows, in_size, out_size, off, idx, s, out);
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}
extern "C" int avvad_count_sketch_backward(const float* grad_out, int64_t rows, int in_size, int out_size,
                                           const int32_t* h, const float* s, float* grad_x, void* stream) {
  AVVAD_CHECK_ARG(grad_out && h && s && grad_x && rows > 0 && in_size > 0 && out_size > 0, "bad argument");
  AVVAD_CHECK_ARG(rows < (1ll << 31), "too many rows");
  count_sketch_bwd_kernel<<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>(grad_out, rows, in_size, out_size, h, s,
                                                                            grad_x);
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}
extern "C" int avvad_mcb_raw_forward(const int32_t* off1, const int32_t* idx1, const float* s1, const int32_t* off2,
                                     const int32_t* idx2, const float* s2, const float* x, const float* y, int64_t rows,
                                     float* out, void* stream) {
  AVVAD_CHECK_ARG(off1 && idx1 && s1 && off2 && idx2 && s2 && x && y && out && rows > 0, "bad argument");
  AVVAD_CHECK_ARG(rows < (1ll << 31), "too many rows");
  const float2* tw = fft_twiddles_device();
  if (!tw) { set_error("twiddle table allocation failed"); return AVVAD_ERR_CUDA; }
  McbTables tb{off1, idx1, s1, off2, idx2, s2};
  mcb_raw_kernel<0><<<(unsigned)rows, kFftThreads, 0, (cudaStream_t)stream>>>(x, y, nullptr, tb, nullptr, tw, out);
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}
extern "C" int avvad_mcb_raw_backward(const int32_t* off1, const int32_t* idx1, const float* s1, const int32_t* h1,
                                      const int32_t* off2, const int32_t* idx2, const float* s2, const int32_t* h2,
                                      const float* x, const float* y, const float* grad_out, int64_t rows, float* grad_x,
                                      float* grad_y, void* stream) {
  AVVAD_CHECK_ARG(off1 && idx1 && s1 && h1 && off2 && idx2 && s2 && h2 && x && y && grad_out && rows > 0, "bad argument");
  AVVAD_CHECK_ARG(rows < (1ll << 31), "too many rows");
  const float2* tw = fft_twiddles_device();
  if (!tw) { set_error("twiddle table allocation failed"); return AVVAD_ERR_CUDA; }
  McbTables tb{off1, idx1, s1, off2, idx2, s2};
  if (grad_x) {
    mcb_raw_kernel<1><<<(unsigned)rows, kFftThreads, 0, (cudaStream_t)stream>>>(x, y, grad_out, tb, h1, tw, grad_x);
    AVVAD_LAUNCHED();
  }
  if (grad_y) {
    mcb_raw_kernel<2><<<(unsigned)rows, kFftThreads, 0, (cudaStream_t)stream>>>(x, y, grad_out, tb, h2, tw, grad_y);
    AVVAD_LAUNCHED();
  }
  return AVVAD_OK;
}
