// Audio front end: peak normalise -> frame/Hann -> 1024-pt rFFT -> |.|^2 -> log(.+eps) -> standardise,
// fused in one kernel (plus a small abs-max reduction); the FFT of each frame runs in shared memory.
//
// Reference semantics: packages/processing/stft.py:123-151, packages/data_handling.py:441,454-457,
// scripts/evaluate_AV_net.py:225-230, packages/utils.py:157-166 (zero padding happens BEFORE the
// standardisation, so padded frames hold (0-mean)/(std+eps)).
#include <math.h>

#include <mutex>

#include "fft.cuh"
#include "fft_reg.cuh"

namespace avvad {
namespace tc {
int prof_begin(cudaStream_t st, void** tok);
void prof_end(cudaStream_t st, void* tok, int cat, double flops);
}  // namespace tc
}  // namespace avvad

namespace avvad {

static float2* g_tw_dev[kMaxDevices] = {};  // one table per device (nn.DataParallel: several devices, one process)
static PerDeviceOnce g_tw_once;

const float2* fft_twiddles_device() {
  int cur = 0;
  if (cudaGetDevice(&cur) != cudaSuccess || cur < 0 || cur >= kMaxDevices) return nullptr;
  const cudaError_t e = g_tw_once.run([cur] {
    static float2 host[kFftTwTotal];
    const double two_pi = 6.283185307179586476925286766559;
    for (int k = 0; k < kFftTwTotal; ++k) host[k] = make_float2(1.f, 0.f);
    for (int r = 0; r < 16; ++r)
      for (int k = 0; k < 16; ++k) {
        double a = -two_pi * (double)(r * k) / 256.0;
        host[kFftTwHann + kFftTwStage + r * 16 + k] = make_float2((float)cos(a), (float)sin(a));
      }
    for (int k = 0; k < 512; ++k) {
      double a = -two_pi * (double)k / 1024.0;
      host[k] = make_float2((float)cos(a), (float)sin(a));
    }
    for (int s = 1; s <= 4; ++s) {
      const int Ns = 1 << (2 * s);
      for (int q = 1; q <= 3; ++q)
        for (int k = 0; k < Ns; ++k) {
          double a = -two_pi * (double)(q * k) / (4.0 * Ns);
          host[kFftTwHann + fft_tw_off(s) + (q - 1) * Ns + k] = make_float2((float)cos(a), (float)sin(a));
        }
    }
    float2* d = nullptr;
    cudaError_t err = cudaMalloc(&d, sizeof(host));
    if (err != cudaSuccess) return err;
    err = cudaMemcpy(d, host, sizeof(host), cudaMemcpyHostToDevice);
    if (err != cudaSuccess) {
      cudaFree(d);
      return err;
    }
    g_tw_dev[cur] = d;
    return cudaSuccess;
  });
  return e == cudaSuccess ? g_tw_dev[cur] : nullptr;
}

// ---- per-utterance max|x| ----------------------------------------------------------------------
__global__ void absmax_kernel(const float* __restrict__ wave, int64_t wave_stride,
                              const int32_t* __restrict__ n_samples, float* __restrict__ peak) {
  const int b = blockIdx.y;
  const int n = n_samples[b];
  const float* x = wave + (int64_t)b * wave_stride;
  float m = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(x[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  __shared__ float sm[8];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    m = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0.f;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    // non-negative floats order like their bit patterns
    if (threadIdx.x == 0) atomicMax(reinterpret_cast<unsigned int*>(peak + b), __float_as_uint(m));
  }
}

// ---- fused STFT / log-power kernel ---------------------------------------------------------------
// One CTA per (frame, utterance): the windowed frame is the real part of a 1024-point complex FFT held in
// shared memory (imaginary part zero), so a frame's features never depend on which other frames share the
// launch (trim / batch invariance is bit-exact).
// MODE 0: standardised log-power (B, t_max, 513);  MODE 1: raw complex STFT (B, 513, t_max, 2).
template <int MODE>
__global__ void __launch_bounds__(kFftThreads)
frontend_kernel(const float* __restrict__ wave, int64_t wave_stride, const int32_t* __restrict__ n_samples,
                const int32_t* __restrict__ n_frames, int t_max, const float* __restrict__ peak,
                const float* __restrict__ mean, const float* __restrict__ stdv, float eps,
                const float2* __restrict__ tw_g, float* __restrict__ out) {
  __shared__ float2 sa[kFftN];
  __shared__ float2 sb[kFftN];
  __shared__ float2 stw[kFftTwStage];

  const int tid = threadIdx.x;
  const int b = blockIdx.y;
  const int t = blockIdx.x;
  const int T = min(n_frames[b], t_max);

  if (t >= T) {
    if (MODE == 0) {
      // collate padding: zeros are padded BEFORE standardisation -> (0 - mean) / (std + eps)
      for (int k = tid; k < 513; k += kFftThreads)
        out[((int64_t)b * t_max + t) * 513 + k] = mean ? (0.f - mean[k]) / (stdv[k] + eps) : 0.f;
    } else {
      for (int k = tid; k < 513; k += kFftThreads)
        reinterpret_cast<float2*>(out)[((int64_t)b * 513 + k) * t_max + t] = make_float2(0.f, 0.f);
    }
    return;
  }

#pragma unroll
  for (int q = 0; q < kFftTwStage / kFftThreads; ++q)
    stw[tid + q * kFftThreads] = tw_g[kFftTwHann + tid + q * kFftThreads];

  const int n = n_samples[b];
  const float* x = wave + (int64_t)b * wave_stride;
  const float pk = peak ? peak[b] : 1.0f;
  const bool norm = peak != nullptr;
  __syncthreads();
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int i = tid + q * kFftThreads;
    // periodic Hann: 0.5 - 0.5*cos(2*pi*i/1024); cos from the twiddle table
    const float c = (i < 512) ? __ldg(&tw_g[i].x) : -__ldg(&tw_g[i - 512].x);
    const float w = 0.5f - 0.5f * c;
    const int i0 = t * 256 + i;
    float v0 = (i0 < n) ? x[i0] : 0.f;  // samples past the end are the pad-at-end zeros
    if (norm) v0 = __fdiv_rn(v0, pk);
    sa[i] = make_float2(v0 * w, 0.f);
  }
  __syncthreads();
  const float2* spec = fft1024_smem(sa, sb, stw, tid);

  for (int k = tid; k < 513; k += kFftThreads) {
    const float2 z = spec[k];
    if (MODE == 0) {
      const float la = logf(z.x * z.x + z.y * z.y + eps);
      out[((int64_t)b * t_max + t) * 513 + k] = mean ? (la - mean[k]) / (stdv[k] + eps) : la;
    } else {
      reinterpret_cast<float2*>(out)[((int64_t)b * 513 + k) * t_max + t] = z;
    }
  }
}

// ---- log-power front end on the register FFT (fft_reg.cuh) -------------------------------------------------------
// Same arithmetic per sample and per bin as frontend_kernel<0> (window from the same twiddle table, __fdiv_rn peak
// normalisation, logf, standardisation), one frame per transform as before (a frame's features never depend on which
// other frames share the launch), but a frame is a 64-thread group with the radix-16 butterflies in registers, CTAs are
// persistent and stage the twiddle tables, the window and the per-bin statistics once instead of 8 KB per frame.
constexpr int kFeGroups = 4;
struct FeSmem {
  float2 buf[kFeGroups][kRfBufEntries];
  float2 twB[kFftTwB];
  float2 twC[kFftTwC];
  float win[kFftN];
  float mean[520];
  float stdv[520];
};

// Output modes of frontend_reg_kernel.  FeOutF32: standardised fp32 rows (B, t_max, 513).  FeOutBf16: the same values
// rounded to bf16 (__float2bfloat16_rn), written straight into an LSTM layer-0 operand of leading dimension `ld` from
// column `col_off` on, with the columns [col_off + 513, ld) of every row zeroed (== the fp32 rows through
// pack_rows_bf16(zero_tail = 1), without the fp32 round trip through HBM).
struct FeOutF32 {
  float* __restrict__ p;
  __device__ float* row(int64_t f) const { return p + f * 513; }
  __device__ static void put(float* o, int k, float v) { o[k] = v; }
  __device__ void tail(float*, int) const {}
};
struct FeOutBf16 {
  __nv_bfloat16* __restrict__ p;
  int64_t ld, col_off;
  __device__ __nv_bfloat16* row(int64_t f) const { return p + f * ld + col_off; }
  __device__ static void put(__nv_bfloat16* o, int k, float v) { o[k] = __float2bfloat16_rn(v); }
  __device__ void tail(__nv_bfloat16* o, int t) const {
    for (int64_t k = 513 + t; k < ld - col_off; k += kRfThreads) o[k] = __float2bfloat16_rn(0.f);
  }
};

template <class Out>
__global__ void __launch_bounds__(kFeGroups * kRfThreads, 3)
frontend_reg_kernel(const float* __restrict__ wave, int64_t wave_stride, const int32_t* __restrict__ n_samples,
                    const int32_t* __restrict__ n_frames, int B, int t_max, const float* __restrict__ peak,
                    const float* __restrict__ mean, const float* __restrict__ stdv, float eps,
                    const float2* __restrict__ tw_g, Out out) {
  extern __shared__ __align__(16) uint8_t fe_smem_raw[];
  FeSmem& sm = *reinterpret_cast<FeSmem*>(fe_smem_raw);
  const int tid = threadIdx.x;
  const int g = tid >> 6, t = tid & 63;
  const int bar_id = 1 + g;
  for (int i = tid; i < kFftTwB; i += blockDim.x) sm.twB[i] = tw_g[kFftTwHann + kFftTwStage + i];
  for (int i = tid; i < kFftTwC; i += blockDim.x) sm.twC[i] = tw_g[kFftTwHann + fft_tw_off(4) + i];
  for (int i = tid; i < kFftN; i += blockDim.x) {
    // periodic Hann: 0.5 - 0.5*cos(2*pi*i/1024); cos from the twiddle table
    const float c = (i < 512) ? tw_g[i].x : -tw_g[i - 512].x;
    sm.win[i] = 0.5f - 0.5f * c;
  }
  for (int i = tid; i < 513; i += blockDim.x) {
    sm.mean[i] = mean ? mean[i] : 0.f;
    sm.stdv[i] = mean ? stdv[i] : 0.f;
  }
  __syncthreads();
  const bool has_stats = mean != nullptr;
  const bool norm = peak != nullptr;
  float2* buf = sm.buf[g];
  const int64_t frames = (int64_t)B * t_max;
  for (int64_t f = (int64_t)blockIdx.x * kFeGroups + g; f < frames; f += (int64_t)gridDim.x * kFeGroups) {
    const int b = (int)(f / t_max), fr = (int)(f - (int64_t)b * t_max);
    auto* o = out.row(f);
    out.tail(o, t);
    if (fr >= min(n_frames[b], t_max)) {
      // collate padding: zeros are padded BEFORE standardisation -> (0 - mean) / (std + eps)
      for (int k = t; k < 513; k += kRfThreads)
        Out::put(o, k, has_stats ? (0.f - sm.mean[k]) / (sm.stdv[k] + eps) : 0.f);
      continue;
    }
    const int n = n_samples[b];
    const float* x = wave + (int64_t)b * wave_stride;
    const float pk = norm ? peak[b] : 1.0f;
    float2 v[16];
#pragma unroll
    for (int m = 0; m < 16; ++m) {
      const int i = t + 64 * m;
      const int i0 = fr * 256 + i;
      float v0 = (i0 < n) ? x[i0] : 0.f;  // samples past the end are the pad-at-end zeros
      if (norm) v0 = __fdiv_rn(v0, pk);
      v[m] = make_float2(v0 * sm.win[i], 0.f);
    }
    fft1024_reg(v, buf, sm.twB, sm.twC, t, bar_id);
#pragma unroll
    for (int m = 0; m <= 8; ++m) {
      const int k = t + 64 * m;
      if (k <= 512) {
        const float la = logf(v[m].x * v[m].x + v[m].y * v[m].y + eps);
        Out::put(o, k, has_stats ? (la - sm.mean[k]) / (sm.stdv[k] + eps) : la);
      }
    }
  }
}

}  // namespace avvad

using namespace avvad;

extern "C" int64_t avvad_stft_num_frames(int64_t n_samples, double fs, double wlen_sec, double hop_percent,
                                         int pad_at_end) {
  // stft.py:123-139, same double-precision expressions in the same order
  if (wlen_sec * fs != (double)(int64_t)(wlen_sec * fs)) return -1;
  const int64_t nfft = (int64_t)(wlen_sec * fs);
  const int64_t hop = (int64_t)(hop_percent * (double)nfft);
  int64_t n = n_samples;
  if (pad_at_end) {
    const double utt_len = (double)n_samples / fs;
    const double q = utt_len / wlen_sec / hop_percent;
    if (ceil(q) != (double)(int64_t)q) n += hop;
  }
  if (n < nfft || hop <= 0) return 0;
  return 1 + (n - nfft) / hop;
}

template <class Out>
static int launch_frontend_reg(const float* wave, int64_t wave_stride, const int32_t* n_samples,
                               const int32_t* n_frames, int32_t B, int32_t t_max, const float* peak,
                               const float* mean, const float* stdv, float eps, const float2* tw, Out out,
                               cudaStream_t st) {
  static PerDeviceOnce attr_once;
  int sms = 0, dev = 0;
  AVVAD_CUDA(cudaGetDevice(&dev));
  AVVAD_CUDA(attr_once.run([] {
    return cudaFuncSetAttribute(frontend_reg_kernel<Out>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)sizeof(FeSmem));
  }));
  AVVAD_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int64_t want = ceil_div((int64_t)B * t_max, (int64_t)kFeGroups);
  const unsigned ctas = (unsigned)std::min<int64_t>(want, (int64_t)sms * 3);
  frontend_reg_kernel<Out><<<ctas, kFeGroups * kRfThreads, sizeof(FeSmem), st>>>(
      wave, wave_stride, n_samples, n_frames, B, t_max, peak, mean, stdv, eps, tw, out);
  return AVVAD_OK;
}

// out_bf16 != NULL (mode 0 only): bf16 operand rows (FeOutBf16) on the register-FFT kernel, whatever AVVAD_FE_REG says.
static int launch_frontend(int mode, const float* wave, int64_t wave_stride, const int32_t* n_samples,
                           const int32_t* n_frames, int32_t B, int32_t t_max, int normalise,
                           const float* mean, const float* stdv, float eps, float* out,
                           float* peak_scratch, cudaStream_t st, void* out_bf16 = nullptr, int64_t ld = 0,
                           int64_t col_off = 0) {
  AVVAD_CHECK_ARG(wave && n_samples && n_frames && (out || out_bf16), "null pointer");
  AVVAD_CHECK_ARG(B > 0 && t_max > 0 && wave_stride > 0, "B, t_max, wave_stride must be positive");
  AVVAD_CHECK_ARG(!out_bf16 || (col_off >= 0 && ld % 8 == 0 && ld >= col_off + 513),
                  "bf16 output: ld must be a multiple of 8 and at least col_off + 513, col_off >= 0");
  AVVAD_CHECK_ARG((mean == nullptr) == (stdv == nullptr), "mean and std must both be given or both NULL");
  AVVAD_CHECK_ARG(normalise >= 0 && normalise <= 2, "normalise must be 0, 1 or 2");
  AVVAD_CHECK_ARG(!normalise || peak_scratch, "peak_scratch required when normalise != 0");
  const float2* tw = fft_twiddles_device();
  if (!tw) {
    set_error("twiddle table allocation failed (no CUDA device?)");
    return AVVAD_ERR_CUDA;
  }
  // profiling category 4 (bench.py: achieved HBM GB/s of the memory-bound stages); "flops" carries the algorithmic bytes:
  // 256 new samples in + 513 (x2 for the raw STFT) floats out per frame (SURVEY 8d)
  void* ptok = nullptr;
  tc::prof_begin(st, &ptok);
  if (normalise == 1) {  // 2: peak_scratch already holds the caller's peaks
    AVVAD_CUDA(cudaMemsetAsync(peak_scratch, 0, sizeof(float) * B, st));
    int chunks = (int)std::min<int64_t>(64, ceil_div(wave_stride, 256 * 16));
    absmax_kernel<<<dim3(chunks, B), 256, 0, st>>>(wave, wave_stride, n_samples, peak_scratch);
    AVVAD_LAUNCHED();
  }
  dim3 grid(t_max, B);
  static int reg_mode = -1;  // AVVAD_FE_REG=0: log-power frames through the radix-4 shared-memory kernel as well
  if (reg_mode < 0) {
    const char* e = getenv("AVVAD_FE_REG");
    reg_mode = (e && e[0] == '0') ? 0 : 1;
  }
  const float* peak = normalise ? peak_scratch : nullptr;
  if (mode == 0 && out_bf16) {
    const int rc = launch_frontend_reg(wave, wave_stride, n_samples, n_frames, B, t_max, peak, mean, stdv, eps, tw,
                                       FeOutBf16{(__nv_bfloat16*)out_bf16, ld, col_off}, st);
    if (rc) return rc;
  } else if (mode == 0 && reg_mode) {
    const int rc = launch_frontend_reg(wave, wave_stride, n_samples, n_frames, B, t_max, peak, mean, stdv, eps, tw,
                                       FeOutF32{out}, st);
    if (rc) return rc;
  } else if (mode == 0)
    frontend_kernel<0><<<grid, kFftThreads, 0, st>>>(wave, wave_stride, n_samples, n_frames, t_max,
                                                     normalise ? peak_scratch : nullptr, mean, stdv, eps, tw, out);
  else
    frontend_kernel<1><<<grid, kFftThreads, 0, st>>>(wave, wave_stride, n_samples, n_frames, t_max, nullptr,
                                                     nullptr, nullptr, 0.f, tw, out);
  AVVAD_LAUNCHED();
  const double out_bytes = out_bf16 ? 2.0 * (double)(ld - col_off) : (mode == 0 ? 2052.0 : 4104.0);
  tc::prof_end(st, ptok, 4, (double)B * t_max * (1024.0 + out_bytes));
  return AVVAD_OK;
}

extern "C" int avvad_frontend_logpower(const float* wave, int64_t wave_stride, const int32_t* n_samples,
                                       const int32_t* n_frames, int32_t B, int32_t t_max, int normalise,
                                       const float* mean, const float* stdv, float eps, float* out,
                                       float* peak_scratch, void* stream) {
  return launch_frontend(0, wave, wave_stride, n_samples, n_frames, B, t_max, normalise, mean, stdv, eps, out,
                         peak_scratch, (cudaStream_t)stream);
}

extern "C" int avvad_frontend_logpower_bf16(const float* wave, int64_t wave_stride, const int32_t* n_samples,
                                            const int32_t* n_frames, int32_t B, int32_t t_max, int normalise,
                                            const float* mean, const float* stdv, float eps, void* out_bf16,
                                            int64_t ld, int64_t col_off, float* peak_scratch, void* stream) {
  AVVAD_CHECK_ARG(out_bf16, "null pointer");
  return launch_frontend(0, wave, wave_stride, n_samples, n_frames, B, t_max, normalise, mean, stdv, eps, nullptr,
                         peak_scratch, (cudaStream_t)stream, out_bf16, ld, col_off);
}

extern "C" int avvad_stft(const float* wave, int64_t wave_stride, const int32_t* n_samples,
                          const int32_t* n_frames, int32_t B, int32_t t_max, float* out_ft2, void* stream) {
  return launch_frontend(1, wave, wave_stride, n_samples, n_frames, B, t_max, 0, nullptr, nullptr, 0.f, out_ft2,
                         nullptr, (cudaStream_t)stream);
}
