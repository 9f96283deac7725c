// WaveNet-style encoder (SURVEY §8a row W1): valid (un-padded) dilated Conv1d stack on the tcgen05 GEMM engine.
//
// Reference semantics: packages/models/wavenet_autoencoder.py:74-93
//   s = Conv1d(q->R,k)(x); for d in dilations: cur = s; s = Conv1d(D->R,1)(relu(Conv1d(R->D,k,dilation=d)(relu(s)))) +
//   cur[..., -L_out:]; s = relu(Conv1d(R->bottleneck,1)(s)); AdaptiveAvgPool1d(pool)(s)
// Mapping: activations are time-major rows [B*L][C padded to 64]; every convolution is a GEMM whose A rows are
// gathered (k dilated taps side by side, optional ReLU, fp32 -> bf16) by a bandwidth kernel; bias / ReLU are fused
// in the GEMM epilogue; the residual stream stays fp32.
#include <vector>

#include <stdlib.h>

#include "wavenet_fused.cuh"

namespace avvad {

static inline int pad64(int c) { return (c + 63) / 64 * 64; }

// W [O][I][k] f32 (torch Conv1d) -> bf16 [Op][k*Ip], column j*Ip + i; zero padding everywhere else
__global__ void wn_pack_w_kernel(const float* __restrict__ w, int O, int I, int k, int Op, int Ip,
                                 __nv_bfloat16* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)Op * k * Ip;
  if (idx >= total) return;
  const int col = (int)(idx % (k * Ip)), o = (int)(idx / (k * Ip));
  const int j = col / Ip, i = col - j * Ip;
  out[idx] = __float2bfloat16_rn((o < O && i < I) ? w[((int64_t)o * I + i) * k + j] : 0.f);
}
__global__ void wn_pack_b_kernel(const float* __restrict__ b, int O, int Op, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < Op) out[i] = (b && i < O) ? b[i] : 0.f;
}
// x (B, C, N) channel-major f32 -> A[b*Lout + t][j*Cp + c] = x[b][c][t + j]   (first, causal layer; dilation 1)
__global__ void wn_gather_cm_kernel(const float* __restrict__ x, int B, int C, int N, int k, int Lout, int Cp,
                                    __nv_bfloat16* __restrict__ A) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)B * Lout * k * Cp;
  if (idx >= total) return;
  const int c = (int)(idx % Cp);
  const int j = (int)((idx / Cp) % k);
  const int64_t row = idx / ((int64_t)Cp * k);
  const int t = (int)(row % Lout), b = (int)(row / Lout);
  A[idx] = __float2bfloat16_rn(c < C ? x[((int64_t)b * C + c) * N + t + j] : 0.f);
}
// s [B][Lin][Cp] f32 -> A[b*Lout + t][j*Cp + c] = act(s[b][t + j*dil][c])
__global__ void wn_gather_kernel(const float* __restrict__ s, int B, int Lin, int Cp, int k, int dil, int Lout, int relu,
                                 __nv_bfloat16* __restrict__ A) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)B * Lout * k * Cp;
  if (idx >= total) return;
  const int c = (int)(idx % Cp);
  const int j = (int)((idx / Cp) % k);
  const int64_t row = idx / ((int64_t)Cp * k);
  const int t = (int)(row % Lout), b = (int)(row / Lout);
  float v = s[((int64_t)b * Lin + t + j * dil) * Cp + c];
  if (relu) v = fmaxf(v, 0.f);
  A[idx] = __float2bfloat16_rn(v);
}
// out[b][t][c] = dense[b][t][c] + cur[b][t + (Lin - Lout)][c]
__global__ void wn_add_slice_kernel(const float* __restrict__ dense, const float* __restrict__ cur, int B, int Lin,
                                    int Lout, int Cp, float* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)B * Lout * Cp;
  if (idx >= total) return;
  const int c = (int)(idx % Cp);
  const int64_t row = idx / Cp;
  const int t = (int)(row % Lout), b = (int)(row / Lout);
  out[idx] = dense[idx] + cur[((int64_t)b * Lin + t + (Lin - Lout)) * Cp + c];
}
// fused path: all weight matrices as one stack of SW128-loadable [64][64] tiles (tap j of a layer = columns j*64.. of its
// packed [64][k*64] matrix), in the order causal taps | per layer: dilated taps, dense | bottleneck
__global__ void wn_stack_tile_kernel(const __nv_bfloat16* __restrict__ w, int k_cols, int tap, __nv_bfloat16* __restrict__ tile) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * 64) return;
  const int o = idx >> 6, i = idx & 63;
  tile[idx] = w[(int64_t)o * k_cols + tap * 64 + i];
}
// AdaptiveAvgPool1d: out[b][c][p] = mean_{t in [floor(p L / P), ceil((p+1) L / P))} s[b][t][c]
__global__ void wn_pool_kernel(const float* __restrict__ s, int B, int L, int Cp, int C, int P, float* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * C * P) return;
  const int p = idx % P, c = (idx / P) % C, b = idx / (P * C);
  const int t0 = (int)(((int64_t)p * L) / P);
  const int t1 = (int)((((int64_t)(p + 1)) * L + P - 1) / P);
  float acc = 0.f;
  for (int t = t0; t < t1; ++t) acc += s[((int64_t)b * L + t) * Cp + c];
  out[idx] = acc / (float)(t1 - t0);
}

}  // namespace avvad

using namespace avvad;

struct WnLayer {
  __nv_bfloat16* w = nullptr;
  float* b = nullptr;
  bool set = false;
};
struct avvad_wavenet {
  int k, q, R, D, bott, pool;
  int qp, Rp, Dp, bp;
  std::vector<int> dil;
  WnLayer causal, bottleneck;
  std::vector<WnLayer> dilated, dense;
  // fused kernel (wavenet_fused.cuh): stacked weight tiles / biases, rebuilt after any set_layer
  __nv_bfloat16* wstack = nullptr;
  float* bstack = nullptr;
  bool stack_ready = false;
};

namespace avvad {
namespace tc {
int encode_weight_map(CUtensorMap* m, const void* ptr, uint64_t K, uint64_t N, uint32_t bn);
bool tma_available();
}  // namespace tc
}  // namespace avvad

static bool wn_fused_enabled() {
  static int v = [] {
    const char* e = getenv("AVVAD_WAVENET_FUSED");
    return (e && atoi(e) == 0) ? 0 : 1;
  }();
  return v != 0;
}
// The fused kernel holds one 64-channel block per tensor and 256 working rows of history per tile.
static bool wn_fused_supported(const avvad_wavenet* h) {
  if (!wn_fused_enabled() || !tc::tma_available()) return false;
  if (h->qp != 64 || h->Rp != 64 || h->Dp != 64 || h->bp != 64) return false;
  if (h->k < 1 || h->k > tc::kWnMaxK || (int)h->dil.size() > tc::kWnMaxLayers) return false;
  int64_t sum = 0;
  for (int d : h->dil) {
    if ((int64_t)(h->k - 1) * d > 128) return false;
    sum += (int64_t)(h->k - 1) * d;
  }
  return sum + h->k <= tc::kWnWork - 1;
}

static int alloc_layer(WnLayer& l, int Op, int K) {
  AVVAD_CUDA(cudaMalloc(&l.w, sizeof(__nv_bfloat16) * (size_t)Op * K));
  AVVAD_CUDA(cudaMalloc(&l.b, sizeof(float) * Op));
  return AVVAD_OK;
}

extern "C" int avvad_wavenet_create(avvad_wavenet** out, int filter_width, int quantization_channel,
                                    const int32_t* dilations, int n_dilations, int residual_channel,
                                    int dilation_channel, int bottleneck_width, int pool_size) {
  AVVAD_CHECK_ARG(out && dilations && n_dilations > 0 && filter_width >= 1, "bad argument");
  AVVAD_CHECK_ARG(quantization_channel > 0 && residual_channel > 0 && dilation_channel > 0 && bottleneck_width > 0 &&
                      pool_size > 0, "bad channel counts");
  avvad_wavenet* h = new avvad_wavenet();
  h->k = filter_width; h->q = quantization_channel; h->R = residual_channel; h->D = dilation_channel;
  h->bott = bottleneck_width; h->pool = pool_size;
  h->qp = pad64(h->q); h->Rp = pad64(h->R); h->Dp = pad64(h->D); h->bp = pad64(h->bott);
  h->dil.assign(dilations, dilations + n_dilations);
  h->dilated.resize(n_dilations);
  h->dense.resize(n_dilations);
  int rc = alloc_layer(h->causal, h->Rp, h->k * h->qp);
  if (rc) return rc;
  rc = alloc_layer(h->bottleneck, h->bp, h->Rp);
  if (rc) return rc;
  for (int i = 0; i < n_dilations; ++i) {
    rc = alloc_layer(h->dilated[i], h->Dp, h->k * h->Rp);
    if (rc) return rc;
    rc = alloc_layer(h->dense[i], h->Rp, h->Dp);
    if (rc) return rc;
  }
  *out = h;
  return AVVAD_OK;
}

extern "C" void avvad_wavenet_destroy(avvad_wavenet* h) {
  if (!h) return;
  auto fr = [](WnLayer& l) { cudaFree(l.w); cudaFree(l.b); };
  cudaFree(h->wstack);
  cudaFree(h->bstack);
  fr(h->causal); fr(h->bottleneck);
  for (auto& l : h->dilated) fr(l);
  for (auto& l : h->dense) fr(l);
  delete h;
}

// kind: 0 = en_causal_layer, 1 = en_dilation_layer_stack[index], 2 = en_dense_layer_stack[index], 3 = bottleneck_layer
// w: torch Conv1d weight [O][I][k] f32; bias [O] f32 or NULL (use_bias=False)
extern "C" int avvad_wavenet_set_layer(avvad_wavenet* h, int kind, int index, const float* w, const float* bias,
                                       void* stream) {
  AVVAD_CHECK_ARG(h && w && kind >= 0 && kind <= 3, "bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  WnLayer* l = nullptr;
  int O = 0, I = 0, k = 1, Op = 0, Ip = 0;
  if (kind == 0) { l = &h->causal; O = h->R; I = h->q; k = h->k; Op = h->Rp; Ip = h->qp; }
  if (kind == 3) { l = &h->bottleneck; O = h->bott; I = h->R; k = 1; Op = h->bp; Ip = h->Rp; }
  if (kind == 1 || kind == 2) {
    AVVAD_CHECK_ARG(index >= 0 && index < (int)h->dil.size(), "bad layer index");
    if (kind == 1) { l = &h->dilated[index]; O = h->D; I = h->R; k = h->k; Op = h->Dp; Ip = h->Rp; }
    else { l = &h->dense[index]; O = h->R; I = h->D; k = 1; Op = h->Rp; Ip = h->Dp; }
  }
  const int64_t total = (int64_t)Op * k * Ip;
  wn_pack_w_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(w, O, I, k, Op, Ip, l->w);
  AVVAD_LAUNCHED();
  wn_pack_b_kernel<<<(unsigned)ceil_div(Op, 256), 256, 0, st>>>(bias, O, Op, l->b);
  AVVAD_LAUNCHED();
  l->set = true;
  h->stack_ready = false;
  return AVVAD_OK;
}

static int64_t wn_out_len(const avvad_wavenet* h, int64_t N) {
  int64_t L = N - (h->k - 1);
  for (int d : h->dil) L -= (int64_t)(h->k - 1) * d;
  return L;
}

extern "C" int64_t avvad_wavenet_encoded_length(const avvad_wavenet* h, int64_t n_samples) {
  return h ? wn_out_len(h, n_samples) : 0;
}

extern "C" size_t avvad_wavenet_workspace_bytes(const avvad_wavenet* h, int64_t B, int64_t N) {
  if (!h || B <= 0 || N < h->k) return 0;
  const int64_t L0 = N - (h->k - 1);
  const int maxC = std::max(std::max(h->qp, h->Rp), std::max(h->Dp, h->bp));
  const size_t rows = (size_t)B * L0;
  // gather buffer (bf16, k*maxC wide), dilated activation (bf16), two fp32 streams + one fp32 temp
  return align_up(rows * h->k * maxC * 2, 256) + align_up(rows * maxC * 2, 256) + 3 * align_up(rows * maxC * 4, 256) + 1024;
}

// Training tape: S_i = the input of dilated layer i (i = 0..n; S_n feeds the bottleneck) as bf16 [B][L_i][Rp], back to
// back; act_i = relu(dilated_i + bias) as bf16 [B][L_{i+1}][Dp], back to back; the bottleneck output relu(...) as f32
// [B][L_n][bp] (the tensor the pool reads).  bf16(relu(S_i)) is exactly the operand the forward fed to dilated layer i
// (ReLU commutes with round-to-nearest), and bf16 keeps fp32's exponent range, so the ReLU masks survive the rounding.
struct WnTape {
  std::vector<int64_t> L;   // L[i] = rows per item of S_i
  std::vector<__nv_bfloat16*> S, act;
  float* out = nullptr;
  size_t bytes = 0;
};
static WnTape wn_tape(const avvad_wavenet* h, int64_t B, int64_t N, void* base) {
  WnTape t;
  const int n = (int)h->dil.size();
  t.L.resize(n + 1);
  t.L[0] = N - (h->k - 1);
  for (int i = 0; i < n; ++i) t.L[i + 1] = t.L[i] - (int64_t)(h->k - 1) * h->dil[i];
  uint8_t* p = (uint8_t*)base;
  size_t off = 0;
  for (int i = 0; i <= n; ++i) {
    t.S.push_back(p ? (__nv_bfloat16*)(p + off) : nullptr);
    off += (size_t)B * t.L[i] * h->Rp * 2;
  }
  off = align_up(off, 256);
  for (int i = 0; i < n; ++i) {
    t.act.push_back(p ? (__nv_bfloat16*)(p + off) : nullptr);
    off += (size_t)B * t.L[i + 1] * h->Dp * 2;
  }
  off = align_up(off, 256);
  t.out = p ? (float*)(p + off) : nullptr;
  t.bytes = off + align_up((size_t)B * t.L[n] * h->bp * 4, 256);
  return t;
}

extern "C" size_t avvad_wavenet_tape_bytes(const avvad_wavenet* h, int64_t B, int64_t N) {
  if (!h || B <= 0 || wn_out_len(h, N) < 1) return 0;
  return wn_tape(h, B, N, nullptr).bytes;
}

static int wn_gemm(const __nv_bfloat16* A, int K, const WnLayer& l, int N, void* C, int ldc, bool c_bf16, bool relu,
                   int64_t M, cudaStream_t st) {
  return avvad_gemm_bf16(A, K, l.w, K, l.b, C, ldc, c_bf16 ? 1 : 0, relu ? 1 : 0, M, N, K, st);
}

static int wn_check(const avvad_wavenet* h, int64_t N) {
  AVVAD_CHECK_ARG(wn_out_len(h, N) >= 1, "input shorter than the receptive field");
  if (!h->causal.set || !h->bottleneck.set) { set_error("wavenet: layers not loaded"); return AVVAD_ERR_STATE; }
  for (size_t i = 0; i < h->dil.size(); ++i)
    if (!h->dilated[i].set || !h->dense[i].set) { set_error("wavenet: layers not loaded"); return AVVAD_ERR_STATE; }
  return AVVAD_OK;
}

template <bool kTape>
static int wn_launch_fused(const tc::WnFusedGeom& g, const CUtensorMap& wmap, int k, int64_t B, cudaStream_t st) {
  const size_t smem = tc::wavenet_fused_smem_bytes(k);
  static PerDeviceOnce once;
  const cudaError_t ae = once.run([] {
    return cudaFuncSetAttribute(tc::wavenet_fused_kernel<kTape>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)tc::wavenet_fused_smem_bytes(tc::kWnMaxK));
  });
  if (ae != cudaSuccess) { set_error(std::string("cudaFuncSetAttribute(wavenet): ") + cudaGetErrorString(ae)); return AVVAD_ERR_CUDA; }
  tc::wavenet_fused_kernel<kTape><<<(unsigned)(B * g.tiles_per_item), tc::kWnThreads, smem, st>>>(wmap, g);
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}

// The forward of both entry points; with a tape (training) it also stores what the backward reads.  The values
// computed are the same either way.
static int wn_encode(avvad_wavenet* h, const float* x, int64_t B, int64_t N, void* workspace, const WnTape* tape,
                     float* out, cudaStream_t st) {
  const int64_t Lfinal = wn_out_len(h, N);
  if (wn_fused_supported(h)) {
    // ---- fused path: one kernel for the whole stack, history in shared memory (wavenet_fused.cuh) ----
    const int n = (int)h->dil.size(), k = h->k;
    const int n_tiles = k + n * (k + 1) + 1;
    if (!h->stack_ready) {
      if (!h->wstack) {
        AVVAD_CUDA(cudaMalloc(&h->wstack, (size_t)n_tiles * 64 * 64 * sizeof(__nv_bfloat16)));
        AVVAD_CUDA(cudaMalloc(&h->bstack, (size_t)(2 + 2 * n) * 64 * sizeof(float)));
      }
      int t = 0;
      auto put = [&](const WnLayer& l, int taps) -> int {
        for (int j = 0; j < taps; ++j, ++t) {
          wn_stack_tile_kernel<<<16, 256, 0, st>>>(l.w, taps * 64, j, h->wstack + (size_t)t * 4096);
          AVVAD_LAUNCHED();
        }
        return AVVAD_OK;
      };
      int rc = put(h->causal, k);
      if (rc) return rc;
      AVVAD_CUDA(cudaMemcpyAsync(h->bstack, h->causal.b, 64 * sizeof(float), cudaMemcpyDeviceToDevice, st));
      for (int i = 0; i < n; ++i) {
        rc = put(h->dilated[i], k);
        if (rc) return rc;
        rc = put(h->dense[i], 1);
        if (rc) return rc;
        AVVAD_CUDA(cudaMemcpyAsync(h->bstack + (1 + 2 * i) * 64, h->dilated[i].b, 64 * sizeof(float),
                                   cudaMemcpyDeviceToDevice, st));
        AVVAD_CUDA(cudaMemcpyAsync(h->bstack + (2 + 2 * i) * 64, h->dense[i].b, 64 * sizeof(float),
                                   cudaMemcpyDeviceToDevice, st));
      }
      rc = put(h->bottleneck, 1);
      if (rc) return rc;
      AVVAD_CUDA(cudaMemcpyAsync(h->bstack + (1 + 2 * n) * 64, h->bottleneck.b, 64 * sizeof(float),
                                 cudaMemcpyDeviceToDevice, st));
      h->stack_ready = true;
    }
    tc::WnFusedGeom g{};
    g.B = (int)B; g.q = h->q; g.N = (int)N; g.k = k; g.n_layers = n;
    int sum = 0;
    for (int i = 0; i < n; ++i) {
      g.dil[i] = h->dil[i];
      sum += (k - 1) * h->dil[i];
    }
    g.sum_shift = sum;
    g.lt = tc::kWnWork - sum - (k - 1);
    g.L_final = (int)Lfinal;
    g.tiles_per_item = (int)ceil_div(Lfinal, g.lt);
    g.x = x;
    g.bias = h->bstack;
    // [B][L_final][64] fp32 (fits: the workspace holds 3 fp32 streams); the tape's copy when training
    float* act = tape ? tape->out : reinterpret_cast<float*>(workspace);
    g.out = act;
    if (tape) {
      g.tape_s = tape->S[0];
      g.tape_act = n > 0 ? tape->act[0] : nullptr;
    }
    CUtensorMap wmap;
    int rc = tc::encode_weight_map(&wmap, h->wstack, 64, (uint64_t)n_tiles * 64, 64);
    if (rc) return rc;
    rc = tape ? wn_launch_fused<true>(g, wmap, k, B, st) : wn_launch_fused<false>(g, wmap, k, B, st);
    if (rc) return rc;
    const int np = (int)(B * h->bott * h->pool);
    wn_pool_kernel<<<(unsigned)ceil_div(np, 128), 128, 0, st>>>(act, (int)B, (int)Lfinal, 64, h->bott, h->pool, out);
    AVVAD_LAUNCHED();
    return AVVAD_OK;
  }
  const int64_t L0 = N - (h->k - 1);
  const int maxC = std::max(std::max(h->qp, h->Rp), std::max(h->Dp, h->bp));
  const size_t rows0 = (size_t)B * L0;
  uint8_t* p = (uint8_t*)workspace;
  __nv_bfloat16* A = (__nv_bfloat16*)p;          p += align_up(rows0 * h->k * maxC * 2, 256);
  __nv_bfloat16* act = (__nv_bfloat16*)p;        p += align_up(rows0 * maxC * 2, 256);
  float* s0 = (float*)p;                         p += align_up(rows0 * maxC * 4, 256);
  float* s1 = (float*)p;                         p += align_up(rows0 * maxC * 4, 256);
  float* tmp = (float*)p;

  // causal layer
  {
    const int64_t tot = (int64_t)B * L0 * h->k * h->qp;
    wn_gather_cm_kernel<<<(unsigned)ceil_div(tot, 256), 256, 0, st>>>(x, (int)B, h->q, (int)N, h->k, (int)L0, h->qp, A);
    AVVAD_LAUNCHED();
    int rc = wn_gemm(A, h->k * h->qp, h->causal, h->Rp, s0, h->Rp, false, false, B * L0, st);
    if (rc) return rc;
    if (tape) {
      rc = avvad_pack_rows_bf16(s0, h->Rp, tape->S[0], h->Rp, 0, B * L0, h->Rp, 0, st);
      if (rc) return rc;
    }
  }
  float* cur = s0;
  float* nxt = s1;
  int64_t L = L0;
  for (size_t i = 0; i < h->dil.size(); ++i) {
    const int d = h->dil[i];
    const int64_t Lo = L - (int64_t)(h->k - 1) * d;
    const int64_t tot = (int64_t)B * Lo * h->k * h->Rp;
    wn_gather_kernel<<<(unsigned)ceil_div(tot, 256), 256, 0, st>>>(cur, (int)B, (int)L, h->Rp, h->k, d, (int)Lo, 1, A);
    AVVAD_LAUNCHED();
    __nv_bfloat16* act_i = tape ? tape->act[i] : act;
    int rc = wn_gemm(A, h->k * h->Rp, h->dilated[i], h->Dp, act_i, h->Dp, true, true, B * Lo, st);  // conv + ReLU
    if (rc) return rc;
    rc = wn_gemm(act_i, h->Dp, h->dense[i], h->Rp, tmp, h->Rp, false, false, B * Lo, st);
    if (rc) return rc;
    const int64_t tot2 = (int64_t)B * Lo * h->Rp;
    wn_add_slice_kernel<<<(unsigned)ceil_div(tot2, 256), 256, 0, st>>>(tmp, cur, (int)B, (int)L, (int)Lo, h->Rp, nxt);
    AVVAD_LAUNCHED();
    if (tape) {
      rc = avvad_pack_rows_bf16(nxt, h->Rp, tape->S[i + 1], h->Rp, 0, B * Lo, h->Rp, 0, st);
      if (rc) return rc;
    }
    float* t = cur; cur = nxt; nxt = t;
    L = Lo;
  }
  {
    const int64_t tot = (int64_t)B * L * h->Rp;
    wn_gather_kernel<<<(unsigned)ceil_div(tot, 256), 256, 0, st>>>(cur, (int)B, (int)L, h->Rp, 1, 1, (int)L, 0, A);
    AVVAD_LAUNCHED();
    float* z = tape ? tape->out : tmp;
    int rc = wn_gemm(A, h->Rp, h->bottleneck, h->bp, z, h->bp, false, true, B * L, st);
    if (rc) return rc;
    const int n = (int)(B * h->bott * h->pool);
    wn_pool_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, st>>>(z, (int)B, (int)L, h->bp, h->bott, h->pool, out);
    AVVAD_LAUNCHED();
  }
  return AVVAD_OK;
}

// x: f32 (B, q, N) channel-major like the reference input; out: f32 (B, bottleneck, pool)
extern "C" int avvad_wavenet_encode(avvad_wavenet* h, const float* x, int64_t B, int64_t N, void* workspace,
                                    size_t workspace_bytes, float* out, void* stream) {
  AVVAD_CHECK_ARG(h && x && workspace && out && B > 0, "bad argument");
  const int rc = wn_check(h, N);
  if (rc) return rc;
  if (workspace_bytes < avvad_wavenet_workspace_bytes(h, B, N)) { set_error("wavenet: workspace too small"); return AVVAD_ERR_WORKSPACE; }
  return wn_encode(h, x, B, N, workspace, nullptr, out, (cudaStream_t)stream);
}

extern "C" int avvad_wavenet_encode_train(avvad_wavenet* h, const float* x, int64_t B, int64_t N, void* workspace,
                                          size_t workspace_bytes, void* tape, size_t tape_bytes, float* out,
                                          void* stream) {
  AVVAD_CHECK_ARG(h && x && workspace && tape && out && B > 0, "bad argument");
  const int rc = wn_check(h, N);
  if (rc) return rc;
  if (workspace_bytes < avvad_wavenet_workspace_bytes(h, B, N)) { set_error("wavenet: workspace too small"); return AVVAD_ERR_WORKSPACE; }
  const WnTape t = wn_tape(h, B, N, tape);
  if (tape_bytes < t.bytes) { set_error("wavenet: tape too small"); return AVVAD_ERR_WORKSPACE; }
  return wn_encode(h, x, B, N, workspace, &t, out, (cudaStream_t)stream);
}

#include "wavenet_bwd.cuh"
