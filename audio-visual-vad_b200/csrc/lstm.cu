// Multi-layer unidirectional LSTM over padded (B,T,I) batches with per-sequence lengths, plus the Linear head,
// sigmoid and 0.5 threshold.
//
// Reference semantics: packages/models/AV_Net.py:127-140 (pack_padded_sequence -> nn.LSTM -> pad_packed_sequence
// -> nn.Linear), scripts/evaluate_AV_net.py:239-240.  nn.LSTM: gates i,f,g,o; c' = s(f)c + s(i)tanh(g);
// h' = s(o)tanh(c'); zero initial state; outputs for t >= len_b are exactly zero so the head emits its bias there.
//
// B200 mapping: the input projection X*W_ih^T (+b_ih+b_hh) of ALL time steps is one tcgen05 GEMM; the recurrence
// of a layer is ONE persistent cooperative kernel (lstm_persist.cuh: W_hh slice resident in shared memory, cell state
// in registers, per-CTA step flags).  When that kernel cannot run (no cooperative launch, H > 1024) every time step
// is one tcgen05 GEMM h_{t-1}*W_hh^T whose epilogue fuses the gate non-linearities, the cell update, the length mask
// and the bf16 store of h_t.  Weight rows are re-ordered gate-interleaved (row 4u+g) so that one epilogue thread owns
// all four gates of a hidden unit.
#include <stdlib.h>

#include <mutex>
#include <string>

#include <vector>

#include "lstm_persist.cuh"
#include "lstm_pair.cuh"

namespace avvad {

// W [4H][I] f32 (PyTorch gate-major: row g*H+u) -> bf16 [4H][ld] with row 4u+g, zero padded to ld
__global__ void pack_lstm_w_kernel(const float* __restrict__ w, int H, int I, int ld, __nv_bfloat16* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)4 * H * ld;
  if (idx >= total) return;
  const int np = (int)(idx / ld), j = (int)(idx - (int64_t)np * ld);
  const int u = np >> 2, g = np & 3;
  out[idx] = __float2bfloat16_rn(j < I ? w[(int64_t)(g * H + u) * I + j] : 0.f);
}
__global__ void pack_lstm_b_kernel(const float* __restrict__ b_ih, const float* __restrict__ b_hh, int H,
                                   float* __restrict__ out) {
  const int np = blockIdx.x * blockDim.x + threadIdx.x;
  if (np >= 4 * H) return;
  const int u = np >> 2, g = np & 3;
  out[np] = b_ih[g * H + u] + b_hh[g * H + u];
}
__global__ void pack_head_kernel(const float* __restrict__ w, int64_t n, float* __restrict__ w32,
                                 __nv_bfloat16* __restrict__ w16) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  w32[i] = w[i];
  w16[i] = __float2bfloat16_rn(w[i]);
}

__device__ __forceinline__ float sigmoid_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

// y_dim == 1 head: one warp per (b,t) row of the last layer's output
__global__ void head1_kernel(const __nv_bfloat16* __restrict__ hseq, int64_t rows, int H, const float* __restrict__ w,
                             const float* __restrict__ b, float* __restrict__ logits, float* __restrict__ post,
                             int32_t* __restrict__ dec) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const __nv_bfloat16* hr = hseq + row * H;
  float acc = 0.f;
  for (int j = lane * 8; j < H; j += 256) {
    const uint4 v = *reinterpret_cast<const uint4*>(hr + j);
    const float4 w0 = *reinterpret_cast<const float4*>(w + j);
    const float4 w1 = *reinterpret_cast<const float4*>(w + j + 4);
    const float2 a = unpack_bf16x2(v.x), c = unpack_bf16x2(v.y), d = unpack_bf16x2(v.z), e = unpack_bf16x2(v.w);
    acc += a.x * w0.x + a.y * w0.y + c.x * w0.z + c.y * w0.w + d.x * w1.x + d.y * w1.y + e.x * w1.z + e.y * w1.w;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) {
    const float l = acc + b[0];
    if (logits) logits[row] = l;
    const float p = sigmoid_acc(l);
    if (post) post[row] = p;
    if (dec) dec[row] = p > 0.5f ? 1 : 0;
  }
}

__global__ void post_dec_kernel(const float* __restrict__ logits, int64_t n, float* __restrict__ post,
                                int32_t* __restrict__ dec) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float p = sigmoid_acc(logits[i]);
  if (post) post[i] = p;
  if (dec) dec[i] = p > 0.5f ? 1 : 0;
}

// hlast[b][:] = hseq[b][len_b - 1][:]
__global__ void gather_last_kernel(const __nv_bfloat16* __restrict__ hseq, const int32_t* __restrict__ lengths, int T,
                                   int H, __nv_bfloat16* __restrict__ hlast) {
  const int b = blockIdx.x;
  int t = lengths[b] - 1;
  t = t < 0 ? 0 : (t >= T ? T - 1 : t);
  const uint4* src = reinterpret_cast<const uint4*>(hseq + ((int64_t)b * T + t) * H);
  uint4* dst = reinterpret_cast<uint4*>(hlast + (int64_t)b * H);
  for (int i = threadIdx.x; i < H / 8; i += blockDim.x) dst[i] = src[i];
}

// Streaming state (avvad_lstm_forward_state): the persistent recurrences run the call's steps at positions 1..T of a
// [B][T+1][H] sequence whose position 0 holds h_in, so their masks see len_b + 1
__global__ void shift_lengths_kernel(const int32_t* __restrict__ lengths, int B, int32_t* __restrict__ out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) out[b] = lengths[b] + 1;
}

// Final state of one layer: h_out[b] = hseq[b][len_b - 1 + shift], c_out[b] = cseq[b][len_b - 1 + shift] (sequences of
// Ts steps), or h_in[b] / c_in[b] (zero when null) when len_b = 0.  Every element is read and written by the same
// thread, so h_out / c_out may alias h_in / c_in.
__global__ void gather_state_kernel(const __nv_bfloat16* __restrict__ hseq, const float* __restrict__ cseq,
                                    const int32_t* __restrict__ lengths, int Ts, int shift, int H,
                                    const __nv_bfloat16* h_in, const float* c_in, __nv_bfloat16* h_out, float* c_out) {
  const int b = blockIdx.x;
  const int len = lengths[b];
  const int64_t src = ((int64_t)b * Ts + len - 1 + shift) * H;
  const int64_t dst = (int64_t)b * H;
  if (h_out) {
    for (int i = threadIdx.x; i < H / 8; i += blockDim.x) {
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (len > 0) v = reinterpret_cast<const uint4*>(hseq + src)[i];
      else if (h_in) v = reinterpret_cast<const uint4*>(h_in + dst)[i];
      reinterpret_cast<uint4*>(h_out + dst)[i] = v;
    }
  }
  if (c_out) {
    for (int i = threadIdx.x; i < H / 4; i += blockDim.x) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (len > 0) v = reinterpret_cast<const float4*>(cseq + src)[i];
      else if (c_in) v = reinterpret_cast<const float4*>(c_in + dst)[i];
      reinterpret_cast<float4*>(c_out + dst)[i] = v;
    }
  }
}

}  // namespace avvad

namespace avvad {
struct BpttGraphCache;
BpttGraphCache* bptt_cache_create();
void bptt_cache_destroy(BpttGraphCache* c);
}  // namespace avvad

using namespace avvad;

struct avvad_lstm {
  int layers, input_size, H, y_dim;
  int64_t ld0;               // padded layer-0 input width
  __nv_bfloat16* w_ih[8];    // [4H][ld_l]
  __nv_bfloat16* w_hh[8];    // [4H][H]
  float* bias[8];            // [4H] gate-interleaved, b_ih + b_hh
  float* head_w32;           // [y_dim][H]
  __nv_bfloat16* head_w16;   // [y_dim][H]
  float* head_b;             // [y_dim]
  bool set[8];
  bool head_set;
  BpttGraphCache* bptt;      // cached CUDA graphs of the backward recurrence (lstm_train.cu)
  // layer overlap (lstm_forward_impl): layer 1 follows layer 0 one chunk of time steps behind on a side stream
  cudaStream_t side = nullptr;
  int side_device = -1;
  cudaEvent_t ev_chunk[32] = {};
  cudaEvent_t ev_done = nullptr;
};

extern "C" int avvad_lstm_create(avvad_lstm** out, int layers, int input_size, int hidden, int y_dim) {
  AVVAD_CHECK_ARG(out, "null out");
  AVVAD_CHECK_ARG(layers >= 1 && layers <= 8, "1..8 layers supported");
  AVVAD_CHECK_ARG(hidden > 0 && hidden % 64 == 0, "hidden size must be a multiple of 64");
  AVVAD_CHECK_ARG(input_size > 0 && y_dim > 0, "bad sizes");
  avvad_lstm* h = new avvad_lstm();
  h->layers = layers;
  h->input_size = input_size;
  h->H = hidden;
  h->y_dim = y_dim;
  h->ld0 = (input_size + 63) / 64 * 64;
  h->head_set = false;
  h->bptt = bptt_cache_create();
  for (int l = 0; l < 8; ++l) {
    h->w_ih[l] = h->w_hh[l] = nullptr;
    h->bias[l] = nullptr;
    h->set[l] = false;
  }
  for (int l = 0; l < layers; ++l) {
    const int64_t ld = l == 0 ? h->ld0 : hidden;
    AVVAD_CUDA(cudaMalloc(&h->w_ih[l], sizeof(__nv_bfloat16) * 4 * hidden * ld));
    AVVAD_CUDA(cudaMalloc(&h->w_hh[l], sizeof(__nv_bfloat16) * 4 * hidden * (int64_t)hidden));
    AVVAD_CUDA(cudaMalloc(&h->bias[l], sizeof(float) * 4 * hidden));
  }
  AVVAD_CUDA(cudaMalloc(&h->head_w32, sizeof(float) * (int64_t)y_dim * hidden));
  AVVAD_CUDA(cudaMalloc(&h->head_w16, sizeof(__nv_bfloat16) * (int64_t)y_dim * hidden));
  AVVAD_CUDA(cudaMalloc(&h->head_b, sizeof(float) * y_dim));
  *out = h;
  return AVVAD_OK;
}

extern "C" void avvad_lstm_destroy(avvad_lstm* h) {
  if (!h) return;
  for (int l = 0; l < 8; ++l) {
    cudaFree(h->w_ih[l]);
    cudaFree(h->w_hh[l]);
    cudaFree(h->bias[l]);
  }
  cudaFree(h->head_w32);
  cudaFree(h->head_w16);
  cudaFree(h->head_b);
  bptt_cache_destroy(h->bptt);
  for (auto e : h->ev_chunk)
    if (e) cudaEventDestroy(e);
  if (h->ev_done) cudaEventDestroy(h->ev_done);
  if (h->side) cudaStreamDestroy(h->side);
  delete h;
}

extern "C" int avvad_lstm_set_layer(avvad_lstm* h, int layer, const float* w_ih, const float* w_hh, const float* b_ih,
                                    const float* b_hh, void* stream) {
  AVVAD_CHECK_ARG(h && layer >= 0 && layer < h->layers, "bad handle/layer");
  AVVAD_CHECK_ARG(w_ih && w_hh && b_ih && b_hh, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int H = h->H;
  const int I = layer == 0 ? h->input_size : H;
  const int ld = layer == 0 ? (int)h->ld0 : H;
  pack_lstm_w_kernel<<<(unsigned)ceil_div((int64_t)4 * H * ld, 256), 256, 0, st>>>(w_ih, H, I, ld, h->w_ih[layer]);
  AVVAD_LAUNCHED();
  pack_lstm_w_kernel<<<(unsigned)ceil_div((int64_t)4 * H * H, 256), 256, 0, st>>>(w_hh, H, H, H, h->w_hh[layer]);
  AVVAD_LAUNCHED();
  pack_lstm_b_kernel<<<(unsigned)ceil_div(4 * H, 256), 256, 0, st>>>(b_ih, b_hh, H, h->bias[layer]);
  AVVAD_LAUNCHED();
  h->set[layer] = true;
  return AVVAD_OK;
}

extern "C" int avvad_lstm_set_head(avvad_lstm* h, const float* w, const float* b, void* stream) {
  AVVAD_CHECK_ARG(h && w && b, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n = (int64_t)h->y_dim * h->H;
  pack_head_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(w, n, h->head_w32, h->head_w16);
  AVVAD_LAUNCHED();
  AVVAD_CUDA(cudaMemcpyAsync(h->head_b, b, sizeof(float) * h->y_dim, cudaMemcpyDeviceToDevice, st));
  h->head_set = true;
  return AVVAD_OK;
}

extern "C" int64_t avvad_lstm_input_ld(const avvad_lstm* h) { return h ? h->ld0 : 0; }

namespace avvad {
namespace tc {
int encode_tiled_bf16(CUtensorMap* m, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                      const uint32_t* box);
}
}  // namespace avvad

namespace avvad {
struct TapeView {
  __nv_bfloat16* gates;
  float* c;
  __nv_bfloat16* hseq;
};
TapeView tape_layer(void* tape, int l, int H, int64_t B, int64_t T);
int lstm_backward_impl(int layers, int input_size, int64_t ld0, int H, int y_dim, __nv_bfloat16* const* w_ih,
                       __nv_bfloat16* const* w_hh, const float* head_w32, const __nv_bfloat16* head_w16,
                       const void* x_bf16, const int32_t* lengths,
                       int64_t B, int64_t T, void* tape, const float* dlogits, void* workspace, size_t workspace_bytes,
                       float* const* dW_ih, float* const* dW_hh, float* const* db, float* dW_head, float* db_head,
                       float* dx, cudaStream_t st, BpttGraphCache* cache);
size_t lstm_backward_workspace(int layers, int input_size, int64_t ld0, int H, int y_dim, int64_t B, int64_t T);
}  // namespace avvad

namespace {
// flag area: [16 batch slices][64] shared lines (lstm_persist.cuh, lstm_pair.cuh) + [2][32][32] private lines (pairs)
constexpr size_t kCounterBytes = 16384;
struct LstmWs {
  float* xproj;
  float* xproj1;  // second input-projection buffer: layer 1's chunks are written while layer 0 still reads its own
  float* c1;
  __nv_bfloat16* hseq[2];
  __nv_bfloat16* hbuf[2];
  float* c;
  __nv_bfloat16* hlast;
  unsigned int* counters;
  // streaming state only: c_t of every step of the layers in flight (f32 [B][T+1][H]) and the shifted lengths
  float* cseq[2];
  int32_t* len1;
  size_t total;
};
// `state`: the layout of avvad_lstm_forward_state, whose sequences have one more step (position 0 holds h_in)
LstmWs carve(const avvad_lstm* h, int64_t B, int64_t T, void* base, bool state = false) {
  LstmWs w{};
  size_t off = 0;
  auto take = [&](size_t bytes) {
    void* p = base ? (uint8_t*)base + off : nullptr;
    off += align_up(bytes, 256);
    return p;
  };
  const int64_t H = h->H;
  if (state) {
    ++T;
    for (int l = 0; l < (h->layers >= 2 ? 2 : 1); ++l) w.cseq[l] = (float*)take((size_t)B * T * H * sizeof(float));
    w.len1 = (int32_t*)take((size_t)B * sizeof(int32_t));
  }
  w.xproj = (float*)take((size_t)((B + 127) / 128 * 128) * T * 4 * H * sizeof(float));  // xT layout pads B to 128
  w.xproj1 = (h->layers >= 2) ? (float*)take((size_t)((B + 127) / 128 * 128) * T * 4 * H * sizeof(float)) : nullptr;
  w.c1 = (float*)take((size_t)B * H * sizeof(float));
  w.hseq[0] = (__nv_bfloat16*)take((size_t)B * T * H * 2);
  w.hseq[1] = (__nv_bfloat16*)take((size_t)B * T * H * 2);
  w.hbuf[0] = (__nv_bfloat16*)take((size_t)B * H * 2);
  w.hbuf[1] = (__nv_bfloat16*)take((size_t)B * H * 2);
  w.c = (float*)take((size_t)B * H * sizeof(float));
  w.hlast = (__nv_bfloat16*)take((size_t)B * H * 2);
  w.counters = (unsigned int*)take(2 * kCounterBytes);  // per-CTA step flags of the persistent recurrences (two layers in flight)
  w.total = off;
  return w;
}
}  // namespace

extern "C" size_t avvad_lstm_workspace_bytes(const avvad_lstm* h, int64_t B, int64_t T) {
  if (!h || B <= 0 || T <= 0) return 0;
  return carve(h, B, T, nullptr).total;
}

extern "C" size_t avvad_lstm_state_workspace_bytes(const avvad_lstm* h, int64_t B, int64_t T) {
  if (!h || B <= 0 || T <= 0) return 0;
  return carve(h, B, T, nullptr, true).total;
}

// ---- persistent recurrence (one cooperative launch per layer and batch group) ---------------------------------
static int persist_mode() {
  static int v = [] {
    const char* e = getenv("AVVAD_LSTM");
    if (e && std::string(e) == "steps") return 0;
    return tc::tma_available() ? 1 : 0;
  }();
  return v;
}

// CTA-pair recurrence (lstm_pair.cuh) for 129..256 batch rows; AVVAD_LSTM_PAIR=0 selects the one-CTA-per-block kernel.
static int pair_mode() {
  static int v = [] {
    const char* e = getenv("AVVAD_LSTM_PAIR");
    return (e && atoi(e) == 0) ? 0 : 1;
  }();
  return v;
}
// debug aid (tools/micro/lstm_ab.py): when set, the next pair launches run the tracing instantiation and write
// [CTA][T][8] globaltimer stamps here
static unsigned long long* g_pair_trace = nullptr;
extern "C" void avvad_debug_lstm_trace(void* buf) { g_pair_trace = (unsigned long long*)buf; }

template <int kEW, int NP>
static int run_pair_cfg(tc::LstmMaps maps, tc::PairGeom g, const __nv_bfloat16* w_hh, unsigned int* counters,
                        cudaStream_t st, double flops) {
  const int H = g.H;
  const size_t smem = (size_t)(H / 64) * (NP / 2) * 128 + tc::kPairStagesOf(NP) * 16384 + 256 + 1024;
  static PerDeviceOnce once;
  AVVAD_CUDA(once.run([] {
    cudaError_t e = cudaFuncSetAttribute(tc::lstm_pair_kernel<false, kEW, NP>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(tc::lstm_pair_kernel<true, kEW, NP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                227 * 1024);
  }));
  g.n_pairs = 4 * H / NP;
  // this CTA's half of a pair's weight slice: NP/2 gate columns per box
  const uint64_t wd[2] = {(uint64_t)H, (uint64_t)4 * H};
  const uint64_t wstr[1] = {(uint64_t)H * 2};
  const uint32_t wbox[2] = {64, NP / 2};
  int rc = tc::encode_tiled_bf16(&maps.w, w_hh, 2, wd, wstr, wbox);
  if (rc) return rc;
  const void* fn = g.trace ? (const void*)tc::lstm_pair_kernel<true, kEW, NP>
                           : (const void*)tc::lstm_pair_kernel<false, kEW, NP>;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * g.n_pairs);
  cfg.blockDim = dim3(tc::kPairThreadsOf(kEW));
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute la[2];
  la[0].id = cudaLaunchAttributeClusterDimension;
  la[0].val.clusterDim.x = 2; la[0].val.clusterDim.y = 1; la[0].val.clusterDim.z = 1;
  la[1].id = cudaLaunchAttributeCooperative;
  la[1].val.cooperative = 1;
  cfg.attrs = la;
  cfg.numAttrs = 1;
  int max_clusters = 0;
  if (cudaOccupancyMaxActiveClusters(&max_clusters, fn, &cfg) != cudaSuccess || max_clusters < g.n_pairs) {
    cudaGetLastError();
    return AVVAD_ERR_STATE;
  }
  // The cooperative attribute guarantees that all CTAs are co-resident (they wait for each other).  ncu cannot launch
  // cooperative cluster kernels ("LaunchFailed"): AVVAD_LSTM_COOP=0 drops the attribute for profiling runs, where the
  // serialised kernel has the GPU to itself anyway.
  static int coop_attr = [] {
    const char* e = getenv("AVVAD_LSTM_COOP");
    return (e && atoi(e) == 0) ? 0 : 1;
  }();
  cfg.numAttrs = coop_attr ? 2 : 1;
  AVVAD_CUDA(cudaMemsetAsync(counters, 0, kCounterBytes, st));
  void* args[2] = {(void*)&maps, (void*)&g};
  void* tok = nullptr;
  tc::prof_begin(st, &tok);
  AVVAD_CUDA(cudaLaunchKernelExC(&cfg, fn, args));
  g_launches.fetch_add(1, std::memory_order_relaxed);
  tc::prof_end(st, tok, 2, flops);
  return AVVAD_OK;
}

static int run_pair(const tc::LstmMaps& maps, const __nv_bfloat16* w_hh, const float4* xT, int64_t Bp,
                    __nv_bfloat16* hseq, const int32_t* lengths, int64_t Bc, int64_t T, int H, unsigned int* counters,
                    cudaStream_t st, __nv_bfloat16* gates_out, float* c_out, int t0, int t1, float* c_state) {
  tc::PairGeom g{};
  g.B = (int)Bc; g.T = (int)T; g.H = H; g.KB = H / 64;
  g.t0 = t0; g.t1 = t1; g.c_state = c_state;
  g.xT = xT;
  g.Bp = (int)Bp;
  g.hseq = hseq;
  g.lengths = lengths;
  g.counters = counters;
  g.gates_out = gates_out;
  g.c_out = c_out;
  g.trace = g_pair_trace;
  static int variant = [] {
    const char* e = getenv("AVVAD_LSTM_VARIANT");
    return e ? atoi(e) : 0;
  }();
  g.variant = variant;
  // AVVAD_LSTM_NP = gate columns per pair (128 | 64), AVVAD_LSTM_EPI_WARPS = cell-update warps per CTA
  static int np = [] {
    const char* e = getenv("AVVAD_LSTM_NP");
    return (e && atoi(e) == 128) ? 128 : (e && atoi(e) == 64) ? 64 : 128;
  }();
  static int epi_warps = [] {
    const char* e = getenv("AVVAD_LSTM_EPI_WARPS");
    return e ? atoi(e) : 8;
  }();
  const double flops = 2.0 * (double)Bc * 4.0 * H * H * (double)(t1 - (t0 > 1 ? t0 : 1));
  if (np == 64 && 4 * H / 64 <= 64) {
    if (epi_warps == 4) return run_pair_cfg<4, 64>(maps, g, w_hh, counters, st, flops);
    return run_pair_cfg<8, 64>(maps, g, w_hh, counters, st, flops);
  }
  if (epi_warps == 16) return run_pair_cfg<16, 128>(maps, g, w_hh, counters, st, flops);
  return run_pair_cfg<8, 128>(maps, g, w_hh, counters, st, flops);
}

static int lstm_num_sms() {
  static int num_sms = [] {
    int dev = 0, v = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v > 0 ? v : 148;
  }();
  return num_sms;
}
// Can the persistent recurrence (one cooperative launch per layer and batch group) run this shape on this device?
static bool persistent_ok(const avvad_lstm* h, int64_t T) {
  const int H = h->H;
  if (!persist_mode() || H % 64 != 0 || H > 1024 || 4 * H / 64 > tc::kLstmMaxSlices || T < 1) return false;
  static int coop = [] {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&v, cudaDevAttrCooperativeLaunch, dev);
    return v;
  }();
  return coop && lstm_num_sms() / (4 * H / 64) >= 1;
}

// xproj: the input projection in the xT layout (tc::launch_tma_gemm_xt) over the whole batch, Bp = B rounded up to 128
// Steps [t0, t1) of layer l; c_state f32 [B][H] carries the cell state between chunks.
static int run_recurrence_persistent(avvad_lstm* h, int l, const float* xproj, __nv_bfloat16* hseq,
                                     const int32_t* lengths, int64_t B, int64_t T, unsigned int* counters,
                                     cudaStream_t st, bool* done, __nv_bfloat16* gates_out, float* c_out, int t0, int t1,
                                     float* c_state) {
  *done = false;
  const int H = h->H;
  if (!persistent_ok(h, T)) return AVVAD_OK;
  const int64_t Bp = (B + 127) / 128 * 128;
  const int num_sms = lstm_num_sms();
  const int n_slices = 4 * H / 64;
  int max_ms = num_sms / n_slices;
  if (max_ms > 16) max_ms = 16;  // flag lines per launch (kCounterBytes)
  const size_t smem = (size_t)(H / 64) * 8192 + tc::kLstmStages * 16384 + 256 + 1024;
  static PerDeviceOnce once;
  AVVAD_CUDA(once.run([] {
    return cudaFuncSetAttribute(tc::lstm_persist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  }));
  const int64_t Bg = (int64_t)max_ms * 128;
  for (int64_t g0 = 0; g0 < B; g0 += Bg) {
    const int64_t Bc = (B - g0 < Bg) ? (B - g0) : Bg;
    const int m_slices = (int)((Bc + 127) / 128);
    tc::LstmMaps maps;
    __nv_bfloat16* hs = hseq + g0 * T * H;
    const uint64_t hd[3] = {(uint64_t)H, (uint64_t)T, (uint64_t)Bc};
    const uint64_t hstr[2] = {(uint64_t)H * 2, (uint64_t)T * H * 2};
    const uint32_t hbox[3] = {64, 1, 128};
    int rc = tc::encode_tiled_bf16(&maps.h, hs, 3, hd, hstr, hbox);
    if (rc) return rc;
    const uint64_t wd[2] = {(uint64_t)H, (uint64_t)4 * H};
    const uint64_t wstr[1] = {(uint64_t)H * 2};
    const uint32_t wbox[2] = {64, 64};
    rc = tc::encode_tiled_bf16(&maps.w, h->w_hh[l], 2, wd, wstr, wbox);
    if (rc) return rc;
    // AVVAD_LSTM_PAIR_MIN: smallest batch (of a group) the pair kernel takes.  With <= 128 rows the second CTA of every
    // pair works on zero-filled rows, but the kernel is still the faster one (full-sector h stores, half the CTAs polling)
    static int pair_min = [] {
      const char* e = getenv("AVVAD_LSTM_PAIR_MIN");
      return e ? atoi(e) : 1;
    }();
    if (pair_mode() && max_ms <= 2 && Bc >= pair_min && n_slices % 2 == 0 && n_slices / 2 <= 32) {
      rc = run_pair(maps, h->w_hh[l], reinterpret_cast<const float4*>(xproj) + g0, Bp, hs, lengths + g0, Bc, T, H, counters, st,
                    gates_out ? gates_out + g0 * T * 4 * H : nullptr, c_out ? c_out + g0 * T * H : nullptr, t0, t1,
                    c_state + g0 * H);
      if (rc == AVVAD_OK) continue;
      if (rc != AVVAD_ERR_STATE) return rc;  // AVVAD_ERR_STATE: the pairs do not fit this device -> one CTA per block
    }
    tc::LstmGeom g{};
    g.B = (int)Bc; g.T = (int)T; g.H = H; g.KB = H / 64; g.n_slices = n_slices;
    g.xT = reinterpret_cast<const float4*>(xproj) + g0;
    g.Bp = (int)Bp;
    g.t0 = t0; g.t1 = t1; g.c_state = c_state + g0 * H;
    g.hseq = hs;
    g.lengths = lengths + g0;
    g.counters = counters;
    static int variant = [] {
      const char* e = getenv("AVVAD_LSTM_VARIANT");
      return e ? atoi(e) : 0;
    }();
    g.variant = variant;
    g.gates_out = gates_out ? gates_out + g0 * T * 4 * H : nullptr;
    g.c_out = c_out ? c_out + g0 * T * H : nullptr;
    AVVAD_CUDA(cudaMemsetAsync(counters, 0, 4096, st));
    // Optional h multicast inside clusters (AVVAD_LSTM_CLUSTER = 2, 4 or 8): cuts the L2 reads of h per step from
    // 32 MB to 32 MB / cluster.  Measured on B200: 7.6 ms (off) vs 10.1 / 7.9 / 8.0 ms (2 / 4 / 8) -- the recurrence is a
    // latency chain, not L2-bandwidth bound, and arming the ring in K order costs more than the traffic saves.  Off
    // by default.
    static int cluster_pref = [] {
      const char* e = getenv("AVVAD_LSTM_CLUSTER");
      return e ? atoi(e) : 1;
    }();
    const int n_ctas = n_slices * m_slices;
    int cluster = 1;
    for (int c = 8; c >= 2; c >>= 1) {
      if (c > cluster_pref || n_slices % c) continue;
      cudaLaunchConfig_t qc = {};
      qc.gridDim = dim3(n_ctas);
      qc.blockDim = dim3(tc::kLstmThreads);
      qc.dynamicSmemBytes = smem;
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = c; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
      qc.attrs = qa;
      qc.numAttrs = 1;
      int max_clusters = 0;
      if (cudaOccupancyMaxActiveClusters(&max_clusters, (const void*)tc::lstm_persist_kernel, &qc) == cudaSuccess &&
          max_clusters * c >= n_ctas) {
        cluster = c;
        break;
      }
      cudaGetLastError();
    }
    g.cluster = cluster;
    void* args[2] = {(void*)&maps, (void*)&g};
    void* tok = nullptr;
    tc::prof_begin(st, &tok);
    if (cluster > 1) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(n_ctas);
      cfg.blockDim = dim3(tc::kLstmThreads);
      cfg.dynamicSmemBytes = smem;
      cfg.stream = st;
      cudaLaunchAttribute la[2];
      la[0].id = cudaLaunchAttributeClusterDimension;
      la[0].val.clusterDim.x = cluster; la[0].val.clusterDim.y = 1; la[0].val.clusterDim.z = 1;
      la[1].id = cudaLaunchAttributeCooperative;
      la[1].val.cooperative = 1;
      cfg.attrs = la;
      cfg.numAttrs = 2;
      AVVAD_CUDA(cudaLaunchKernelExC(&cfg, (const void*)tc::lstm_persist_kernel, args));
    } else {
      AVVAD_CUDA(cudaLaunchCooperativeKernel((const void*)tc::lstm_persist_kernel, dim3(n_ctas),
                                             dim3(tc::kLstmThreads), args, smem, st));
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    tc::prof_end(st, tok, 2, 2.0 * (double)Bc * 4.0 * H * H * (double)(t1 - (t0 > 1 ? t0 : 1)));
  }
  *done = true;
  return AVVAD_OK;
}

static int run_head(avvad_lstm* h, const __nv_bfloat16* hs, int64_t rows, float* logits, float* post, int32_t* dec,
                    cudaStream_t st) {
  const int H = h->H;
  if (h->y_dim == 1) {
    head1_kernel<<<(unsigned)ceil_div(rows * 32, 256), 256, 0, st>>>(hs, rows, H, h->head_w32, h->head_b, logits, post,
                                                                     dec);
    AVVAD_LAUNCHED();
    return AVVAD_OK;
  }
  AVVAD_CHECK_ARG(logits, "logits buffer required when y_dim > 1");
  int rc = avvad_gemm_bf16(hs, H, h->head_w16, H, h->head_b, logits, h->y_dim, 0, 0, rows, h->y_dim, H, st);
  if (rc) return rc;
  if (post || dec) {
    const int64_t n = rows * h->y_dim;
    post_dec_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(logits, n, post, dec);
    AVVAD_LAUNCHED();
  }
  return AVVAD_OK;
}

namespace {
// Recurrent state of avvad_lstm_forward_state: h bf16 [L][B][H], c f32 [L][B][H]; null inputs mean zero
struct LstmStateIO {
  const __nv_bfloat16* h_in;
  const float* c_in;
  __nv_bfloat16* h_out;
  float* c_out;
};
}  // namespace

static int lstm_forward_impl(avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T,
                             void* workspace, size_t workspace_bytes, float* logits, float* post, int32_t* dec,
                             float* last_logits, void* tape, void* stream, const LstmStateIO* sio = nullptr) {
  AVVAD_CHECK_ARG(h && x_bf16 && lengths && workspace && B > 0 && T > 0, "bad argument");
  const bool want_head = logits || post || dec || last_logits;
  AVVAD_CHECK_ARG(want_head || (sio && (sio->h_out || sio->c_out)), "no output requested");
  AVVAD_CHECK_ARG(!(sio && tape), "lstm: the training forward takes no initial state");
  for (int l = 0; l < h->layers; ++l)
    if (!h->set[l]) {
      set_error("lstm: layer " + std::to_string(l) + " not loaded");
      return AVVAD_ERR_STATE;
    }
  if (!h->head_set) {
    set_error("lstm: head not loaded");
    return AVVAD_ERR_STATE;
  }
  if (workspace_bytes < (sio ? avvad_lstm_state_workspace_bytes(h, B, T) : avvad_lstm_workspace_bytes(h, B, T))) {
    set_error("lstm: workspace too small");
    return AVVAD_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int H = h->H;
  const int H4 = 4 * H;
  LstmWs ws = carve(h, B, T, workspace, sio != nullptr);
  const int64_t rows = B * T;

  const __nv_bfloat16* layer_in = (const __nv_bfloat16*)x_bf16;
  int64_t ld_in = h->ld0;
  int64_t in_stride = T;  // steps per batch row of layer_in
  __nv_bfloat16* layer_out = nullptr;
  const bool persistent = persistent_ok(h, T);

  // ---- streaming state.  The persistent recurrences run this call's steps at positions s = 1 .. T of [B][T+1][H]
  // sequences whose position 0 holds h_in, with c_in in c_state: exactly the hand-over between two chunks of one layer,
  // so the kernels are the ones the stateless call runs.  They record c_t of every step (the training tape's c store),
  // from which the final state is gathered at len_b - 1.  The per-step fallback seeds its h operand instead (s = 0).
  const int s = (sio && persistent) ? 1 : 0;
  const int64_t Ts = T + s;
  const int64_t Bp = (B + 127) / 128 * 128;
  const int32_t* lens_rec = lengths;  // lengths the recurrence masks with (positions, not steps)
  if (s) {
    shift_lengths_kernel<<<(unsigned)ceil_div(B, 256), 256, 0, st>>>(lengths, (int)B, ws.len1);
    AVVAD_LAUNCHED();
    lens_rec = ws.len1;
  }
  // layer l's initial state: h_in[l] -> position 0 of `hs` (rows `pitch` steps apart), c_in[l] -> c_state
  auto seed = [&](int l, __nv_bfloat16* hs, int64_t pitch, float* c_state) -> int {
    const size_t hrow = (size_t)H * 2, crow = (size_t)H * sizeof(float);
    const int64_t off = (int64_t)l * B * H;
    if (sio->h_in)
      AVVAD_CUDA(cudaMemcpy2DAsync(hs, pitch * hrow, sio->h_in + off, hrow, hrow, B, cudaMemcpyDeviceToDevice, st));
    else
      AVVAD_CUDA(cudaMemset2DAsync(hs, pitch * hrow, 0, hrow, B, st));
    if (sio->c_in)
      AVVAD_CUDA(cudaMemcpyAsync(c_state, sio->c_in + off, B * crow, cudaMemcpyDeviceToDevice, st));
    else
      AVVAD_CUDA(cudaMemsetAsync(c_state, 0, B * crow, st));
    return AVVAD_OK;
  };
  // layer l's final state from its output sequence and its record of c
  auto emit = [&](int l, const __nv_bfloat16* hs, const float* cseq) -> int {
    const int64_t off = (int64_t)l * B * H;
    gather_state_kernel<<<(unsigned)B, 128, 0, st>>>(hs, cseq, lengths, (int)Ts, s, H,
                                                     sio->h_in ? sio->h_in + off : nullptr,
                                                     sio->c_in ? sio->c_in + off : nullptr,
                                                     sio->h_out ? sio->h_out + off : nullptr,
                                                     sio->c_out ? sio->c_out + off : nullptr);
    AVVAD_LAUNCHED();
    return AVVAD_OK;
  };

  // ---- two layers, chunked: layer 1 follows layer 0 one chunk of time steps behind on a side stream.  Both recurrences
  // are latency chains on 64 SMs each, so they overlap almost perfectly; layer 1's input projection of a chunk (a GEMM
  // over the chunk's h0 rows) runs on the SMs layer 0 leaves free.  AVVAD_LSTM_CHUNKS = 1 runs the layers back to back.
  static int n_chunks_pref = [] {
    const char* e = getenv("AVVAD_LSTM_CHUNKS");
    int v = e ? atoi(e) : 8;
    return v < 1 ? 1 : (v > 32 ? 32 : v);
  }();
  int n_chunks = n_chunks_pref;
  while (n_chunks > 1 && T / n_chunks < 16) --n_chunks;
  if (persistent && h->layers == 2 && n_chunks > 1) {
    int dev = 0;
    AVVAD_CUDA(cudaGetDevice(&dev));
    if (!h->side || h->side_device != dev) {
      if (h->side) cudaStreamDestroy(h->side);
      for (auto& e : h->ev_chunk) {
        if (e) cudaEventDestroy(e);
        e = nullptr;
      }
      if (h->ev_done) cudaEventDestroy(h->ev_done);
      h->ev_done = nullptr;
      AVVAD_CUDA(cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking));
      for (auto& e : h->ev_chunk) AVVAD_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      AVVAD_CUDA(cudaEventCreateWithFlags(&h->ev_done, cudaEventDisableTiming));
      h->side_device = dev;
    }
    __nv_bfloat16* out0 = ws.hseq[0];
    __nv_bfloat16* out1 = ws.hseq[1];
    float* crec0 = ws.cseq[0];
    float* crec1 = ws.cseq[1];
    TapeView tv0{}, tv1{};
    if (tape) {
      tv0 = tape_layer(tape, 0, H, B, T);
      tv1 = tape_layer(tape, 1, H, B, T);
      out0 = tv0.hseq;
      out1 = tv1.hseq;
      crec0 = tv0.c;
      crec1 = tv1.c;
    }
    int rc;
    if (sio) {  // on `st` before the first chunk's event: the side stream sees layer 1's seed too
      if ((rc = seed(0, out0, Ts, ws.c)) || (rc = seed(1, out1, Ts, ws.c1))) return rc;
    }
    rc = tc::launch_tma_gemm_xt(layer_in, ld_in, h->w_ih[0], ld_in, B, T, T, H4, (int)ld_in, h->bias[0],
                                ws.xproj + s * H4 * Bp, st);
    if (rc) return rc;
    const int free_sms = lstm_num_sms() - 2 * (4 * H / 128);  // SMs a layer-0 pair launch leaves to the projection GEMM
    for (int c = 0; c < n_chunks; ++c) {
      const int t0 = s + (int)(T * c / n_chunks), t1 = s + (int)(T * (c + 1) / n_chunks);
      bool done = false;
      rc = run_recurrence_persistent(h, 0, ws.xproj, out0, lens_rec, B, Ts, ws.counters, st, &done, tv0.gates, crec0,
                                     t0, t1, ws.c);
      if (rc) return rc;
      if (!done) {
        set_error("lstm: persistent recurrence unavailable");
        return AVVAD_ERR_STATE;
      }
      AVVAD_CUDA(cudaEventRecord(h->ev_chunk[c], st));
      AVVAD_CUDA(cudaStreamWaitEvent(h->side, h->ev_chunk[c], 0));
      rc = tc::launch_tma_gemm_xt(out0 + (int64_t)t0 * H, H, h->w_ih[1], H, B, t1 - t0, Ts, H4, H, h->bias[1],
                                  ws.xproj1 + (int64_t)t0 * H4 * Bp, h->side, free_sms > 16 ? free_sms : 0);
      if (rc) return rc;
      rc = run_recurrence_persistent(h, 1, ws.xproj1, out1, lens_rec, B, Ts, ws.counters + kCounterBytes / 4, h->side,
                                     &done, tv1.gates, crec1, t0, t1, ws.c1);
      if (rc) return rc;
    }
    AVVAD_CUDA(cudaEventRecord(h->ev_done, h->side));
    AVVAD_CUDA(cudaStreamWaitEvent(st, h->ev_done, 0));
    if (sio) {
      if ((rc = emit(0, out0, crec0)) || (rc = emit(1, out1, crec1))) return rc;
    }
    layer_out = out1;
  } else {
  for (int l = 0; l < h->layers; ++l) {
    layer_out = ws.hseq[l & 1];
    float* crec = ws.cseq[l & 1];
    TapeView tv{};
    if (tape) {
      tv = tape_layer(tape, l, H, B, T);
      layer_out = tv.hseq;
      crec = tv.c;
    }
    int rc;
    if (s && (rc = seed(l, layer_out, Ts, ws.c))) return rc;
    // (1) input projection for every (b,t): xproj = X * W_ih'^T + (b_ih + b_hh)'.  The persistent recurrences read it
    // time-major and unit-major (xT[t][u][b][4]: lane = batch row -> coalesced), the per-step fallback row-major.
    rc = persistent ? tc::launch_tma_gemm_xt(layer_in, ld_in, h->w_ih[l], ld_in, B, T, in_stride, H4, (int)ld_in,
                                             h->bias[l], ws.xproj + s * H4 * Bp, st)
                    : avvad_gemm_bf16(layer_in, ld_in, h->w_ih[l], ld_in, h->bias[l], ws.xproj, H4, 0, 0, rows, H4,
                                      ld_in, st);
    if (rc) return rc;
    // (2) recurrence: one persistent cooperative kernel per layer, or (fallback) one GEMM launch per time step
    bool done = false;
    rc = run_recurrence_persistent(h, l, ws.xproj, layer_out, lens_rec, B, Ts, ws.counters, st, &done, tv.gates, crec,
                                   s, (int)Ts, ws.c);
    if (rc) return rc;
    if (persistent && !done) {
      set_error("lstm: persistent recurrence unavailable after the xT input projection");
      return AVVAD_ERR_STATE;
    }
    if (tape && !done) {
      set_error("lstm: the training forward needs the persistent recurrence (TMA + cooperative launch, H <= 1024)");
      return AVVAD_ERR_STATE;
    }
    if (done) {
      if (sio && (rc = emit(l, layer_out, crec))) return rc;
      layer_in = layer_out + (int64_t)s * H;
      ld_in = H;
      in_stride = Ts;
      continue;
    }
    if (sio) {
      if ((rc = seed(l, ws.hbuf[0], 1, ws.c))) return rc;
    } else {
      AVVAD_CUDA(cudaMemsetAsync(ws.hbuf[0], 0, (size_t)B * H * 2, st));
      AVVAD_CUDA(cudaMemsetAsync(ws.c, 0, (size_t)B * H * sizeof(float), st));
    }
    for (int t = 0; t < (int)T; ++t) {
      tc::EpiParams ep{};
      ep.xproj = ws.xproj;
      ep.c_state = ws.c;
      ep.h_next = ws.hbuf[(t + 1) & 1];
      ep.hseq = layer_out;
      ep.lengths = lengths;
      ep.t = t;
      ep.T = (int)T;
      ep.H4 = H4;
      rc = tc::gemm_dispatch(ws.hbuf[t & 1], H, h->w_hh[l], H, B, H4, H, ep, tc::EPI_LSTM, 64, st);
      if (rc) return rc;
      if (sio)  // the epilogue keeps updating c past the length: record c_t for the final-state gather
        AVVAD_CUDA(cudaMemcpy2DAsync(crec + (int64_t)t * H, (size_t)T * H * sizeof(float), ws.c, (size_t)H * sizeof(float),
                                     (size_t)H * sizeof(float), B, cudaMemcpyDeviceToDevice, st));
    }
    if (sio && (rc = emit(l, layer_out, crec))) return rc;
    layer_in = layer_out;
    ld_in = H;
  }
  }
  if (!want_head) return AVVAD_OK;
  if (s) {  // the head reads [B][T][H] rows: drop position 0 into the sequence buffer the last layer did not use
    __nv_bfloat16* compact = layer_out == ws.hseq[0] ? ws.hseq[1] : ws.hseq[0];
    AVVAD_CUDA(cudaMemcpy2DAsync(compact, (size_t)T * H * 2, layer_out + H, (size_t)Ts * H * 2, (size_t)T * H * 2, B,
                                 cudaMemcpyDeviceToDevice, st));
    layer_out = compact;
  }
  if (logits || post || dec) {
    float* lg = logits;
    int rc = run_head(h, layer_out, rows, lg, post, dec, st);
    if (rc) return rc;
  }
  if (last_logits) {
    gather_last_kernel<<<(unsigned)B, 128, 0, st>>>(layer_out, lengths, (int)T, H, ws.hlast);
    AVVAD_LAUNCHED();
    int rc = run_head(h, ws.hlast, B, last_logits, nullptr, nullptr, st);
    if (rc) return rc;
  }
  return AVVAD_OK;
}


extern "C" int avvad_lstm_forward(avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T,
                                  void* workspace, size_t workspace_bytes, float* logits, float* post, int32_t* dec,
                                  float* last_logits, void* stream) {
  return lstm_forward_impl(h, x_bf16, lengths, B, T, workspace, workspace_bytes, logits, post, dec, last_logits, nullptr,
                           stream);
}

extern "C" int avvad_lstm_forward_state(avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T,
                                        const void* h_in, const float* c_in, void* h_out, float* c_out,
                                        void* workspace, size_t workspace_bytes, float* logits, float* post,
                                        int32_t* dec, float* last_logits, void* stream) {
  const LstmStateIO sio{(const __nv_bfloat16*)h_in, c_in, (__nv_bfloat16*)h_out, c_out};
  return lstm_forward_impl(h, x_bf16, lengths, B, T, workspace, workspace_bytes, logits, post, dec, last_logits, nullptr,
                           stream, &sio);
}

extern "C" size_t avvad_lstm_tape_bytes(int layers, int hidden, int64_t B, int64_t T);

// Training forward: identical arithmetic, but every layer's output sequence, post-activation gates and cell states
// are kept in `tape` (avvad_lstm_tape_bytes) for avvad_lstm_backward.
extern "C" int avvad_lstm_forward_train(avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T,
                                        void* workspace, size_t workspace_bytes, void* tape, size_t tape_bytes,
                                        float* logits, void* stream) {
  AVVAD_CHECK_ARG(h && tape && logits, "bad argument");
  if (tape_bytes < avvad_lstm_tape_bytes(h->layers, h->H, B, T)) {
    set_error("lstm: tape too small");
    return AVVAD_ERR_WORKSPACE;
  }
  return lstm_forward_impl(h, x_bf16, lengths, B, T, workspace, workspace_bytes, logits, nullptr, nullptr, nullptr, tape,
                           stream);
}

extern "C" size_t avvad_lstm_backward_workspace_bytes(const avvad_lstm* h, int64_t B, int64_t T) {
  if (!h || B <= 0 || T <= 0) return 0;
  return lstm_backward_workspace(h->layers, h->input_size, h->ld0, h->H, h->y_dim, B, T);
}

// dlogits f32 [B][T][1] (e.g. from avvad_bce_loss).  Gradients in PyTorch layout, fp32: dW_ih[l] [4H][I_l],
// dW_hh[l] [4H][H], db[l] [4H] (= grad of bias_ih_l and of bias_hh_l), dW_head [1][H], db_head [1];
// dx optional f32 [B][T][input_size] (gradient w.r.t. the layer-0 input).
extern "C" int avvad_lstm_backward(avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T,
                                   void* tape, const float* dlogits, void* workspace, size_t workspace_bytes,
                                   float* const* dW_ih, float* const* dW_hh, float* const* db, float* dW_head,
                                   float* db_head, float* dx, void* stream) {
  AVVAD_CHECK_ARG(h && x_bf16 && lengths && tape && dlogits && workspace && dW_ih && dW_hh && db && dW_head && db_head,
                  "null pointer");
  return lstm_backward_impl(h->layers, h->input_size, h->ld0, h->H, h->y_dim, h->w_ih, h->w_hh, h->head_w32,
                            h->head_w16, x_bf16,
                            lengths, B, T, tape, dlogits, workspace, workspace_bytes, dW_ih, dW_hh, db, dW_head, db_head,
                            dx, (cudaStream_t)stream, h->bptt);
}
