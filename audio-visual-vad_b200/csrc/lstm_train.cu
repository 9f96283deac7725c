// Training step of the LSTM + Linear head (SURVEY §8a row O1): back-propagation through time, weight-gradient GEMMs
// and a fused Adam update.  The forward that feeds it is avvad_lstm_forward with a non-null `tape` (the persistent
// recurrence then also stores the post-activation gates and the cell states).
//
// Reference semantics: autograd of packages/models/AV_Net.py:127-140 / Audio_Net.py:50-59 (nn.LSTM + nn.Linear over
// packed sequences) and torch.optim.Adam(lr, betas=(0.9,0.999)) (scripts/train_AV_net.py:238,305-307).
//
//   per layer, t = T-1 .. 0 : cell kernel  (dY_t + dh_rec, dc) -> dgates_t (bf16, gate-interleaved), dc
//                             tcgen05 GEMM  dh_rec = dgates_t * W_hh          (B operand: W_hh^T, K = 4H)
//   after the loop          : dX  = dG * W_ih                                  (GEMM, K = 4H)
//                             dW_ih = dG^T * X, dW_hh = dG^T * H_prev          (GEMMs over K = B*T on transposed copies)
//                             db = column sums of dG
// Gradients are returned in PyTorch's layout (gate-major rows i,f,g,o), fp32.
#include <vector>

#include "gemm_tma.cuh"

namespace avvad {

__device__ __forceinline__ float bf16lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }

// one thread per (b, u)
__global__ void lstm_bwd_cell_kernel(const __nv_bfloat16* __restrict__ gates, const float* __restrict__ cst,
                                     const float* __restrict__ dY, const float* __restrict__ dl,
                                     const float* __restrict__ w_head, const float* __restrict__ dh_rec,
                                     float* __restrict__ dc, const int32_t* __restrict__ lengths, int B, int T, int H,
                                     int t, int has_rec, __nv_bfloat16* __restrict__ dG) {
  // dh_rec holds `has_rec` split-K partial products [has_rec][B][H] of the recurrent GEMM of step t+1
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * H) return;
  const int b = idx / H, u = idx - b * H;
  const int64_t row = (int64_t)b * T + t;
  uint2* out = reinterpret_cast<uint2*>(dG + row * 4 * H + 4 * u);
  if (t >= lengths[b]) {  // padded step: no gradient flows (packed-sequence semantics)
    *out = make_uint2(0u, 0u);
    dc[idx] = 0.f;
    return;
  }
  const uint2 gp = *reinterpret_cast<const uint2*>(gates + row * 4 * H + 4 * u);
  const float gi = bf16lo(gp.x), gf = bf16hi(gp.x), gg = bf16lo(gp.y), go = bf16hi(gp.y);
  const float c = cst[row * H + u];
  const float cp = t > 0 ? cst[(row - 1) * H + u] : 0.f;
  float dh = dY ? dY[row * H + u] : dl[row] * w_head[u];
  for (int sp = 0; sp < has_rec; ++sp) dh += dh_rec[(int64_t)sp * B * H + idx];
  const float tc = tanhf(c);
  const float d_o = dh * tc * go * (1.f - go);
  const float dcc = dh * go * (1.f - tc * tc) + dc[idx];
  const float d_i = dcc * gg * gi * (1.f - gi);
  const float d_g = dcc * gi * (1.f - gg * gg);
  const float d_f = dcc * cp * gf * (1.f - gf);
  dc[idx] = dcc * gf;
  uint2 o;
  o.x = pack_bf16x2(d_i, d_f);
  o.y = pack_bf16x2(d_g, d_o);
  *out = o;
}

// ---- two-layer wavefront (small per-rank batches): layer 1 at step t1 = T-1-s and layer 0 at step t0 = T-s run in the
// SAME launches, so the dependent chain is T+1 (cell, GEMM) pairs instead of 2T.  One GEMM per iteration does all three
// products on a block-structured operand:
//   A [2B][2*4H]:  rows 0..B-1   = [ dG1_t1 | 0 ],   rows B..2B-1 = [ 0 | dG0_t0 ]
//   W [2H][2*4H]:  rows 0..H-1   = [ W_hh1^T | W_hh0^T ],   rows H..2H-1 = [ W_ih1^T | 0 ]
//   C [2B][2H]  :  rows 0..B-1   = [ dh_rec1 | dY0_t1 ],    rows B..2B-1 = [ dh_rec0 | 0 ]
// which the next iteration's cell launch consumes (layer 0 then sits at the step layer 1 just left).
__global__ void lstm_bwd_cell_wf_kernel(const __nv_bfloat16* __restrict__ gates1, const float* __restrict__ cst1,
                                        const __nv_bfloat16* __restrict__ gates0, const float* __restrict__ cst0,
                                        const float* __restrict__ dY1, const float* __restrict__ dl,
                                        const float* __restrict__ w_head, const float* __restrict__ Cpart, int nsplit,
                                        float* __restrict__ dc2, const int32_t* __restrict__ lengths, int B, int T, int H,
                                        int s, __nv_bfloat16* __restrict__ dG1, __nv_bfloat16* __restrict__ dG0,
                                        __nv_bfloat16* __restrict__ Abuf) {
  const int layer = 1 - (int)blockIdx.y;   // blockIdx.y 0 -> layer 1, 1 -> layer 0
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * H) return;
  const int b = idx / H, u = idx - b * H;
  const int t = (layer == 1) ? (T - 1 - s) : (T - s);
  const int64_t K2 = 8ll * H;              // row length of Abuf (null: the GEMMs read dG1 / dG0 directly)
  uint2* aout = Abuf ? reinterpret_cast<uint2*>(Abuf + (int64_t)(layer == 1 ? b : B + b) * K2 + (layer == 1 ? 0 : 4 * H) + 4 * u)
                     : nullptr;
  if (t < 0 || t > T - 1) {                // this layer is idle in iteration s: contribute nothing to the GEMM
    if (aout) *aout = make_uint2(0u, 0u);
    return;
  }
  const int64_t row = (int64_t)b * T + t;
  __nv_bfloat16* dG = layer == 1 ? dG1 : dG0;
  uint2* gout = reinterpret_cast<uint2*>(dG + row * 4 * H + 4 * u);
  float* dc = dc2 + (int64_t)layer * B * H;
  if (t >= lengths[b]) {
    *gout = make_uint2(0u, 0u);
    if (aout) *aout = make_uint2(0u, 0u);
    dc[idx] = 0.f;
    return;
  }
  const __nv_bfloat16* gates = layer == 1 ? gates1 : gates0;
  const float* cst = layer == 1 ? cst1 : cst0;
  const uint2 gp = *reinterpret_cast<const uint2*>(gates + row * 4 * H + 4 * u);
  const float gi = bf16lo(gp.x), gf = bf16hi(gp.x), gg = bf16lo(gp.y), go = bf16hi(gp.y);
  const float c = cst[row * H + u];
  const float cp = t > 0 ? cst[(row - 1) * H + u] : 0.f;
  const int64_t cstride = 2ll * B * 2 * H;  // one split-K partial of C
  float dh;
  if (layer == 1) {
    dh = dY1 ? dY1[row * H + u] : dl[row] * w_head[u];
    if (s > 0)
      for (int sp = 0; sp < nsplit; ++sp) dh += Cpart[sp * cstride + (int64_t)b * 2 * H + u];
  } else {
    dh = 0.f;
    for (int sp = 0; sp < nsplit; ++sp) {
      dh += Cpart[sp * cstride + (int64_t)b * 2 * H + H + u];                      // dY0_t = dG1_t * W_ih1
      if (t < T - 1) dh += Cpart[sp * cstride + (int64_t)(B + b) * 2 * H + u];      // recurrent term from step t+1
    }
  }
  const float tc = tanhf(c);
  const float d_o = dh * tc * go * (1.f - go);
  const float dcc = dh * go * (1.f - tc * tc) + dc[idx];
  const float d_i = dcc * gg * gi * (1.f - gi);
  const float d_g = dcc * gi * (1.f - gg * gg);
  const float d_f = dcc * cp * gf * (1.f - gf);
  dc[idx] = dcc * gf;
  uint2 o;
  o.x = pack_bf16x2(d_i, d_f);
  o.y = pack_bf16x2(d_g, d_o);
  *gout = o;
  if (aout) *aout = o;
}
// Wcat [2H][8H] from the gate-interleaved packed weights W' [4H][ld] (see the layout above)
__global__ void lstm_wf_pack_w_kernel(const __nv_bfloat16* __restrict__ whh1, const __nv_bfloat16* __restrict__ wih1,
                                      const __nv_bfloat16* __restrict__ whh0, int H, __nv_bfloat16* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t K2 = 8ll * H;
  if (idx >= 2ll * H * K2) return;
  const int n = (int)(idx / K2);
  const int k = (int)(idx - (int64_t)n * K2);
  __nv_bfloat16 v = __float2bfloat16_rn(0.f);
  if (n < H) v = (k < 4 * H) ? whh1[(int64_t)k * H + n] : whh0[(int64_t)(k - 4 * H) * H + n];
  else if (k < 4 * H) v = wih1[(int64_t)k * H + (n - H)];
  out[idx] = v;
}

// bf16 [R][ld] (first C columns) -> [C][Rp] with zero fill for r >= R; `shift` > 0 reads row r - shift*? (see below)
// mode 0: plain transpose.  mode 1: H_prev transpose: out[c][b*T + t] = in[b*T + t - 1][c] for t > 0, else 0.
__global__ void transpose_bf16_kernel(const __nv_bfloat16* __restrict__ in, int64_t R, int C, int64_t ld, int64_t Rp,
                                      int mode, int T, __nv_bfloat16* __restrict__ out) {
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

// W' (gate-interleaved rows 4u+g) bf16 [4H][ld] -> W'^T bf16 [cols][4H]
__global__ void transpose_w_kernel(const __nv_bfloat16* __restrict__ w, int rows, int cols, int ld,
                                   __nv_bfloat16* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)rows * cols) return;
  const int c = (int)(idx / rows), r = (int)(idx - (int64_t)c * rows);
  out[idx] = w[(int64_t)r * ld + c];
}

// dW' f32 [4H][ldw] (interleaved rows) -> torch layout f32 [4H][I] (row g*H+u), first I columns
__global__ void deinterleave_w_kernel(const float* __restrict__ dwp, int H, int I, int ldw, float* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)4 * H * I) return;
  const int i = (int)(idx % I);
  const int rt = (int)(idx / I);  // torch row g*H+u
  const int g = rt / H, u = rt - g * H;
  out[idx] = dwp[(int64_t)(4 * u + g) * ldw + i];
}

// db[g*H+u] = sum_r dG[r][4u+g].  Two deterministic stages: (column block of 256, row chunk) partial sums with 16-byte
// loads (thread = 8 columns x one of 8 row lanes), then a fixed-order sum over the row chunks.
constexpr int kBiasChunks = 64;
__global__ void __launch_bounds__(256) bias_grad_partial_kernel(const __nv_bfloat16* __restrict__ dG, int64_t R, int H4,
                                                                float* __restrict__ partial) {
  __shared__ float sm[8][256];
  const int grp = threadIdx.x & 31, ln = threadIdx.x >> 5;
  const int col = blockIdx.x * 256 + grp * 8;
  const int64_t rows_per = (R + kBiasChunks - 1) / kBiasChunks;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per;
  const int64_t r1 = (r0 + rows_per < R) ? r0 + rows_per : R;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int64_t r = r0 + ln; r < r1; r += 8) {
    const uint4 v = *reinterpret_cast<const uint4*>(dG + r * H4 + col);
    acc[0] += bf16lo(v.x); acc[1] += bf16hi(v.x); acc[2] += bf16lo(v.y); acc[3] += bf16hi(v.y);
    acc[4] += bf16lo(v.z); acc[5] += bf16hi(v.z); acc[6] += bf16lo(v.w); acc[7] += bf16hi(v.w);
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) sm[ln][grp * 8 + e] = acc[e];
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int l = 0; l < 8; ++l) t += sm[l][threadIdx.x];
  partial[(int64_t)blockIdx.y * H4 + blockIdx.x * 256 + threadIdx.x] = t;
}
__global__ void bias_grad_final_kernel(const float* __restrict__ partial, int H, float* __restrict__ db) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= 4 * H) return;
  float t = 0.f;
  for (int c = 0; c < kBiasChunks; ++c) t += partial[(int64_t)c * 4 * H + col];
  const int u = col >> 2, g = col & 3;
  db[g * H + u] = t;
}

// W_head bf16 [y][H] -> W_head^T as the GEMM's B operand [N = H][K = yp] (zero columns past y)
__global__ void head_wt_kernel(const __nv_bfloat16* __restrict__ w, int y, int H, int yp, __nv_bfloat16* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)H * yp) return;
  const int u = (int)(idx / yp), k = (int)(idx - (int64_t)u * yp);
  out[idx] = (k < y) ? w[(int64_t)k * H + u] : __float2bfloat16_rn(0.f);
}
// out[c] = sum_r x[r][c]  (fp32, 64 columns per block, fixed-order reduction over four row lanes)
__global__ void __launch_bounds__(256) colsum_f32_kernel(const float* __restrict__ x, int64_t R, int Ccols,
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

// y_dim == 1 head: dW[u] = sum_r dl[r] * h[r][u]; db = sum_r dl[r].  Two-stage deterministic reduction.
__global__ void __launch_bounds__(256) head_grad_partial_kernel(const float* __restrict__ dl,
                                                                const __nv_bfloat16* __restrict__ h, int64_t R, int H,
                                                                int rows_per_block, float* __restrict__ partial) {
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = (r0 + rows_per_block < R) ? r0 + rows_per_block : R;
  for (int u = threadIdx.x; u < H; u += 256) {
    float acc = 0.f;
    for (int64_t r = r0; r < r1; ++r) acc += dl[r] * __bfloat162float(h[r * H + u]);
    partial[(int64_t)blockIdx.x * (H + 1) + u] = acc;
  }
  if (threadIdx.x == 0) {
    float acc = 0.f;
    for (int64_t r = r0; r < r1; ++r) acc += dl[r];
    partial[(int64_t)blockIdx.x * (H + 1) + H] = acc;
  }
}
__global__ void head_grad_final_kernel(const float* __restrict__ partial, int nblocks, int H, float* __restrict__ dw,
                                       float* __restrict__ db) {
  const int u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u > H) return;
  float acc = 0.f;
  for (int i = 0; i < nblocks; ++i) acc += partial[(int64_t)i * (H + 1) + u];
  if (u < H) dw[u] = acc; else db[0] = acc;
}

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, int64_t n, float lr, float b1, float b2, float eps, float bc1,
                            float bc2_sqrt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gi = g[i];
  const float mi = b1 * m[i] + (1.f - b1) * gi;
  const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  const float denom = sqrtf(vi) / bc2_sqrt + eps;
  p[i] -= (lr / bc1) * (mi / denom);
}

}  // namespace avvad

using namespace avvad;

// ---- tape / workspace geometry (shared with lstm.cu through these helpers) --------------------------------------
// Per layer l the tape holds, each region 256-byte aligned: gates bf16 [B][T][4H] (gate-interleaved, element 4u+g),
// c f32 [B][T][H], hseq bf16 [B][T][H].  tape_offsets() is the one place that lays it out.
namespace avvad {
struct TapeOffsets {
  size_t gates, c, hseq, per_layer;
};
static TapeOffsets tape_offsets(int l, int H, int64_t B, int64_t T) {
  const size_t g = align_up((size_t)B * T * 4 * H * 2, 256), c = align_up((size_t)B * T * H * 4, 256),
               h = align_up((size_t)B * T * H * 2, 256);
  const size_t base = (size_t)l * (g + c + h);
  return TapeOffsets{base, base + g, base + g + c, g + c + h};
}
}  // namespace avvad

extern "C" size_t avvad_lstm_tape_bytes(int layers, int hidden, int64_t B, int64_t T) {
  if (layers <= 0 || hidden <= 0 || B <= 0 || T <= 0) return 0;
  return tape_offsets(0, hidden, B, T).per_layer * layers + 256;
}

// Byte offsets of the tape's tensors (inspection hook used by the state tests): offsets[3l + {0, 1, 2}] = gates, c and
// hseq of layer l.
extern "C" int avvad_lstm_tape_layout(int layers, int hidden, int64_t B, int64_t T, int64_t* offsets, int count) {
  AVVAD_CHECK_ARG(layers >= 1 && layers <= 8 && hidden > 0 && B > 0 && T > 0, "bad sizes");
  AVVAD_CHECK_ARG(offsets && count == 3 * layers, "offsets must hold 3 entries per layer");
  for (int l = 0; l < layers; ++l) {
    const TapeOffsets o = tape_offsets(l, hidden, B, T);
    offsets[3 * l + 0] = (int64_t)o.gates;
    offsets[3 * l + 1] = (int64_t)o.c;
    offsets[3 * l + 2] = (int64_t)o.hseq;
  }
  return AVVAD_OK;
}

extern "C" int avvad_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                               float beta1, float beta2, float eps, int64_t step, void* stream) {
  AVVAD_CHECK_ARG(param && grad && exp_avg && exp_avg_sq && n > 0 && step >= 1, "bad argument");
  const float bc1 = 1.f - powf(beta1, (float)step);
  const float bc2 = 1.f - powf(beta2, (float)step);
  adam_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1,
                                                                            beta2, eps, bc1, sqrtf(bc2));
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}

namespace avvad {
// The backward recurrence is 2 launches per time step and layer (1,268 for T = 317, two layers), each a few
// microseconds of work: issued one by one the step is bound by launch latency.  The T-step loop of a layer is therefore
// captured once into a CUDA graph and replayed while every pointer baked into its kernel parameters is unchanged (the
// key below); the per-call inputs that PyTorch re-allocates (lengths, dlogits) are first copied into the caller's
// workspace so that a steady-state training loop always hits the cache.  AVVAD_BPTT_GRAPH=0 disables it.
constexpr int kBpttSlots = 40;      // graphs: per layer (0, 1), wavefront (2), per (layer, chunk) of the overlapped chains
constexpr int kBpttMaxChunks = 16;
struct BpttGraphCache {
  cudaGraphExec_t exec[kBpttSlots] = {};
  std::vector<uintptr_t> key[kBpttSlots];
  size_t nodes[kBpttSlots] = {};
  // overlapped two-layer backward: layer 0's chain runs on `side`, one chunk of time steps behind layer 1
  cudaStream_t side = nullptr;
  cudaEvent_t ev_chunk[kBpttMaxChunks] = {};
  cudaEvent_t ev_side_done = nullptr;
  // Capture happens on a private stream: PyTorch's default current stream is the legacy NULL stream, which cannot be
  // captured; the instantiated graph is then launched into the caller's stream (any stream, the NULL stream included).
  cudaStream_t cap_stream = nullptr;
  cudaStream_t cap_stream2 = nullptr;  // forked branch of the two-GEMM wavefront
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int cap_device = -1;
  ~BpttGraphCache() {
    for (auto e : exec)
      if (e) cudaGraphExecDestroy(e);
    if (cap_stream) cudaStreamDestroy(cap_stream);
    if (cap_stream2) cudaStreamDestroy(cap_stream2);
    if (ev_fork) cudaEventDestroy(ev_fork);
    if (ev_join) cudaEventDestroy(ev_join);
    if (side) cudaStreamDestroy(side);
    for (auto e : ev_chunk)
      if (e) cudaEventDestroy(e);
    if (ev_side_done) cudaEventDestroy(ev_side_done);
  }
};
BpttGraphCache* bptt_cache_create() { return new BpttGraphCache(); }
void bptt_cache_destroy(BpttGraphCache* c) { delete c; }

// exposed to lstm.cu
int lstm_backward_impl(int layers, int input_size, int64_t ld0, int H, int y_dim, __nv_bfloat16* const* w_ih,
                       __nv_bfloat16* const* w_hh, const float* head_w32, const __nv_bfloat16* head_w16,
                       const void* x_bf16, const int32_t* lengths,
                       int64_t B, int64_t T, void* tape, const float* dlogits, void* workspace, size_t workspace_bytes,
                       float* const* dW_ih, float* const* dW_hh, float* const* db, float* dW_head, float* db_head,
                       float* dx, cudaStream_t st, BpttGraphCache* cache);
// split-K factor of the per-step recurrent-gradient GEMMs (AVVAD_BPTT_SPLIT = 1..8, buffers are sized for 8)
constexpr int kBpttSplitMax = 8;
// Default: 8 for per-rank batches up to 64 rows (one m-tile: 256 CTAs instead of 128, backward 6.0 -> 5.4 ms at B = 32),
// 4 above (B = 256: 16.7 ms with 4, 17.0 with 8, 19.7 with 2).
static int bptt_split(int64_t B) {
  static int v = [] {
    const char* e = getenv("AVVAD_BPTT_SPLIT");
    int x = e ? atoi(e) : 0;
    return x < 0 ? 0 : (x > kBpttSplitMax ? kBpttSplitMax : x);
  }();
  return v ? v : (B <= 64 ? 8 : 4);
}

// Two layers run as a wavefront (layer 0 one step behind layer 1): T + 1 dependent iterations instead of 2T.
//   mode 1 (2B <= 128): one block-structured GEMM per iteration (both layers in one 128-row MMA block)
//   mode 2 (larger batches): two GEMMs per iteration on forked streams of the captured graph
// AVVAD_BPTT_WAVEFRONT=0 disables both, =1 (default) allows only mode 1, =2 both.  Measured (B200, T = 317, backward of
// 2 x LSTM-1024): mode 1 7.9 -> 6.1 ms at B = 32 and 8.8 -> 7.3 ms at B = 64; mode 2 with the GEMMs in order 9.9 -> 9.5 ms
// at B = 96, 11.9 -> 11.8 at B = 128 and 15.5 -> 19.0 ms at B = 256 (the merged cell kernel and the extra N = H columns
// cost more than the shorter chain saves once a step fills the GPU), forked onto two captured streams 43.7 ms.
static int bptt_wavefront(int layers, int64_t B) {
  static int v = [] {
    const char* e = getenv("AVVAD_BPTT_WAVEFRONT");
    return e ? atoi(e) : 1;
  }();
  if (v == 0 || layers != 2) return 0;
  if (2 * B <= 128) return 1;
  return v >= 2 ? 2 : 0;
}

static bool bptt_graph_enabled() {
  static int v = [] {
    const char* e = getenv("AVVAD_BPTT_GRAPH");
    return (e && atoi(e) == 0) ? 0 : 1;
  }();
  return v != 0;
}

size_t lstm_backward_workspace(int layers, int input_size, int64_t ld0, int H, int y_dim, int64_t B, int64_t T);

struct TapeView {
  __nv_bfloat16* gates;
  float* c;
  __nv_bfloat16* hseq;
};
TapeView tape_layer(void* tape, int l, int H, int64_t B, int64_t T) {
  const TapeOffsets o = tape_offsets(l, H, B, T);
  uint8_t* p = (uint8_t*)tape;
  TapeView v;
  v.gates = (__nv_bfloat16*)(p + o.gates);
  v.c = (float*)(p + o.c);
  v.hseq = (__nv_bfloat16*)(p + o.hseq);
  return v;
}

static int64_t head_pad(int y_dim) { return ((int64_t)y_dim + 63) / 64 * 64; }

size_t lstm_backward_workspace(int layers, int input_size, int64_t ld0, int H, int y_dim, int64_t B, int64_t T) {
  (void)input_size;
  const int64_t BT = B * T, BTp = (BT + 63) / 64 * 64;
  const int64_t maxI = ld0 > H ? ld0 : H;
  size_t s = 0;
  s += align_up((size_t)BT * 4 * H * 2, 256);          // dG
  s += align_up((size_t)4 * H * BTp * 2, 256);         // dG^T
  s += align_up((size_t)maxI * BTp * 2, 256);          // X^T / H_prev^T
  s += 2 * align_up((size_t)BT * maxI * 4, 256);       // dY ping-pong (f32)
  s += (kBpttSplitMax + 1) * align_up((size_t)B * H * 4, 256);  // dh_rec split-K partials, dc
  s += align_up((size_t)4 * H * maxI * 4, 256);        // dW' (interleaved)
  s += align_up((size_t)maxI * 4 * H * 2, 256);        // W^T (bf16)
  s += align_up((size_t)1024 * (H + 1) * 4, 256);      // head partials
  s += align_up((size_t)B * 4, 256) + align_up((size_t)BT * 4, 256);  // stable copies of lengths / dlogits (y_dim == 1)
  if (bptt_wavefront(layers, B)) {
    const int64_t rows = 2 * B > 128 ? 2 * B : 128;
    s += align_up((size_t)BT * 4 * H * 2, 256);                        // second dG (both layers are live at once)
    s += align_up((size_t)128 * 8 * H * 2, 256);                       // A [2B <= 128][8H] (mode 1)
    s += align_up((size_t)2 * H * 8 * H * 2, 256);                     // Wcat [2H][8H]
    s += align_up((size_t)kBpttSplitMax * rows * 2 * H * 4, 256);         // C partials [split][2B][2H]
    s += align_up((size_t)2 * B * H * 4, 256);                         // dc of both layers
  }
  if (layers == 2 && !bptt_wavefront(layers, B)) {     // overlapped chains (see lstm_backward_impl)
    s += align_up((size_t)BT * 4 * H * 2, 256);                        // second dG
    s += (kBpttSplitMax + 1) * align_up((size_t)B * H * 4, 256);       // layer 0's dh_rec partials, dc
    s += 2 * align_up((size_t)H * 4 * H * 2, 256);                     // W_hh0'^T, W_ih1'^T
  }
  if (y_dim > 1) {
    const int64_t yp = head_pad(y_dim);
    s += align_up((size_t)BT * yp * 2, 256);           // dlogits bf16, padded columns
    s += align_up((size_t)yp * BTp * 2, 256);          // its transpose
    s += align_up((size_t)H * yp * 2, 256);            // W_head^T bf16 [H][yp]
  }
  return s + 1024;
}

// Runs `steps(stream)` -- a long chain of tiny dependent launches -- either directly (cache == nullptr) or as a CUDA graph
// captured once on the cache's private stream and replayed while `key` (every pointer / size baked into the kernel
// parameters) is unchanged.
static int bptt_cache_streams(BpttGraphCache* cache) {
  int dev = 0;
  AVVAD_CUDA(cudaGetDevice(&dev));
  if (!cache->cap_stream || cache->cap_device != dev) {
    if (cache->cap_stream) cudaStreamDestroy(cache->cap_stream);
    if (cache->cap_stream2) cudaStreamDestroy(cache->cap_stream2);
    if (cache->ev_fork) cudaEventDestroy(cache->ev_fork);
    if (cache->ev_join) cudaEventDestroy(cache->ev_join);
    cache->cap_stream = cache->cap_stream2 = nullptr;
    cache->ev_fork = cache->ev_join = nullptr;
    AVVAD_CUDA(cudaStreamCreateWithFlags(&cache->cap_stream, cudaStreamNonBlocking));
    AVVAD_CUDA(cudaStreamCreateWithFlags(&cache->cap_stream2, cudaStreamNonBlocking));
    AVVAD_CUDA(cudaEventCreateWithFlags(&cache->ev_fork, cudaEventDisableTiming));
    AVVAD_CUDA(cudaEventCreateWithFlags(&cache->ev_join, cudaEventDisableTiming));
    if (cache->side) cudaStreamDestroy(cache->side);
    cache->side = nullptr;
    AVVAD_CUDA(cudaStreamCreateWithFlags(&cache->side, cudaStreamNonBlocking));
    for (auto& e : cache->ev_chunk) {
      if (e) cudaEventDestroy(e);
      e = nullptr;
      AVVAD_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    if (cache->ev_side_done) cudaEventDestroy(cache->ev_side_done);
    AVVAD_CUDA(cudaEventCreateWithFlags(&cache->ev_side_done, cudaEventDisableTiming));
    cache->cap_device = dev;
    for (auto& e : cache->exec) {  // graphs belong to the previous device
      if (e) cudaGraphExecDestroy(e);
      e = nullptr;
    }
  }
  return AVVAD_OK;
}

template <class Warm, class Steps>
static int run_captured(BpttGraphCache* cache, int slot, std::vector<uintptr_t> key, Warm&& warm, Steps&& steps,
                        cudaStream_t st) {
  if (!cache) return steps(st);
  int rcs = bptt_cache_streams(cache);
  if (rcs) return rcs;
  key.push_back((uintptr_t)cache->cap_device);
  if (!cache->exec[slot] || cache->key[slot] != key) {
    if (cache->exec[slot]) {
      cudaGraphExecDestroy(cache->exec[slot]);
      cache->exec[slot] = nullptr;
    }
    int rc0 = warm();
    if (rc0) return rc0;
    const uint64_t before = g_launches.load();
    AVVAD_CUDA(cudaStreamBeginCapture(cache->cap_stream, cudaStreamCaptureModeThreadLocal));
    int rc = steps(cache->cap_stream);
    cudaGraph_t graph = nullptr;
    cudaError_t ce = cudaStreamEndCapture(cache->cap_stream, &graph);
    if (rc) {
      if (graph) cudaGraphDestroy(graph);
      return rc;
    }
    if (ce != cudaSuccess) {
      set_error(std::string("BPTT graph capture failed: ") + cudaGetErrorString(ce));
      return AVVAD_ERR_CUDA;
    }
    ce = cudaGraphInstantiate(&cache->exec[slot], graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) {
      cache->exec[slot] = nullptr;
      set_error(std::string("BPTT graph instantiation failed: ") + cudaGetErrorString(ce));
      return AVVAD_ERR_CUDA;
    }
    cache->key[slot] = key;
    cache->nodes[slot] = (size_t)(g_launches.load() - before);  // launches counted while capturing = kernel nodes
  } else {
    g_launches.fetch_add(cache->nodes[slot], std::memory_order_relaxed);  // a replay launches every captured kernel
  }
  AVVAD_CUDA(cudaGraphLaunch(cache->exec[slot], st));
  return AVVAD_OK;
}

int lstm_backward_impl(int layers, int input_size, int64_t ld0, int H, int y_dim, __nv_bfloat16* const* w_ih,
                       __nv_bfloat16* const* w_hh, const float* head_w32, const __nv_bfloat16* head_w16,
                       const void* x_bf16, const int32_t* lengths,
                       int64_t B, int64_t T, void* tape, const float* dlogits, void* workspace, size_t workspace_bytes,
                       float* const* dW_ih, float* const* dW_hh, float* const* db, float* dW_head, float* db_head,
                       float* dx, cudaStream_t st, BpttGraphCache* cache) {
  AVVAD_CHECK_ARG(y_dim >= 1, "bad y_dim");
  AVVAD_CHECK_ARG(workspace_bytes >= lstm_backward_workspace(layers, input_size, ld0, H, y_dim, B, T),
                  "workspace too small");
  const int64_t BT = B * T, BTp = (BT + 63) / 64 * 64;
  const int64_t maxI = ld0 > H ? ld0 : H;
  const int H4 = 4 * H;
  uint8_t* p = (uint8_t*)workspace;
  auto take = [&](size_t bytes) { void* q = p; p += align_up(bytes, 256); return q; };
  __nv_bfloat16* dG = (__nv_bfloat16*)take((size_t)BT * H4 * 2);
  __nv_bfloat16* dGT = (__nv_bfloat16*)take((size_t)H4 * BTp * 2);
  __nv_bfloat16* XT = (__nv_bfloat16*)take((size_t)maxI * BTp * 2);
  float* dYa = (float*)take((size_t)BT * maxI * 4);
  float* dYb = (float*)take((size_t)BT * maxI * 4);
  float* dh_rec = (float*)take((size_t)kBpttSplitMax * align_up((size_t)B * H * 4, 256));
  float* dc = (float*)take((size_t)B * H * 4);
  float* dWp = (float*)take((size_t)H4 * maxI * 4);
  __nv_bfloat16* WT = (__nv_bfloat16*)take((size_t)maxI * H4 * 2);
  float* partial = (float*)take((size_t)1024 * (H + 1) * 4);
  int32_t* len_st = (int32_t*)take((size_t)B * 4);
  float* dl_st = (float*)take((size_t)BT * 4);
  // stable-address copies of the per-call inputs the step kernels read (see BpttGraphCache)
  AVVAD_CUDA(cudaMemcpyAsync(len_st, lengths, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
  if (y_dim == 1) AVVAD_CUDA(cudaMemcpyAsync(dl_st, dlogits, (size_t)BT * 4, cudaMemcpyDeviceToDevice, st));
  const float* dl_step = (y_dim == 1) ? dl_st : dlogits;
  const bool use_graph = cache && bptt_graph_enabled() && !tc::profiling_on() && !sync_debug();
  const int kBpttSplit = bptt_split(B);  // split-K factor of the per-step GEMMs of this call

  const float* dY_head = nullptr;  // y_dim > 1: gradient of the top layer's output through the head (GEMM)
  if (y_dim == 1) {
    // ---- head gradients (y_dim == 1): dl = dlogits [BT]
    TapeView top = tape_layer(tape, layers - 1, H, B, T);
    int nblocks = (int)std::min<int64_t>(1024, ceil_div(BT, 64));
    int rows_per_block = (int)ceil_div(BT, nblocks);
    nblocks = (int)ceil_div(BT, rows_per_block);
    head_grad_partial_kernel<<<nblocks, 256, 0, st>>>(dlogits, top.hseq, BT, H, rows_per_block, partial);
    AVVAD_LAUNCHED();
    head_grad_final_kernel<<<(unsigned)ceil_div(H + 1, 256), 256, 0, st>>>(partial, nblocks, H, dW_head, db_head);
    AVVAD_LAUNCHED();
  } else {
    // ---- head gradients (IBM head, y_dim = 513): three GEMMs on bf16 copies of dlogits
    //   dY_top [BT][H]   = dL [BT][yp] * W_head [yp][H]
    //   dW_head [y][H]   = dL^T [yp][BT] * h_top [BT][H]
    //   db_head [y]      = column sums of dL (fp32)
    const int64_t yp = head_pad(y_dim);
    __nv_bfloat16* dl16 = (__nv_bfloat16*)take((size_t)BT * yp * 2);
    __nv_bfloat16* dlT = (__nv_bfloat16*)take((size_t)yp * BTp * 2);
    __nv_bfloat16* WTh = (__nv_bfloat16*)take((size_t)H * yp * 2);
    TapeView top = tape_layer(tape, layers - 1, H, B, T);
    int rc = avvad_pack_rows_bf16(dlogits, y_dim, dl16, yp, 0, BT, y_dim, 1, st);
    if (rc) return rc;
    head_wt_kernel<<<(unsigned)ceil_div((int64_t)H * yp, 256), 256, 0, st>>>(head_w16, y_dim, H, (int)yp, WTh);
    AVVAD_LAUNCHED();
    {
      tc::EpiParams ep{};
      ep.C = dYa;
      ep.ldc = H;
      rc = tc::gemm_dispatch(dl16, yp, WTh, yp, BT, H, (int)yp, ep, tc::EPI_F32, 0, st);
      if (rc) return rc;
      dY_head = dYa;
    }
    {
      dim3 grid((unsigned)ceil_div(BTp, 32), (unsigned)ceil_div(yp, 32));
      transpose_bf16_kernel<<<grid, dim3(32, 8), 0, st>>>(dl16, BT, (int)yp, yp, BTp, 0, (int)T, dlT);
      AVVAD_LAUNCHED();
      dim3 grid2((unsigned)ceil_div(BTp, 32), (unsigned)ceil_div(H, 32));
      transpose_bf16_kernel<<<grid2, dim3(32, 8), 0, st>>>(top.hseq, BT, H, H, BTp, 0, (int)T, XT);
      AVVAD_LAUNCHED();
      tc::EpiParams ep{};
      ep.C = dWp;
      ep.ldc = H;
      rc = tc::gemm_dispatch(dlT, BTp, XT, BTp, yp, H, (int)BTp, ep, tc::EPI_F32, 0, st);
      if (rc) return rc;
      AVVAD_CUDA(cudaMemcpyAsync(dW_head, dWp, (size_t)y_dim * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    colsum_f32_kernel<<<(unsigned)ceil_div(y_dim, 64), 256, 0, st>>>(dlogits, BT, y_dim, db_head);
    AVVAD_LAUNCHED();
  }

  // ---- parameter gradients of layer l from its complete gate gradients dGl [BT][4H]; optionally dX = dGl * W_ih'
  auto weight_grads = [&](int l, const __nv_bfloat16* dGl, float* dx_dst) -> int {
    TapeView tv = tape_layer(tape, l, H, B, T);
    const int64_t ld_in = (l == 0) ? ld0 : H;
    const int I = (l == 0) ? input_size : H;
    const __nv_bfloat16* Xin = (l == 0) ? (const __nv_bfloat16*)x_bf16 : tape_layer(tape, l - 1, H, B, T).hseq;
    // db (= db_ih = db_hh)
    bias_grad_partial_kernel<<<dim3(H4 / 256, kBiasChunks), 256, 0, st>>>(dGl, BT, H4, dWp);  // dWp is free here
    AVVAD_LAUNCHED();
    bias_grad_final_kernel<<<(unsigned)ceil_div(H4, 256), 256, 0, st>>>(dWp, H, db[l]);
    AVVAD_LAUNCHED();
    // dG^T [4H][BTp]
    {
      dim3 grid((unsigned)ceil_div(BTp, 32), (unsigned)ceil_div(H4, 32));
      transpose_bf16_kernel<<<grid, dim3(32, 8), 0, st>>>(dGl, BT, H4, H4, BTp, 0, (int)T, dGT);
      AVVAD_LAUNCHED();
    }
    // dW_ih' = dG^T * X  -> [4H][ld_in]
    {
      dim3 grid((unsigned)ceil_div(BTp, 32), (unsigned)ceil_div(ld_in, 32));
      transpose_bf16_kernel<<<grid, dim3(32, 8), 0, st>>>(Xin, BT, (int)ld_in, ld_in, BTp, 0, (int)T, XT);
      AVVAD_LAUNCHED();
      tc::EpiParams ep{};
      ep.C = dWp;
      ep.ldc = ld_in;
      int rc = tc::gemm_dispatch(dGT, BTp, XT, BTp, H4, (int)ld_in, (int)BTp, ep, tc::EPI_F32, 0, st);
      if (rc) return rc;
      deinterleave_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * I, 256), 256, 0, st>>>(dWp, H, I, (int)ld_in, dW_ih[l]);
      AVVAD_LAUNCHED();
    }
    // dW_hh' = dG^T * H_prev -> [4H][H]
    {
      dim3 grid((unsigned)ceil_div(BTp, 32), (unsigned)ceil_div(H, 32));
      transpose_bf16_kernel<<<grid, dim3(32, 8), 0, st>>>(tv.hseq, BT, H, H, BTp, 1, (int)T, XT);
      AVVAD_LAUNCHED();
      tc::EpiParams ep{};
      ep.C = dWp;
      ep.ldc = H;
      int rc = tc::gemm_dispatch(dGT, BTp, XT, BTp, H4, H, (int)BTp, ep, tc::EPI_F32, 0, st);
      if (rc) return rc;
      deinterleave_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * H, 256), 256, 0, st>>>(dWp, H, H, H, dW_hh[l]);
      AVVAD_LAUNCHED();
    }
    if (dx_dst) {
      transpose_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * ld_in, 256), 256, 0, st>>>(w_ih[l], H4, (int)ld_in,
                                                                                       (int)ld_in, WT);
      AVVAD_LAUNCHED();
      tc::EpiParams ep{};
      ep.C = dx_dst;
      ep.ldc = (l == 0) ? I : ld_in;
      // l == 0: only the first I (un-padded) columns are written (N guard in the epilogue)
      int rc = tc::gemm_dispatch(dGl, H4, WT, H4, BT, (l == 0) ? I : (int)ld_in, H4, ep, tc::EPI_F32, 0, st);
      if (rc) return rc;
    }
    return AVVAD_OK;
  };

  const int wf_mode = bptt_wavefront(layers, B);
  if (wf_mode) {
    // ---- both layers as one wavefront: T + 1 dependent iterations instead of 2T (see lstm_bwd_cell_wf_kernel)
    const int64_t rows = 2 * B > 128 ? 2 * B : 128;
    __nv_bfloat16* dG0 = (__nv_bfloat16*)take((size_t)BT * H4 * 2);
    __nv_bfloat16* Abuf = (__nv_bfloat16*)take((size_t)128 * 8 * H * 2);
    __nv_bfloat16* Wcat = (__nv_bfloat16*)take((size_t)2 * H * 8 * H * 2);
    float* Cpart = (float*)take((size_t)kBpttSplitMax * rows * 2 * H * 4);
    float* dc2 = (float*)take((size_t)2 * B * H * 4);
    TapeView t1 = tape_layer(tape, 1, H, B, T), t0 = tape_layer(tape, 0, H, B, T);
    lstm_wf_pack_w_kernel<<<(unsigned)ceil_div((int64_t)2 * H * 8 * H, 256), 256, 0, st>>>(w_hh[1], w_ih[1], w_hh[0], H,
                                                                                          Wcat);
    AVVAD_LAUNCHED();
    AVVAD_CUDA(cudaMemsetAsync(dc2, 0, (size_t)2 * B * H * 4, st));
    if (wf_mode == 1) AVVAD_CUDA(cudaMemsetAsync(Abuf, 0, (size_t)128 * 8 * H * 2, st));  // rows 2B..127 stay zero
    const int64_t cstride = 2 * B * 2 * H;
    // mode 1: C [2B][2H] = A [2B][8H] * Wcat^T
    auto wf_gemm = [&](cudaStream_t s2) -> int {
      tc::EpiParams ep{};
      ep.C = Cpart;
      ep.ldc = 2 * H;
      return tc::launch_tma_gemm(Abuf, 8 * H, Wcat, 8 * H, 2 * B, 2 * H, 8 * H, ep, tc::EPI_F32, 64, s2, kBpttSplit,
                                 cstride);
    };
    // mode 2: rows 0..B-1 = dG1_t [B][4H] * [W_hh1^T | W_ih1^T] (N = 2H); rows B..2B-1 = dG0_t * W_hh0^T (N = H); both
    // read the first / second 4H columns of Wcat's rows
    auto gemm_l1 = [&](int t, cudaStream_t s2) -> int {
      tc::EpiParams ep{};
      ep.C = Cpart;
      ep.ldc = 2 * H;
      return tc::launch_tma_gemm(dG + (int64_t)t * H4, (int64_t)T * H4, Wcat, 8 * H, B, 2 * H, H4, ep, tc::EPI_F32, 64, s2,
                                 kBpttSplit, cstride);
    };
    auto gemm_l0 = [&](int t, cudaStream_t s2) -> int {
      tc::EpiParams ep{};
      ep.C = Cpart + B * 2 * H;
      ep.ldc = 2 * H;
      return tc::launch_tma_gemm(dG0 + (int64_t)t * H4, (int64_t)T * H4, Wcat + H4, 8 * H, B, H, H4, ep, tc::EPI_F32, 64, s2,
                                 kBpttSplit, cstride);
    };
    auto run_wf = [&](cudaStream_t s1) -> int {
      // Forking the layer-0 GEMM onto a second captured stream was measured 3-4x SLOWER than issuing both GEMMs in order
      // (B = 256: 43.7 ms against 15.5 ms for the layer-by-layer loop): AVVAD_BPTT_FORK=1 keeps the experiment reachable.
      static int fork_pref = [] {
        const char* e = getenv("AVVAD_BPTT_FORK");
        return e ? atoi(e) : 0;
      }();
      cudaStream_t s2 = (use_graph && wf_mode == 2 && fork_pref) ? cache->cap_stream2 : nullptr;
      for (int s = 0; s <= (int)T; ++s) {
        lstm_bwd_cell_wf_kernel<<<dim3((unsigned)ceil_div(B * H, 256), 2), 256, 0, s1>>>(
            t1.gates, t1.c, t0.gates, t0.c, dY_head, dl_step, head_w32, Cpart, kBpttSplit, dc2, len_st, (int)B, (int)T, H,
            s, dG, dG0, wf_mode == 1 ? Abuf : nullptr);
        AVVAD_LAUNCHED();
        if (s >= (int)T) break;
        if (wf_mode == 1) {
          int rc = wf_gemm(s1);
          if (rc) return rc;
          continue;
        }
        const int tl1 = (int)T - 1 - s, tl0 = (int)T - s;   // the steps the layers just finished
        const bool need0 = s >= 1 && tl0 > 0;               // layer 0's recurrent term for step tl0 - 1
        if (need0 && s2) {
          AVVAD_CUDA(cudaEventRecord(cache->ev_fork, s1));
          AVVAD_CUDA(cudaStreamWaitEvent(s2, cache->ev_fork, 0));
          int rc = gemm_l0(tl0, s2);
          if (rc) return rc;
          AVVAD_CUDA(cudaEventRecord(cache->ev_join, s2));
        }
        int rc = gemm_l1(tl1, s1);
        if (rc) return rc;
        if (need0) {
          if (s2) AVVAD_CUDA(cudaStreamWaitEvent(s1, cache->ev_join, 0));
          else {
            rc = gemm_l0(tl0, s1);
            if (rc) return rc;
          }
        }
      }
      return AVVAD_OK;
    };
    const std::vector<uintptr_t> key = {(uintptr_t)t1.gates, (uintptr_t)t1.c, (uintptr_t)t0.gates, (uintptr_t)t0.c,
                                        (uintptr_t)dY_head, (uintptr_t)dl_step, (uintptr_t)head_w32, (uintptr_t)Cpart,
                                        (uintptr_t)dc2, (uintptr_t)len_st, (uintptr_t)dG, (uintptr_t)dG0,
                                        (uintptr_t)Abuf, (uintptr_t)Wcat, (uintptr_t)B, (uintptr_t)T, (uintptr_t)H,
                                        (uintptr_t)wf_mode};
    auto warm = [&]() -> int {
      if (wf_mode == 1) return wf_gemm(st);
      int rc = gemm_l1(0, st);
      return rc ? rc : gemm_l0(0, st);
    };
    int rc = run_captured(use_graph ? cache : nullptr, 2, key, warm, run_wf, st);
    if (rc) return rc;
    rc = weight_grads(1, dG, nullptr);
    if (rc) return rc;
    return weight_grads(0, dG0, dx);
  }

  // ---- two layers, larger batches: the recurrences of both layers as chunked chains on two streams.  Layer 1 runs its
  // steps in chunks (t descending); after each chunk the input gradient of that chunk (dY0 = dG1 * W_ih1, one time-major
  // GEMM) and then layer 0's steps of the same chunk run on a side stream while layer 1 continues: every step is a
  // latency-bound (cell kernel, split-K GEMM) pair, so the two chains overlap.  AVVAD_BPTT_CHUNKS=1 disables it.
  static int chunks_pref = [] {
    const char* e = getenv("AVVAD_BPTT_CHUNKS");
    int v = e ? atoi(e) : 8;
    return v < 1 ? 1 : (v > kBpttMaxChunks ? kBpttMaxChunks : v);
  }();
  int n_chunks = chunks_pref;
  while (n_chunks > 1 && T / n_chunks < 16) --n_chunks;
  if (layers == 2 && n_chunks > 1 && cache && !tc::profiling_on() && !sync_debug()) {
    int rcs = bptt_cache_streams(cache);
    if (rcs) return rcs;
    __nv_bfloat16* dG0 = (__nv_bfloat16*)take((size_t)BT * H4 * 2);
    float* dh_rec0 = (float*)take((size_t)kBpttSplitMax * align_up((size_t)B * H * 4, 256));
    float* dc0 = (float*)take((size_t)B * H * 4);
    __nv_bfloat16* WT0 = (__nv_bfloat16*)take((size_t)H * H4 * 2);
    __nv_bfloat16* WTi = (__nv_bfloat16*)take((size_t)H * H4 * 2);
    float* dY0 = dY_head ? dYb : dYa;  // [BT][H] fp32: gradient w.r.t. layer 0's output, written chunk by chunk
    TapeView tv1 = tape_layer(tape, 1, H, B, T), tv0 = tape_layer(tape, 0, H, B, T);
    transpose_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * H, 256), 256, 0, st>>>(w_hh[1], H4, H, H, WT);
    AVVAD_LAUNCHED();
    transpose_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * H, 256), 256, 0, st>>>(w_hh[0], H4, H, H, WT0);
    AVVAD_LAUNCHED();
    transpose_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * H, 256), 256, 0, st>>>(w_ih[1], H4, H, H, WTi);
    AVVAD_LAUNCHED();
    AVVAD_CUDA(cudaMemsetAsync(dc, 0, (size_t)B * H * 4, st));
    AVVAD_CUDA(cudaMemsetAsync(dc0, 0, (size_t)B * H * 4, st));
    // steps te-1 .. tb of one layer: (cell, recurrent split-K GEMM) pairs
    auto steps_of = [&](const TapeView& tv, const float* dYl, float* dh, float* dcl, __nv_bfloat16* dGl,
                        const __nv_bfloat16* WTl, int tb, int te, cudaStream_t s2) -> int {
      for (int t = te - 1; t >= tb; --t) {
        const int has_rec = (t < (int)T - 1) ? kBpttSplit : 0;
        lstm_bwd_cell_kernel<<<(unsigned)ceil_div(B * H, 256), 256, 0, s2>>>(tv.gates, tv.c, dYl, dl_step, head_w32, dh, dcl,
                                                                            len_st, (int)B, (int)T, H, t, has_rec, dGl);
        AVVAD_LAUNCHED();
        if (t > 0) {
          tc::EpiParams ep{};
          ep.C = dh;
          ep.ldc = H;
          int rc = tc::launch_tma_gemm(dGl + (int64_t)t * H4, (int64_t)T * H4, WTl, H4, B, H, H4, ep, tc::EPI_F32, 64, s2,
                                       kBpttSplit, (int64_t)B * H);
          if (rc) return rc;
        }
      }
      return AVVAD_OK;
    };
    auto warm_of = [&](float* dh, const __nv_bfloat16* dGl, const __nv_bfloat16* WTl, cudaStream_t s2) -> int {
      tc::EpiParams ep{};
      ep.C = dh;
      ep.ldc = H;
      return tc::launch_tma_gemm(dGl, (int64_t)T * H4, WTl, H4, B, H, H4, ep, tc::EPI_F32, 64, s2, kBpttSplit,
                                 (int64_t)B * H);
    };
    cudaStream_t side = cache->side;
    // one real launch of the step GEMM before any capture (kernel attributes are set on first use, which cannot be
    // captured); it must not run between chunks: dh_rec carries the recurrent term from one chunk to the next
    {
      int rcw = warm_of(dh_rec, dG, WT, st);
      if (rcw) return rcw;
    }
    auto no_warm = []() -> int { return 0; };
    for (int c = n_chunks - 1; c >= 0; --c) {
      const int tb = (int)(T * c / n_chunks), te = (int)(T * (c + 1) / n_chunks);
      {  // layer 1, chunk c, on the caller's stream
        const std::vector<uintptr_t> key = {(uintptr_t)tv1.gates, (uintptr_t)tv1.c, (uintptr_t)dY_head, (uintptr_t)dl_step,
                                            (uintptr_t)head_w32, (uintptr_t)dh_rec, (uintptr_t)dc, (uintptr_t)len_st,
                                            (uintptr_t)dG, (uintptr_t)WT, (uintptr_t)B, (uintptr_t)T, (uintptr_t)H,
                                            (uintptr_t)tb, (uintptr_t)te, (uintptr_t)kBpttSplit};
        int rc = run_captured(use_graph ? cache : nullptr, 3 + c, key, no_warm,
                              [&](cudaStream_t s2) { return steps_of(tv1, dY_head, dh_rec, dc, dG, WT, tb, te, s2); }, st);
        if (rc) return rc;
      }
      AVVAD_CUDA(cudaEventRecord(cache->ev_chunk[c], st));
      AVVAD_CUDA(cudaStreamWaitEvent(side, cache->ev_chunk[c], 0));
      // dY0 of the chunk: rows (b, t in [tb, te)) of dG1 times W_ih1
      int rc = tc::launch_tma_gemm_tm(dG + (int64_t)tb * H4, H4, WTi, H4, B, te - tb, T, H, H4, dY0 + (int64_t)tb * H, H, side);
      if (rc) return rc;
      {  // layer 0, chunk c, on the side stream
        const std::vector<uintptr_t> key = {(uintptr_t)tv0.gates, (uintptr_t)tv0.c, (uintptr_t)dY0, (uintptr_t)dl_step,
                                            (uintptr_t)head_w32, (uintptr_t)dh_rec0, (uintptr_t)dc0, (uintptr_t)len_st,
                                            (uintptr_t)dG0, (uintptr_t)WT0, (uintptr_t)B, (uintptr_t)T, (uintptr_t)H,
                                            (uintptr_t)tb, (uintptr_t)te, (uintptr_t)kBpttSplit};
        rc = run_captured(use_graph ? cache : nullptr, 3 + kBpttMaxChunks + c, key, no_warm,
                          [&](cudaStream_t s2) { return steps_of(tv0, dY0, dh_rec0, dc0, dG0, WT0, tb, te, s2); }, side);
        if (rc) return rc;
      }
    }
    AVVAD_CUDA(cudaEventRecord(cache->ev_side_done, side));
    // layer 1's parameter gradients (large GEMMs over K = B*T) while layer 0's last chunks still run on the side stream
    int rc = weight_grads(1, dG, nullptr);
    if (rc) return rc;
    AVVAD_CUDA(cudaStreamWaitEvent(st, cache->ev_side_done, 0));
    return weight_grads(0, dG0, dx);
  }

  const float* dY = dY_head;  // null (y_dim == 1): the top layer takes dl * w_head on the fly
  float* dX_out = dY_head ? dYb : dYa;
  for (int l = layers - 1; l >= 0; --l) {
    TapeView tv = tape_layer(tape, l, H, B, T);

    // W_hh'^T [H][4H] for the recurrent gradient GEMM
    transpose_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * H, 256), 256, 0, st>>>(w_hh[l], H4, H, H, WT);
    AVVAD_LAUNCHED();
    AVVAD_CUDA(cudaMemsetAsync(dc, 0, (size_t)B * H * 4, st));
    auto run_steps = [&](cudaStream_t st) -> int {   // `st`: the caller's stream, or the capture stream
      for (int t = (int)T - 1; t >= 0; --t) {
        const int has_rec = (t < (int)T - 1) ? kBpttSplit : 0;  // number of partial products to sum
        lstm_bwd_cell_kernel<<<(unsigned)ceil_div(B * H, 256), 256, 0, st>>>(tv.gates, tv.c, dY, dl_step, head_w32, dh_rec,
                                                                            dc, len_st, (int)B, (int)T, H, t, has_rec, dG);
        AVVAD_LAUNCHED();
        if (t > 0) {
          tc::EpiParams ep{};
          ep.C = dh_rec;
          ep.ldc = H;
          // M = B is tiny: split K = 4H over kBpttSplit CTAs per output tile so the step fills the GPU
          int rc = tc::launch_tma_gemm(dG + (int64_t)t * H4, (int64_t)T * H4, WT, H4, B, H, H4, ep, tc::EPI_F32, 64, st,
                                       kBpttSplit, (int64_t)B * H);
          if (rc) return rc;
        }
      }
      return AVVAD_OK;
    };
    {
      const std::vector<uintptr_t> key = {(uintptr_t)tv.gates, (uintptr_t)tv.c, (uintptr_t)dY, (uintptr_t)dl_step,
                                          (uintptr_t)head_w32, (uintptr_t)dh_rec, (uintptr_t)dc, (uintptr_t)len_st,
                                          (uintptr_t)dG, (uintptr_t)WT, (uintptr_t)B, (uintptr_t)T, (uintptr_t)H};
      auto warm = [&]() -> int {   // the kernels' one-time attribute setup is not capturable: one real split-K launch
        tc::EpiParams ep{};
        ep.C = dh_rec;
        ep.ldc = H;
        return tc::launch_tma_gemm(dG, (int64_t)T * H4, WT, H4, B, H, H4, ep, tc::EPI_F32, 64, st, kBpttSplit,
                                   (int64_t)B * H);
      };
      int rc = run_captured(use_graph ? cache : nullptr, l, key, warm, run_steps, st);
      if (rc) return rc;
    }
    float* dst = (l == 0) ? dx : dX_out;
    int rc = weight_grads(l, dG, (l > 0 || dx) ? dst : nullptr);
    if (rc) return rc;
    if (l > 0 || dx) {
      dY = dst;
      dX_out = (dX_out == dYa) ? dYb : dYa;
    }
  }
  return AVVAD_OK;
}
}  // namespace avvad
