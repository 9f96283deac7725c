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
// With a carried state (avvad_lstm_backward_state) the same schedules run over a tape of T + 1 positions whose position 0
// holds the initial state; see the kState instantiations of the cell kernels and lstm_backward_state_impl.
#include <vector>

#include "bwd_common.cuh"
#include "gemm_tma.cuh"
#include "lstm_internal.cuh"

namespace avvad {

__device__ __forceinline__ float bf16lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }

// ---- stateful BPTT (avvad_lstm_backward_state).  The tape has T + 1 positions per row and lengths are shifted by one:
// position 0 holds the initial state (h_in in hseq, c_in in c) and is frozen -- read, never differentiated.  The cell
// kernels below take it as their kState instantiation:
//   * position t >= 1 reads cp = c[t-1], so the first step's forget-gate term uses c_in
//   * at the last valid position len_b (shifted) - 1 the incoming state gradients dh_out / dc_out [B][H] are added
//   * at position 0 nothing is written to dG but zeros; the state gradients leave as dh_in = the recurrent term of
//     step 1 (dG_1 * W_hh) and dc_in = dc after step 1.  A row of length 0 has its last valid position at 0, where
//     the recurrent term is exactly zero: dh_in = dh_out and dc_in = dc_out.
struct BwdStateArgs {
  const float* dh_out;  // [B][H] of this layer (zero-filled when the caller passes none)
  const float* dc_out;
  float* dh_in;         // null: no state gradient requested
  float* dc_in;
};
// One cell step backward: gate gradients (bf16, gate-interleaved) from dh and the cell-state gradient *dc, which is
// read in place and replaced by its value for step t-1.  The stateless kernels pass dc in global memory, so that the
// load stays where the arithmetic needs it.
__device__ __forceinline__ uint2 lstm_cell_bwd(uint2 gp, float c, float cp, float dh, float* dc) {
  const float gi = bf16lo(gp.x), gf = bf16hi(gp.x), gg = bf16lo(gp.y), go = bf16hi(gp.y);
  const float tc = tanhf(c);
  const float d_o = dh * tc * go * (1.f - go);
  const float dcc = dh * go * (1.f - tc * tc) + *dc;
  const float d_i = dcc * gg * gi * (1.f - gi);
  const float d_g = dcc * gi * (1.f - gg * gg);
  const float d_f = dcc * cp * gf * (1.f - gf);
  *dc = dcc * gf;
  uint2 o;
  o.x = pack_bf16x2(d_i, d_f);
  o.y = pack_bf16x2(d_g, d_o);
  return o;
}
// position 0 of a stateful tape: dh_rec_sum = the recurrent term from step 1 (exactly zero for a row of length 0)
__device__ __forceinline__ void lstm_state_grad_out(const BwdStateArgs& sa, int idx, bool last, float dh_rec_sum,
                                                    float dc) {
  if (sa.dh_in) sa.dh_in[idx] = (last ? sa.dh_out[idx] : 0.f) + dh_rec_sum;
  if (sa.dc_in) sa.dc_in[idx] = dc + (last ? sa.dc_out[idx] : 0.f);
}

// one thread per (b, u); `sa` is unused without kState
template <bool kState>
__global__ void lstm_bwd_cell_kernel(const __nv_bfloat16* __restrict__ gates, const float* __restrict__ cst,
                                     const float* __restrict__ dY, const float* __restrict__ dl,
                                     const float* __restrict__ w_head, const float* __restrict__ dh_rec,
                                     float* __restrict__ dc, const int32_t* __restrict__ lengths, int B, int T, int H,
                                     int t, int has_rec, __nv_bfloat16* __restrict__ dG, BwdStateArgs sa) {
  // dh_rec holds `has_rec` split-K partial products [has_rec][B][H] of the recurrent GEMM of step t+1
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * H) return;
  const int b = idx / H, u = idx - b * H;
  const int64_t row = (int64_t)b * T + t;
  uint2* out = reinterpret_cast<uint2*>(dG + row * 4 * H + 4 * u);
  const int len = lengths[b];
  if (kState && t == 0) {  // frozen initial state
    float rec = 0.f;
    for (int sp = 0; sp < has_rec; ++sp) rec += dh_rec[(int64_t)sp * B * H + idx];
    lstm_state_grad_out(sa, idx, len == 1, rec, dc[idx]);
    *out = make_uint2(0u, 0u);
    return;
  }
  if (t >= len) {  // padded step: no gradient flows (packed-sequence semantics)
    *out = make_uint2(0u, 0u);
    dc[idx] = 0.f;
    return;
  }
  const uint2 gp = *reinterpret_cast<const uint2*>(gates + row * 4 * H + 4 * u);
  const float c = cst[row * H + u];
  const float cp = (kState || t > 0) ? cst[(row - 1) * H + u] : 0.f;
  float dh = dY ? dY[row * H + u] : dl[row] * w_head[u];
  for (int sp = 0; sp < has_rec; ++sp) dh += dh_rec[(int64_t)sp * B * H + idx];
  if constexpr (kState) {
    float dcv = dc[idx];
    if (t == len - 1) {
      dh += sa.dh_out[idx];
      dcv += sa.dc_out[idx];
    }
    *out = lstm_cell_bwd(gp, c, cp, dh, &dcv);
    dc[idx] = dcv;
  } else {
    *out = lstm_cell_bwd(gp, c, cp, dh, dc + idx);
  }
}

// ---- two-layer wavefront (small per-rank batches): layer 1 at step t1 = T-1-s and layer 0 at step t0 = T-s run in the
// SAME launches, so the dependent chain is T+1 (cell, GEMM) pairs instead of 2T.  One GEMM per iteration does all three
// products on a block-structured operand:
//   A [2B][2*4H]:  rows 0..B-1   = [ dG1_t1 | 0 ],   rows B..2B-1 = [ 0 | dG0_t0 ]
//   W [2H][2*4H]:  rows 0..H-1   = [ W_hh1^T | W_hh0^T ],   rows H..2H-1 = [ W_ih1^T | 0 ]
//   C [2B][2H]  :  rows 0..B-1   = [ dh_rec1 | dY0_t1 ],    rows B..2B-1 = [ dh_rec0 | 0 ]
// which the next iteration's cell launch consumes (layer 0 then sits at the step layer 1 just left).  With kState it
// runs over T + 1 positions; sa0 / sa1: layer 0 / layer 1.
template <bool kState>
__global__ void lstm_bwd_cell_wf_kernel(const __nv_bfloat16* __restrict__ gates1, const float* __restrict__ cst1,
                                        const __nv_bfloat16* __restrict__ gates0, const float* __restrict__ cst0,
                                        const float* __restrict__ dY1, const float* __restrict__ dl,
                                        const float* __restrict__ w_head, const float* __restrict__ Cpart, int nsplit,
                                        float* __restrict__ dc2, const int32_t* __restrict__ lengths, int B, int T, int H,
                                        int s, __nv_bfloat16* __restrict__ dG1, __nv_bfloat16* __restrict__ dG0,
                                        __nv_bfloat16* __restrict__ Abuf, BwdStateArgs sa1, BwdStateArgs sa0) {
  const int layer = 1 - (int)blockIdx.y;   // blockIdx.y 0 -> layer 1, 1 -> layer 0
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * H) return;
  const int b = idx / H, u = idx - b * H;
  const int t = (layer == 1) ? (T - 1 - s) : (T - s);
  // Abuf is never null.  Its null tests and the two copies of cstride below keep the instructions of the kernels this
  // template replaced: without the tests ptxas schedules the stateless instantiation differently, and forward +
  // backward of 2 x LSTM-1024 at B = 32, T = 317 measured 8.97 -> 9.18 ms (one B200 at 1000 W).
  const int64_t K2 = 8ll * H;              // row length of Abuf
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
  const int64_t cstride0 = 2ll * B * 2 * H;  // one split-K partial of C
  const int len = lengths[b];
  if (kState && t == 0) {  // frozen initial state: the recurrent term of step 1 is dh_in
    float rec = 0.f;
    if (layer == 1) {
      if (s > 0)
        for (int sp = 0; sp < nsplit; ++sp) rec += Cpart[sp * cstride0 + (int64_t)b * 2 * H + u];
    } else if (T > 1) {
      for (int sp = 0; sp < nsplit; ++sp) rec += Cpart[sp * cstride0 + (int64_t)(B + b) * 2 * H + u];
    }
    lstm_state_grad_out(layer == 1 ? sa1 : sa0, idx, len == 1, rec, dc[idx]);
    *gout = make_uint2(0u, 0u);
    if (aout) *aout = make_uint2(0u, 0u);
    return;
  }
  if (t >= len) {
    *gout = make_uint2(0u, 0u);
    if (aout) *aout = make_uint2(0u, 0u);
    dc[idx] = 0.f;
    return;
  }
  const __nv_bfloat16* gates = layer == 1 ? gates1 : gates0;
  const float* cst = layer == 1 ? cst1 : cst0;
  const uint2 gp = *reinterpret_cast<const uint2*>(gates + row * 4 * H + 4 * u);
  const float c = cst[row * H + u];
  const float cp = (kState || t > 0) ? cst[(row - 1) * H + u] : 0.f;
  const int64_t cstride = 2ll * B * 2 * H;
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
  uint2 o;
  if constexpr (kState) {
    float dcv = dc[idx];
    if (t == len - 1) {
      const BwdStateArgs& sa = layer == 1 ? sa1 : sa0;
      dh += sa.dh_out[idx];
      dcv += sa.dc_out[idx];
    }
    o = lstm_cell_bwd(gp, c, cp, dh, &dcv);
    dc[idx] = dcv;
  } else {
    o = lstm_cell_bwd(gp, c, cp, dh, dc + idx);
  }
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
constexpr int kBpttChunks = 8;  // chunks of layer 1's chain in the overlapped two-layer schedule (fewer for short T)
// graphs: per layer (slot l, up to 8 layers), wavefront (2), per (layer, chunk) of the overlapped chains (3 + ...)
constexpr int kBpttSlots = 3 + 2 * kBpttChunks;
struct BpttGraphCache {
  cudaGraphExec_t exec[kBpttSlots] = {};
  std::vector<uintptr_t> key[kBpttSlots];
  size_t nodes[kBpttSlots] = {};
  // overlapped two-layer backward: layer 0's chain runs on `side`, one chunk of time steps behind layer 1
  cudaStream_t side = nullptr;
  cudaEvent_t ev_chunk[kBpttChunks] = {};
  cudaEvent_t ev_side_done = nullptr;
  // Capture happens on a private stream: PyTorch's default current stream is the legacy NULL stream, which cannot be
  // captured; the instantiated graph is then launched into the caller's stream (any stream, the NULL stream included).
  cudaStream_t cap_stream = nullptr;
  int cap_device = -1;
  ~BpttGraphCache() {
    for (auto e : exec)
      if (e) cudaGraphExecDestroy(e);
    if (cap_stream) cudaStreamDestroy(cap_stream);
    if (side) cudaStreamDestroy(side);
    for (auto e : ev_chunk)
      if (e) cudaEventDestroy(e);
    if (ev_side_done) cudaEventDestroy(ev_side_done);
  }
};
BpttGraphCache* bptt_cache_create() { return new BpttGraphCache(); }
void bptt_cache_destroy(BpttGraphCache* c) { delete c; }

// Stateful backward (the tape and `lengths` of lstm_backward_impl are then those of T + 1 positions, position 0 =
// state): the state gradients in f32 [L][B][H], all at stable workspace addresses so that the captured graphs replay.
// dh_in / dc_in null: no state gradient requested, and the recurrent GEMM of step 1 is skipped.
struct BpttState {
  const float* dh_out;
  const float* dc_out;
  float* dh_in;
  float* dc_in;
  BwdStateArgs layer(int l, int64_t B, int H) const {
    const int64_t o = (int64_t)l * B * H;
    return BwdStateArgs{dh_out + o, dc_out + o, dh_in ? dh_in + o : nullptr, dc_in ? dc_in + o : nullptr};
  }
};

// split-K factor of the per-step recurrent-gradient GEMMs: 8 for per-rank batches up to 64 rows (one m-tile: 256 CTAs
// instead of 128), 4 above (DESIGN.md §3 has the measurements); the partial-product buffers are sized for 8
constexpr int kBpttSplitMax = 8;
static int bptt_split(int64_t B) { return B <= 64 ? 8 : 4; }

// Two layers at per-rank batches 2B <= 128 run as a wavefront (layer 0 one step behind layer 1, both in one 128-row MMA
// block per GEMM): T + 1 dependent iterations instead of 2T.  Measured (B200, T = 317, backward of 2 x LSTM-1024):
// 7.9 -> 6.1 ms at B = 32 and 8.8 -> 7.3 ms at B = 64.  AVVAD_BPTT_WAVEFRONT=0 runs the layers one after the other.
static bool bptt_wavefront(int layers, int64_t B) {
  static const bool on = [] {
    const char* e = getenv("AVVAD_BPTT_WAVEFRONT");
    return !e || atoi(e) != 0;
  }();
  return on && layers == 2 && 2 * B <= 128;
}

// Two layers at larger batches run as chunked chains on two streams (lstm_backward_impl); AVVAD_BPTT_CHUNKS=1 runs
// them one after the other.
static bool bptt_chains_enabled() {
  static const bool on = [] {
    const char* e = getenv("AVVAD_BPTT_CHUNKS");
    return !e || atoi(e) > 1;
  }();
  return on;
}

static bool bptt_graph_enabled() {
  static int v = [] {
    const char* e = getenv("AVVAD_BPTT_GRAPH");
    return (e && atoi(e) == 0) ? 0 : 1;
  }();
  return v != 0;
}

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

// The workspace of lstm_backward_impl, each buffer 256-byte aligned; with a null base only `total` is meaningful.
struct BpttWs {
  __nv_bfloat16* dG;       // [BT][4H] (layer 1's in the two-layer schedules)
  __nv_bfloat16* dGT;      // dG^T [4H][BTp]
  __nv_bfloat16* XT;       // X^T / H_prev^T [maxI][BTp]
  float *dYa, *dYb;        // dY ping-pong [BT][maxI]
  float* dh_rec;           // split-K partials of the recurrent term [kBpttSplitMax][B][H] (each 256-byte aligned)
  float* dc;               // [B][H]
  float* dWp;              // dW' (interleaved) [4H][maxI]
  __nv_bfloat16* WT;       // W^T [maxI][4H]
  float* partial;          // head / bias partial sums
  int32_t* len_st;         // stable copies of lengths / dlogits (y_dim == 1), see BpttGraphCache
  float* dl_st;
  __nv_bfloat16 *dl16, *dlT, *WTh;  // y_dim > 1: dlogits bf16 [BT][yp], its transpose, W_head^T [H][yp]
  __nv_bfloat16* dG0;               // two layers: layer 0's dG (both layers are live at once)
  __nv_bfloat16 *Abuf, *Wcat;       // wavefront: A [128][8H], Wcat [2H][8H],
  float *Cpart, *dc2;               //   C partials [kBpttSplitMax][128][2H], dc of both layers
  float *dh_rec0, *dc0;             // chunked chains: layer 0's dh_rec partials and dc,
  __nv_bfloat16 *WT0, *WTi;         //   W_hh0'^T and W_ih1'^T [H][4H]
  size_t total;
};
static BpttWs carve_bptt(const avvad_lstm* h, int64_t B, int64_t T, void* base) {
  BpttWs w{};
  size_t off = 0;
  auto take = [&](size_t bytes) {
    void* p = base ? (uint8_t*)base + off : nullptr;
    off += align_up(bytes, 256);
    return p;
  };
  const int H = h->H;
  const int64_t BT = B * T, BTp = (BT + 63) / 64 * 64;
  const int64_t maxI = h->ld0 > H ? h->ld0 : H;
  const size_t bh = (size_t)B * H * 4;
  w.dG = (__nv_bfloat16*)take((size_t)BT * 4 * H * 2);
  w.dGT = (__nv_bfloat16*)take((size_t)4 * H * BTp * 2);
  w.XT = (__nv_bfloat16*)take((size_t)maxI * BTp * 2);
  w.dYa = (float*)take((size_t)BT * maxI * 4);
  w.dYb = (float*)take((size_t)BT * maxI * 4);
  w.dh_rec = (float*)take(kBpttSplitMax * align_up(bh, 256));
  w.dc = (float*)take(bh);
  w.dWp = (float*)take((size_t)4 * H * maxI * 4);
  w.WT = (__nv_bfloat16*)take((size_t)maxI * 4 * H * 2);
  w.partial = (float*)take((size_t)1024 * (H + 1) * 4);
  w.len_st = (int32_t*)take((size_t)B * 4);
  w.dl_st = (float*)take((size_t)BT * 4);
  if (h->y_dim > 1) {
    const int64_t yp = head_pad(h->y_dim);
    w.dl16 = (__nv_bfloat16*)take((size_t)BT * yp * 2);
    w.dlT = (__nv_bfloat16*)take((size_t)yp * BTp * 2);
    w.WTh = (__nv_bfloat16*)take((size_t)H * yp * 2);
  }
  if (h->layers == 2) {
    w.dG0 = (__nv_bfloat16*)take((size_t)BT * 4 * H * 2);
    if (bptt_wavefront(h->layers, B)) {
      w.Abuf = (__nv_bfloat16*)take((size_t)128 * 8 * H * 2);
      w.Wcat = (__nv_bfloat16*)take((size_t)2 * H * 8 * H * 2);
      w.Cpart = (float*)take((size_t)kBpttSplitMax * 128 * 2 * H * 4);
      w.dc2 = (float*)take(2 * bh);
    } else {  // also sized when the chains do not run (AVVAD_BPTT_CHUNKS=1, short T, profiling)
      w.dh_rec0 = (float*)take(kBpttSplitMax * align_up(bh, 256));
      w.dc0 = (float*)take(bh);
      w.WT0 = (__nv_bfloat16*)take((size_t)H * 4 * H * 2);
      w.WTi = (__nv_bfloat16*)take((size_t)H * 4 * H * 2);
    }
  }
  w.total = off + 1024;
  return w;
}

size_t lstm_backward_workspace(const avvad_lstm* h, int64_t B, int64_t T) { return carve_bptt(h, B, T, nullptr).total; }

// Runs `steps(stream)` -- a long chain of tiny dependent launches -- either directly (cache == nullptr) or as a CUDA graph
// captured once on the cache's private stream and replayed while `key` (every pointer / size baked into the kernel
// parameters) is unchanged.
static int bptt_cache_streams(BpttGraphCache* cache) {
  int dev = 0;
  AVVAD_CUDA(cudaGetDevice(&dev));
  if (!cache->cap_stream || cache->cap_device != dev) {
    if (cache->cap_stream) cudaStreamDestroy(cache->cap_stream);
    cache->cap_stream = nullptr;
    AVVAD_CUDA(cudaStreamCreateWithFlags(&cache->cap_stream, cudaStreamNonBlocking));
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

int lstm_backward_impl(const avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T, void* tape,
                       const float* dlogits, void* workspace, size_t workspace_bytes, float* const* dW_ih,
                       float* const* dW_hh, float* const* db, float* dW_head, float* db_head, float* dx, cudaStream_t st,
                       const BpttState* bs) {
  const int layers = h->layers, H = h->H, y_dim = h->y_dim;
  AVVAD_CHECK_ARG(y_dim >= 1, "bad y_dim");
  const BpttWs w = carve_bptt(h, B, T, workspace);
  AVVAD_CHECK_ARG(workspace_bytes >= w.total, "workspace too small");
  const int64_t BT = B * T, BTp = (BT + 63) / 64 * 64;
  const int H4 = 4 * H;
  BpttGraphCache* cache = h->bptt;
  // stable-address copies of the per-call inputs the step kernels read (see BpttGraphCache)
  AVVAD_CUDA(cudaMemcpyAsync(w.len_st, lengths, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
  if (y_dim == 1) AVVAD_CUDA(cudaMemcpyAsync(w.dl_st, dlogits, (size_t)BT * 4, cudaMemcpyDeviceToDevice, st));
  const float* dl_step = (y_dim == 1) ? w.dl_st : dlogits;
  const bool use_graph = bptt_graph_enabled() && !tc::profiling_on() && !sync_debug();
  const int kBpttSplit = bptt_split(B);  // split-K factor of the per-step GEMMs of this call
  // stateful: the last position visited (0 when state gradients leave through the frozen position 0, else 1)
  const int t_min = (bs && !bs->dh_in) ? 1 : 0;
  const auto state_args = [&](int l) { return bs ? bs->layer(l, B, H) : BwdStateArgs{}; };
  // stateful: position 0 of dG is never differentiated; zero it once so the weight-gradient GEMMs see zero rows even
  // where the recurrence stops at position 1
  auto zero_pos0 = [&](__nv_bfloat16* dGl) -> int {
    if (bs) AVVAD_CUDA(cudaMemset2DAsync(dGl, (size_t)T * H4 * 2, 0, (size_t)H4 * 2, (size_t)B, st));
    return AVVAD_OK;
  };
  // the state's kernel-parameter pointers join the graph keys (a stateless key is shorter, so the two never match)
  auto state_key = [&](std::vector<uintptr_t> key) {
    if (bs)
      for (uintptr_t v : {(uintptr_t)bs->dh_out, (uintptr_t)bs->dc_out, (uintptr_t)bs->dh_in, (uintptr_t)bs->dc_in})
        key.push_back(v);
    return key;
  };

  const float* dY_head = nullptr;  // y_dim > 1: gradient of the top layer's output through the head (GEMM)
  if (y_dim == 1) {
    // ---- head gradients (y_dim == 1): dl = dlogits [BT]
    TapeView top = tape_layer(tape, layers - 1, H, B, T);
    int nblocks = (int)std::min<int64_t>(1024, ceil_div(BT, 64));
    int rows_per_block = (int)ceil_div(BT, nblocks);
    nblocks = (int)ceil_div(BT, rows_per_block);
    head_grad_partial_kernel<<<nblocks, 256, 0, st>>>(dlogits, top.hseq, BT, H, rows_per_block, w.partial);
    AVVAD_LAUNCHED();
    head_grad_final_kernel<<<(unsigned)ceil_div(H + 1, 256), 256, 0, st>>>(w.partial, nblocks, H, dW_head, db_head);
    AVVAD_LAUNCHED();
  } else {
    // ---- head gradients (IBM head, y_dim = 513): three GEMMs on bf16 copies of dlogits
    //   dY_top [BT][H]   = dL [BT][yp] * W_head [yp][H]
    //   dW_head [y][H]   = dL^T [yp][BT] * h_top [BT][H]
    //   db_head [y]      = column sums of dL (fp32)
    const int64_t yp = head_pad(y_dim);
    TapeView top = tape_layer(tape, layers - 1, H, B, T);
    int rc = avvad_pack_rows_bf16(dlogits, y_dim, w.dl16, yp, 0, BT, y_dim, 1, st);
    if (rc) return rc;
    head_wt_kernel<<<(unsigned)ceil_div((int64_t)H * yp, 256), 256, 0, st>>>(h->head_w16, y_dim, H, (int)yp, w.WTh);
    AVVAD_LAUNCHED();
    {
      tc::EpiParams ep{};
      ep.C = w.dYa;
      ep.ldc = H;
      rc = tc::gemm_dispatch(w.dl16, yp, w.WTh, yp, BT, H, (int)yp, ep, tc::EPI_F32, 0, st);
      if (rc) return rc;
      dY_head = w.dYa;
    }
    {
      dim3 grid((unsigned)ceil_div(BTp, 32), (unsigned)ceil_div(yp, 32));
      transpose_bf16_kernel<<<grid, dim3(32, 8), 0, st>>>(w.dl16, BT, (int)yp, yp, BTp, 0, (int)T, w.dlT);
      AVVAD_LAUNCHED();
      dim3 grid2((unsigned)ceil_div(BTp, 32), (unsigned)ceil_div(H, 32));
      transpose_bf16_kernel<<<grid2, dim3(32, 8), 0, st>>>(top.hseq, BT, H, H, BTp, 0, (int)T, w.XT);
      AVVAD_LAUNCHED();
      tc::EpiParams ep{};
      ep.C = w.dWp;
      ep.ldc = H;
      rc = tc::gemm_dispatch(w.dlT, BTp, w.XT, BTp, yp, H, (int)BTp, ep, tc::EPI_F32, 0, st);
      if (rc) return rc;
      AVVAD_CUDA(cudaMemcpyAsync(dW_head, w.dWp, (size_t)y_dim * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    colsum_f32_kernel<<<(unsigned)ceil_div(y_dim, 64), 256, 0, st>>>(dlogits, BT, y_dim, db_head);
    AVVAD_LAUNCHED();
  }

  // ---- parameter gradients of layer l from its complete gate gradients dGl [BT][4H]; optionally dX = dGl * W_ih'
  auto weight_grads = [&](int l, const __nv_bfloat16* dGl, float* dx_dst) -> int {
    TapeView tv = tape_layer(tape, l, H, B, T);
    const int64_t ld_in = (l == 0) ? h->ld0 : H;
    const int I = (l == 0) ? h->input_size : H;
    const __nv_bfloat16* Xin = (l == 0) ? (const __nv_bfloat16*)x_bf16 : tape_layer(tape, l - 1, H, B, T).hseq;
    // db (= db_ih = db_hh)
    bias_grad_partial_kernel<<<dim3(H4 / 256, kBiasChunks), 256, 0, st>>>(dGl, BT, H4, w.dWp);  // dWp is free here
    AVVAD_LAUNCHED();
    bias_grad_final_kernel<<<(unsigned)ceil_div(H4, 256), 256, 0, st>>>(w.dWp, H, db[l]);
    AVVAD_LAUNCHED();
    // dG^T [4H][BTp]
    {
      dim3 grid((unsigned)ceil_div(BTp, 32), (unsigned)ceil_div(H4, 32));
      transpose_bf16_kernel<<<grid, dim3(32, 8), 0, st>>>(dGl, BT, H4, H4, BTp, 0, (int)T, w.dGT);
      AVVAD_LAUNCHED();
    }
    // dW_ih' = dG^T * X  -> [4H][ld_in]
    {
      dim3 grid((unsigned)ceil_div(BTp, 32), (unsigned)ceil_div(ld_in, 32));
      transpose_bf16_kernel<<<grid, dim3(32, 8), 0, st>>>(Xin, BT, (int)ld_in, ld_in, BTp, 0, (int)T, w.XT);
      AVVAD_LAUNCHED();
      tc::EpiParams ep{};
      ep.C = w.dWp;
      ep.ldc = ld_in;
      int rc = tc::gemm_dispatch(w.dGT, BTp, w.XT, BTp, H4, (int)ld_in, (int)BTp, ep, tc::EPI_F32, 0, st);
      if (rc) return rc;
      deinterleave_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * I, 256), 256, 0, st>>>(w.dWp, H, I, (int)ld_in, dW_ih[l]);
      AVVAD_LAUNCHED();
    }
    // dW_hh' = dG^T * H_prev -> [4H][H]
    {
      dim3 grid((unsigned)ceil_div(BTp, 32), (unsigned)ceil_div(H, 32));
      transpose_bf16_kernel<<<grid, dim3(32, 8), 0, st>>>(tv.hseq, BT, H, H, BTp, 1, (int)T, w.XT);
      AVVAD_LAUNCHED();
      tc::EpiParams ep{};
      ep.C = w.dWp;
      ep.ldc = H;
      int rc = tc::gemm_dispatch(w.dGT, BTp, w.XT, BTp, H4, H, (int)BTp, ep, tc::EPI_F32, 0, st);
      if (rc) return rc;
      deinterleave_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * H, 256), 256, 0, st>>>(w.dWp, H, H, H, dW_hh[l]);
      AVVAD_LAUNCHED();
    }
    if (dx_dst) {
      transpose_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * ld_in, 256), 256, 0, st>>>(h->w_ih[l], H4, (int)ld_in,
                                                                                       (int)ld_in, w.WT);
      AVVAD_LAUNCHED();
      tc::EpiParams ep{};
      ep.C = dx_dst;
      ep.ldc = (l == 0) ? I : ld_in;
      // l == 0: only the first I (un-padded) columns are written (N guard in the epilogue)
      int rc = tc::gemm_dispatch(dGl, H4, w.WT, H4, BT, (l == 0) ? I : (int)ld_in, H4, ep, tc::EPI_F32, 0, st);
      if (rc) return rc;
    }
    return AVVAD_OK;
  };

  // ---- the recurrent-gradient GEMM of one step: split-K partials dh [kBpttSplit][B][H] of dG_t [B][4H] (rows T * 4H
  // apart) times W_l'.  M = B is tiny: K = 4H is split over kBpttSplit CTAs per output tile so that a step fills the GPU.
  auto step_gemm = [&](float* dh, const __nv_bfloat16* dGt, const __nv_bfloat16* WTl, cudaStream_t s) -> int {
    tc::EpiParams ep{};
    ep.C = dh;
    ep.ldc = H;
    return tc::launch_tma_gemm(dGt, (int64_t)T * H4, WTl, H4, B, H, H4, ep, tc::EPI_F32, 64, s, kBpttSplit,
                               (int64_t)B * H);
  };
  // one real launch of the step GEMM before any capture: the kernels' one-time attribute setup is not capturable
  auto warm = [&]() -> int { return step_gemm(w.dh_rec, w.dG, w.WT, st); };
  // steps te-1 .. tb of layer l, not below t_min: (cell, recurrent GEMM) pairs on stream s
  auto steps = [&](int l, const TapeView& tv, const float* dYl, float* dh, float* dcl, __nv_bfloat16* dGl,
                   const __nv_bfloat16* WTl, int tb, int te, cudaStream_t s) -> int {
    const auto cell = bs ? &lstm_bwd_cell_kernel<true> : &lstm_bwd_cell_kernel<false>;
    const BwdStateArgs sa = state_args(l);
    for (int t = te - 1; t >= tb && t >= t_min; --t) {
      const int has_rec = (t < (int)T - 1) ? kBpttSplit : 0;  // number of partial products to sum
      cell<<<(unsigned)ceil_div(B * H, 256), 256, 0, s>>>(tv.gates, tv.c, dYl, dl_step, h->head_w32, dh, dcl, w.len_st,
                                                          (int)B, (int)T, H, t, has_rec, dGl, sa);
      AVVAD_LAUNCHED();
      if (t > t_min) {
        int rc = step_gemm(dh, dGl + (int64_t)t * H4, WTl, s);
        if (rc) return rc;
      }
    }
    return AVVAD_OK;
  };

  if (bptt_wavefront(layers, B)) {
    // ---- both layers as one wavefront: T + 1 dependent iterations instead of 2T (see lstm_bwd_cell_wf_kernel)
    TapeView t1 = tape_layer(tape, 1, H, B, T), t0 = tape_layer(tape, 0, H, B, T);
    lstm_wf_pack_w_kernel<<<(unsigned)ceil_div((int64_t)2 * H * 8 * H, 256), 256, 0, st>>>(h->w_hh[1], h->w_ih[1],
                                                                                          h->w_hh[0], H, w.Wcat);
    AVVAD_LAUNCHED();
    AVVAD_CUDA(cudaMemsetAsync(w.dc2, 0, (size_t)2 * B * H * 4, st));
    if (int rcz = zero_pos0(w.dG)) return rcz;
    if (int rcz = zero_pos0(w.dG0)) return rcz;
    AVVAD_CUDA(cudaMemsetAsync(w.Abuf, 0, (size_t)128 * 8 * H * 2, st));  // rows 2B..127 stay zero
    // C [2B][2H] = A [2B][8H] * Wcat^T
    auto wf_gemm = [&](cudaStream_t s) -> int {
      tc::EpiParams ep{};
      ep.C = w.Cpart;
      ep.ldc = 2 * H;
      return tc::launch_tma_gemm(w.Abuf, 8 * H, w.Wcat, 8 * H, 2 * B, 2 * H, 8 * H, ep, tc::EPI_F32, 64, s, kBpttSplit,
                                 2 * B * 2 * H);
    };
    const auto cell = bs ? &lstm_bwd_cell_wf_kernel<true> : &lstm_bwd_cell_wf_kernel<false>;
    const BwdStateArgs sa1 = state_args(1), sa0 = state_args(0);
    auto run_wf = [&](cudaStream_t s1) -> int {
      // stateful: layer 0 reaches position 1 in iteration T - 1 and the frozen position 0 in iteration T
      for (int s = 0; s <= (int)T; ++s) {
        cell<<<dim3((unsigned)ceil_div(B * H, 256), 2), 256, 0, s1>>>(
            t1.gates, t1.c, t0.gates, t0.c, dY_head, dl_step, h->head_w32, w.Cpart, kBpttSplit, w.dc2, w.len_st, (int)B,
            (int)T, H, s, w.dG, w.dG0, w.Abuf, sa1, sa0);
        AVVAD_LAUNCHED();
        if (s >= (int)T - t_min) break;
        int rc = wf_gemm(s1);
        if (rc) return rc;
      }
      return AVVAD_OK;
    };
    const std::vector<uintptr_t> key = state_key(
        {(uintptr_t)t1.gates, (uintptr_t)t1.c, (uintptr_t)t0.gates, (uintptr_t)t0.c, (uintptr_t)dY_head,
         (uintptr_t)dl_step, (uintptr_t)h->head_w32, (uintptr_t)w.Cpart, (uintptr_t)w.dc2, (uintptr_t)w.len_st,
         (uintptr_t)w.dG, (uintptr_t)w.dG0, (uintptr_t)w.Abuf, (uintptr_t)w.Wcat, (uintptr_t)B, (uintptr_t)T,
         (uintptr_t)H});
    int rc = run_captured(use_graph ? cache : nullptr, 2, key, [&]() { return wf_gemm(st); }, run_wf, st);
    if (rc) return rc;
    rc = weight_grads(1, w.dG, nullptr);
    if (rc) return rc;
    return weight_grads(0, w.dG0, dx);
  }

  // ---- two layers, larger batches: the recurrences of both layers as chunked chains on two streams.  Layer 1 runs its
  // steps in chunks (t descending); after each chunk the input gradient of that chunk (dY0 = dG1 * W_ih1, one time-major
  // GEMM) and then layer 0's steps of the same chunk run on a side stream while layer 1 continues: every step is a
  // latency-bound (cell kernel, split-K GEMM) pair, so the two chains overlap.
  int n_chunks = bptt_chains_enabled() ? kBpttChunks : 1;
  while (n_chunks > 1 && T / n_chunks < 16) --n_chunks;
  if (layers == 2 && n_chunks > 1 && !tc::profiling_on() && !sync_debug()) {
    int rcs = bptt_cache_streams(cache);
    if (rcs) return rcs;
    float* dY0 = dY_head ? w.dYb : w.dYa;  // [BT][H] fp32: gradient w.r.t. layer 0's output, written chunk by chunk
    TapeView tv1 = tape_layer(tape, 1, H, B, T), tv0 = tape_layer(tape, 0, H, B, T);
    transpose_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * H, 256), 256, 0, st>>>(h->w_hh[1], H4, H, H, w.WT);
    AVVAD_LAUNCHED();
    transpose_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * H, 256), 256, 0, st>>>(h->w_hh[0], H4, H, H, w.WT0);
    AVVAD_LAUNCHED();
    transpose_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * H, 256), 256, 0, st>>>(h->w_ih[1], H4, H, H, w.WTi);
    AVVAD_LAUNCHED();
    AVVAD_CUDA(cudaMemsetAsync(w.dc, 0, (size_t)B * H * 4, st));
    AVVAD_CUDA(cudaMemsetAsync(w.dc0, 0, (size_t)B * H * 4, st));
    if (int rcz = zero_pos0(w.dG)) return rcz;
    if (int rcz = zero_pos0(w.dG0)) return rcz;
    cudaStream_t side = cache->side;
    // the warm-up runs here, not between chunks: dh_rec carries the recurrent term from one chunk to the next
    {
      int rcw = warm();
      if (rcw) return rcw;
    }
    auto no_warm = []() -> int { return 0; };
    for (int c = n_chunks - 1; c >= 0; --c) {
      const int tb = (int)(T * c / n_chunks), te = (int)(T * (c + 1) / n_chunks);
      {  // layer 1, chunk c, on the caller's stream
        const std::vector<uintptr_t> key = state_key({(uintptr_t)tv1.gates, (uintptr_t)tv1.c, (uintptr_t)dY_head,
                                                      (uintptr_t)dl_step, (uintptr_t)h->head_w32, (uintptr_t)w.dh_rec,
                                                      (uintptr_t)w.dc, (uintptr_t)w.len_st, (uintptr_t)w.dG,
                                                      (uintptr_t)w.WT, (uintptr_t)B, (uintptr_t)T, (uintptr_t)H,
                                                      (uintptr_t)tb, (uintptr_t)te, (uintptr_t)kBpttSplit});
        int rc = run_captured(use_graph ? cache : nullptr, 3 + c, key, no_warm,
                              [&](cudaStream_t s2) { return steps(1, tv1, dY_head, w.dh_rec, w.dc, w.dG, w.WT, tb, te, s2); },
                              st);
        if (rc) return rc;
      }
      AVVAD_CUDA(cudaEventRecord(cache->ev_chunk[c], st));
      AVVAD_CUDA(cudaStreamWaitEvent(side, cache->ev_chunk[c], 0));
      // dY0 of the chunk: rows (b, t in [tb, te)) of dG1 times W_ih1
      int rc = tc::launch_tma_gemm_tm(w.dG + (int64_t)tb * H4, H4, w.WTi, H4, B, te - tb, T, H, H4, dY0 + (int64_t)tb * H,
                                      H, side);
      if (rc) return rc;
      {  // layer 0, chunk c, on the side stream
        const std::vector<uintptr_t> key = state_key({(uintptr_t)tv0.gates, (uintptr_t)tv0.c, (uintptr_t)dY0,
                                                      (uintptr_t)dl_step, (uintptr_t)h->head_w32, (uintptr_t)w.dh_rec0,
                                                      (uintptr_t)w.dc0, (uintptr_t)w.len_st, (uintptr_t)w.dG0,
                                                      (uintptr_t)w.WT0, (uintptr_t)B, (uintptr_t)T, (uintptr_t)H,
                                                      (uintptr_t)tb, (uintptr_t)te, (uintptr_t)kBpttSplit});
        rc = run_captured(use_graph ? cache : nullptr, 3 + kBpttChunks + c, key, no_warm,
                          [&](cudaStream_t s2) { return steps(0, tv0, dY0, w.dh_rec0, w.dc0, w.dG0, w.WT0, tb, te, s2); },
                          side);
        if (rc) return rc;
      }
    }
    AVVAD_CUDA(cudaEventRecord(cache->ev_side_done, side));
    // layer 1's parameter gradients (large GEMMs over K = B*T) while layer 0's last chunks still run on the side stream
    int rc = weight_grads(1, w.dG, nullptr);
    if (rc) return rc;
    AVVAD_CUDA(cudaStreamWaitEvent(st, cache->ev_side_done, 0));
    return weight_grads(0, w.dG0, dx);
  }

  const float* dY = dY_head;  // null (y_dim == 1): the top layer takes dl * w_head on the fly
  float* dX_out = dY_head ? w.dYb : w.dYa;
  for (int l = layers - 1; l >= 0; --l) {
    TapeView tv = tape_layer(tape, l, H, B, T);

    // W_hh'^T [H][4H] for the recurrent gradient GEMM
    transpose_w_kernel<<<(unsigned)ceil_div((int64_t)H4 * H, 256), 256, 0, st>>>(h->w_hh[l], H4, H, H, w.WT);
    AVVAD_LAUNCHED();
    AVVAD_CUDA(cudaMemsetAsync(w.dc, 0, (size_t)B * H * 4, st));
    if (int rcz = zero_pos0(w.dG)) return rcz;
    const std::vector<uintptr_t> key = state_key({(uintptr_t)tv.gates, (uintptr_t)tv.c, (uintptr_t)dY,
                                                  (uintptr_t)dl_step, (uintptr_t)h->head_w32, (uintptr_t)w.dh_rec,
                                                  (uintptr_t)w.dc, (uintptr_t)w.len_st, (uintptr_t)w.dG, (uintptr_t)w.WT,
                                                  (uintptr_t)B, (uintptr_t)T, (uintptr_t)H});
    int rc = run_captured(use_graph ? cache : nullptr, l, key, warm,
                          [&](cudaStream_t s) { return steps(l, tv, dY, w.dh_rec, w.dc, w.dG, w.WT, 0, (int)T, s); }, st);
    if (rc) return rc;
    float* dst = (l == 0) ? dx : dX_out;
    rc = weight_grads(l, w.dG, (l > 0 || dx) ? dst : nullptr);
    if (rc) return rc;
    if (l > 0 || dx) {
      dY = dst;
      dX_out = (dX_out == w.dYa) ? w.dYb : w.dYa;
    }
  }
  return AVVAD_OK;
}

// ---- stateful backward (avvad_lstm_backward_state) over a tape of T + 1 positions per row.  The per-call tensors of
// T steps are laid out once more with a leading position 0 -- zero rows of x and dlogits, lengths + 1 -- so that
// lstm_backward_impl runs its schedules unchanged over T + 1 positions; dx is read back from positions 1..T.
namespace {
struct StateBwdWs {
  int32_t* len1;
  __nv_bfloat16* x1;  // [B][T+1][ld0]
  float* dl1;         // [B][T+1][y_dim]
  float* dx1;         // [B][T+1][input_size]
  float *dh_out, *dc_out, *dh_in, *dc_in;  // [L][B][H]
  uint8_t* inner;     // lstm_backward_impl's workspace
  size_t total;
};
StateBwdWs carve_state_bwd(const avvad_lstm* h, int64_t B, int64_t T, void* base) {
  StateBwdWs w{};
  size_t off = 0;
  auto take = [&](size_t bytes) {
    void* p = base ? (uint8_t*)base + off : nullptr;
    off += align_up(bytes, 256);
    return p;
  };
  const int64_t T1 = T + 1;
  const size_t st = (size_t)h->layers * B * h->H * sizeof(float);
  w.len1 = (int32_t*)take((size_t)B * 4);
  w.x1 = (__nv_bfloat16*)take((size_t)B * T1 * h->ld0 * 2);
  w.dl1 = (float*)take((size_t)B * T1 * h->y_dim * 4);
  w.dx1 = (float*)take((size_t)B * T1 * h->input_size * 4);
  w.dh_out = (float*)take(st);
  w.dc_out = (float*)take(st);
  w.dh_in = (float*)take(st);
  w.dc_in = (float*)take(st);
  w.inner = (uint8_t*)take(0);
  w.total = off + lstm_backward_workspace(h, B, T1);
  return w;
}
}  // namespace

size_t lstm_backward_state_workspace(const avvad_lstm* h, int64_t B, int64_t T) {
  return carve_state_bwd(h, B, T, nullptr).total;
}

int lstm_backward_state_impl(const avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T,
                             void* tape, const float* dlogits, const float* dh_out, const float* dc_out, float* dh_in,
                             float* dc_in, void* workspace, size_t workspace_bytes, float* const* dW_ih,
                             float* const* dW_hh, float* const* db, float* dW_head, float* db_head, float* dx,
                             cudaStream_t st) {
  AVVAD_CHECK_ARG(B > 0 && T > 0, "bad sizes");
  const StateBwdWs w = carve_state_bwd(h, B, T, workspace);
  AVVAD_CHECK_ARG(workspace_bytes >= w.total, "workspace too small");
  const int64_t T1 = T + 1;
  shift_lengths_kernel<<<(unsigned)ceil_div(B, 256), 256, 0, st>>>(lengths, (int)B, w.len1);
  AVVAD_LAUNCHED();
  // [B][T][n] -> [B][T+1][n] with a zero row at position 0
  auto widen = [&](void* dst, const void* src, size_t row_bytes) -> int {
    AVVAD_CUDA(cudaMemset2DAsync(dst, T1 * row_bytes, 0, row_bytes, (size_t)B, st));
    AVVAD_CUDA(cudaMemcpy2DAsync((uint8_t*)dst + row_bytes, T1 * row_bytes, src, T * row_bytes, T * row_bytes, (size_t)B,
                                 cudaMemcpyDeviceToDevice, st));
    return AVVAD_OK;
  };
  int rc = widen(w.x1, x_bf16, (size_t)h->ld0 * 2);
  if (!rc) rc = widen(w.dl1, dlogits, (size_t)h->y_dim * 4);
  if (rc) return rc;
  // the state gradients at stable addresses (inputs copied first, so outputs may alias them)
  const size_t sbytes = (size_t)h->layers * B * h->H * sizeof(float);
  if (dh_out) AVVAD_CUDA(cudaMemcpyAsync(w.dh_out, dh_out, sbytes, cudaMemcpyDeviceToDevice, st));
  else AVVAD_CUDA(cudaMemsetAsync(w.dh_out, 0, sbytes, st));
  if (dc_out) AVVAD_CUDA(cudaMemcpyAsync(w.dc_out, dc_out, sbytes, cudaMemcpyDeviceToDevice, st));
  else AVVAD_CUDA(cudaMemsetAsync(w.dc_out, 0, sbytes, st));
  const bool want = dh_in || dc_in;
  const BpttState bs{w.dh_out, w.dc_out, want ? w.dh_in : nullptr, want ? w.dc_in : nullptr};
  rc = lstm_backward_impl(h, w.x1, w.len1, B, T1, tape, w.dl1, w.inner,
                          workspace_bytes - (size_t)(w.inner - (uint8_t*)workspace), dW_ih, dW_hh, db, dW_head, db_head,
                          dx ? w.dx1 : nullptr, st, &bs);
  if (rc) return rc;
  if (dx) {
    const size_t row = (size_t)h->input_size * 4;
    AVVAD_CUDA(cudaMemcpy2DAsync(dx, T * row, (uint8_t*)w.dx1 + row, T1 * row, T * row, (size_t)B,
                                 cudaMemcpyDeviceToDevice, st));
  }
  if (dh_in) AVVAD_CUDA(cudaMemcpyAsync(dh_in, w.dh_in, sbytes, cudaMemcpyDeviceToDevice, st));
  if (dc_in) AVVAD_CUDA(cudaMemcpyAsync(dc_in, w.dc_in, sbytes, cudaMemcpyDeviceToDevice, st));
  return AVVAD_OK;
}
}  // namespace avvad
