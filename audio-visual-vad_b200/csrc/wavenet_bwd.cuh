// Back-propagation through the WaveNet encoder (included at the end of wavenet.cu: it uses the handle and the tape
// layout defined there).
//
// Reference semantics: autograd of packages/models/wavenet_autoencoder.py:74-93 (_encode).
//
// The forward with a tape (avvad_wavenet_encode_train) keeps S_i (bf16, every layer input), act_i (bf16, every dense
// operand) and the bottleneck output (f32).  The backward runs in reverse:
//   pool + bottleneck : AdaptiveAvgPool1d backward as a gather over every bin that contains t (bins overlap when
//                       L % P != 0), the ReLU mask out > 0, then g_n = dZ . W_bott, dW_bott = dZ^T . S_n, db = sum dZ
//   dilated layer i   : d act = g_{i+1} . W_dense, dW_dense = g_{i+1}^T . act_i;  d pre = [act_i > 0] d act;
//                       dA = d pre . W_dil (one Rp-wide block per tap), dW_dil = d pre^T . im2col(relu(S_i));
//                       g_i[t] = [S_i[t] > 0] sum_j dA[t - j d][tap j] + g_{i+1}[t - (k-1) d]   (a gather: no atomics)
//   causal layer      : dW_causal = g_0^T . im2col(x); dx (when asked) = the tap gather of g_0 . W_causal
// GEMM operands are bf16 with fp32 accumulation; the residual-stream gradient g_i stays fp32 from layer to layer (it is
// the sum along the skip path) with a bf16 copy for the GEMMs.  Weight gradients reduce over K = B * L rows: transposed
// copies of both operands and a split-K tcgen05 GEMM over the SMs, summed in a fixed order.  Bias gradients are fp32
// column sums in a fixed order.  Two identical calls therefore give bit-identical gradients.
#include "bwd_common.cuh"

namespace avvad {

// d out (B, bott, P) f32 -> dZ = [z > 0] * d relu-output, z [B][L][bp] the tape's bottleneck output; f32 and bf16 copies.
// Row t belongs to bins p in [floor(t P / L), ceil((t + 1) P / L) - 1], each of size ceil((p+1)L/P) - floor(pL/P).
__global__ void wn_pool_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ z, int B, int L, int Cp,
                                   int C, int P, float* __restrict__ dz, __nv_bfloat16* __restrict__ dz16) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)B * L * Cp) return;
  const int c = (int)(idx % Cp);
  const int64_t row = idx / Cp;
  const int t = (int)(row % L), b = (int)(row / L);
  float acc = 0.f;
  if (c < C && z[idx] > 0.f) {
    const int p0 = (int)(((int64_t)t * P) / L);
    const int p1 = (int)((((int64_t)t + 1) * P + L - 1) / L);
    for (int p = p0; p < p1; ++p) {
      const int t0 = (int)(((int64_t)p * L) / P);
      const int t1 = (int)((((int64_t)(p + 1)) * L + P - 1) / P);
      acc += dout[((int64_t)b * C + c) * P + p] / (float)(t1 - t0);
    }
  }
  dz[idx] = acc;
  dz16[idx] = __float2bfloat16_rn(acc);
}
__device__ __forceinline__ void wn_load8(const float* p, float v[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
// v -> 8 f32 at p and their bf16 copy at p16
__device__ __forceinline__ void wn_store8(const float v[8], float* p, __nv_bfloat16* p16) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
  *reinterpret_cast<uint4*>(p16) = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]),
                                              pack_bf16x2(v[6], v[7]));
}
__device__ __forceinline__ void wn_unpack8(uint4 u, float v[8]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 f = unpack_bf16x2(w[e]);
    v[2 * e] = f.x;
    v[2 * e + 1] = f.y;
  }
}

// d pre = [act > 0] * d act, in place (f32), and its bf16 copy; 8 elements per thread (n % 8 == 0)
__global__ void wn_relu_mask_kernel(float* __restrict__ d, const __nv_bfloat16* __restrict__ act, int64_t n,
                                    __nv_bfloat16* __restrict__ d16) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (i >= n) return;
  float a[8], v[8];
  wn_unpack8(*reinterpret_cast<const uint4*>(act + i), a);
  wn_load8(d + i, v);
#pragma unroll
  for (int e = 0; e < 8; ++e) v[e] = a[e] > 0.f ? v[e] : 0.f;
  wn_store8(v, d + i, d16 + i);
}
// g_in[b][t][c] = [S[b][t][c] > 0] sum_j dA[b][t - j d][j Cp + c] + (t >= shift ? g_out[b][t - shift][c] : 0),
// shift = (k-1) d; f32 and bf16 copies; 8 channels per thread
__global__ void wn_grad_gather_kernel(const float* __restrict__ dA, const float* __restrict__ g_out,
                                      const __nv_bfloat16* __restrict__ S, int B, int Lin, int Lo, int k, int d, int Cp,
                                      float* __restrict__ g_in, __nv_bfloat16* __restrict__ g16) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int groups = Cp >> 3;
  if (idx >= (int64_t)B * Lin * groups) return;
  const int64_t row = idx / groups;
  const int c = (int)(idx - row * groups) * 8;
  const int b = (int)(row / Lin), t = (int)(row - (int64_t)b * Lin);
  float s[8], acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  wn_unpack8(*reinterpret_cast<const uint4*>(S + row * Cp + c), s);
  for (int j = 0; j < k; ++j) {
    const int to = t - j * d;
    if (to >= 0 && to < Lo) {
      float v[8];
      wn_load8(dA + ((int64_t)b * Lo + to) * k * Cp + j * Cp + c, v);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] += v[e];
    }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] = s[e] > 0.f ? acc[e] : 0.f;
  const int shift = (k - 1) * d;
  if (t >= shift) {
    float v[8];
    wn_load8(g_out + ((int64_t)b * Lo + t - shift) * Cp + c, v);
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] += v[e];
  }
  wn_store8(acc, g_in + row * Cp + c, g16 + row * Cp + c);
}
// dx (B, C, N) f32 channel-major: dx[b][c][t] = sum_j dX[b][t - j][j Cp + c] over 0 <= t - j < L0
__global__ void wn_dx_gather_kernel(const float* __restrict__ dX, int B, int C, int N, int k, int L0, int Cp,
                                    float* __restrict__ dx) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)B * C * N) return;
  const int t = (int)(idx % N);
  const int64_t bc = idx / N;
  const int c = (int)(bc % C), b = (int)(bc / C);
  float acc = 0.f;
  for (int j = 0; j < k; ++j) {
    const int to = t - j;
    if (to >= 0 && to < L0) acc += dX[((int64_t)b * L0 + to) * k * Cp + j * Cp + c];
  }
  dx[idx] = acc;
}
// transposed im2col of a time-major bf16 layer input: out[j Cp + c][m] = act(S[b][t + j d][c]) for m = b Lo + t < M,
// zero for M <= m < Mp (act = ReLU when relu != 0).  32 x 32 tiles through shared memory.
__global__ void wn_im2col_t_kernel(const __nv_bfloat16* __restrict__ S, int64_t M, int Lo, int Lin, int Cp, int d,
                                   int relu, int64_t Mp, __nv_bfloat16* __restrict__ out) {
  __shared__ __nv_bfloat16 tile[32][33];
  const int64_t m0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32, j = blockIdx.z;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int64_t m = m0 + i;
    __nv_bfloat16 v = __float2bfloat16_rn(0.f);
    if (m < M) {
      const int64_t b = m / Lo, t = m - b * Lo;
      v = S[(b * Lin + t + (int64_t)j * d) * Cp + c0 + threadIdx.x];
      if (relu && !(__bfloat162float(v) > 0.f)) v = __float2bfloat16_rn(0.f);
    }
    tile[i][threadIdx.x] = v;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int64_t m = m0 + threadIdx.x;
    if (m < Mp) out[((int64_t)j * Cp + c0 + i) * Mp + m] = tile[threadIdx.x][i];
  }
}
// transposed im2col of the channel-major input: out[j Cp + c][b L0 + t] = bf16(x[b][c][t + j]) (zero for c >= C and
// for columns past B L0)
__global__ void wn_im2col_cm_t_kernel(const float* __restrict__ x, int B, int C, int N, int k, int L0, int Cp,
                                      int64_t Mp, __nv_bfloat16* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)k * Cp * Mp) return;
  const int64_t m = idx % Mp;
  const int col = (int)(idx / Mp);
  const int j = col / Cp, c = col - j * Cp;
  float v = 0.f;
  if (c < C && m < (int64_t)B * L0) {
    const int64_t b = m / L0, t = m - b * L0;
    v = x[(b * C + c) * N + t + j];
  }
  out[idx] = __float2bfloat16_rn(v);
}
// acc [Op][k Ip] f32 (column j Ip + i) -> PyTorch Conv1d layout [O][I][k]
__global__ void wn_unpack_w_kernel(const float* __restrict__ acc, int O, int I, int k, int Ip, float* __restrict__ dw) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)O * I * k) return;
  const int j = (int)(idx % k);
  const int i = (int)((idx / k) % I);
  const int o = (int)(idx / ((int64_t)k * I));
  dw[idx] = acc[(int64_t)o * k * Ip + j * Ip + i];
}

constexpr int kWnColGroups = 512;                  // row groups of the first column-sum stage
constexpr size_t kWnPartFloats = 8u << 20;         // split-K partials (32 MB)

struct WnBwdWs {
  float* g[2];             // residual-stream gradient, f32 [B*L0][Rp]
  __nv_bfloat16* g16;      // its bf16 copy
  float* d;                // d pre / dZ, f32 [B*L0][max(Dp, bp)]
  __nv_bfloat16* d16;      // its bf16 copy
  float* dA;               // per-tap data gradient, f32 [B*L0][k * max(Rp, qp)]
  __nv_bfloat16* T1;       // transposed gradient [max C][Pp]
  __nv_bfloat16* T2;       // transposed operand [kcw][Pp], kcw = max(k * max(Rp, qp), max C)
  __nv_bfloat16* wT;       // transposed weight [kcw][max C]
  float* part;             // split-K partials
  float* acc;              // weight gradient before the layout change [max C][kcw]
  float* cs;               // column-sum scratch [2 * kWnColGroups + 1][max C]
  int64_t Pp;              // B * L0 rounded up to 64 (K of the weight-gradient GEMMs)
  size_t bytes;
};
static WnBwdWs wn_bwd_ws(const avvad_wavenet* h, int64_t B, int64_t N, void* base) {
  WnBwdWs w{};
  const size_t M0 = (size_t)B * (N - (h->k - 1));
  w.Pp = (int64_t)(M0 + 63) / 64 * 64;
  const size_t cmax = std::max(std::max(h->qp, h->Rp), std::max(h->Dp, h->bp));
  const size_t kc = (size_t)h->k * std::max(h->Rp, h->qp);
  const size_t kcw = std::max(kc, cmax);   // widest weight-gradient GEMM (N) / transposed weight (rows)
  const size_t dw = std::max(h->Dp, h->bp);
  uint8_t* p = (uint8_t*)base;
  size_t off = 0;
  auto take = [&](size_t n) -> void* {
    void* q = p ? p + off : nullptr;
    off += align_up(n, 256);
    return q;
  };
  w.g[0] = (float*)take(M0 * h->Rp * 4);
  w.g[1] = (float*)take(M0 * h->Rp * 4);
  w.g16 = (__nv_bfloat16*)take(M0 * h->Rp * 2);
  w.d = (float*)take(M0 * dw * 4);
  w.d16 = (__nv_bfloat16*)take(M0 * dw * 2);
  w.dA = (float*)take(M0 * kc * 4);
  w.T1 = (__nv_bfloat16*)take(cmax * w.Pp * 2);
  w.T2 = (__nv_bfloat16*)take(kcw * w.Pp * 2);
  w.wT = (__nv_bfloat16*)take(kcw * cmax * 2);
  w.part = (float*)take(kWnPartFloats * 4);
  w.acc = (float*)take(cmax * kcw * 4);
  w.cs = (float*)take((2 * kWnColGroups + 1) * cmax * 4);
  w.bytes = off;
  return w;
}

extern "C" size_t avvad_wavenet_backward_workspace_bytes(const avvad_wavenet* h, int64_t B, int64_t N) {
  if (!h || B <= 0 || wn_out_len(h, N) < 1) return 0;
  return wn_bwd_ws(h, B, N, nullptr).bytes;
}

namespace {

struct WnBwd {
  const avvad_wavenet* h;
  WnBwdWs w;
  cudaStream_t st;

  // bf16 [R][C] -> [C][Rp] (zero columns past R)
  int transpose(const __nv_bfloat16* in, int64_t R, int C, int64_t Rp, __nv_bfloat16* out) const {
    dim3 grid((unsigned)ceil_div(Rp, 32), (unsigned)ceil_div(C, 32));
    transpose_bf16_kernel<<<grid, dim3(32, 8), 0, st>>>(in, R, C, C, Rp, 0, 1, out);
    AVVAD_LAUNCHED();
    return AVVAD_OK;
  }
  // out[c] = sum_r x[r][c] for c < O: column sums over kWnColGroups row groups (x viewed as [R / G][G * C]), then over
  // the group sums and the R % G leftover rows
  int colsum(const float* x, int64_t R, int C, float* out, int O) const {
    if (!out) return AVVAD_OK;
    const int64_t G = kWnColGroups, R1 = R / G * G;
    int64_t rows = R - R1;
    float* left = w.cs;
    if (R1 > 0) {
      colsum_f32_kernel<<<(unsigned)ceil_div(G * C, 64), 256, 0, st>>>(x, R1 / G, (int)(G * C), w.cs);
      AVVAD_LAUNCHED();
      rows += G;
      left += G * C;
    }
    if (R > R1) AVVAD_CUDA(cudaMemcpyAsync(left, x + R1 * C, (R - R1) * C * sizeof(float), cudaMemcpyDeviceToDevice, st));
    float* tot = w.cs + 2 * G * C;
    colsum_f32_kernel<<<(unsigned)ceil_div(C, 64), 256, 0, st>>>(w.cs, rows, C, tot);
    AVVAD_LAUNCHED();
    AVVAD_CUDA(cudaMemcpyAsync(out, tot, O * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return AVVAD_OK;
  }
  // dw (PyTorch layout [O][I][k]) = AT [M][Pp] . BT [k Ip][Pp]^T, split K over the SMs
  int wgrad(const __nv_bfloat16* AT, int M, const __nv_bfloat16* BT, int O, int I, int k, int Ip, float* dw) const {
    const int N = k * Ip;
    const int bn = (N % 256 == 0 && M >= 128) ? 256 : 64;
    const int tiles = (int)(ceil_div(M, 128) * ceil_div(N, bn));
    const int64_t kblocks = w.Pp / 64;
    int ksplit = (int)std::min<int64_t>(std::max<int64_t>(1, 296 / tiles), kblocks);
    const size_t per = (size_t)M * N;
    if ((size_t)ksplit * per > kWnPartFloats) ksplit = (int)std::max<size_t>(1, kWnPartFloats / per);
    ksplit = (int)ceil_div(kblocks, ceil_div(kblocks, ksplit));   // every split owns at least one K block
    tc::EpiParams ep{};
    ep.C = w.part;
    ep.ldc = N;
    int rc = tc::launch_tma_gemm(AT, w.Pp, BT, w.Pp, M, N, (int)w.Pp, ep, tc::EPI_F32, bn, st, ksplit, (int64_t)per);
    if (rc) return rc;
    sum_partials_kernel<<<(unsigned)ceil_div(per, 256), 256, 0, st>>>(w.part, ksplit, (int64_t)per, 0, w.acc);
    AVVAD_LAUNCHED();
    const int64_t total = (int64_t)O * I * k;
    wn_unpack_w_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(w.acc, O, I, k, Ip, dw);
    AVVAD_LAUNCHED();
    return AVVAD_OK;
  }
  // C [M][Kw] f32 = A [M][Kin] . Wp [Kin-rows][Kw]: the data gradient through packed weights Wp [Op = Kin][Kw]
  int dgrad(const __nv_bfloat16* A, int64_t M, const WnLayer& l, int Op, int Kw, float* C) const {
    int rc = transpose(l.w, Op, Kw, Op, w.wT);
    if (rc) return rc;
    return avvad_gemm_bf16(A, Op, w.wT, Op, nullptr, C, Kw, 0, 0, M, Kw, Op, st);
  }
};

}  // namespace

}  // namespace avvad

// dw[i] / db[i], i = 0 causal, 1 + 2j dilated_j, 2 + 2j dense_j, 1 + 2n bottleneck: f32 [O][I][k] / [O].
extern "C" int avvad_wavenet_backward(avvad_wavenet* h, const float* x, int64_t B, int64_t N, const void* tape,
                                      size_t tape_bytes, const float* dout, float* dx, float* const* dw,
                                      float* const* db, void* workspace, size_t workspace_bytes, void* stream) {
  AVVAD_CHECK_ARG(h && x && tape && dout && dw && workspace && B > 0, "bad argument");
  const int n = (int)h->dil.size(), k = h->k;
  for (int i = 0; i < 2 + 2 * n; ++i) AVVAD_CHECK_ARG(dw[i], "null weight-gradient pointer");
  int rc = wn_check(h, N);
  if (rc) return rc;
  const WnTape t = wn_tape(h, B, N, const_cast<void*>(tape));
  if (tape_bytes < t.bytes) { set_error("wavenet: tape too small"); return AVVAD_ERR_WORKSPACE; }
  WnBwd c{h, wn_bwd_ws(h, B, N, workspace), (cudaStream_t)stream};
  if (workspace_bytes < c.w.bytes) { set_error("wavenet: backward workspace too small"); return AVVAD_ERR_WORKSPACE; }
  if (!tc::tma_available()) {
    set_error("cuTensorMapEncodeTiled driver entry point unavailable: libavvad needs a CUDA 12 driver");
    return AVVAD_ERR_CUDA;
  }
  const WnBwdWs& w = c.w;
  cudaStream_t st = c.st;
  auto bias_out = [&](int i) -> float* { return db ? db[i] : nullptr; };

  // ---- pool, bottleneck ReLU and the bottleneck layer ----
  const int64_t Mf = B * t.L[n];
  wn_pool_bwd_kernel<<<(unsigned)ceil_div(Mf * h->bp, 256), 256, 0, st>>>(dout, t.out, (int)B, (int)t.L[n], h->bp,
                                                                          h->bott, h->pool, w.d, w.d16);
  AVVAD_LAUNCHED();
  if ((rc = c.colsum(w.d, Mf, h->bp, bias_out(1 + 2 * n), h->bott))) return rc;
  if ((rc = c.transpose(w.d16, Mf, h->bp, w.Pp, w.T1))) return rc;
  if ((rc = c.transpose(t.S[n], Mf, h->Rp, w.Pp, w.T2))) return rc;
  if ((rc = c.wgrad(w.T1, h->bp, w.T2, h->bott, h->R, 1, h->Rp, dw[1 + 2 * n]))) return rc;
  int gi = 0;   // w.g[gi] holds g_{i+1} (f32) and w.g16 its bf16 copy
  if ((rc = c.dgrad(w.d16, Mf, h->bottleneck, h->bp, h->Rp, w.g[gi]))) return rc;
  if ((rc = avvad_pack_rows_bf16(w.g[gi], h->Rp, w.g16, h->Rp, 0, Mf, h->Rp, 0, st))) return rc;

  // ---- dilated layers in reverse ----
  for (int i = n - 1; i >= 0; --i) {
    const int d = h->dil[i];
    const int64_t Lin = t.L[i], Lo = t.L[i + 1], Mo = B * Lo;
    // dense 1x1: bias and weight gradients, then d act -> d pre
    if ((rc = c.colsum(w.g[gi], Mo, h->Rp, bias_out(2 + 2 * i), h->R))) return rc;
    if ((rc = c.transpose(w.g16, Mo, h->Rp, w.Pp, w.T1))) return rc;
    if ((rc = c.transpose(t.act[i], Mo, h->Dp, w.Pp, w.T2))) return rc;
    if ((rc = c.wgrad(w.T1, h->Rp, w.T2, h->R, h->D, 1, h->Dp, dw[2 + 2 * i]))) return rc;
    if ((rc = c.dgrad(w.g16, Mo, h->dense[i], h->Rp, h->Dp, w.d))) return rc;
    wn_relu_mask_kernel<<<(unsigned)ceil_div(Mo * h->Dp / 8, 256), 256, 0, st>>>(w.d, t.act[i], Mo * h->Dp, w.d16);
    AVVAD_LAUNCHED();
    // dilated conv: bias and weight gradients against im2col(relu(S_i)), then the per-tap data gradient
    if ((rc = c.colsum(w.d, Mo, h->Dp, bias_out(1 + 2 * i), h->D))) return rc;
    if ((rc = c.transpose(w.d16, Mo, h->Dp, w.Pp, w.T1))) return rc;
    {
      dim3 grid((unsigned)(w.Pp / 32), (unsigned)(h->Rp / 32), (unsigned)k);
      wn_im2col_t_kernel<<<grid, dim3(32, 8), 0, st>>>(t.S[i], Mo, (int)Lo, (int)Lin, h->Rp, d, 1, w.Pp, w.T2);
      AVVAD_LAUNCHED();
    }
    if ((rc = c.wgrad(w.T1, h->Dp, w.T2, h->D, h->R, k, h->Rp, dw[1 + 2 * i]))) return rc;
    if ((rc = c.dgrad(w.d16, Mo, h->dilated[i], h->Dp, k * h->Rp, w.dA))) return rc;
    // g_i: the ReLU-masked tap gather plus the residual path
    const int64_t tot = B * Lin * h->Rp / 8;
    wn_grad_gather_kernel<<<(unsigned)ceil_div(tot, 256), 256, 0, st>>>(w.dA, w.g[gi], t.S[i], (int)B, (int)Lin, (int)Lo,
                                                                        k, d, h->Rp, w.g[gi ^ 1], w.g16);
    AVVAD_LAUNCHED();
    gi ^= 1;
  }

  // ---- causal layer ----
  const int64_t L0 = t.L[0], M0 = B * L0;
  if ((rc = c.colsum(w.g[gi], M0, h->Rp, bias_out(0), h->R))) return rc;
  if ((rc = c.transpose(w.g16, M0, h->Rp, w.Pp, w.T1))) return rc;
  {
    const int64_t tot = (int64_t)k * h->qp * w.Pp;
    wn_im2col_cm_t_kernel<<<(unsigned)ceil_div(tot, 256), 256, 0, st>>>(x, (int)B, h->q, (int)N, k, (int)L0, h->qp,
                                                                         w.Pp, w.T2);
    AVVAD_LAUNCHED();
  }
  if ((rc = c.wgrad(w.T1, h->Rp, w.T2, h->R, h->q, k, h->qp, dw[0]))) return rc;
  if (dx) {
    if ((rc = c.dgrad(w.g16, M0, h->causal, h->Rp, k * h->qp, w.dA))) return rc;
    const int64_t tot = B * h->q * N;
    wn_dx_gather_kernel<<<(unsigned)ceil_div(tot, 256), 256, 0, st>>>(w.dA, (int)B, h->q, (int)N, k, (int)L0, h->qp, dx);
    AVVAD_LAUNCHED();
  }
  return AVVAD_OK;
}
