// Host launchers for the tcgen05 engine + the exported GEMM / NHWC-conv / row-pack entry points.
#include <stdlib.h>

#include <mutex>
#include <vector>

#include "conv_slab.cuh"

namespace avvad {
namespace tc {

// ---- optional per-launch timing (bench.py roofline): CUDA events on the launching stream ----------------
struct ProfRec {
  cudaEvent_t beg, end;
  int cat;
  double flops;
};
static std::mutex g_prof_mu;
static bool g_prof_on = false;
static std::vector<ProfRec> g_prof;
static std::vector<cudaEvent_t> g_prof_pool;

bool profiling_on() {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  return g_prof_on;
}

static cudaEvent_t prof_event() {
  if (!g_prof_pool.empty()) {
    cudaEvent_t e = g_prof_pool.back();
    g_prof_pool.pop_back();
    return e;
  }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}

// Per-launch records are only taken in detailed mode (AVVAD_PROFILE_PER_LAUNCH=1); by default the trunk brackets
// each chunk's 19 convolution launches with ONE event pair (prof_group_*), which keeps the timed region of bench.py
// free of ~1800 extra event records per step.
static bool per_launch_mode() {
  static int v = [] {
    const char* e = getenv("AVVAD_PROFILE_PER_LAUNCH");
    return (e && atoi(e) != 0) ? 1 : 0;
  }();
  return v != 0;
}
static thread_local int t_group_depth = 0;

int prof_group_begin(cudaStream_t st, void** tok) {
  *tok = nullptr;
  if (per_launch_mode()) return 0;
  int rc = 0;
  {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (!g_prof_on) return 0;
    ProfRec* r = new ProfRec();
    r->beg = prof_event();
    r->end = prof_event();
    cudaEventRecord(r->beg, st);
    *tok = r;
    rc = 1;
  }
  ++t_group_depth;
  return rc;
}
void prof_group_end(cudaStream_t st, void* tok, int cat, double flops) {
  if (!tok) return;
  --t_group_depth;
  ProfRec* r = static_cast<ProfRec*>(tok);
  cudaEventRecord(r->end, st);
  r->cat = cat;
  r->flops = flops;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof.push_back(*r);
  delete r;
}

// generic begin/end used by both engines
int prof_begin(cudaStream_t st, void** tok) {
  *tok = nullptr;
  if (t_group_depth > 0) return 0;  // covered by the enclosing group record
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (!g_prof_on) return 0;
  ProfRec* r = new ProfRec();
  r->beg = prof_event();
  r->end = prof_event();
  cudaEventRecord(r->beg, st);
  *tok = r;
  return 1;
}
void prof_end(cudaStream_t st, void* tok, int cat, double flops) {
  if (!tok) return;
  ProfRec* r = static_cast<ProfRec*>(tok);
  cudaEventRecord(r->end, st);
  r->cat = cat;
  r->flops = flops;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof.push_back(*r);
  delete r;
}

// Plain GEMM on the TMA-fed engine.  cuTensorMapEncodeTiled is fetched from the driver at run time; a driver without
// it cannot run this library (there is no second engine).
int gemm_dispatch(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* Wt, int64_t ldw, int64_t M, int N, int K,
                  const EpiParams& ep, int epi_mode, int bn_hint, cudaStream_t st) {
  if (!tma_available()) {
    set_error("cuTensorMapEncodeTiled driver entry point unavailable: libavvad needs a CUDA 12 driver");
    return AVVAD_ERR_CUDA;
  }
  AVVAD_CHECK_ARG(K > 0 && K % BK == 0, "K must be a positive multiple of 64");
  AVVAD_CHECK_ARG((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(Wt) & 15) == 0,
                  "operands must be 16-byte aligned");
  if (epi_mode == EPI_LSTM) AVVAD_CHECK_ARG(N % 32 == 0, "LSTM epilogue needs N % 32 == 0");
  return launch_tma_gemm(A, lda, Wt, ldw, M, N, K, ep, epi_mode, bn_hint, st);
}

__global__ void pack_rows_kernel(const float* __restrict__ src, int64_t ld_src, __nv_bfloat16* __restrict__ dst,
                                 int64_t ld_dst, int64_t col_off, int64_t rows, int64_t cols, int64_t width) {
  // one thread per destination element in [col_off, col_off + width)
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * width) return;
  const int64_t r = idx / width, j = idx - r * width;
  const float v = (j < cols) ? src[r * ld_src + j] : 0.f;
  dst[r * ld_dst + col_off + j] = __float2bfloat16_rn(v);
}

}  // namespace tc
}  // namespace avvad

using namespace avvad;

extern "C" int avvad_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(tc::g_prof_mu);
  tc::g_prof_on = on != 0;
  return AVVAD_OK;
}

// Sums the recorded tensor-core launches of category `cat` (0 = implicit-GEMM conv, 1 = plain GEMM,
// 2 = LSTM step) since the last call, then clears ALL records.  Synchronises the device.
extern "C" int avvad_profile_read(int cat, double* ms, double* flops, uint64_t* launches) {
  AVVAD_CHECK_ARG(ms && flops && launches, "null pointer");
  AVVAD_CUDA(cudaDeviceSynchronize());
  std::lock_guard<std::mutex> lk(tc::g_prof_mu);
  double t = 0, f = 0;
  uint64_t n = 0;
  for (auto& r : tc::g_prof) {
    if (r.cat == cat) {
      float e = 0.f;
      if (cudaEventElapsedTime(&e, r.beg, r.end) == cudaSuccess) {
        t += e;
        f += r.flops;
        ++n;
      }
    }
  }
  *ms = t;
  *flops = f;
  *launches = n;
  return AVVAD_OK;
}

// Per-launch records of one category, in launch order: ms[i], flops[i]; returns the count (<= max_n).
extern "C" int64_t avvad_profile_dump(int cat, double* ms, double* flops, int64_t max_n) {
  if (!ms || !flops || max_n <= 0) return 0;
  if (cudaDeviceSynchronize() != cudaSuccess) return 0;
  std::lock_guard<std::mutex> lk(tc::g_prof_mu);
  int64_t n = 0;
  for (auto& r : tc::g_prof) {
    if (r.cat != cat || n >= max_n) continue;
    float e = 0.f;
    if (cudaEventElapsedTime(&e, r.beg, r.end) != cudaSuccess) continue;
    ms[n] = e;
    flops[n] = r.flops;
    ++n;
  }
  return n;
}

extern "C" int avvad_profile_clear(void) {
  std::lock_guard<std::mutex> lk(tc::g_prof_mu);
  for (auto& r : tc::g_prof) {
    tc::g_prof_pool.push_back(r.beg);
    tc::g_prof_pool.push_back(r.end);
  }
  tc::g_prof.clear();
  return AVVAD_OK;
}

extern "C" int avvad_gemm_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, void* Cp,
                               int64_t ldc, int c_is_bf16, int relu, int64_t M, int64_t N, int64_t K, void* stream) {
  AVVAD_CHECK_ARG(A && W && Cp, "null pointer");
  AVVAD_CHECK_ARG(M > 0 && N > 0 && N < (1 << 30), "bad M/N");
  tc::EpiParams ep{};
  ep.bias = bias;
  ep.C = Cp;
  ep.ldc = ldc;
  ep.relu = relu;
  return tc::gemm_dispatch((const __nv_bfloat16*)A, lda, (const __nv_bfloat16*)W, ldw, M, (int)N, (int)K, ep,
                           c_is_bf16 ? tc::EPI_BF16 : tc::EPI_F32, 0, (cudaStream_t)stream);
}

extern "C" int avvad_conv2d_nhwc_bf16(const void* in, const void* w, const float* bias, const void* residual,
                                      void* out, int64_t n, int H, int W, int Cin, int Cout, int R, int S, int stride,
                                      int pad, int relu, void* stream) {
  AVVAD_CHECK_ARG(in && w && out, "null pointer");
  AVVAD_CHECK_ARG(n > 0 && H > 0 && W > 0 && R > 0 && S > 0 && stride > 0 && pad >= 0, "bad conv shape");
  AVVAD_CHECK_ARG(Cin % 64 == 0 && Cout % 32 == 0, "Cin must be a multiple of 64 and Cout of 32");
  const int OH = (H + 2 * pad - R) / stride + 1;
  const int OW = (W + 2 * pad - S) / stride + 1;
  AVVAD_CHECK_ARG(OH > 0 && OW > 0, "empty output");
  tc::EpiParams ep{};
  ep.bias = bias;
  ep.residual = (const __nv_bfloat16*)residual;
  ep.C = out;
  ep.ldc = Cout;
  ep.relu = relu;
  if (!tc::tma_available()) {
    set_error("cuTensorMapEncodeTiled driver entry point unavailable: libavvad needs a CUDA 12 driver");
    return AVVAD_ERR_CUDA;
  }
  AVVAD_CHECK_ARG(OW <= 128, "output width above 128 is not supported by the TMA box tiling");
  // the slab epilogue uses 256-bit residual loads / output stores: rows must be 32-byte aligned
  const bool aligned32 = ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(residual)) & 31) == 0;
  if (aligned32 && tc::slab_supported(H, W, Cin, Cout, R, S, stride, pad))
    return tc::launch_slab_conv((const __nv_bfloat16*)in, (const __nv_bfloat16*)w, ep, n, H, Cin, Cout,
                                (cudaStream_t)stream);
  return tc::launch_tma_conv((const __nv_bfloat16*)in, (const __nv_bfloat16*)w, ep, n, H, W, Cin, Cout, R, S, stride,
                             pad, 0, (cudaStream_t)stream);
}

extern "C" int avvad_conv2d_nhwc_bf16_dual(const void* in, const void* in2, const void* w, const float* bias, void* out,
                                           int64_t n, int H, int W, int Cin, int H2, int W2, int Cin2, int stride2,
                                           int Cout, int R, int S, int stride, int pad, int relu, void* stream) {
  AVVAD_CHECK_ARG(in && in2 && w && out, "null pointer");
  AVVAD_CHECK_ARG(n > 0 && H > 0 && W > 0 && H2 > 0 && W2 > 0 && R > 0 && S > 0 && stride > 0 && stride2 > 0 && pad >= 0,
                  "bad conv shape");
  AVVAD_CHECK_ARG(Cin % 64 == 0 && Cin2 % 64 == 0 && Cout % 32 == 0, "Cin, Cin2 multiples of 64 and Cout of 32");
  if (!tc::tma_available()) {
    set_error("cuTensorMapEncodeTiled driver entry point unavailable: libavvad needs a CUDA 12 driver");
    return AVVAD_ERR_CUDA;
  }
  tc::EpiParams ep{};
  ep.bias = bias;
  ep.C = out;
  ep.ldc = Cout;
  ep.relu = relu;
  tc::SecondOperand so;
  so.in2 = (const __nv_bfloat16*)in2;
  so.H2 = H2; so.W2 = W2; so.Cin2 = Cin2; so.stride2 = stride2;
  return tc::launch_tma_conv((const __nv_bfloat16*)in, (const __nv_bfloat16*)w, ep, n, H, W, Cin, Cout, R, S, stride,
                             pad, 0, (cudaStream_t)stream, 0, 0.0, &so);
}

extern "C" int avvad_pack_rows_bf16(const float* src, int64_t ld_src, void* dst, int64_t ld_dst, int64_t col_off,
                                    int64_t rows, int64_t cols, int zero_tail, void* stream) {
  AVVAD_CHECK_ARG(src && dst && rows > 0 && cols > 0 && col_off >= 0 && col_off + cols <= ld_dst, "bad argument");
  const int64_t width = zero_tail ? (ld_dst - col_off) : cols;
  const int64_t total = rows * width;
  tc::pack_rows_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, (cudaStream_t)stream>>>(
      src, ld_src, (__nv_bfloat16*)dst, ld_dst, col_off, rows, cols, width);
  AVVAD_LAUNCHED();
  return AVVAD_OK;
}
