// Shared pieces of the bf16 tensor-core engine for sm_100a (C[M][N] = A[M][K] * W[N][K]^T, fp32 accumulation in TMEM):
// PTX wrappers (mbarrier, tcgen05.alloc / mma / commit / ld, UMMA descriptors), the epilogue parameter block and the
// generic per-chunk epilogue (bias / residual / ReLU / LSTM cell).  The kernels live in gemm_tma.cuh (TMA-fed
// implicit GEMM), conv_slab.cuh (3x3 slab convolution), stem_s2d.cuh (stem) and lstm_persist.cuh (recurrence).
#pragma once
#include "common.cuh"

namespace avvad {
namespace tc {

constexpr int BM = 128;
constexpr int BK = 64;  // bf16 elements per K block = 128 bytes = one swizzle row
// EPI_XT: fp32 output of the LSTM input projection in the recurrence's layout xT[t][u][b][4] (see launch_tma_gemm_xt)
enum EpiMode { EPI_BF16 = 0, EPI_F32 = 1, EPI_LSTM = 2, EPI_XT = 3 };

struct EpiParams {
  const float* bias;              // [N] or null
  const __nv_bfloat16* residual;  // [M][ldc] or null (EPI_BF16)
  void* C;                        // bf16 or f32 [M][ldc]
  int64_t ldc;
  int relu;
  // EPI_LSTM: accumulator column n = 4*u + gate (i,f,g,o); row = batch index b
  const float* xproj;     // [B][T][4H] gate-interleaved input projection (+ both biases)
  float* c_state;         // [B][H]
  __nv_bfloat16* h_next;  // [B][H]   A operand of the next step
  __nv_bfloat16* hseq;    // [B][T][H] layer output (zero for t >= len_b)
  const int32_t* lengths;
  int t, T, H4;
};

// ---- PTX wrappers ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (reported as a CUDA error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 24)) __trap();
  }
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem), "r"(cols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout):
//   [0,14) start address >> 4 | [16,30) LBO >> 4 (=1, unused for swizzled K-major) |
//   [32,46) SBO >> 4 (=1024 B between 8-row groups) | [46,48) version = 1 | [61,64) layout = 2 (SW128)
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor: D=f32 (bit4), A=B=bf16 (bits 7,10), K-major A and B, N>>3 at [17,23),
// M>>4 at [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accum)
      : "memory");
}
// Same instruction with the two descriptors given as (low word, shared high word): the high word of a K-major
// SWIZZLE_128B descriptor (SBO, version, layout) is constant, so stepping a descriptor is one 32-bit add on the
// low word ((address >> 4) | LBO << 16) -- keeps the single issuing thread ahead of 48-cycle MMAs.
constexpr uint32_t kDescHi = (64u) | (1u << 14) | (2u << 29);  // SBO=1024>>4 | version 1 | SWIZZLE_128B
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr) { return ((saddr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ void umma_f16_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc,
                                            uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accum), "r"(kDescHi)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets row (lane base + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 16 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
// One elected lane of a fully converged warp (deterministic for a given mask).  Issuing tcgen05.mma / commit / TMA from
// `if (elect_one_sync())` inside warp-uniform control flow lets the compiler keep descriptors in uniform registers and
// emit the instructions back to back; the older `if (lane == 0) { whole loop }` form made every issue pay ~10-20
// scalar instructions (R2UR, ELECT, BRA.U.ANY loops), which was the bound for N <= 128 tiles (48-64 cycle MMAs).
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- epilogue for one 32-column chunk held by one thread (row m, columns n0..n0+31) ----------------
__device__ __forceinline__ void epilogue_chunk(const EpiParams& ep, int mode, const uint32_t (&v)[32], int64_t m,
                                               int n0, int N) {
  if (mode == EPI_LSTM) {
    // 8 hidden units x (i,f,g,o)
    const int b = (int)m;
    const int u0 = n0 >> 2;
    const int H = ep.H4 >> 2;
    const float* xp = ep.xproj + ((int64_t)b * ep.T + ep.t) * ep.H4 + n0;
    float* cs = ep.c_state + (int64_t)b * H + u0;
    const bool live = ep.t < ep.lengths[b];
    float hv[8];
    float4 c_lo = *reinterpret_cast<const float4*>(cs);
    float4 c_hi = *reinterpret_cast<const float4*>(cs + 4);
    float cv[8] = {c_lo.x, c_lo.y, c_lo.z, c_lo.w, c_hi.x, c_hi.y, c_hi.z, c_hi.w};
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const float4 x4 = *reinterpret_cast<const float4*>(xp + 4 * u);
      const float gi = __uint_as_float(v[4 * u + 0]) + x4.x;
      const float gf = __uint_as_float(v[4 * u + 1]) + x4.y;
      const float gg = __uint_as_float(v[4 * u + 2]) + x4.z;
      const float go = __uint_as_float(v[4 * u + 3]) + x4.w;
      const float c = sigmoidf_fast(gf) * cv[u] + sigmoidf_fast(gi) * tanhf_fast(gg);
      cv[u] = c;
      hv[u] = sigmoidf_fast(go) * tanhf_fast(c);
    }
    *reinterpret_cast<float4*>(cs) = make_float4(cv[0], cv[1], cv[2], cv[3]);
    *reinterpret_cast<float4*>(cs + 4) = make_float4(cv[4], cv[5], cv[6], cv[7]);
    uint4 hp;
    hp.x = pack_bf16x2(hv[0], hv[1]);
    hp.y = pack_bf16x2(hv[2], hv[3]);
    hp.z = pack_bf16x2(hv[4], hv[5]);
    hp.w = pack_bf16x2(hv[6], hv[7]);
    *reinterpret_cast<uint4*>(ep.h_next + (int64_t)b * H + u0) = hp;
    if (!live) hp = make_uint4(0u, 0u, 0u, 0u);
    *reinterpret_cast<uint4*>(ep.hseq + ((int64_t)b * ep.T + ep.t) * H + u0) = hp;
    return;
  }
  // NOTE: every access to f[] below uses a compile-time index (fully unrolled loops with predicates); a runtime
  // index would push the array to local memory and turn the whole epilogue into L1 traffic.
  float f[32];
#pragma unroll
  for (int q = 0; q < 32; ++q) f[q] = __uint_as_float(v[q]);
  const bool full = (n0 + 32 <= N);
  if (ep.bias) {
    if (full) {
      const float4* bp = reinterpret_cast<const float4*>(ep.bias + n0);  // n0 % 32 == 0 -> 16-byte aligned
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float4 b4 = __ldg(bp + q);
        f[4 * q + 0] += b4.x; f[4 * q + 1] += b4.y; f[4 * q + 2] += b4.z; f[4 * q + 3] += b4.w;
      }
    } else {
#pragma unroll
      for (int q = 0; q < 32; ++q)
        if (n0 + q < N) f[q] += __ldg(ep.bias + n0 + q);
    }
  }
  if (mode == EPI_BF16) {
    __nv_bfloat16* crow = reinterpret_cast<__nv_bfloat16*>(ep.C) + m * ep.ldc + n0;
    if (full) {
      if (ep.residual) {
        const uint4* rp = reinterpret_cast<const uint4*>(ep.residual + m * ep.ldc + n0);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint4 r = rp[q];
          float2 a = unpack_bf16x2(r.x), b2 = unpack_bf16x2(r.y), c2 = unpack_bf16x2(r.z), d2 = unpack_bf16x2(r.w);
          f[8 * q + 0] += a.x;  f[8 * q + 1] += a.y;  f[8 * q + 2] += b2.x; f[8 * q + 3] += b2.y;
          f[8 * q + 4] += c2.x; f[8 * q + 5] += c2.y; f[8 * q + 6] += d2.x; f[8 * q + 7] += d2.y;
        }
      }
      if (ep.relu) {
#pragma unroll
        for (int q = 0; q < 32; ++q) f[q] = fmaxf(f[q], 0.f);
      }
      uint4* cp = reinterpret_cast<uint4*>(crow);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint4 o;
        o.x = pack_bf16x2(f[8 * q + 0], f[8 * q + 1]);
        o.y = pack_bf16x2(f[8 * q + 2], f[8 * q + 3]);
        o.z = pack_bf16x2(f[8 * q + 4], f[8 * q + 5]);
        o.w = pack_bf16x2(f[8 * q + 6], f[8 * q + 7]);
        cp[q] = o;
      }
    } else {
#pragma unroll
      for (int q = 0; q < 32; ++q) {
        if (n0 + q < N) {
          float x = f[q];
          if (ep.residual) x += __bfloat162float(ep.residual[m * ep.ldc + n0 + q]);
          if (ep.relu) x = fmaxf(x, 0.f);
          crow[q] = __float2bfloat16_rn(x);
        }
      }
    }
  } else {  // EPI_F32
    float* crow = reinterpret_cast<float*>(ep.C) + m * ep.ldc + n0;
    if (ep.relu) {
#pragma unroll
      for (int q = 0; q < 32; ++q) f[q] = fmaxf(f[q], 0.f);
    }
    if (full && ((reinterpret_cast<uintptr_t>(crow) & 15) == 0)) {
      float4* cp = reinterpret_cast<float4*>(crow);
#pragma unroll
      for (int q = 0; q < 8; ++q) cp[q] = make_float4(f[4 * q], f[4 * q + 1], f[4 * q + 2], f[4 * q + 3]);
    } else {
#pragma unroll
      for (int q = 0; q < 32; ++q)
        if (n0 + q < N) crow[q] = f[q];
    }
  }
}

// ---- host-side launcher -----------------------------------------------------------------------------
bool profiling_on();
int prof_begin(cudaStream_t st, void** tok);
void prof_end(cudaStream_t st, void* tok, int cat, double flops);
int prof_group_begin(cudaStream_t st, void** tok);
void prof_group_end(cudaStream_t st, void* tok, int cat, double flops);
int gemm_dispatch(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* Wt, int64_t ldw, int64_t M, int N, int K,
                  const EpiParams& ep, int epi_mode, int bn_hint, cudaStream_t st);

}  // namespace tc
}  // namespace avvad
