// TMA-fed variant of the tcgen05 engine (sm_100a): operands are staged by the Tensor Memory Accelerator instead of
// per-thread cp.async gathers, so operand delivery costs one instruction per box instead of ~2000 per K block.
//
//   warp 0 (lane 0) : TMA producer.  Per K block it arms full[s] with the expected byte count and issues
//                     cp.async.bulk.tensor: a 4-D box {64 ch, OW, hb, F} of the NHWC activation for the A
//                     operand (the box IS the im2col tile of one filter tap: the tap only shifts the box
//                     coordinates, out-of-image pixels are zero-filled by the hardware, stride-2 convolutions use
//                     the map's traversal strides) and a 2-D box {64, BN} of the packed weights for B.  Both land
//                     in the canonical K-major SWIZZLE_128B layout the UMMA descriptors expect.
//   warp 1          : TMEM allocation; lane 0 issues tcgen05.mma / tcgen05.commit (as in gemm_tc.cuh).
//   warps 2-9       : epilogue (TMEM -> registers -> bias / residual / ReLU / LSTM cell -> global).  Two warps per
//                     TMEM lane quarter split the 32-column chunks of a tile; the residual of a thread's chunks is
//                     requested BEFORE the wait on the accumulator and the bias sits in shared memory, so no global
//                     latency is left on the drain path.
//
// K-concatenated second operand (ResNet downsample blocks): after the KB blocks of the main convolution the producer
// appends KB2 blocks of a 1x1 / stride-s2 convolution over a SECOND activation tensor (maps.a2) into the same
// accumulator -- out = conv3x3(y) + conv1x1_s2(x) + bias -- so the downsample branch costs neither a launch nor an
// output/residual round trip.  The packed weight rows are [9*C | Cin2] wide.
//
// An output tile is F whole frames x a band of hb output rows (F*hb*OW <= 128 accumulator rows).  Up to two
// "phases" with different (hb, F) cover a frame (e.g. 17x17: two 7-row bands per frame + one 3-row band over
// two frames = 90 % of the 128 MMA rows; 9x9: 7 rows x 2 frames + 2 rows x 7 frames = 98 %).  A plain GEMM is the
// degenerate case C=K, W=M, H=1.
#pragma once
#include <cuda.h>

#include "gemm_tc.cuh"

namespace avvad {
namespace tc {

constexpr int kTmaThreads = 320;
constexpr int kTmaEpiWarps = 8;
// bias entries staged in shared memory (N <= this), else read through L1: the BN = 256 configuration runs one CTA per
// SM and can afford the 4096 columns of the LSTM input projection, the two-CTA configurations keep 1024
template <int BN>
struct TmaBias {
  static constexpr int kEntries = (BN == 256) ? 4096 : 1024;
};

struct TmaGeom {
  int mode;             // 0 = plain GEMM rows, 1 = convolution boxes
  int n_tiles;          // tiles along N
  int64_t total_tiles;  // all (super m, n) tiles of the launch
  int64_t m_tiles;      // 128-row blocks (both phases)
  int64_t tiles0;       // m-tiles of phase 0 (conv)
  int h0[2], hb[2], nb[2], F[2];  // per phase: first output row, band height, bands per frame, frames per tile
  int OH, OW, stride, pad, S, cpb, KB;
  int KB2, stride2;     // K-concatenated 1x1 / stride2 / pad 0 second operand (0 = none)
  // split-K (plain GEMM, fp32 output, no bias): split s covers K blocks [s*kb_split, (s+1)*kb_split) and writes its
  // partial product to C + s*split_stride; the consumer sums the partials (tiny-M GEMMs such as the BPTT step would
  // otherwise run on 32 CTAs with a 64-block K loop each)
  int ksplit, kb_split;
  int64_t split_stride, m_supers;
  int64_t n_frames;     // conv: frames in this launch; gemm: M
  int N;
  // time-major GEMM over a [B][T][K] operand (launch_tma_gemm_xt): row index m = t * tm_bp + b, tm_bp = B rounded up to
  // 128, so that a 128-row tile is 128 consecutive batch items of ONE time step (0 = plain row order)
  int tm_bp, tm_b;
  int64_t tm_tstride;   // time-major GEMM with a row-major output (launch_tma_gemm_tm): output row = b * tm_tstride + t
  int pair;      // host only: launch on CTA pairs (decided where the weight map is encoded: its box is BN/2 rows then)
  int grid_cap;  // host only: at most this many CTAs (0 = all SMs) -- for launches that share the GPU with a recurrence
  uint32_t bytesA[2];   // TMA box bytes per phase
  uint32_t bytesB;
};

struct TmaMaps {
  CUtensorMap a[2];
  CUtensorMap a2[2];  // second operand (per phase), valid when TmaGeom::KB2 > 0
  CUtensorMap b;
};

__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3,
                                            uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void umma_f16_lo2(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc,
                                             uint32_t accum, uint32_t hi) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accum), "r"(hi)
      : "memory");
}
// ---- CTA-pair (tcgen05 cta_group::2) primitives: both CTAs of a cluster of two execute the loads, the transaction bytes
// complete on the LEADER's barrier (cluster address `bar_leader`); rank 0 issues the M = 256 MMAs; commits are multicast
__device__ __forceinline__ void tma_load_4d_2sm(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3,
                                                uint32_t bar_leader) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%2, %3, %4, %5}], [%6];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar_leader)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar_leader) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar_leader)
      : "memory");
}
__device__ __forceinline__ void umma2_f16_lo2(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc,
                                              uint32_t accum, uint32_t hi) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accum), "r"(hi)
      : "memory");
}
__device__ __forceinline__ void umma2_commit_mc2(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"((uint16_t)3)
      : "memory");
}
__device__ __forceinline__ uint32_t pair_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t pair_mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void pair_arrive(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void pair_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// kind::f16 instruction descriptor, M = 256 over the pair
__host__ __device__ constexpr uint32_t make_idesc_m256(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// KE = bf16 elements per K block: 64 (128-byte rows, SWIZZLE_128B, four K16 UMMAs per block) or 16 (32-byte rows,
// SWIZZLE_32B, one UMMA per block -- used by the stem convolution whose packed input has 16 "channels").
// MB = accumulator blocks (128 rows each) per tile that share one weight box per K block.  A 128x128 tile moves
// 32 KB through L2 -> SMEM per 256 MMA cycles (128 B/clk/SM, more than L2 delivers to 148 SMs at once: the N = 128
// layers sat at 51-57 % tensor activity with L2 at 62-65 %); MB = 2 makes it 48 KB per 512 cycles (96 B/clk), the
// ratio of the 128x256 tiles.  TMEM: 2 (double buffer) x MB x BN columns <= 512.
// CG = 2: the tile is two accumulator blocks x BN columns computed by a CTA PAIR (tcgen05 cta_group::2, M = 256): each CTA
// stages its own block of A and HALF of the weight box (the tensor cores of both SMs read both halves), so a K block
// costs 32 KB of L2 -> SMEM traffic per SM instead of 48 KB and the same shared memory holds six stages instead of four.
template <int BN, int KE = 64, int MB = 1, int CG = 1>
struct TmaCfg {
  static constexpr uint32_t kRowBytes = KE * 2;
  static constexpr uint32_t kABytes = BM * kRowBytes;
  static constexpr uint32_t kBBytes = (BN / CG) * kRowBytes;  // per CTA
  static constexpr uint32_t kStageBytes = MB * kABytes + kBBytes;
  static constexpr int kCtasPerSm = (BN == 256 || MB > 1 || CG == 2) ? 1 : 2;
  // ring depth: fill ~200 KB per SM
  static constexpr int kStages =
      (CG == 2) ? (int)((200u * 1024u) / kStageBytes)
                : ((KE == 16) ? 8 : ((BN == 256) ? 4 : ((BN == 128) ? (MB > 1 ? 4 : 3) : 4)));
  static_assert(CG == 1 || (KE == 64 && (BN == 256 || BN == 128)), "pair mode: BN = 256 or 128");
  static constexpr uint32_t kSmemBytes = kStages * kStageBytes + 1024 + 256 + TmaBias<BN>::kEntries * 4;
  // descriptor high word: SBO (8 rows) >> 4 | version 1 << 14 | layout (2 = SW128, 6 = SW32) << 29
  static constexpr uint32_t kDescHiWord = ((8 * kRowBytes) >> 4) | (1u << 14) | ((KE == 64 ? 2u : 6u) << 29);
  static_assert(2 * MB * BN <= 512, "TMEM: two accumulator stages of MB x BN columns");
};

struct TileCoord {
  int phase;
  int64_t n0;   // conv: first frame; gemm: first row
  int hstart;   // conv: first output row of the band
  bool valid;   // false: block index past the last m-tile (operands of the last valid block are loaded, nothing is stored)
};

// m-tile index -> coordinates (clamped to the last m-tile)
__device__ __forceinline__ TileCoord decode_block(const TmaGeom& g, int64_t mt) {
  TileCoord t;
  t.valid = mt < g.m_tiles;
  if (!t.valid) mt = g.m_tiles - 1;
  if (g.mode == 0) {
    t.phase = 0;
    t.n0 = mt * BM;
    t.hstart = 0;
    return t;
  }
  t.phase = (mt < g.tiles0) ? 0 : 1;
  if (t.phase) mt -= g.tiles0;
  const int nb = g.nb[t.phase];
  const int band = (int)(mt % nb);
  t.n0 = (mt / nb) * g.F[t.phase];
  t.hstart = g.h0[t.phase] + band * g.hb[t.phase];
  return t;
}

template <int BN, int KE, int MB, int CG = 1>
__global__ void __launch_bounds__(kTmaThreads, TmaCfg<BN, KE, MB, CG>::kCtasPerSm)
tc_tma_kernel(const __grid_constant__ TmaMaps maps, const __grid_constant__ TmaGeom g, const EpiParams ep,
              const int epi_mode) {
  using C = TmaCfg<BN, KE, MB, CG>;
  constexpr int S = C::kStages;
  constexpr int MBT = CG * MB;  // accumulator blocks per tile (over the pair when CG == 2)
  // pair mode: CTA `rank` owns blocks rank*MB .. rank*MB + MB-1 of every tile (MMA mb pairs block mb of both CTAs into
  // one M = 256 instruction); tiles are distributed over clusters
  const uint32_t rank = (CG == 2) ? pair_rank() : 0u;
  const int64_t tile0 = (CG == 2) ? (int64_t)(blockIdx.x >> 1) : (int64_t)blockIdx.x;
  const int64_t tile_step = (CG == 2) ? (int64_t)(gridDim.x >> 1) : (int64_t)gridDim.x;
  constexpr uint32_t kAccCols = MB * BN;       // columns of one accumulator stage
  constexpr uint32_t kTmemCols = 2 * kAccCols;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw);
  const uint32_t bar0 = base + S * C::kStageBytes;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + S * C::kStageBytes + 8 * (2 * S + 4));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(bar0 + 8 * s, 1);        // full: the producer's arrive.expect_tx (+ TMA transaction bytes)
      mbar_init(bar0 + 8 * (S + s), 1);  // empty: tcgen05.commit
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar0 + 8 * (2 * S + a), 1);      // tmem full
      mbar_init(bar0 + 8 * (2 * S + 2 + a), CG * kTmaEpiWarps);  // tmem empty: one arrival per epilogue warp (of the pair)
    }
    fence_barrier_init();
    tma_prefetch_desc(&maps.a[0]);
    tma_prefetch_desc(&maps.a[1]);
    if (g.KB2 > 0) {
      tma_prefetch_desc(&maps.a2[0]);
      tma_prefetch_desc(&maps.a2[1]);
    }
    tma_prefetch_desc(&maps.b);
  }
  // bias -> shared memory (behind the barriers and the TMEM slot); zero when absent
  float* bias_s = reinterpret_cast<float*>(smem + S * C::kStageBytes + 256);
  const bool bias_in_smem = g.N <= TmaBias<BN>::kEntries;
  if (bias_in_smem)
    for (int i = threadIdx.x; i < g.N; i += kTmaThreads) bias_s[i] = ep.bias ? ep.bias[i] : 0.f;
  if (warp == 1) {
    if (CG == 2) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                       smem_u32(const_cast<uint32_t*>(tmem_slot))),
                   "r"(kTmemCols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), kTmemCols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CG == 2) pair_sync();  // the peer's barriers are initialised and its TMEM allocated before anything targets them
  tc_fence_after();
  const uint32_t tmem_acc = *tmem_slot;
  const uint32_t bar0_leader = (CG == 2) ? pair_mapa(bar0, 0) : bar0;

  // tile = (n-tile fastest, super m-tile); super m-tile sm covers m-tiles sm*MBT .. sm*MBT + MBT-1
  if (warp == 0) {
    // ================= TMA producer (warp-converged; one elected lane issues) =================
    uint32_t it = 0;
    for (int64_t tile = tile0; tile < g.total_tiles; tile += tile_step) {
      const int n_base = (int)(tile % g.n_tiles) * BN + (int)rank * (BN / CG);  // pair mode: this CTA's half of the box
      const int64_t sm = (tile / g.n_tiles) % g.m_supers;
      const int split = (int)(tile / (g.n_tiles * g.m_supers));
      const int kb0 = split * g.kb_split;
      const int kb1 = (kb0 + g.kb_split < g.KB) ? kb0 + g.kb_split : g.KB;
      TileCoord t[MB];
      uint32_t bytes = g.bytesB;  // pair mode: the leader expects both halves of the weight box and both A blocks
#pragma unroll
      for (int mb = 0; mb < MB; ++mb) {
        t[mb] = decode_block(g, sm * MBT + mb + (CG == 2 ? (int)rank * MB : 0));
        bytes += g.bytesA[t[mb].phase];
      }
      if (CG == 2) {
#pragma unroll
        for (int mb = 0; mb < MB; ++mb) bytes += g.bytesA[decode_block(g, sm * MBT + mb + (1 - (int)rank) * MB).phase];
      }
      int cb = 0, fr = 0, fs = 0;
      for (int kb = kb0; kb < kb1; ++kb, ++it) {  // conv mode: kb0 = 0, kb1 = KB
        const int s = it % S;
        const uint32_t ph = (it / S) & 1u;
        mbar_wait(bar0 + 8 * (S + s), ph ^ 1u);
        if (elect_one_sync()) {
          const uint32_t sa = base + s * C::kStageBytes;
          if (CG == 2) {
            const uint32_t full = bar0_leader + 8 * s;
            if (rank == 0) mbar_arrive_expect_tx(bar0 + 8 * s, bytes);
#pragma unroll
            for (int mb = 0; mb < MB; ++mb) {
              const uint32_t da = sa + mb * C::kABytes;
              if (g.mode == 0) {
                if (g.tm_bp)
                  tma_load_4d_2sm(da, &maps.a[0], kb * KE, (int)(t[mb].n0 % g.tm_bp), (int)(t[mb].n0 / g.tm_bp), 0, full);
                else
                  tma_load_4d_2sm(da, &maps.a[0], kb * KE, (int)t[mb].n0, 0, 0, full);
              } else {
                tma_load_4d_2sm(da, &maps.a[t[mb].phase], cb * KE, fs - g.pad, t[mb].hstart * g.stride + fr - g.pad,
                                (int)t[mb].n0, full);
              }
            }
            tma_load_2d_2sm(sa + MB * C::kABytes, &maps.b, kb * KE, n_base, full);
          } else {
          const uint32_t full = bar0 + 8 * s;
          mbar_arrive_expect_tx(full, bytes);
#pragma unroll
          for (int mb = 0; mb < MB; ++mb) {
            if (g.mode == 0) {
              if (g.tm_bp)
                tma_load_4d(sa + mb * C::kABytes, &maps.a[0], kb * KE, (int)(t[mb].n0 % g.tm_bp),
                            (int)(t[mb].n0 / g.tm_bp), 0, full);
              else
                tma_load_4d(sa + mb * C::kABytes, &maps.a[0], kb * KE, (int)t[mb].n0, 0, 0, full);
            } else {
              tma_load_4d(sa + mb * C::kABytes, &maps.a[t[mb].phase], cb * KE, fs - g.pad,
                          t[mb].hstart * g.stride + fr - g.pad, (int)t[mb].n0, full);
            }
          }
          tma_load_2d(sa + MB * C::kABytes, &maps.b, kb * KE, n_base, full);
          }
        }
        __syncwarp();
        if (++cb == g.cpb) {
          cb = 0;
          if (++fs == g.S) {
            fs = 0;
            ++fr;
          }
        }
      }
      for (int kb2 = 0; kb2 < g.KB2; ++kb2, ++it) {
        const int s = it % S;
        const uint32_t ph = (it / S) & 1u;
        mbar_wait(bar0 + 8 * (S + s), ph ^ 1u);
        if (elect_one_sync()) {
          const uint32_t sa = base + s * C::kStageBytes;
          if (CG == 2) {
            const uint32_t full = bar0_leader + 8 * s;
            if (rank == 0) mbar_arrive_expect_tx(bar0 + 8 * s, bytes);
#pragma unroll
            for (int mb = 0; mb < MB; ++mb)
              tma_load_4d_2sm(sa + mb * C::kABytes, &maps.a2[t[mb].phase], kb2 * KE, 0, t[mb].hstart * g.stride2,
                              (int)t[mb].n0, full);
            tma_load_2d_2sm(sa + MB * C::kABytes, &maps.b, (g.KB + kb2) * KE, n_base, full);
          } else {
          const uint32_t full = bar0 + 8 * s;
          mbar_arrive_expect_tx(full, bytes);
#pragma unroll
          for (int mb = 0; mb < MB; ++mb)
            tma_load_4d(sa + mb * C::kABytes, &maps.a2[t[mb].phase], kb2 * KE, 0, t[mb].hstart * g.stride2,
                        (int)t[mb].n0, full);
          tma_load_2d(sa + MB * C::kABytes, &maps.b, (g.KB + kb2) * KE, n_base, full);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (warp-converged; one elected lane issues MMAs and commits) =================
    constexpr uint32_t idesc = (CG == 2) ? make_idesc_m256(BN) : make_idesc(BN);
    uint32_t it = 0, tl = 0;
    if (CG == 1 || rank == 0)  // pair mode: the leader issues for both CTAs
    for (int64_t tile = tile0; tile < g.total_tiles; tile += tile_step, ++tl) {
      const uint32_t acc = tl & 1u, aph = (tl >> 1) & 1u;
      const int split = (int)(tile / (g.n_tiles * g.m_supers));
      const int kbs = split * g.kb_split;
      const int kb_total = ((kbs + g.kb_split < g.KB) ? g.kb_split : g.KB - kbs) + g.KB2;
      mbar_wait(bar0 + 8 * (2 * S + 2 + acc), aph ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_acc + acc * kAccCols;
      for (int kb = 0; kb < kb_total; ++kb, ++it) {
        const int s = it % S;
        const uint32_t ph = (it / S) & 1u;
        mbar_wait(bar0 + 8 * s, ph);
        tc_fence_after();
        if (elect_one_sync()) {
          const uint32_t a0 = desc_lo(base + s * C::kStageBytes);
          const uint32_t b_lo = a0 + ((MB * C::kABytes) >> 4);
#pragma unroll
          for (int mb = 0; mb < MB; ++mb) {
            const uint32_t a_lo = a0 + ((mb * C::kABytes) >> 4);
            const uint32_t d = d_tmem + mb * BN;
            if (CG == 2) {
              umma2_f16_lo2(d, a_lo, b_lo, idesc, kb != 0, C::kDescHiWord);
              umma2_f16_lo2(d, a_lo + 2, b_lo + 2, idesc, 1, C::kDescHiWord);
              umma2_f16_lo2(d, a_lo + 4, b_lo + 4, idesc, 1, C::kDescHiWord);
              umma2_f16_lo2(d, a_lo + 6, b_lo + 6, idesc, 1, C::kDescHiWord);
              continue;
            }
            umma_f16_lo2(d, a_lo, b_lo, idesc, kb != 0, C::kDescHiWord);
            if (KE == 64) {
              umma_f16_lo2(d, a_lo + 2, b_lo + 2, idesc, 1, C::kDescHiWord);
              umma_f16_lo2(d, a_lo + 4, b_lo + 4, idesc, 1, C::kDescHiWord);
              umma_f16_lo2(d, a_lo + 6, b_lo + 6, idesc, 1, C::kDescHiWord);
            }
          }
          if (CG == 2) {
            umma2_commit_mc2(bar0 + 8 * (S + s));
            if (kb == kb_total - 1) umma2_commit_mc2(bar0 + 8 * (2 * S + acc));
          } else {
            umma_commit(bar0 + 8 * (S + s));
            if (kb == kb_total - 1) umma_commit(bar0 + 8 * (2 * S + acc));
          }
        }
        __syncwarp();
      }
    }
  } else {
    // ================= epilogue warps 2..9 =================
    const int q = warp & 3;             // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;   // chunk parity handled by this warp
    constexpr int kJ = BN / 32;         // 32-column chunks per accumulator block
    constexpr int kMine = (kJ + 1) / 2;  // chunks per warp and block
    const bool fast = (epi_mode == EPI_BF16) && bias_in_smem && (g.N % 32 == 0);
    const bool fast32 = (epi_mode == EPI_F32) && bias_in_smem && (g.N % 32 == 0) && (ep.ldc % 4 == 0) &&
                        ((reinterpret_cast<uintptr_t>(ep.C) & 15) == 0);
    uint32_t tl = 0;
    for (int64_t tile = tile0; tile < g.total_tiles; tile += tile_step, ++tl) {
      const int n_base = (int)(tile % g.n_tiles) * BN;
      const int64_t sm = (tile / g.n_tiles) % g.m_supers;
      const int64_t c_off = (tile / (g.n_tiles * g.m_supers)) * g.split_stride;  // split-K partial (fp32 paths)
      const uint32_t acc = tl & 1u, aph = (tl >> 1) & 1u;
      // output row of accumulator row r = q*32 + lane of every block
      const int r = q * 32 + lane;
      int64_t m[MB];
#pragma unroll
      for (int mb = 0; mb < MB; ++mb) {
        const TileCoord t = decode_block(g, sm * MBT + mb + (CG == 2 ? (int)rank * MB : 0));
        m[mb] = -1;
        if (!t.valid) continue;
        if (g.mode == 0) {
          if (t.n0 + r < g.n_frames) m[mb] = t.n0 + r;
          if (g.tm_bp && epi_mode != EPI_XT && m[mb] >= 0) {  // time-major tile order, row-major [b][t] output
            const int64_t tt = m[mb] / g.tm_bp, bb = m[mb] - tt * g.tm_bp;
            m[mb] = (bb < g.tm_b) ? bb * g.tm_tstride + tt : -1;
          }
        } else {
          const int hb = g.hb[t.phase];
          const int per_frame = hb * g.OW;
          const int f = r / per_frame;
          const int rem = r - f * per_frame;
          const int hh = rem / g.OW;
          const int ww = rem - hh * g.OW;
          const int oh = t.hstart + hh;
          if (f < g.F[t.phase] && t.n0 + f < g.n_frames && oh < g.OH)
            m[mb] = ((t.n0 + f) * g.OH + oh) * g.OW + ww;
        }
      }
      const uint32_t t_row = tmem_acc + acc * kAccCols + ((uint32_t)(q * 32) << 16);
      if (fast) {
        // residual of this thread's chunks: in flight while the tile's MMAs run
        u32x8 rb[MB * kMine][2] = {};
        const bool wide = ((reinterpret_cast<uintptr_t>(ep.C) | reinterpret_cast<uintptr_t>(ep.residual)) & 31) == 0 &&
                          (ep.ldc % 16 == 0);  // 32-byte aligned rows: 256-bit loads / stores
        if (ep.residual) {
#pragma unroll
          for (int mb = 0; mb < MB; ++mb)
#pragma unroll
            for (int i = 0; i < kMine; ++i) {
              const int n0 = n_base + (2 * i + half) * 32;
              if (m[mb] >= 0 && 2 * i + half < kJ && n0 < g.N) {
                const __nv_bfloat16* rp = ep.residual + m[mb] * ep.ldc + n0;
                if (wide) {
                  rb[mb * kMine + i][0] = ld_global_256(rp);
                  rb[mb * kMine + i][1] = ld_global_256(rp + 16);
                } else {
                  const uint4* r4 = reinterpret_cast<const uint4*>(rp);
#pragma unroll
                  for (int c = 0; c < 4; ++c) {
                    const uint4 t4 = r4[c];
                    rb[mb * kMine + i][c >> 1].v[4 * (c & 1) + 0] = t4.x;
                    rb[mb * kMine + i][c >> 1].v[4 * (c & 1) + 1] = t4.y;
                    rb[mb * kMine + i][c >> 1].v[4 * (c & 1) + 2] = t4.z;
                    rb[mb * kMine + i][c >> 1].v[4 * (c & 1) + 3] = t4.w;
                  }
                }
              }
            }
        }
        mbar_wait(bar0 + 8 * (2 * S + acc), aph);
        tc_fence_after();
        // pin the prefetched residual behind the wait (otherwise the unpack is hoisted right behind the loads and their
        // latency is paid before the wait instead of under the tile's MMAs)
#pragma unroll
        for (int i = 0; i < MB * kMine; ++i)
#pragma unroll
          for (int c = 0; c < 2; ++c)
#pragma unroll
            for (int e = 0; e < 8; ++e) asm volatile("" : "+r"(rb[i][c].v[e]));
#pragma unroll
        for (int mb = 0; mb < MB; ++mb)
#pragma unroll
          for (int i = 0; i < kMine; ++i) {
            const int j = 2 * i + half;
            if (j < kJ) {  // warp-uniform
              uint32_t v[32];
              tmem_ld32(t_row + mb * BN + j * 32, v);
              tmem_ld_wait();
              const int n0 = n_base + j * 32;
              if (m[mb] >= 0 && n0 < g.N) {
                float f32[32];
                const float4* bp = reinterpret_cast<const float4*>(bias_s + n0);
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                  const float4 b4 = bp[c];
                  f32[4 * c + 0] = __uint_as_float(v[4 * c + 0]) + b4.x;
                  f32[4 * c + 1] = __uint_as_float(v[4 * c + 1]) + b4.y;
                  f32[4 * c + 2] = __uint_as_float(v[4 * c + 2]) + b4.z;
                  f32[4 * c + 3] = __uint_as_float(v[4 * c + 3]) + b4.w;
                }
                if (ep.residual) {
#pragma unroll
                  for (int e = 0; e < 16; ++e) {  // bf16 -> f32 is a 16-bit shift / mask
                    const uint32_t w = rb[mb * kMine + i][e >> 3].v[e & 7];
                    f32[2 * e + 0] += __uint_as_float(w << 16);
                    f32[2 * e + 1] += __uint_as_float(w & 0xFFFF0000u);
                  }
                }
                __nv_bfloat16* cp = reinterpret_cast<__nv_bfloat16*>(ep.C) + m[mb] * ep.ldc + n0;
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                  u32x8 o;
#pragma unroll
                  for (int e = 0; e < 8; ++e)
                    o.v[e] = ep.relu ? pack_relu_bf16x2(f32[16 * c + 2 * e], f32[16 * c + 2 * e + 1])
                                     : pack_bf16x2(f32[16 * c + 2 * e], f32[16 * c + 2 * e + 1]);
                  if (wide) {
                    st_global_256(cp + 16 * c, o);
                  } else {
                    uint4* c4 = reinterpret_cast<uint4*>(cp + 16 * c);
                    c4[0] = make_uint4(o.v[0], o.v[1], o.v[2], o.v[3]);
                    c4[1] = make_uint4(o.v[4], o.v[5], o.v[6], o.v[7]);
                  }
                }
              }
            }
          }
      } else if (epi_mode == EPI_XT) {
        // LSTM input projection in the recurrence's layout: xT[t][u][b][4] (u = hidden unit, the four floats are its
        // gates): lane = batch item, so every 16-byte store of a warp lands in one contiguous 512-byte run, and the
        // recurrence reads it back the same way
        mbar_wait(bar0 + 8 * (2 * S + acc), aph);
        tc_fence_after();
        const int U = g.N >> 2;
#pragma unroll
        for (int mb = 0; mb < MB; ++mb) {
          const int tt = (m[mb] >= 0) ? (int)(m[mb] / g.tm_bp) : 0;
          const int bb = (m[mb] >= 0) ? (int)(m[mb] - (int64_t)tt * g.tm_bp) : g.tm_b;
#pragma unroll 1
          for (int j = half; j < kJ; j += 2) {
            uint32_t v[32];
            tmem_ld32(t_row + mb * BN + j * 32, v);
            tmem_ld_wait();
            const int n0 = n_base + j * 32;
            if (bb < g.tm_b && n0 < g.N) {
              float4* dst = reinterpret_cast<float4*>(ep.C) + ((int64_t)tt * U + (n0 >> 2)) * g.tm_bp + bb;
#pragma unroll
              for (int c = 0; c < 8; ++c) {
                float4 b4;
                if (bias_in_smem) b4 = reinterpret_cast<const float4*>(bias_s + n0)[c];
                else b4 = ep.bias ? __ldg(reinterpret_cast<const float4*>(ep.bias + n0) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
                dst[(int64_t)c * g.tm_bp] = make_float4(__uint_as_float(v[4 * c + 0]) + b4.x, __uint_as_float(v[4 * c + 1]) + b4.y,
                                                        __uint_as_float(v[4 * c + 2]) + b4.z, __uint_as_float(v[4 * c + 3]) + b4.w);
              }
            }
          }
        }
      } else if (fast32) {
        // fp32 output (LSTM input projection): smem bias, 8 x 16-byte stores per 32-column chunk
        mbar_wait(bar0 + 8 * (2 * S + acc), aph);
        tc_fence_after();
#pragma unroll
        for (int mb = 0; mb < MB; ++mb) {
#pragma unroll 1
          for (int j = half; j < kJ; j += 2) {
            uint32_t v[32];
            tmem_ld32(t_row + mb * BN + j * 32, v);
            tmem_ld_wait();
            const int n0 = n_base + j * 32;
            if (m[mb] >= 0 && n0 < g.N) {
              const float4* bp = reinterpret_cast<const float4*>(bias_s + n0);
              float* crow = reinterpret_cast<float*>(ep.C) + c_off + m[mb] * ep.ldc + n0;
              const bool wide32 = (reinterpret_cast<uintptr_t>(crow) & 31) == 0;  // 256-bit stores when aligned
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                const float4 ba = bp[2 * c], bb = bp[2 * c + 1];
                float o[8] = {__uint_as_float(v[8 * c + 0]) + ba.x, __uint_as_float(v[8 * c + 1]) + ba.y,
                              __uint_as_float(v[8 * c + 2]) + ba.z, __uint_as_float(v[8 * c + 3]) + ba.w,
                              __uint_as_float(v[8 * c + 4]) + bb.x, __uint_as_float(v[8 * c + 5]) + bb.y,
                              __uint_as_float(v[8 * c + 6]) + bb.z, __uint_as_float(v[8 * c + 7]) + bb.w};
                if (ep.relu) {
#pragma unroll
                  for (int e = 0; e < 8; ++e) o[e] = fmaxf(o[e], 0.f);
                }
                if (wide32) {
                  u32x8 w;
#pragma unroll
                  for (int e = 0; e < 8; ++e) w.v[e] = __float_as_uint(o[e]);
                  st_global_256(crow + 8 * c, w);
                } else {
                  reinterpret_cast<float4*>(crow + 8 * c)[0] = make_float4(o[0], o[1], o[2], o[3]);
                  reinterpret_cast<float4*>(crow + 8 * c)[1] = make_float4(o[4], o[5], o[6], o[7]);
                }
              }
            }
          }
        }
      } else {
        mbar_wait(bar0 + 8 * (2 * S + acc), aph);
        tc_fence_after();
#pragma unroll
        for (int mb = 0; mb < MB; ++mb) {
#pragma unroll 1
          for (int j = half; j < kJ; j += 2) {
            uint32_t v[32];
            tmem_ld32(t_row + mb * BN + j * 32, v);
            tmem_ld_wait();
            const int n0 = n_base + j * 32;
            if (m[mb] >= 0 && n0 < g.N) {
              EpiParams e2 = ep;
              if (epi_mode == EPI_F32) e2.C = reinterpret_cast<float*>(ep.C) + c_off;
              epilogue_chunk(e2, epi_mode, v, m[mb], n0, g.N);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CG == 2) pair_arrive(bar0_leader + 8 * (2 * S + 2 + acc));  // the leader's MMAs overwrite both CTAs' TMEM
        else mbar_arrive(bar0 + 8 * (2 * S + 2 + acc));
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (CG == 2) pair_sync();  // no CTA exits (or frees TMEM) while the peer may still signal it or read its operands
  if (warp == 1) {
    __syncwarp();
    if (CG == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "r"(kTmemCols) : "memory");
    else tmem_dealloc(tmem_acc, kTmemCols);
  }
}

// host side (gemm_tma.cu)
bool tma_available();
// Optional K-concatenated second operand: `in2` NHWC [n][H2][W2][Cin2] convolved 1x1 / stride2 / pad 0 (same output
// grid required); the weight rows are then [R*S*Cin | Cin2] wide.
struct SecondOperand {
  const __nv_bfloat16* in2 = nullptr;
  int H2 = 0, W2 = 0, Cin2 = 0, stride2 = 1;
};
int launch_tma_conv(const __nv_bfloat16* in, const __nv_bfloat16* w, const EpiParams& ep, int64_t n, int H, int W,
                    int Cin, int Cout, int R, int S, int stride, int pad, int bn_hint, cudaStream_t st, int cat = 0,
                    double flops_override = 0.0, const SecondOperand* second = nullptr);
int launch_tma_gemm(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* Wt, int64_t ldw, int64_t M, int N, int K,
                    const EpiParams& ep, int epi_mode, int bn_hint, cudaStream_t st, int ksplit = 1,
                    int64_t split_stride = 0);
// xT[t][u][b][4] (fp32, b < Bp = B rounded up to 128) = X[b][t][:] * Wt[4u+g][:]^T + bias[4u+g] for an operand X laid out
// [B][T][lda]: the LSTM input projection in the layout the persistent recurrences read (N = 4H, N % 32 == 0)
// X points at time step 0 of the chunk, T = steps in the chunk, T_stride = steps between consecutive batch items of X
int launch_tma_gemm_xt(const __nv_bfloat16* X, int64_t lda, const __nv_bfloat16* Wt, int64_t ldw, int64_t B, int64_t T,
                       int64_t T_stride, int N, int K, const float* bias, float* xT, cudaStream_t st, int grid_cap = 0);
// Same time-major traversal of a [B][T][lda] operand chunk, fp32 output in the operand's own row order:
// C[(b * T_stride + t) * ldc + n] = sum_k X[b][t][k] * Wt[n][k]   (the input gradient of an LSTM layer for a chunk of steps)
int launch_tma_gemm_tm(const __nv_bfloat16* X, int64_t lda, const __nv_bfloat16* Wt, int64_t ldw, int64_t B, int64_t T,
                       int64_t T_stride, int N, int K, float* C, int64_t ldc, cudaStream_t st, int grid_cap = 0);

}  // namespace tc
}  // namespace avvad
