// "Slab" convolution for 3x3 / stride 1 / pad 1 layers on sm_100a: the input of a tile is loaded ONCE, with its
// halo, as one TMA box per 64-channel block ({64, OW+2, hb+2, F}; the zero border comes from TMA out-of-bounds
// fill), and the nine filter taps are nine row-shifted views of that resident slab: the UMMA A descriptor of tap
// (r,s) simply starts (r*(OW+2)+s) rows further down.  GEMM rows are positions of the padded grid, so a few rows
// per image row (the two border columns) and per band (the two border rows) are computed and dropped -- in exchange
// the A operand crosses L2 once instead of nine times and one weight K-block feeds `mb` accumulator blocks.
// The weights stay resident in shared memory (64 -> 64 channels: 9 x [64][64] bf16 = 72 KB, loaded once per CTA).
//
//   warp 0  : TMA producer (the one-off weight load, then the slabs)
//   warp 1  : TMEM alloc + tcgen05.mma issue (mb accumulator blocks x 9 taps x cpb channel blocks x 4 K16 steps)
//   warps 2-9: two epilogue groups (TMEM -> bias / residual / ReLU -> NHWC bf16), accumulators double-buffered
#pragma once
#include "gemm_tma.cuh"

namespace avvad {
namespace tc {

constexpr int kSlabThreads = 320;
constexpr int kSlabEpiWarps = 8;

struct SlabGeom {
  int64_t n_frames, total_tiles;
  int OH, OW, Wp, Hs, hb, F, nb, mb, cpb, n_tiles, N;
  int slab_rows;        // rows allocated per slab buffer (>= mb*128 + 2*Wp + 2)
  uint32_t slab_tx;     // bytes one slab TMA box delivers
};

struct SlabMaps {
  CUtensorMap a;
  CUtensorMap b;
};

// dynamic smem: [slab 0][slab 1][weights: KB resident tiles][barriers, TMEM slot, bias]
// MBC > 0: the number of accumulator blocks per tile is a compile-time constant (3 for the 17x17 maps of layer1), so the
// 9 x MBC x 4 MMAs of a channel block are straight-line code with immediate descriptor offsets -- the issuing thread
// was spending ~45 % of its slots on short-scoreboard stalls (constant-bank reloads, loop arithmetic) between
// 48-cycle MMAs.  MBC = 0 keeps the generic loops.
template <int BN, int MBC = 0>
__global__ void __launch_bounds__(kSlabThreads)
tc_slab_kernel(const __grid_constant__ SlabMaps maps, const SlabGeom g, const EpiParams ep) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw);
  const uint32_t slab_bytes = ((uint32_t)g.slab_rows * 128u + 1023u) & ~1023u;
  const uint32_t b_tile = BN * 128u;
  const int KB = 9 * g.cpb;
  const uint32_t w_base = base + 2 * slab_bytes;
  const uint32_t bar0 = w_base + (uint32_t)KB * b_tile;
  // barriers: slab_full[2] | slab_empty[2] | tfull[2] | tempty[2] | b_full, in 192 reserved bytes; then the TMEM slot
  // and, 16-byte aligned, the bias
  auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  const int kBarBFull = 8;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + (bar0 - base) + 8 * 24);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t acc_cols = (uint32_t)g.mb * BN;  // columns of one accumulator stage
  uint32_t tmem_cols = 32;
  while (tmem_cols < 2 * acc_cols) tmem_cols <<= 1;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(BAR(0 + i), 1);              // slab full (expect_tx)
      mbar_init(BAR(2 + i), 1);              // slab empty (tcgen05.commit)
      mbar_init(BAR(4 + i), 1);              // tmem full
      mbar_init(BAR(6 + i), kSlabEpiWarps);  // tmem empty
    }
    mbar_init(BAR(kBarBFull), 1);
    fence_barrier_init();
    tma_prefetch_desc(&maps.a);
    tma_prefetch_desc(&maps.b);
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), tmem_cols);
    tmem_relinquish();
  }
  {  // folded-BN bias -> shared memory (zero when absent); the region sits behind the barriers
    float* bs = reinterpret_cast<float*>(smem + (bar0 - base) + 8 * 24 + 16);
    for (int i = threadIdx.x; i < g.N; i += kSlabThreads) bs[i] = ep.bias ? ep.bias[i] : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_acc = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer (warp-converged; one elected lane issues) =================
    // all weight K blocks, once (n_tiles == 1)
    if (elect_one_sync()) {
      mbar_arrive_expect_tx(BAR(kBarBFull), (uint32_t)KB * b_tile);
      for (int kb = 0; kb < KB; ++kb) tma_load_2d(w_base + kb * b_tile, &maps.b, kb * BK, 0, BAR(kBarBFull));
    }
    __syncwarp();
    uint32_t si = 0;  // slab counter
    for (int64_t tile = blockIdx.x; tile < g.total_tiles; tile += gridDim.x) {
      const int64_t mt = tile / g.n_tiles;
      const int band = (int)(mt % g.nb);
      const int n0 = (int)((mt / g.nb) * g.F);
      const int hstart = band * g.hb;
      for (int cb = 0; cb < g.cpb; ++cb, ++si) {
        const int sb = si & 1;
        mbar_wait(BAR(2 + sb), ((si >> 1) & 1u) ^ 1u);
        if (elect_one_sync()) {
          mbar_arrive_expect_tx(BAR(0 + sb), g.slab_tx);
          tma_load_4d(base + sb * slab_bytes, &maps.a, cb * BK, -1, hstart - 1, n0, BAR(0 + sb));
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (warp-converged; one elected lane issues MMAs and commits) =================
    constexpr uint32_t idesc = make_idesc(BN);
    uint32_t si = 0, tl = 0;
    mbar_wait(BAR(kBarBFull), 0);
    tc_fence_after();
    for (int64_t tile = blockIdx.x; tile < g.total_tiles; tile += gridDim.x, ++tl) {
      const uint32_t acc = tl & 1u, aph = (tl >> 1) & 1u;
      mbar_wait(BAR(6 + acc), aph ^ 1u);
      tc_fence_after();
      for (int cb = 0; cb < g.cpb; ++cb, ++si) {
        const int sb = si & 1;
        mbar_wait(BAR(0 + sb), (si >> 1) & 1u);
        tc_fence_after();
        const uint32_t slab_lo = desc_lo(base + sb * slab_bytes);
        // every tap of this channel block in one elected region: 9 x mb x 4 MMAs issued back to back
        if (elect_one_sync()) {
          const int Wp = g.Wp, cpb = g.cpb;
          const uint32_t d0 = tmem_acc + acc * acc_cols;
          if (MBC > 0) {
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
              const uint32_t w_lo = desc_lo(w_base + (uint32_t)(tap * cpb + cb) * b_tile);
              const int fr = tap / 3, fs = tap - fr * 3;
              // descriptor low words count 16-byte units: one slab row = 8, one accumulator block (128 rows) = 1024
              const uint32_t a0 = slab_lo + (uint32_t)(fr * Wp + fs) * 8u;
              const uint32_t first = (cb | tap) != 0;
#pragma unroll
              for (int m = 0; m < MBC; ++m) {
                umma_f16_lo(d0 + m * BN, a0 + m * 1024u, w_lo, idesc, first);
                umma_f16_lo(d0 + m * BN, a0 + m * 1024u + 2, w_lo + 2, idesc, 1);
                umma_f16_lo(d0 + m * BN, a0 + m * 1024u + 4, w_lo + 4, idesc, 1);
                umma_f16_lo(d0 + m * BN, a0 + m * 1024u + 6, w_lo + 6, idesc, 1);
              }
            }
          } else {
            const int mb = g.mb;
#pragma unroll 1
            for (int tap = 0; tap < 9; ++tap) {
              const uint32_t w_lo = desc_lo(w_base + (uint32_t)(tap * cpb + cb) * b_tile);
              const int fr = tap / 3, fs = tap - fr * 3;
              uint32_t a_lo = slab_lo + (uint32_t)(fr * Wp + fs) * 8u;
              uint32_t d_tmem = d0;
              const uint32_t first = (cb | tap) != 0;
              for (int m = 0; m < mb; ++m, a_lo += 1024u, d_tmem += BN) {
                umma_f16_lo(d_tmem, a_lo, w_lo, idesc, first);
                umma_f16_lo(d_tmem, a_lo + 2, w_lo + 2, idesc, 1);
                umma_f16_lo(d_tmem, a_lo + 4, w_lo + 4, idesc, 1);
                umma_f16_lo(d_tmem, a_lo + 6, w_lo + 6, idesc, 1);
              }
            }
          }
          umma_commit(BAR(2 + sb));
          if (cb == g.cpb - 1) umma_commit(BAR(4 + acc));
        }
        __syncwarp();
      }
    }
  } else {
    // ================= epilogue: warps 2..9 =================
    // A tile has mb * (BN/32) units of 128 rows x 32 columns; unit u = (m, j) is handled by the four warps of
    // group (u & 1) (one TMEM lane quarter each).  The position -> (frame, y, x) mapping of a thread's rows is the
    // same for every tile, so it is computed once; per tile only the frame / band base is added.  The residual of
    // every unit a thread owns is requested BEFORE the wait on the accumulator (and pinned behind it), so its latency
    // hides behind the tile's MMAs; the folded-BN bias sits in smem; ReLU is fused into the bf16 pack.
    const int q = warp & 3;
    const int grp = (warp - 2) >> 2;  // 0 or 1
    uint32_t tl = 0;
    const int per_frame = g.Hs * g.Wp;
    constexpr int kJ = BN / 32;
    constexpr int kMaxUnits = 4;  // per warp and tile (mb * kJ <= 8)
    const float* bias_s = reinterpret_cast<const float*>(smem + (bar0 - base) + 8 * 24 + 16);
    const int units = g.mb * kJ;
    // tile-invariant part: local output offset (elements) and the (frame, row) of each owned unit row; -1 = padding
    int loc[kMaxUnits], lf[kMaxUnits], ly[kMaxUnits], ncol[kMaxUnits];
#pragma unroll
    for (int i = 0; i < kMaxUnits; ++i) {
      const int u = grp + 2 * i;
      loc[i] = -1; lf[i] = 0; ly[i] = 0; ncol[i] = 0;
      if (u < units) {
        const int m = u / kJ, j = u - m * kJ;
        const int p = m * 128 + q * 32 + lane;  // position in the padded grid of the slab
        const int f = p / per_frame;
        const int rem = p - f * per_frame;
        const int y = rem / g.Wp;
        const int x = rem - y * g.Wp;
        ncol[i] = j * 32;
        if (f < g.F && y < g.hb && x < g.OW) {
          loc[i] = ((f * g.OH + y) * g.OW + x) * (int)ep.ldc + j * 32;
          lf[i] = f;
          ly[i] = y;
        }
      }
    }
    const __nv_bfloat16* resp = ep.residual;
    __nv_bfloat16* outp = reinterpret_cast<__nv_bfloat16*>(ep.C);
    const bool relu = ep.relu != 0;
    for (int64_t tile = blockIdx.x; tile < g.total_tiles; tile += gridDim.x, ++tl) {
      const int n_base = (int)(tile % g.n_tiles) * BN;
      const int64_t mt = tile / g.n_tiles;
      const int band = (int)(mt % g.nb);
      const int64_t n0 = (mt / g.nb) * g.F;
      const int hstart = band * g.hb;
      const uint32_t acc = tl & 1u, aph = (tl >> 1) & 1u;
      const int64_t tile_off = ((n0 * g.OH + hstart) * g.OW) * ep.ldc + n_base;
      bool ok[kMaxUnits];
      u32x8 rb[kMaxUnits][2] = {};  // activations are 128-byte rows at 1 KB aligned bases: 256-bit accesses are legal
#pragma unroll
      for (int i = 0; i < kMaxUnits; ++i) {
        ok[i] = loc[i] >= 0 && n0 + lf[i] < g.n_frames && hstart + ly[i] < g.OH;
        if (ok[i] && resp) {
          rb[i][0] = ld_global_256(resp + tile_off + loc[i]);
          rb[i][1] = ld_global_256(resp + tile_off + loc[i] + 16);
        }
      }
      mbar_wait(BAR(4 + acc), aph);
      tc_fence_after();
      // pin the prefetched residual registers behind the wait: without this the compiler hoists the bf16 unpack
      // right behind the loads and every unit's load latency is paid synchronously before the wait
#pragma unroll
      for (int i = 0; i < kMaxUnits; ++i)
#pragma unroll
        for (int c = 0; c < 2; ++c)
#pragma unroll
          for (int e = 0; e < 8; ++e) asm volatile("" : "+r"(rb[i][c].v[e]));
#pragma unroll
      for (int i = 0; i < kMaxUnits; ++i) {
        const int u = grp + 2 * i;
        if (u < units) {  // warp-uniform
          const int m = u / kJ;
          uint32_t v[32];
          tmem_ld32(tmem_acc + acc * acc_cols + (uint32_t)m * BN + (uint32_t)ncol[i] + ((uint32_t)(q * 32) << 16), v);
          tmem_ld_wait();
          if (ok[i]) {
            const int nc = n_base + ncol[i];
            float f32[32];
            const float4* bp = reinterpret_cast<const float4*>(bias_s + nc);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const float4 b4 = bp[c];
              f32[4 * c + 0] = __uint_as_float(v[4 * c + 0]) + b4.x;
              f32[4 * c + 1] = __uint_as_float(v[4 * c + 1]) + b4.y;
              f32[4 * c + 2] = __uint_as_float(v[4 * c + 2]) + b4.z;
              f32[4 * c + 3] = __uint_as_float(v[4 * c + 3]) + b4.w;
            }
            if (resp) {
#pragma unroll
              for (int e = 0; e < 16; ++e) {  // bf16 -> f32 is a 16-bit shift / mask
                const uint32_t w = rb[i][e >> 3].v[e & 7];
                f32[2 * e + 0] += __uint_as_float(w << 16);
                f32[2 * e + 1] += __uint_as_float(w & 0xFFFF0000u);
              }
            }
            __nv_bfloat16* cp = outp + tile_off + loc[i];
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              u32x8 o;
#pragma unroll
              for (int e = 0; e < 8; ++e)
                o.v[e] = relu ? pack_relu_bf16x2(f32[16 * c + 2 * e], f32[16 * c + 2 * e + 1])
                              : pack_bf16x2(f32[16 * c + 2 * e], f32[16 * c + 2 * e + 1]);
              st_global_256(cp + 16 * c, o);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(BAR(6 + acc));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_acc, tmem_cols);
  }
}

int launch_slab_conv(const __nv_bfloat16* in, const __nv_bfloat16* w, const EpiParams& ep, int64_t n, int H, int Cin,
                     int Cout, cudaStream_t st);
bool slab_supported(int H, int W, int Cin, int Cout, int R, int S, int stride, int pad);

}  // namespace tc
}  // namespace avvad
