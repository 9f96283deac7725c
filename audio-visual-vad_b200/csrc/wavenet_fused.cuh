// Fused WaveNet encoder stack (SURVEY §8a row W1, BASELINE.json north_star §2): the causal layer, EVERY dilated
// residual layer and the bottleneck in ONE kernel -- the receptive-field history of a time tile stays in shared memory
// across all dilation levels, the dilated taps are row-shifted tcgen05 descriptors on that resident history, and the
// ReLU / 1x1 dense projection / residual add are the epilogues of the two MMAs of a layer.  HBM sees the input waveform
// features once and the bottleneck activations once; the per-layer variant in wavenet.cu writes an im2col copy and
// three activation tensors per layer instead.
//
// Reference semantics: packages/models/wavenet_autoencoder.py:74-93
//   s = causal(x);  for d: s = dense(relu(dilated_d(relu(s)))) + s[..., -L_out:];  relu(bottleneck(s)) -> avg-pool
// Valid (un-padded) convolutions: an output at position t of a layer reads its input at t, t+d, .., t+(k-1)d and the
// residual at t+(k-1)d, so with the row index kept fixed through the stack a tile of `lt` final outputs starting at o0
// needs the causal output rows [o0, o0 + lt + sum_i (k-1)d_i) and nothing else: tiles are independent (halo recompute).
//
// Shapes: every channel count padded to 64 (one 128-byte SWIZZLE_128B row per time step); requires q, R, D, bottleneck
// <= 64 and sum (k-1)d <= 128 -- otherwise avvad_wavenet_encode keeps the per-layer path.
//
// Shared memory (one CTA = one (batch item, time tile), 256 threads):
//   S      fp32 [256][68]   residual stream (pitch 68 floats: conflict-free float4 rows), updated in place
//   A      bf16 [384][64]   SW128 operand: relu(S) (or the input features for the causal layer, S for the bottleneck)
//   A2     bf16 [128][64]   SW128 operand of the dense 1x1 GEMM: relu(dilated conv) of the current 128-row block
//   W      bf16 2 x (k+1) x [64][64]   weight tiles of the current / next layer (TMA, double buffered)
// TMEM: 128 columns (two 128x64 fp32 accumulators).
#pragma once
#include "gemm_tma.cuh"

namespace avvad {
namespace tc {

constexpr int kWnThreads = 256;
constexpr int kWnRows = 384;        // history rows held per tile (256 working rows + 128 rows of tap slack)
constexpr int kWnWork = 256;        // working rows: lt + sum shifts + (k-1) <= 256
constexpr int kWnSPitch = 68;       // floats
constexpr int kWnMaxLayers = 32;
constexpr int kWnMaxK = 4;

struct WnFusedGeom {
  int B, q, N;               // input (B, q, N) fp32 channel-major
  int k, n_layers;
  int dil[kWnMaxLayers];
  int lt;                    // final outputs per tile
  int tiles_per_item;
  int L_final;               // final sequence length
  int sum_shift;             // sum_i (k-1) d_i
  const float* x;
  const float* bias;         // [1 + 2*n_layers + 1][64]: causal, (dilated_i, dense_i)..., bottleneck
  float* out;                // [B][L_final][64] fp32: relu(bottleneck), time-major
  // training forward (kTape): S_i for i = 0..n_layers, [B][L_i][64] each, back to back; act_i for i < n_layers,
  // [B][L_{i+1}][64] each, back to back (see avvad_wavenet_tape_bytes)
  __nv_bfloat16* tape_s;
  __nv_bfloat16* tape_act;
};

__device__ __forceinline__ uint32_t wn_sw128_off(int row, int chunk16) {
  return (uint32_t)row * 128u + (uint32_t)((chunk16 ^ (row & 7)) << 4);
}

// kTape: also store the tile's OWNED rows of every layer input S_i (bf16, before the ReLU) and of every act_i =
// relu(dilated_i + bias) (bf16: the dense GEMM's operand) -- rows [o0, o0 + lt) of a non-last tile, [o0, L_i) of the
// last tile of an item, so every row is written exactly once.  The arithmetic is the same in both instantiations.
template <bool kTape>
__global__ void __launch_bounds__(kWnThreads)
wavenet_fused_kernel(const __grid_constant__ CUtensorMap wmap, const WnFusedGeom g) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw);
  // layout
  const uint32_t offA = 0;                                   // 384 * 128 = 49152
  const uint32_t offA2 = offA + kWnRows * 128u;              // 16384
  const uint32_t offW = offA2 + 128u * 128u;                 // 2 * (k+1) * 8192
  const uint32_t wbuf_bytes = (uint32_t)(g.k + 1) * 8192u;
  const uint32_t offS = offW + 2u * wbuf_bytes;              // 256 * 68 * 4 = 69632 (S[r + shift] stays below 256)
  const uint32_t offBar = offS + kWnWork * kWnSPitch * 4u;
  float* S = reinterpret_cast<float*>(smem + offS);
  uint8_t* A = smem + offA;
  uint8_t* A2 = smem + offA2;
  auto BAR = [&](int i) { return base + offBar + 8u * (uint32_t)i; };   // 0,1: weights full; 2: mma1 done; 3: mma2 done
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + offBar + 64);
  float* bias_s = reinterpret_cast<float*>(smem + offBar + 128);        // [2][64] of the current layer

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x / g.tiles_per_item, tile = blockIdx.x % g.tiles_per_item;
  const int o0 = tile * g.lt;
  const int n_out = min(g.lt, g.L_final - o0);         // valid final outputs of this tile
  const int rows0 = n_out + g.sum_shift;               // causal-layer output rows needed
  const int rows_x = rows0 + (g.k - 1);                // input rows needed

  if (threadIdx.x == 0) {
    mbar_init(BAR(0), 1);
    mbar_init(BAR(1), 1);
    mbar_init(BAR(2), 1);
    mbar_init(BAR(3), 1);
    fence_barrier_init();
    tma_prefetch_desc(&wmap);
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), 128);
    tmem_relinquish();
  }
  // weight tiles of a "layer slot": slot 0 = causal (k tiles), slot 1+i = layer i (k dilated taps + dense), last = bottleneck
  auto slot_first_tile = [&](int slot) { return slot == 0 ? 0 : g.k + (slot - 1) * (g.k + 1); };
  auto slot_tiles = [&](int slot) { return slot == 0 ? g.k : (slot == g.n_layers + 1 ? 1 : g.k + 1); };
  auto load_weights = [&](int slot) {   // one thread
    const int buf = slot & 1, nt = slot_tiles(slot), t0 = slot_first_tile(slot);
    mbar_arrive_expect_tx(BAR(buf), (uint32_t)nt * 8192u);
    for (int t = 0; t < nt; ++t) tma_load_2d(base + offW + buf * wbuf_bytes + t * 8192u, &wmap, 0, (t0 + t) * 64, BAR(buf));
  };
  // input features -> A (bf16, SW128): A[r][c] = x[item][c][o0 + r]; zero rows beyond rows_x and channels beyond q
  for (int idx = threadIdx.x; idx < kWnRows * 8; idx += kWnThreads) {
    const int r = idx % kWnRows, ch = idx / kWnRows;   // lanes walk rows: coalesced global reads per channel
    uint32_t pk[4] = {0u, 0u, 0u, 0u};
    if (r < rows_x) {
      float v[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int c = ch * 8 + e;
        v[e] = (c < g.q) ? g.x[((int64_t)item * g.q + c) * g.N + o0 + r] : 0.f;
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) pk[e] = pack_bf16x2(v[2 * e], v[2 * e + 1]);
    }
    *reinterpret_cast<uint4*>(A + wn_sw128_off(r, ch)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
  }
  if (threadIdx.x == 0) load_weights(0);
  tc_fence_before();
  fence_proxy_async();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_acc = *tmem_slot;
  constexpr uint32_t idesc = make_idesc(64);
  uint32_t wphase[2] = {0u, 0u}, p1 = 0u, p2 = 0u;

  // epilogue geometry: warp w reads TMEM lanes 32*(w&3) .. +31 (row = lane), columns 32*(w>>2) .. +31
  const int q4 = warp & 3, half = warp >> 2;
  const int erow = q4 * 32 + lane;

  int rows_in = rows0 + (g.k - 1);  // rows of the CURRENT layer's input (for the causal layer: rows_x)
  const bool last_tile = tile == g.tiles_per_item - 1;
  int L_in = g.L_final + g.sum_shift;   // kTape: global length of the current layer's input (S_0 for slot 1)
  __nv_bfloat16* tape_s = g.tape_s;     // kTape: S_{slot-1} of this item
  __nv_bfloat16* tape_a = g.tape_act;   // kTape: act_{slot-1} of this item
  for (int slot = 0; slot <= g.n_layers + 1; ++slot) {
    const bool causal = slot == 0, bott = slot == g.n_layers + 1;
    const int d = (causal || bott) ? 1 : g.dil[slot - 1];
    const int taps = bott ? 1 : g.k;
    const int shift = bott ? 0 : (g.k - 1) * d;
    const int rows_out = rows_in - shift;
    const int buf = slot & 1;
    // prefetch the next layer's weights into the other buffer (its previous user finished one layer ago)
    if (threadIdx.x == 0 && slot + 1 <= g.n_layers + 1) load_weights(slot + 1);
    // this layer's biases -> shared memory
    if (threadIdx.x < 128) {
      const int which = threadIdx.x >> 6, c = threadIdx.x & 63;
      const int vec = causal ? 0 : (bott ? 1 + 2 * g.n_layers : 1 + 2 * (slot - 1) + which);
      bias_s[threadIdx.x] = (which == 0 || (!causal && !bott)) ? g.bias[vec * 64 + c] : 0.f;
    }
    if (!causal) {
      // A = bf16(relu(S)) (bottleneck: no ReLU), all rows of the layer input
      for (int idx = threadIdx.x; idx < rows_in * 8; idx += kWnThreads) {
        const int r = idx >> 3, ch = idx & 7;
        const float4 a = *reinterpret_cast<const float4*>(S + r * kWnSPitch + ch * 8);
        const float4 b = *reinterpret_cast<const float4*>(S + r * kWnSPitch + ch * 8 + 4);
        uint4 o;
        if (bott) {
          o.x = pack_bf16x2(a.x, a.y); o.y = pack_bf16x2(a.z, a.w); o.z = pack_bf16x2(b.x, b.y); o.w = pack_bf16x2(b.z, b.w);
        } else {
          o.x = pack_relu_bf16x2(a.x, a.y); o.y = pack_relu_bf16x2(a.z, a.w);
          o.z = pack_relu_bf16x2(b.x, b.y); o.w = pack_relu_bf16x2(b.z, b.w);
        }
        *reinterpret_cast<uint4*>(A + wn_sw128_off(r, ch)) = o;
        if constexpr (kTape) {
          if (r < (last_tile ? rows_in : g.lt))
            *reinterpret_cast<uint4*>(tape_s + ((int64_t)item * L_in + o0 + r) * 64 + ch * 8) =
                make_uint4(pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w), pack_bf16x2(b.x, b.y), pack_bf16x2(b.z, b.w));
        }
      }
    }
    fence_proxy_async();
    __syncthreads();
    mbar_wait(BAR(buf), wphase[buf]);
    wphase[buf] ^= 1u;
    const uint32_t wbase = base + offW + buf * wbuf_bytes;

    const int n_blocks = (rows_out + 127) / 128;
    for (int mb = 0; mb < n_blocks; ++mb) {
      const int m0 = mb * 128;
      // ---- MMA 1: taps = row-shifted views of the resident history ----
      if (warp == 1) {
        tc_fence_after();
        if (elect_one_sync()) {
          for (int j = 0; j < taps; ++j) {
            const uint32_t a_lo = desc_lo(base + offA + (uint32_t)(m0 + j * d) * 128u);
            const uint32_t b_lo = desc_lo(wbase + (uint32_t)j * 8192u);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) umma_f16_lo(tmem_acc, a_lo + 2 * kk, b_lo + 2 * kk, idesc, (j | kk) != 0);
          }
          umma_commit(BAR(2));
        }
        __syncwarp();
      }
      mbar_wait(BAR(2), p1);
      p1 ^= 1u;
      tc_fence_after();
      uint32_t v[32];
      tmem_ld32(tmem_acc + (uint32_t)(half * 32) + ((uint32_t)(q4 * 32) << 16), v);
      tmem_ld_wait();
      const int r = m0 + erow;
      if (causal || bott) {
        // causal: S[r] = acc + bias;  bottleneck: out[o0 + r] = relu(acc + bias)
        if (r < rows_out) {
          float f[32];
#pragma unroll
          for (int e = 0; e < 32; ++e) f[e] = __uint_as_float(v[e]) + bias_s[half * 32 + e];
          if (causal) {
            float4* dst = reinterpret_cast<float4*>(S + r * kWnSPitch + half * 32);
#pragma unroll
            for (int e = 0; e < 8; ++e) dst[e] = make_float4(f[4 * e], f[4 * e + 1], f[4 * e + 2], f[4 * e + 3]);
          } else if (r < n_out) {
            float4* dst = reinterpret_cast<float4*>(g.out + ((int64_t)item * g.L_final + o0 + r) * 64 + half * 32);
#pragma unroll
            for (int e = 0; e < 8; ++e)
              dst[e] = make_float4(fmaxf(f[4 * e], 0.f), fmaxf(f[4 * e + 1], 0.f), fmaxf(f[4 * e + 2], 0.f),
                                   fmaxf(f[4 * e + 3], 0.f));
          }
        }
        tc_fence_before();
        __syncthreads();   // accumulator drained (and S rows written) before the next block's MMA / next layer's pass
        continue;
      }
      // ---- epilogue 1: relu(dilated conv + bias) -> A2 (bf16, SW128), the operand of the dense 1x1 GEMM ----
      {
        uint32_t pk[16];
#pragma unroll
        for (int e = 0; e < 16; ++e)
          pk[e] = pack_relu_bf16x2(__uint_as_float(v[2 * e]) + bias_s[half * 32 + 2 * e],
                                   __uint_as_float(v[2 * e + 1]) + bias_s[half * 32 + 2 * e + 1]);
#pragma unroll
        for (int cq = 0; cq < 4; ++cq)
          *reinterpret_cast<uint4*>(A2 + wn_sw128_off(erow, half * 4 + cq)) =
              make_uint4(pk[4 * cq], pk[4 * cq + 1], pk[4 * cq + 2], pk[4 * cq + 3]);
        if constexpr (kTape) {
          if (r < (last_tile ? rows_out : g.lt)) {
            uint4* dst = reinterpret_cast<uint4*>(tape_a + ((int64_t)item * (L_in - shift) + o0 + r) * 64 + half * 32);
#pragma unroll
            for (int cq = 0; cq < 4; ++cq) dst[cq] = make_uint4(pk[4 * cq], pk[4 * cq + 1], pk[4 * cq + 2], pk[4 * cq + 3]);
          }
        }
      }
      tc_fence_before();
      fence_proxy_async();
      __syncthreads();
      // ---- MMA 2: dense 1x1 (D -> R) ----
      if (warp == 1) {
        tc_fence_after();
        if (elect_one_sync()) {
          const uint32_t a_lo = desc_lo(base + offA2);
          const uint32_t b_lo = desc_lo(wbase + (uint32_t)g.k * 8192u);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) umma_f16_lo(tmem_acc + 64u, a_lo + 2 * kk, b_lo + 2 * kk, idesc, kk != 0);
          umma_commit(BAR(3));
        }
        __syncwarp();
      }
      mbar_wait(BAR(3), p2);
      p2 ^= 1u;
      tc_fence_after();
      tmem_ld32(tmem_acc + 64u + (uint32_t)(half * 32) + ((uint32_t)(q4 * 32) << 16), v);
      tmem_ld_wait();
      // ---- epilogue 2: + bias + residual S[r + shift]; in place (all reads of the block happen before its writes) ----
      float f[32];
      if (r < rows_out) {
        const float4* res = reinterpret_cast<const float4*>(S + (r + shift) * kWnSPitch + half * 32);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float4 rr = res[e];
          f[4 * e] = __uint_as_float(v[4 * e]) + bias_s[64 + half * 32 + 4 * e] + rr.x;
          f[4 * e + 1] = __uint_as_float(v[4 * e + 1]) + bias_s[64 + half * 32 + 4 * e + 1] + rr.y;
          f[4 * e + 2] = __uint_as_float(v[4 * e + 2]) + bias_s[64 + half * 32 + 4 * e + 2] + rr.z;
          f[4 * e + 3] = __uint_as_float(v[4 * e + 3]) + bias_s[64 + half * 32 + 4 * e + 3] + rr.w;
        }
      }
      tc_fence_before();
      __syncthreads();
      if (r < rows_out) {
        float4* dst = reinterpret_cast<float4*>(S + r * kWnSPitch + half * 32);
#pragma unroll
        for (int e = 0; e < 8; ++e) dst[e] = make_float4(f[4 * e], f[4 * e + 1], f[4 * e + 2], f[4 * e + 3]);
      }
      __syncthreads();
    }
    rows_in = rows_out;
    if constexpr (kTape) {
      if (!causal) {
        tape_s += (int64_t)g.B * L_in * 64;
        tape_a += (int64_t)g.B * (L_in - shift) * 64;
        L_in -= shift;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_acc, 128);
  }
}

static inline size_t wavenet_fused_smem_bytes(int k) {
  return 1024 + (size_t)kWnRows * 128 + 128 * 128 + 2 * (size_t)(k + 1) * 8192 + (size_t)kWnWork * kWnSPitch * 4 + 128 + 512;
}

}  // namespace tc
}  // namespace avvad
