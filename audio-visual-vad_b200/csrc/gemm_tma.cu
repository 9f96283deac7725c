// Host side of the TMA-fed tcgen05 engine: tensor-map encoding (driver entry point fetched at run time, libcuda
// is not linked), tile-phase selection and launch.
#include <cudaTypedefs.h>
#include <stdlib.h>

#include <mutex>

#include "gemm_tma.cuh"

namespace avvad {
namespace tc {

int prof_begin(cudaStream_t st, void** tok);
void prof_end(cudaStream_t st, void* tok, int cat, double flops);

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}

bool tma_available() { return encode_fn() != nullptr; }

// rank-4 bf16 tensor, dims innermost first
static int encode4(CUtensorMap* m, const void* ptr, const uint64_t dims[4], const uint64_t strides_bytes[3],
                   const uint32_t box[4], const uint32_t estr[4], bool sw32 = false) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point unavailable");
    return AVVAD_ERR_CUDA;
  }
  cuuint64_t gd[4] = {dims[0], dims[1], dims[2], dims[3]};
  cuuint64_t gs[3] = {strides_bytes[0], strides_bytes[1], strides_bytes[2]};
  cuuint32_t bx[4] = {box[0], box[1], box[2], box[3]};
  cuuint32_t es[4] = {estr[0], estr[1], estr[2], estr[3]};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), gd, gs, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, sw32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(rank 4) failed with CUresult " + std::to_string((int)r) + " dims=" +
              std::to_string(dims[0]) + "," + std::to_string(dims[1]) + "," + std::to_string(dims[2]) + "," +
              std::to_string(dims[3]) + " box=" + std::to_string(box[0]) + "," + std::to_string(box[1]) + "," +
              std::to_string(box[2]) + "," + std::to_string(box[3]));
    return AVVAD_ERR_CUDA;
  }
  return AVVAD_OK;
}

static int encode2(CUtensorMap* m, const void* ptr, uint64_t inner, uint64_t outer, uint64_t stride_bytes,
                   uint32_t box_inner, uint32_t box_outer, bool sw32 = false) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point unavailable");
    return AVVAD_ERR_CUDA;
  }
  cuuint64_t gd[2] = {inner, outer};
  cuuint64_t gs[1] = {stride_bytes};
  cuuint32_t bx[2] = {box_inner, box_outer};
  cuuint32_t es[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gd, gs, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, sw32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(rank 2) failed with CUresult " + std::to_string((int)r));
    return AVVAD_ERR_CUDA;
  }
  return AVVAD_OK;
}

// generic rank-N (<= 5) bf16 SWIZZLE_128B map, unit traversal strides
int encode_tiled_bf16(CUtensorMap* m, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                      const uint32_t* box) {
  EncodeTiledFn fn = encode_fn();
  if (!fn || rank < 1 || rank > 5) {
    set_error("cuTensorMapEncodeTiled unavailable or bad rank");
    return AVVAD_ERR_CUDA;
  }
  cuuint64_t gd[5], gs[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gd[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i < rank - 1) gs[i] = strides_bytes[i];
  }
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(ptr), gd, gs, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(rank " + std::to_string(rank) + ") failed with CUresult " +
              std::to_string((int)r));
    return AVVAD_ERR_CUDA;
  }
  return AVVAD_OK;
}

int encode_act_map(CUtensorMap* m, const void* ptr, int Cin, int W, int H, int64_t n, const uint32_t box[4],
                   const uint32_t estr[4]) {
  const uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)n};
  const uint64_t strides[3] = {(uint64_t)Cin * 2, (uint64_t)W * Cin * 2, (uint64_t)H * W * Cin * 2};
  return encode4(m, ptr, dims, strides, box, estr);
}
int encode_weight_map(CUtensorMap* m, const void* ptr, uint64_t K, uint64_t N, uint32_t bn) {
  return encode2(m, ptr, K, N, K * 2, 64, bn);
}

// N = 256 tiles run on CTA pairs (tcgen05 cta_group::2) unless AVVAD_CG2=0; split-K launches and the per-step LSTM
// epilogue keep the one-CTA kernel.  The weight map of a pair launch has a BN/2-row box (each CTA loads its half).
static bool pair_enabled() {
  static int v = [] {
    const char* e = getenv("AVVAD_CG2");
    return (e && atoi(e) == 0) ? 0 : 1;
  }();
  return v != 0;
}
// kb = K blocks of the launch: short K loops (layer2's first convolution, K = 576) measured slower on pairs of
// two-block CTAs (307 us against 266 us per 20,288-frame pass), so N = 128 pairs need at least 16 K blocks
static bool use_pair(int bn, int ksplit, int epi_mode, int kb) {
  if (!pair_enabled() || ksplit > 1 || epi_mode == EPI_LSTM) return false;
  return bn == 256 || (bn == 128 && kb >= 16);
}

template <int BN, int KE = 64, int MB = 1, int CG = 1>
static int launch_bn(const TmaMaps& maps, TmaGeom g, const EpiParams& ep, int epi_mode, int cat, double flops,
                     cudaStream_t st) {
  using C = TmaCfg<BN, KE, MB, CG>;
  constexpr int MBT = CG * MB;
  if (g.ksplit < 1) g.ksplit = 1;
  if (g.ksplit == 1) g.kb_split = g.KB;
  g.m_supers = (g.m_tiles + MBT - 1) / MBT;
  g.total_tiles = g.m_supers * g.n_tiles * g.ksplit;
  static PerDeviceOnce once;
  const cudaError_t attr_err = once.run([] {
    return cudaFuncSetAttribute(tc_tma_kernel<BN, KE, MB, CG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)C::kSmemBytes);
  });
  if (attr_err != cudaSuccess) {
    set_error(std::string("cudaFuncSetAttribute(smem): ") + cudaGetErrorString(attr_err));
    return AVVAD_ERR_CUDA;
  }
  static int num_sms = [] {
    int dev = 0, n = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n > 0 ? n : 148;
  }();
  if (g.total_tiles <= 0) return AVVAD_OK;
  void* tok = nullptr;
  if (CG == 2) {
    int64_t pairs = num_sms / 2;
    if (g.grid_cap > 0 && g.grid_cap / 2 < pairs) pairs = g.grid_cap / 2 > 0 ? g.grid_cap / 2 : 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2u * (unsigned)(g.total_tiles < pairs ? g.total_tiles : pairs));
    cfg.blockDim = dim3(kTmaThreads);
    cfg.dynamicSmemBytes = C::kSmemBytes;
    cfg.stream = st;
    cudaLaunchAttribute la[1];
    la[0].id = cudaLaunchAttributeClusterDimension;
    la[0].val.clusterDim.x = 2; la[0].val.clusterDim.y = 1; la[0].val.clusterDim.z = 1;
    cfg.attrs = la;
    cfg.numAttrs = 1;
    prof_begin(st, &tok);
    cudaError_t le = cudaLaunchKernelEx(&cfg, tc_tma_kernel<BN, KE, MB, CG>, maps, g, ep, epi_mode);
    if (le != cudaSuccess) {
      set_error(std::string("pair launch failed: ") + cudaGetErrorString(le));
      return AVVAD_ERR_CUDA;
    }
    AVVAD_LAUNCHED();
    prof_end(st, tok, cat, flops);
    return AVVAD_OK;
  }
  int64_t resident = (int64_t)num_sms * C::kCtasPerSm;
  if (g.grid_cap > 0 && g.grid_cap < resident) resident = g.grid_cap;
  const unsigned grid = (unsigned)(g.total_tiles < resident ? g.total_tiles : resident);
  prof_begin(st, &tok);
  tc_tma_kernel<BN, KE, MB, CG><<<grid, kTmaThreads, C::kSmemBytes, st>>>(maps, g, ep, epi_mode);
  AVVAD_LAUNCHED();
  prof_end(st, tok, cat, flops);
  return AVVAD_OK;
}

static int dispatch(int bn, const TmaMaps& maps, const TmaGeom& g, const EpiParams& ep, int epi_mode, int cat,
                    double flops, cudaStream_t st) {
  switch (bn) {
    case 64: return launch_bn<64>(maps, g, ep, epi_mode, cat, flops, st);
    case 128:
      // two accumulator blocks per weight box (see TmaCfg); the per-step LSTM epilogue keeps one
      if (g.pair) return launch_bn<128, 64, 2, 2>(maps, g, ep, epi_mode, cat, flops, st);
      if (epi_mode != EPI_LSTM) return launch_bn<128, 64, 2>(maps, g, ep, epi_mode, cat, flops, st);
      return launch_bn<128>(maps, g, ep, epi_mode, cat, flops, st);
    case 256:
      if (g.pair) return launch_bn<256, 64, 1, 2>(maps, g, ep, epi_mode, cat, flops, st);
      return launch_bn<256>(maps, g, ep, epi_mode, cat, flops, st);
  }
  set_error("bad BN");
  return AVVAD_ERR_ARG;
}

static int pick_bn(int N, int hint) {
  if (hint == 64 || hint == 128 || hint == 256) {
    if (N % hint == 0 || hint == 64) return hint;
  }
  if (N <= 64) return 64;
  if (N % 256 == 0) return 256;
  if (N % 128 == 0) return 128;
  return 64;
}

int launch_tma_conv(const __nv_bfloat16* in, const __nv_bfloat16* w, const EpiParams& ep, int64_t n, int H, int W,
                    int Cin, int Cout, int R, int S, int stride, int pad, int bn_hint, cudaStream_t st, int cat,
                    double flops_override, const SecondOperand* second) {
  const int OH = (H + 2 * pad - R) / stride + 1;
  const int OW = (W + 2 * pad - S) / stride + 1;
  const int KE = (Cin % 64 == 0) ? 64 : 16;  // 16-channel inputs (packed stem) use 32-byte K blocks
  AVVAD_CHECK_ARG(OW <= 128 && Cin % KE == 0, "TMA conv: OW <= 128 and Cin % 64 == 0 (or Cin == 16) required");
  AVVAD_CHECK_ARG(KE == 64 || Cout == 64, "16-channel TMA conv supports Cout == 64 only");
  const bool dual = second && second->in2;
  if (dual) {
    AVVAD_CHECK_ARG(KE == 64 && second->Cin2 % 64 == 0 && second->stride2 >= 1, "second operand: Cin2 % 64 == 0 required");
    AVVAD_CHECK_ARG((second->H2 - 1) / second->stride2 + 1 == OH && (second->W2 - 1) / second->stride2 + 1 == OW,
                    "second operand: output grid mismatch");
  }
  TmaGeom g{};
  g.mode = 1;
  g.OH = OH; g.OW = OW; g.stride = stride; g.pad = pad; g.S = S; g.cpb = Cin / KE; g.KB = R * S * (Cin / KE);
  g.n_frames = n;
  g.N = Cout;
  g.KB2 = dual ? second->Cin2 / 64 : 0;
  g.stride2 = dual ? second->stride2 : 1;
  const int bn = pick_bn(Cout, bn_hint);
  g.n_tiles = (Cout + bn - 1) / bn;
  // choose up to two (band height, frames per tile) phases maximising the fill of the 128 accumulator rows
  double best = -1;
  int bh0 = 1, bF0 = 1, bnb0 = OH, brem = 0, bF1 = 1;
  for (int hb0 = 1; hb0 <= OH; ++hb0) {
    if (hb0 * OW > 128) break;
    const int nb0 = OH / hb0;
    const int rem = OH - nb0 * hb0;
    int F0 = (nb0 == 1 && rem == 0) ? 128 / (hb0 * OW) : 128 / (hb0 * OW);
    if (F0 < 1) continue;
    if (nb0 > 1) F0 = 1;  // several bands per frame: one frame per tile keeps the tile enumeration simple
    if (F0 > 256) F0 = 256;
    double tiles_per_frame = (double)nb0 / F0;
    int F1 = 1;
    if (rem > 0) {
      F1 = 128 / (rem * OW);
      if (F1 < 1) continue;
      if (F1 > 256) F1 = 256;
      tiles_per_frame += 1.0 / F1;
    }
    const double eff = (double)OH * OW / (128.0 * tiles_per_frame);
    if (eff > best + 1e-9) {
      best = eff; bh0 = hb0; bF0 = F0; bnb0 = nb0; brem = rem; bF1 = F1;
    }
  }
  AVVAD_CHECK_ARG(best > 0, "TMA conv: no valid tiling");
  g.h0[0] = 0; g.hb[0] = bh0; g.nb[0] = bnb0; g.F[0] = bF0;
  g.tiles0 = ((n + bF0 - 1) / bF0) * bnb0;
  int64_t tiles1 = 0;
  g.h0[1] = bnb0 * bh0; g.hb[1] = brem > 0 ? brem : 1; g.nb[1] = 1; g.F[1] = bF1;
  if (brem > 0) tiles1 = (n + bF1 - 1) / bF1;
  g.m_tiles = g.tiles0 + tiles1;
  g.total_tiles = g.m_tiles * g.n_tiles;

  TmaMaps maps;
  const uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)n};
  const uint64_t strides[3] = {(uint64_t)Cin * 2, (uint64_t)W * Cin * 2, (uint64_t)H * W * Cin * 2};
  const uint32_t estr[4] = {1, (uint32_t)stride, (uint32_t)stride, 1};
  for (int p = 0; p < 2; ++p) {
    const int hb = g.hb[p], F = g.F[p];
    const uint32_t box[4] = {(uint32_t)KE, (uint32_t)((OW - 1) * stride + 1), (uint32_t)((hb - 1) * stride + 1),
                             (uint32_t)F};
    int rc = encode4(&maps.a[p], in, dims, strides, box, estr, KE == 16);
    if (rc) return rc;
    g.bytesA[p] = (uint32_t)F * hb * OW * (uint32_t)(KE * 2);
    if (dual) {
      const int s2 = second->stride2;
      const uint64_t dims2[4] = {(uint64_t)second->Cin2, (uint64_t)second->W2, (uint64_t)second->H2, (uint64_t)n};
      const uint64_t strides2[3] = {(uint64_t)second->Cin2 * 2, (uint64_t)second->W2 * second->Cin2 * 2,
                                    (uint64_t)second->H2 * second->W2 * second->Cin2 * 2};
      const uint32_t estr2[4] = {1, (uint32_t)s2, (uint32_t)s2, 1};
      const uint32_t box2[4] = {64, (uint32_t)((OW - 1) * s2 + 1), (uint32_t)((hb - 1) * s2 + 1), (uint32_t)F};
      rc = encode4(&maps.a2[p], second->in2, dims2, strides2, box2, estr2, false);
      if (rc) return rc;
    } else {
      maps.a2[p] = maps.a[p];
    }
  }
  const int K = R * S * Cin + (dual ? second->Cin2 : 0);
  const bool pair = KE == 64 && use_pair(bn, 1, EPI_BF16, g.KB + g.KB2);
  g.pair = pair ? 1 : 0;
  int rc = encode2(&maps.b, w, (uint64_t)K, (uint64_t)Cout, (uint64_t)K * 2, (uint32_t)KE, (uint32_t)(pair ? bn / 2 : bn),
                   KE == 16);
  if (rc) return rc;
  g.bytesB = (uint32_t)bn * (uint32_t)(KE * 2);
  const double flops = flops_override > 0 ? flops_override : 2.0 * (double)n * OH * OW * Cout * K;
  if (KE == 16) return launch_bn<64, 16>(maps, g, ep, EPI_BF16, cat, flops, st);
  return dispatch(bn, maps, g, ep, EPI_BF16, cat, flops, st);
}

int launch_tma_gemm(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* Wt, int64_t ldw, int64_t M, int N, int K,
                    const EpiParams& ep, int epi_mode, int bn_hint, cudaStream_t st, int ksplit, int64_t split_stride) {
  AVVAD_CHECK_ARG(K % 64 == 0 && lda % 8 == 0 && ldw % 8 == 0, "TMA gemm: K % 64, lda % 8, ldw % 8 required");
  AVVAD_CHECK_ARG(ksplit >= 1 && (ksplit == 1 || (epi_mode == EPI_F32 && !ep.bias && !ep.relu)),
                  "split-K needs fp32 output without bias / ReLU");
  TmaGeom g{};
  g.ksplit = ksplit;
  g.kb_split = (K / 64 + ksplit - 1) / ksplit;
  // every split must own at least one K block: a CTA with an empty K range would wait for an accumulator that no MMA
  // ever commits (the bounded barrier wait then traps)
  AVVAD_CHECK_ARG((int64_t)(ksplit - 1) * g.kb_split < K / 64, "split-K: empty split (choose ksplit = ceil(KB / ceil(KB / ksplit)))");
  g.split_stride = split_stride;
  g.mode = 0;
  g.KB = K / 64;
  g.cpb = g.KB;  // never wraps
  g.S = 1;
  g.n_frames = M;
  g.N = N;
  int bn = pick_bn(N, bn_hint);
  g.n_tiles = (N + bn - 1) / bn;
  g.m_tiles = (M + BM - 1) / BM;
  g.total_tiles = g.m_tiles * g.n_tiles;
  g.tiles0 = g.m_tiles;
  g.hb[0] = g.hb[1] = 1; g.nb[0] = g.nb[1] = 1; g.F[0] = g.F[1] = 1; g.OW = 128; g.OH = 1;
  TmaMaps maps;
  const uint64_t dims[4] = {(uint64_t)K, (uint64_t)M, 1, 1};
  const uint64_t strides[3] = {(uint64_t)lda * 2, (uint64_t)lda * 2 * (uint64_t)M, (uint64_t)lda * 2 * (uint64_t)M};
  const uint32_t box[4] = {64, 128, 1, 1};
  const uint32_t estr[4] = {1, 1, 1, 1};
  int rc = encode4(&maps.a[0], A, dims, strides, box, estr);
  if (rc) return rc;
  maps.a[1] = maps.a[0];
  maps.a2[0] = maps.a2[1] = maps.a[0];
  g.bytesA[0] = g.bytesA[1] = 128u * 128u;
  g.pair = use_pair(bn, ksplit, epi_mode, g.KB) ? 1 : 0;
  rc = encode2(&maps.b, Wt, (uint64_t)K, (uint64_t)N, (uint64_t)ldw * 2, 64, (uint32_t)(g.pair ? bn / 2 : bn));
  if (rc) return rc;
  g.bytesB = (uint32_t)bn * 128u;
  const double flops = 2.0 * (double)M * N * K;
  return dispatch(bn, maps, g, ep, epi_mode, epi_mode == EPI_LSTM ? 2 : 1, flops, st);
}

int launch_tma_gemm_xt(const __nv_bfloat16* X, int64_t lda, const __nv_bfloat16* Wt, int64_t ldw, int64_t B, int64_t T,
                       int64_t T_stride, int N, int K, const float* bias, float* xT, cudaStream_t st, int grid_cap) {
  AVVAD_CHECK_ARG(K % 64 == 0 && lda % 8 == 0 && ldw % 8 == 0 && N % 32 == 0, "TMA gemm (xT): K % 64, lda % 8, N % 32");
  const int64_t Bp = (B + 127) / 128 * 128;
  AVVAD_CHECK_ARG(T * Bp < (1ll << 31), "TMA gemm (xT): T * B too large");
  TmaGeom g{};
  g.ksplit = 1;
  g.kb_split = K / 64;
  g.mode = 0;
  g.KB = K / 64;
  g.cpb = g.KB;
  g.S = 1;
  g.n_frames = T * Bp;
  g.N = N;
  g.tm_bp = (int)Bp;
  g.tm_b = (int)B;
  g.grid_cap = grid_cap;
  const int bn = pick_bn(N, 0);
  g.n_tiles = (N + bn - 1) / bn;
  g.m_tiles = T * Bp / BM;
  g.total_tiles = g.m_tiles * g.n_tiles;
  g.tiles0 = g.m_tiles;
  g.hb[0] = g.hb[1] = 1; g.nb[0] = g.nb[1] = 1; g.F[0] = g.F[1] = 1; g.OW = 128; g.OH = 1;
  TmaMaps maps;
  // (k, b, t): a box is 128 batch items of one time step; rows past B are zero-filled by the hardware
  const uint64_t dims[4] = {(uint64_t)K, (uint64_t)B, (uint64_t)T, 1};
  const uint64_t strides[3] = {(uint64_t)lda * 2 * (uint64_t)T_stride, (uint64_t)lda * 2,
                               (uint64_t)lda * 2 * (uint64_t)T_stride * (uint64_t)B};
  const uint32_t box[4] = {64, 128, 1, 1};
  const uint32_t estr[4] = {1, 1, 1, 1};
  int rc = encode4(&maps.a[0], X, dims, strides, box, estr);
  if (rc) return rc;
  maps.a[1] = maps.a[0];
  maps.a2[0] = maps.a2[1] = maps.a[0];
  g.bytesA[0] = g.bytesA[1] = 128u * 128u;
  g.pair = use_pair(bn, 1, EPI_XT, g.KB) ? 1 : 0;
  rc = encode2(&maps.b, Wt, (uint64_t)K, (uint64_t)N, (uint64_t)ldw * 2, 64, (uint32_t)(g.pair ? bn / 2 : bn));
  if (rc) return rc;
  g.bytesB = (uint32_t)bn * 128u;
  EpiParams ep{};
  ep.bias = bias;
  ep.C = xT;
  ep.ldc = N;
  return dispatch(bn, maps, g, ep, EPI_XT, 1, 2.0 * (double)B * T * N * K, st);
}

int launch_tma_gemm_tm(const __nv_bfloat16* X, int64_t lda, const __nv_bfloat16* Wt, int64_t ldw, int64_t B, int64_t T,
                       int64_t T_stride, int N, int K, float* C, int64_t ldc, cudaStream_t st, int grid_cap) {
  AVVAD_CHECK_ARG(K % 64 == 0 && lda % 8 == 0 && ldw % 8 == 0 && N % 32 == 0, "TMA gemm (tm): K % 64, lda % 8, N % 32");
  const int64_t Bp = (B + 127) / 128 * 128;
  AVVAD_CHECK_ARG(T * Bp < (1ll << 31), "TMA gemm (xT): T * B too large");
  TmaGeom g{};
  g.ksplit = 1;
  g.kb_split = K / 64;
  g.mode = 0;
  g.KB = K / 64;
  g.cpb = g.KB;
  g.S = 1;
  g.n_frames = T * Bp;
  g.N = N;
  g.tm_bp = (int)Bp;
  g.tm_b = (int)B;
  g.tm_tstride = T_stride;
  g.grid_cap = grid_cap;
  const int bn = pick_bn(N, 0);
  g.n_tiles = (N + bn - 1) / bn;
  g.m_tiles = T * Bp / BM;
  g.total_tiles = g.m_tiles * g.n_tiles;
  g.tiles0 = g.m_tiles;
  g.hb[0] = g.hb[1] = 1; g.nb[0] = g.nb[1] = 1; g.F[0] = g.F[1] = 1; g.OW = 128; g.OH = 1;
  TmaMaps maps;
  // (k, b, t): a box is 128 batch items of one time step; rows past B are zero-filled by the hardware
  const uint64_t dims[4] = {(uint64_t)K, (uint64_t)B, (uint64_t)T, 1};
  const uint64_t strides[3] = {(uint64_t)lda * 2 * (uint64_t)T_stride, (uint64_t)lda * 2,
                               (uint64_t)lda * 2 * (uint64_t)T_stride * (uint64_t)B};
  const uint32_t box[4] = {64, 128, 1, 1};
  const uint32_t estr[4] = {1, 1, 1, 1};
  int rc = encode4(&maps.a[0], X, dims, strides, box, estr);
  if (rc) return rc;
  maps.a[1] = maps.a[0];
  maps.a2[0] = maps.a2[1] = maps.a[0];
  g.bytesA[0] = g.bytesA[1] = 128u * 128u;
  g.pair = use_pair(bn, 1, EPI_F32, g.KB) ? 1 : 0;
  rc = encode2(&maps.b, Wt, (uint64_t)K, (uint64_t)N, (uint64_t)ldw * 2, 64, (uint32_t)(g.pair ? bn / 2 : bn));
  if (rc) return rc;
  g.bytesB = (uint32_t)bn * 128u;
  EpiParams ep{};
  ep.C = C;
  ep.ldc = ldc;
  return dispatch(bn, maps, g, ep, EPI_F32, 1, 2.0 * (double)B * T * N * K, st);
}


}  // namespace tc
}  // namespace avvad
