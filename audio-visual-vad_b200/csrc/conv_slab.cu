// Host side of the slab convolution: geometry search, tensor maps, launch.
#include <cudaTypedefs.h>
#include <stdlib.h>

#include <mutex>

#include "conv_slab.cuh"
#include "conv_block.cuh"

namespace avvad {
namespace tc {

int prof_begin(cudaStream_t st, void** tok);
void prof_end(cudaStream_t st, void* tok, int cat, double flops);
int encode_act_map(CUtensorMap* m, const void* ptr, int Cin, int W, int H, int64_t n, const uint32_t box[4],
                   const uint32_t estr[4]);
int encode_weight_map(CUtensorMap* m, const void* ptr, uint64_t K, uint64_t N, uint32_t bn);

// 64 -> 64 channels (layer1): the 72 KB of weights stay resident in shared memory
bool slab_supported(int H, int W, int Cin, int Cout, int R, int S, int stride, int pad) {
  return tma_available() && R == 3 && S == 3 && stride == 1 && pad == 1 && H == W && Cin == 64 && Cout == 64;
}

struct SlabPlan {
  int F, hb, mb, bn;
  size_t smem;
  double eff;
};

static bool plan(int H, int Cin, int Cout, SlabPlan* out) {
  const int OW = H, OH = H, Wp = OW + 2;
  const int cpb = Cin / 64;
  SlabPlan best{};
  best.eff = -1;
  const int bn = 64;
  for (int hb = 1; hb <= OH; ++hb) {
    const int Hs = hb + 2;
    if (Hs > 256 || Wp > 256) continue;
    const int fmax = (hb == OH) ? 64 : 1;  // several frames per slab only for whole-frame bands
    for (int F = 1; F <= fmax; ++F) {
      const int rows = F * Hs * Wp;
      const int P = rows - 2 * Wp - 2;
      const int mb = (P + 127) / 128;
      if (2 * mb * bn > 512) break;
      const int slab_rows = mb * 128 + 2 * Wp + 2;
      if (slab_rows < rows) continue;
      const size_t slab_bytes = ((size_t)slab_rows * 128 + 1023) / 1024 * 1024;
      const size_t wbytes = (size_t)9 * cpb * bn * 128;
      const size_t smem = 2 * slab_bytes + wbytes + 256 + 1024 + (size_t)Cout * 4;
      if (smem > 225 * 1024) continue;
      const int nb = (OH + hb - 1) / hb;
      // valid outputs per frame / MMA rows per frame
      const double eff = (double)OH * OW / ((double)nb * mb * 128.0 / F);
      // prefer higher efficiency, then more accumulator blocks per weight load
      if (eff > best.eff + 1e-9 || (eff > best.eff - 1e-9 && mb > best.mb)) {
        best.F = F; best.hb = hb; best.mb = mb; best.bn = bn; best.smem = smem; best.eff = eff;
      }
    }
  }
  if (best.eff <= 0) return false;
  *out = best;
  return true;
}

template <int MBC = 0>
static int launch_k(const SlabMaps& maps, const SlabGeom& g, const EpiParams& ep, size_t smem, double flops,
                    cudaStream_t st) {
  static std::mutex mu;
  static size_t attr_set[kMaxDevices] = {};  // per device: function attributes live in the device's context
  {
    int dev = 0;
    AVVAD_CUDA(cudaGetDevice(&dev));
    AVVAD_CHECK_ARG(dev >= 0 && dev < kMaxDevices, "device index out of range");
    std::lock_guard<std::mutex> lk(mu);
    if (smem > attr_set[dev]) {
      AVVAD_CUDA(cudaFuncSetAttribute(tc_slab_kernel<64, MBC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr_set[dev] = smem;
    }
  }
  static int num_sms = [] {
    int dev = 0, n = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n > 0 ? n : 148;
  }();
  void* tok = nullptr;
  const unsigned grid = (unsigned)(g.total_tiles < num_sms ? g.total_tiles : num_sms);
  prof_begin(st, &tok);
  tc_slab_kernel<64, MBC><<<grid, kSlabThreads, smem, st>>>(maps, g, ep);
  AVVAD_LAUNCHED();
  prof_end(st, tok, 0, flops);
  return AVVAD_OK;
}

int launch_slab_conv(const __nv_bfloat16* in, const __nv_bfloat16* w, const EpiParams& ep, int64_t n, int H, int Cin,
                     int Cout, cudaStream_t st) {
  SlabPlan p;
  if (!plan(H, Cin, Cout, &p)) {
    set_error("slab conv: no feasible plan");
    return AVVAD_ERR_ARG;
  }
  SlabGeom g{};
  g.n_frames = n;
  g.OH = H; g.OW = H; g.Wp = H + 2; g.hb = p.hb; g.Hs = p.hb + 2; g.F = p.F; g.mb = p.mb;
  g.nb = (H + p.hb - 1) / p.hb;
  g.cpb = Cin / 64;
  g.N = Cout;
  g.n_tiles = Cout / p.bn;
  g.total_tiles = ((n + p.F - 1) / p.F) * g.nb * g.n_tiles;
  g.slab_rows = p.mb * 128 + 2 * g.Wp + 2;
  g.slab_tx = (uint32_t)p.F * g.Hs * g.Wp * 128u;
  SlabMaps maps;
  const uint32_t box[4] = {64, (uint32_t)g.Wp, (uint32_t)g.Hs, (uint32_t)p.F};
  const uint32_t estr[4] = {1, 1, 1, 1};
  int rc = encode_act_map(&maps.a, in, Cin, H, H, n, box, estr);
  if (rc) return rc;
  rc = encode_weight_map(&maps.b, w, (uint64_t)9 * Cin, (uint64_t)Cout, (uint32_t)p.bn);
  if (rc) return rc;
  const double flops = 2.0 * (double)n * H * H * Cout * 9.0 * Cin;
  if (p.mb == 3) return launch_k<3>(maps, g, ep, p.smem, flops, st);
  return launch_k(maps, g, ep, p.smem, flops, st);
}

// ---- fused BasicBlock of layer1 (conv_block.cuh); AVVAD_BLOCK17=0 keeps the two slab convolutions
bool block17_enabled() {
  static int v = [] {
    const char* e = getenv("AVVAD_BLOCK17");
    return (e && atoi(e) == 0) ? 0 : 1;
  }();
  return v != 0 && tma_available();
}

int launch_block17(const __nv_bfloat16* x, const __nv_bfloat16* wa, const float* bias_a, const __nv_bfloat16* wb,
                   const float* bias_b, __nv_bfloat16* z, int64_t n, cudaStream_t st) {
  AVVAD_CHECK_ARG(x && wa && wb && z && n > 0, "block17: bad argument");
  AVVAD_CHECK_ARG(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(z)) & 31) == 0, "block17: 32-byte aligned activations");
  static PerDeviceOnce once;
  AVVAD_CUDA(once.run([] {
    return cudaFuncSetAttribute(tc_block17_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBlkSmem);
  }));
  static int num_sms = [] {
    int dev = 0, v = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v > 0 ? v : 148;
  }();
  BlockMaps maps;
  const uint32_t box[4] = {64, (uint32_t)kBlkWp, (uint32_t)kBlkWp, 1};
  const uint32_t estr[4] = {1, 1, 1, 1};
  int rc = encode_act_map(&maps.x, x, 64, kBlkW, kBlkW, n, box, estr);
  if (rc) return rc;
  rc = encode_weight_map(&maps.wa, wa, 576, 64, 32);
  if (rc) return rc;
  rc = encode_weight_map(&maps.wb, wb, 576, 64, 32);
  if (rc) return rc;
  BlockGeom g{};
  g.n_frames = n;
  const int64_t want = (n + 1) / 2, pairs = num_sms / 2;
  g.n_pairs = (int)(want < pairs ? want : pairs);
  g.bias_a = bias_a;
  g.bias_b = bias_b;
  g.x = x;
  g.z = z;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2u * (unsigned)g.n_pairs);
  cfg.blockDim = dim3(kBlkThreads);
  cfg.dynamicSmemBytes = kBlkSmem;
  cfg.stream = st;
  cudaLaunchAttribute la[1];
  la[0].id = cudaLaunchAttributeClusterDimension;
  la[0].val.clusterDim.x = 2; la[0].val.clusterDim.y = 1; la[0].val.clusterDim.z = 1;
  cfg.attrs = la;
  cfg.numAttrs = 1;
  void* tok = nullptr;
  prof_begin(st, &tok);
  cudaError_t le = cudaLaunchKernelEx(&cfg, tc_block17_kernel, maps, g);
  if (le != cudaSuccess) {
    set_error(std::string("block17 launch failed: ") + cudaGetErrorString(le));
    return AVVAD_ERR_CUDA;
  }
  AVVAD_LAUNCHED();
  prof_end(st, tok, 0, 2.0 * 2.0 * (double)n * kBlkW * kBlkW * 64.0 * 576.0);
  return AVVAD_OK;
}

}  // namespace tc
}  // namespace avvad
