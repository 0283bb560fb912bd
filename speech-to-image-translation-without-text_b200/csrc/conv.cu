// Host side of the convolution entry points: tap tables, TMA tensor maps, launch geometry.
// Reference constructs replaced: nn.Conv2d 3x3 (model.py:125-128), nn.Upsample+conv3x3 (model.py:133-140),
// nn.Conv2d 4x4 s2 (model.py:369-398) — forward, data gradient and weight gradient.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "../../include/sg2b200.h"
#ifdef SG2_BUILD_PROBES
#include "../../include/sg2b200_probes.h"
#endif
#include "common.cuh"
#include "igemm.cuh"
#include "igemm_pair.cuh"
#ifdef SG2_BUILD_PROBES
#include "halo_probe.cuh"
#endif
#include "tile_conv.cuh"
#include "tile_wgrad.cuh"

namespace sg2 {

thread_local char g_err[512] = "";

// ------------------------------------------------------------------------------------------ driver entry
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// A strided NHWC view: element (b, y, x, c) lives at base[b*sb + y*sy + x*sx + c] (bf16 elements).
struct View {
  const __nv_bfloat16* base;
  int C, W, H, B;
  long long sx, sy, sb;
};
static View dense_view(const void* p, int B, int H, int W, int C) {
  return View{reinterpret_cast<const __nv_bfloat16*>(p), C, W, H, B, (long long)C, (long long)W * C,
              (long long)H * W * C};
}
// Parity plane (py, px) of a view with even H, W: pixels (2i+py, 2j+px).
static View plane_view(const View& v, int py, int px) {
  View r = v;
  r.base = v.base + py * v.sy + px * v.sx;
  r.W = v.W / 2;
  r.H = v.H / 2;
  r.sx = 2 * v.sx;
  r.sy = 2 * v.sy;
  return r;
}

static CUtensorMapSwizzle sw_enum(int bytes) {
  return bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                      : (bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                     : (bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE));
}

static int make_act_map(CUtensorMap* m, const View& v, int boxC, int tw, int th, int nb) {
  EncodeTiledFn enc = get_encode();
  if (!enc) SG2_FAIL(SG2_EDRIVER, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[4] = {(cuuint64_t)v.C, (cuuint64_t)v.W, (cuuint64_t)v.H, (cuuint64_t)v.B};
  cuuint64_t strides[3] = {(cuuint64_t)v.sx * 2, (cuuint64_t)v.sy * 2, (cuuint64_t)v.sb * 2};
  cuuint32_t box[4] = {(cuuint32_t)boxC, (cuuint32_t)tw, (cuuint32_t)th, (cuuint32_t)nb};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  if ((reinterpret_cast<uintptr_t>(v.base) & 15) || (strides[0] & 15) || (strides[1] & 15) || (strides[2] & 15))
    SG2_FAIL(SG2_EINVAL, "activation view not 16-byte aligned (C=%d)", v.C);
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<__nv_bfloat16*>(v.base), dims, strides, box,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw_enum(boxC * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    SG2_FAIL(SG2_EDRIVER, "cuTensorMapEncodeTiled(act) failed: %d (C=%d W=%d H=%d B=%d box=%d,%d,%d,%d)", (int)r,
             v.C, v.W, v.H, v.B, boxC, tw, th, nb);
  return 0;
}

static int make_w_map(CUtensorMap* m, const void* w, long long rows, long long K, int bk, int bn) {
  EncodeTiledFn enc = get_encode();
  if (!enc) SG2_FAIL(SG2_EDRIVER, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {(cuuint32_t)bk, (cuuint32_t)bn};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(w), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw_enum(bk * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    SG2_FAIL(SG2_EDRIVER, "cuTensorMapEncodeTiled(weights) failed: %d (rows=%lld K=%lld box=%d,%d)", (int)r, rows, K,
             bk, bn);
  return 0;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is per device (context): remember it per device ordinal, not per process.
static bool attr_needed(bool (&done)[64]) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
  if (done[dev]) return false;
  done[dev] = true;
  return true;
}

// Pipeline depth: as many stages as fit the per-CTA shared-memory budget (default 100 KB so that two CTAs
// co-reside per SM and one's epilogue overlaps the other's main loop); SG2_SMEM_BUDGET_KB overrides.
static int max_stages(int stage_bytes) {
  static int budget_kb = [] {
    const char* e = getenv("SG2_SMEM_BUDGET_KB");
    int v = e ? atoi(e) : 100;
    return v < 16 ? 16 : (v > 220 ? 220 : v);
  }();
  // small tiles are latency-bound: prefer four co-resident CTAs per SM over a deep pipeline
  const int kb = stage_bytes < 24 * 1024 ? (budget_kb < 48 ? budget_kb : 48) : budget_kb;
  int s = kb * 1024 / stage_bytes;
  return s > 8 ? 8 : (s < 2 ? 2 : s);
}

// pixel tile {tw, th, nb} with tw*th*nb == npix over a Wg x Hg grid
static int pick_tile(int Wg, int Hg, int npix, int* tw, int* th, int* nb) {
  int w = (Hg == 1) ? (Wg < npix ? Wg : npix) : (Wg < 16 ? Wg : 16);
  int h = npix / w;
  if (h > Hg) h = Hg;
  if (w <= 0 || h <= 0 || npix % (w * h)) SG2_FAIL(SG2_EINVAL, "no %d-pixel tile for a %dx%d grid", npix, Wg, Hg);
  *tw = w;
  *th = h;
  *nb = npix / (w * h);
  return 0;
}

// ------------------------------------------------------------------------------------------ gather launch
struct GatherDesc {
  View a[4];
  int nmaps;
  TapF taps[4][kMaxTaps];
  int ntaps, ngroups;
  int Cin;  // channels per tap (K per tap)
  const void* w;
  int N;          // output channels (weight rows per group)
  int Wg, Hg, B;  // logical output grid per group
  void* out;
  long long out_off[4], osx, osy, osb;
  int out_mode, splitk;
  long long split_stride;  // elements between the split-K slabs of an OUT_F32_STORE output
  double* stats;
  int stats_bg;  // images per statistics group (0: one)
  int act;  // epilogue activation (tile kernel only): 0 none, 2 LeakyReLU(0.2)
  const float* bias9;  // [B][9][N] border-region bias (tile kernel only)
  const void* epi_src;  // epilogue operand, layout of the output (tile kernel only)
  int epi_mode;         // 0 none, SG2_EPI_ADD, SG2_EPI_LRELU_MASK
  const float* bias;    // [N] per-channel bias (plain gather kernel only)
  int tw, th, nb;       // pixel tile of the plain gather kernel (0: pick_tile's 128-pixel tile)
};

// two pixel tiles per CTA on the gather kernels' 256-channel instances (FpropCfg). Off by default: measured 8.05 vs 7.70
// ms/step (fewer, longer CTAs and a higher split factor cost more than the saved weight bytes); SG2_IGEMM_MT2=1 enables it
static bool igemm_mt2() {
  static const bool on = [] {
    const char* e = getenv("SG2_IGEMM_MT2");
    return e ? atoi(e) != 0 : false;
  }();
  return on;
}

template <int BN, int BK, int MT = 1>
static int launch_fprop_t(const GatherDesc& d, cudaStream_t st) {
  using Cfg = FpropCfg<BN, BK, MT>;
  FpropParams p;
  memset(&p, 0, sizeof(p));
  int rc;
  if (d.tw) {
    p.tw = d.tw, p.th = d.th, p.nb = d.nb;
  } else if ((rc = pick_tile(d.Wg, d.Hg, kBlockM, &p.tw, &p.th, &p.nb))) {
    return rc;
  }
  for (int i = 0; i < d.nmaps; ++i)
    if ((rc = make_act_map(&p.tmA[i], d.a[i], BK, p.tw, p.th, p.nb))) return rc;
  const long long K = (long long)d.ntaps * d.Cin;
  if ((rc = make_w_map(&p.tmB, d.w, (long long)d.ngroups * d.N, K, BK, BN))) return rc;
  memcpy(p.taps, d.taps, sizeof(p.taps));
  p.ntaps = d.ntaps;
  p.kchunks = d.Cin / BK;
  p.ngroups = d.ngroups;
  p.bias = d.bias;
  const int KB = p.ntaps * p.kchunks;
  p.splitk = d.splitk < 1 ? 1 : (d.splitk > KB ? KB : d.splitk);
  if (p.splitk > 1 && d.out_mode == OUT_BF16) SG2_FAIL(SG2_EINVAL, "split-K needs an fp32 output mode");
  if (p.splitk != d.splitk && d.splitk > 1 && d.out_mode == OUT_F32_STORE)
    SG2_FAIL(SG2_EINVAL, "split-K slabs: %d splits requested, only %d K blocks", d.splitk, KB);
  p.split_stride = d.split_stride;
  p.tiles_x = (d.Wg + p.tw - 1) / p.tw;
  p.tiles_y = (d.Hg + p.th - 1) / p.th;
  p.tiles_b = (d.B + p.nb - 1) / p.nb;
  p.Wo = d.Wg;
  p.Ho = d.Hg;
  p.B = d.B;
  p.N = d.N;
  for (int g = 0; g < 4; ++g) p.out_off[g] = d.out_off[g];
  p.sb = d.osb;
  p.sy = d.osy;
  p.sx = d.osx;
  p.out = d.out;
  p.out_mode = d.out_mode;
  p.stats = d.stats;
  p.stats_bg = d.stats_bg;
  p.act = d.act;
  if (d.stats && d.stats_bg > 0 && (d.stats_bg % p.nb))
    SG2_FAIL(SG2_ENOFUSE, "fused BN statistics: a %d-image tile would straddle statistics groups of %d images", p.nb, d.stats_bg);
  // MT = 2 fills the 512 TMEM columns of an SM by itself: one CTA per SM, as deep a ring as shared memory allows
  const int smax = MT == 2 ? (int)((200 * 1024) / Cfg::kStageBytes) : max_stages(Cfg::kStageBytes);
  int stages = smax;
  if (stages > KB / p.splitk + 1) stages = KB / p.splitk + 1;
  if (stages < 2) stages = 2;
  p.stages = stages;
  const size_t smem = Cfg::smem_bytes(stages);
  static bool attr_done[64] = {};
  if (attr_needed(attr_done)) {
    cudaError_t e = cudaFuncSetAttribute(igemm_fprop_kernel<BN, BK, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)Cfg::smem_bytes(smax));
    if (e != cudaSuccess) SG2_FAIL((int)e, "cudaFuncSetAttribute(fprop<%d,%d>): %s", BN, BK, cudaGetErrorString(e));
  }
  const int pix_tiles = p.tiles_x * p.tiles_y * p.tiles_b;
  dim3 grid((pix_tiles + MT - 1) / MT, (d.N + BN - 1) / BN, p.ngroups * p.splitk);
  igemm_fprop_kernel<BN, BK, MT><<<grid, kNumThreads, smem, st>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) SG2_FAIL((int)e, "fprop<%d,%d> launch: %s", BN, BK, cudaGetErrorString(e));
  return 0;
}

// ------------------------------------------------------------------------------------------ cluster split-K launch
template <int BN, int BK, int MT = 1>
static int launch_fprop_cluster_t(const GatherDesc& d, cudaStream_t st) {
  using Cfg = FpropCfg<BN, BK, MT>;
  using CC = ClusterCfg<BN, BK, MT>;
  FpropParams p;
  memset(&p, 0, sizeof(p));
  int rc;
  if ((rc = pick_tile(d.Wg, d.Hg, kBlockM, &p.tw, &p.th, &p.nb))) return rc;
  for (int i = 0; i < d.nmaps; ++i)
    if ((rc = make_act_map(&p.tmA[i], d.a[i], BK, p.tw, p.th, p.nb))) return rc;
  const long long K = (long long)d.ntaps * d.Cin;
  if ((rc = make_w_map(&p.tmB, d.w, (long long)d.ngroups * d.N, K, BK, BN))) return rc;
  memcpy(p.taps, d.taps, sizeof(p.taps));
  p.ntaps = d.ntaps;
  p.kchunks = d.Cin / BK;
  p.ngroups = d.ngroups;
  const int KB = p.ntaps * p.kchunks;
  p.splitk = d.splitk > KB ? KB : d.splitk;
  if (p.splitk < 2 || p.splitk > 16) SG2_FAIL(SG2_ENOFUSE, "cluster split-K: %d splits (2..16)", p.splitk);
  p.tiles_x = (d.Wg + p.tw - 1) / p.tw;
  p.tiles_y = (d.Hg + p.th - 1) / p.th;
  p.tiles_b = (d.B + p.nb - 1) / p.nb;
  p.Wo = d.Wg;
  p.Ho = d.Hg;
  p.B = d.B;
  p.N = d.N;
  for (int g = 0; g < 4; ++g) p.out_off[g] = d.out_off[g];
  p.sb = d.osb;
  p.sy = d.osy;
  p.sx = d.osx;
  p.out = d.out;
  p.out_mode = OUT_BF16;
  p.stats = d.stats;
  p.stats_bg = d.stats_bg;
  p.act = d.act;
  p.epi_src = d.epi_src;
  p.epi_mode = d.epi_mode;
  if (d.stats && d.stats_bg > 0 && (d.stats_bg % p.nb))
    SG2_FAIL(SG2_ENOFUSE, "fused BN statistics: a %d-image tile would straddle statistics groups of %d images", p.nb, d.stats_bg);
  int stages = (int)((200 * 1024) / Cfg::kStageBytes);
  if (stages > 8) stages = 8;
  if (stages > KB / p.splitk + 1) stages = KB / p.splitk + 1;
  if (stages < 2) stages = 2;
  p.stages = stages;
  static bool attr_done[64] = {};
  if (attr_needed(attr_done)) {
    cudaError_t e = cudaFuncSetAttribute(igemm_fprop_cluster_kernel<BN, BK, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)CC::smem_bytes(8 < (int)((200 * 1024) / Cfg::kStageBytes) ? 8 : (int)((200 * 1024) / Cfg::kStageBytes)));
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(igemm_fprop_cluster_kernel<BN, BK, MT>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) SG2_FAIL((int)e, "cudaFuncSetAttribute(fprop_cluster<%d,%d>): %s", BN, BK, cudaGetErrorString(e));
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((p.tiles_x * p.tiles_y * p.tiles_b + MT - 1) / MT, d.N / BN, p.ngroups * p.splitk);
  cfg.blockDim = dim3(kNumThreads);
  cfg.dynamicSmemBytes = CC::smem_bytes(stages);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = p.splitk;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, igemm_fprop_cluster_kernel<BN, BK, MT>, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    SG2_FAIL((int)e, "fprop_cluster<%d,%d> launch (cluster %d): %s", BN, BK, p.splitk, cudaGetErrorString(e));
  }
  return 0;
}

// ------------------------------------------------------------------------------------------ CTA-pair launch (cta_group::2)
// SG2_PAIR=0 / SG2_PAIR_WGRAD=0 switch the pair kernels off (the cluster / plain gather kernels take their layers again).
// History (profiles/r02_pair_deadlock.md): in the multi-stream train step the first version deadlocked about once in a few
// hundred steps — the two CTAs of a pair issued tcgen05.alloc.cta_group::2 as soon as each of them started, and next to
// other streams' kernels the CTAs of a cluster start at different times. With a cluster barrier in front of the
// allocation (igemm_pair.cuh) tools/stress_replay.py LOAD=1 ran 2 x 2 500 replays clean where every earlier process
// hung within 500.
static int g_pair_override = -1;   // sg2_set_pair_kernels: -1 = the environment decides
static bool igemm_pair() {
  static const bool on = [] {
    const char* e = getenv("SG2_PAIR");
    return e ? atoi(e) != 0 : true;
  }();
  return g_pair_override >= 0 ? g_pair_override != 0 : on;
}

// One hypothesis for that deadlock: a cta_group::2 TMEM allocation takes columns on both SMs of the pair, so two pair CTAs
// resident on the same SM couple could each hold one SM's columns while waiting for the other's. Every pair launch asks for
// more than half of an SM's shared memory (at most one pair CTA per SM; SG2_PAIR_SMEM_KB). Kept as a precaution: the hang
// persisted with it, so this is not (the whole) cause.
static size_t pair_exclusive_smem(size_t need) {
  static const size_t floor_ = [] {
    const char* e = getenv("SG2_PAIR_SMEM_KB");
    return (size_t)(e ? atoi(e) : 118) * 1024;
  }();
  return need > floor_ ? need : floor_;
}

static bool igemm_pair_wgrad() {
  static const int env = [] {
    const char* e = getenv("SG2_PAIR_WGRAD");
    return e ? (atoi(e) != 0 ? 1 : 0) : -1;
  }();
  return g_pair_override >= 0 ? g_pair_override != 0 : (env >= 0 ? env != 0 : igemm_pair());
}

template <int BN, int BK, bool kDirect>
static int launch_fprop_pair_t(const GatherDesc& d, cudaStream_t st) {
  using Cfg = PairCfg<BN, BK>;
  FpropParams p;
  memset(&p, 0, sizeof(p));
  int rc;
  if ((rc = pick_tile(d.Wg, d.Hg, kBlockM, &p.tw, &p.th, &p.nb))) return rc;
  for (int i = 0; i < d.nmaps; ++i)
    if ((rc = make_act_map(&p.tmA[i], d.a[i], BK, p.tw, p.th, p.nb))) return rc;
  const long long K = (long long)d.ntaps * d.Cin;
  if ((rc = make_w_map(&p.tmB, d.w, (long long)d.ngroups * d.N, K, BK, BN / 2))) return rc;   // each CTA stages half of the channels
  memcpy(p.taps, d.taps, sizeof(p.taps));
  p.ntaps = d.ntaps;
  p.kchunks = d.Cin / BK;
  p.ngroups = d.ngroups;
  const int KB = p.ntaps * p.kchunks;
  p.splitk = d.splitk < 1 ? 1 : (d.splitk > KB ? KB : d.splitk);
  if (p.splitk > 8 || (kDirect && p.splitk != 1)) SG2_FAIL(SG2_ENOFUSE, "pair kernel: %d splits", p.splitk);
  p.tiles_x = (d.Wg + p.tw - 1) / p.tw;
  p.tiles_y = (d.Hg + p.th - 1) / p.th;
  p.tiles_b = (d.B + p.nb - 1) / p.nb;
  p.Wo = d.Wg;
  p.Ho = d.Hg;
  p.B = d.B;
  p.N = d.N;
  for (int g = 0; g < 4; ++g) p.out_off[g] = d.out_off[g];
  p.sb = d.osb;
  p.sy = d.osy;
  p.sx = d.osx;
  p.out = d.out;
  p.out_mode = OUT_BF16;
  p.stats = d.stats;
  p.stats_bg = d.stats_bg;
  p.act = d.act;
  p.epi_src = d.epi_src;
  p.epi_mode = d.epi_mode;
  if (d.stats && d.stats_bg > 0 && (d.stats_bg % p.nb))
    SG2_FAIL(SG2_ENOFUSE, "fused BN statistics: a %d-image tile would straddle statistics groups of %d images", p.nb, d.stats_bg);
  const int smax = kDirect ? Cfg::kDirectStages : Cfg::kMaxStages;
  int stages = smax;
  if (stages > KB / p.splitk + 1) stages = KB / p.splitk + 1;
  if (stages < 2) stages = 2;
  p.stages = stages;
  static bool attr_done[64] = {};
  if (attr_needed(attr_done)) {
    cudaError_t e = cudaFuncSetAttribute(igemm_fprop_pair_kernel<BN, BK, kDirect>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)pair_exclusive_smem(kDirect ? Cfg::smem_bytes_direct(smax) : Cfg::smem_bytes(smax)));
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(igemm_fprop_pair_kernel<BN, BK, kDirect>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) SG2_FAIL((int)e, "cudaFuncSetAttribute(fprop_pair<%d,%d>): %s", BN, BK, cudaGetErrorString(e));
  }
  const int pix_tiles = p.tiles_x * p.tiles_y * p.tiles_b;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(2 * ((pix_tiles + 1) / 2), d.N / BN, p.ngroups * p.splitk);
  cfg.blockDim = dim3(kNumThreads);
  cfg.dynamicSmemBytes = pair_exclusive_smem(kDirect ? Cfg::smem_bytes_direct(stages) : Cfg::smem_bytes(stages));
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = p.splitk;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, igemm_fprop_pair_kernel<BN, BK, kDirect>, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    SG2_FAIL((int)e, "fprop_pair<%d,%d> launch (cluster 2x%d): %s", BN, BK, p.splitk, cudaGetErrorString(e));
  }
  return 0;
}

// ------------------------------------------------------------------------------------------ tile-resident launch
static long long* g_tile_dbg = nullptr;
static int tile_mode() {
  static int m = [] {
    const char* e = getenv("SG2_TILE");
    return e ? atoi(e) : 1;
  }();
  return m;
}

// SMs the persistent kernels leave free (sg2_set_sm_reserve): in a data-parallel run NCCL's all-reduce CTAs must find a
// free SM while a one-CTA-per-SM convolution is running, or the reduction only advances in the gaps between kernels.
static int g_sm_reserve = 0;
static int num_sms() {
  static int n = [] {
    int dev = 0, v = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v > 0 ? v : 148;
  }();
  const int r = n - g_sm_reserve;
  return r > 16 ? r : 16;
}

static bool tile_eligible(const GatherDesc& d) {
  return tile_mode() && d.out_mode == OUT_BF16 && d.splitk <= 1 && d.Wg >= kTileW && d.Hg >= kTileH;
}

struct TilePlan {
  TileParams p;
  int bn, bk;
  size_t smem;
};

// Decide tile shape, weight residency, units and pipeline depths. Returns 0 (planned), 1 (use the gather kernel), <0 error.
static int plan_tile(const GatherDesc& d, TilePlan& pl) {
  TileParams& p = pl.p;
  memset(&p, 0, sizeof(p));
  const int bk = (d.Cin % 64 == 0) ? 64 : ((d.Cin % 32 == 0) ? 32 : 16);
  const int row_b = bk * 2;
  // ---- per-source window extents over all groups' taps; taps sorted by source
  int mny[4], mxy[4], mnx[4], mxx[4], cnt[4] = {0, 0, 0, 0};
  for (int s = 0; s < 4; ++s) mny[s] = mnx[s] = 127, mxy[s] = mxx[s] = -127;
  for (int g = 0; g < d.ngroups; ++g)
    for (int t = 0; t < d.ntaps; ++t) {
      const TapF& tp = d.taps[g][t];
      mny[tp.map] = tp.dy < mny[tp.map] ? tp.dy : mny[tp.map];
      mxy[tp.map] = tp.dy > mxy[tp.map] ? tp.dy : mxy[tp.map];
      mnx[tp.map] = tp.dx < mnx[tp.map] ? tp.dx : mnx[tp.map];
      mxx[tp.map] = tp.dx > mxx[tp.map] ? tp.dx : mxx[tp.map];
      if (g == 0) ++cnt[tp.map];
    }
  int ex = 0, ey = 0;
  for (int s = 0; s < d.nmaps; ++s) {
    if (cnt[s] == 0 || cnt[s] != cnt[0]) return 1;
    ex = (mxx[s] - mnx[s]) > ex ? (mxx[s] - mnx[s]) : ex;
    ey = (mxy[s] - mny[s]) > ey ? (mxy[s] - mny[s]) : ey;
    p.org_x[s] = mnx[s];
    p.org_y[s] = mny[s];
  }
  p.pitch = kTileW + ex;
  p.ph = kTileH + ey;
  p.nsrc = d.nmaps;
  p.ntaps = d.ntaps;
  p.ngroups = d.ngroups;
  p.kchunks = d.Cin / bk;
  p.src_begin[0] = 0;
  for (int s = 0; s < d.nmaps; ++s) p.src_begin[s + 1] = p.src_begin[s] + cnt[s];
  for (int g = 0; g < d.ngroups; ++g) {
    int fill[4] = {0, 0, 0, 0};
    for (int t = 0; t < d.ntaps; ++t) {
      const TapF& tp = d.taps[g][t];
      const int slot = p.src_begin[tp.map] + fill[tp.map]++;
      if (slot >= p.src_begin[tp.map + 1]) return 1;  // groups disagree on taps per source
      p.tap_off16[g][slot] = (uint32_t)(((tp.dy - p.org_y[tp.map]) * p.pitch + (tp.dx - p.org_x[tp.map])) * row_b) >> 4;
      p.tap_kblk[g][slot] = t;
    }
  }
  p.box_bytes = p.pitch * p.ph * row_b;
  p.a_box_bytes = (p.box_bytes + 1023) & ~1023;
  p.tiles_x = (d.Wg + kTileW - 1) / kTileW;
  p.tiles_y = (d.Hg + kTileH - 1) / kTileH;
  p.magic_img = (uint32_t)((0x100000000ULL + (unsigned)(p.tiles_x * p.tiles_y) - 1) / (unsigned)(p.tiles_x * p.tiles_y));
  p.magic_x = (uint32_t)((0x100000000ULL + (unsigned)p.tiles_x - 1) / (unsigned)p.tiles_x);
  p.B = d.B;
  p.Wo = d.Wg;
  p.Ho = d.Hg;
  p.N = d.N;
  for (int g = 0; g < 4; ++g) p.out_off[g] = d.out_off[g];
  p.sb = d.osb;
  p.sy = d.osy;
  p.sx = d.osx;
  p.out = d.out;
  p.stats = d.stats;
  p.stats_bg = d.stats_bg;
  p.act = d.act;
  p.bias9 = d.bias9;
  p.epi_src = d.epi_src;
  p.epi_mode = d.epi_mode;
  {
    const char* e = getenv("SG2_TILE_DBG");
    p.dbg = e ? atoi(e) : 0;
    if (p.dbg & 64) {
      static long long* buf = nullptr;
      if (!buf) cudaMalloc(&buf, 1024 * 16 * sizeof(long long));
      p.dbg_out = buf;
      g_tile_dbg = buf;
    }
  }
  const int pix_tiles = p.tiles_x * p.tiles_y * p.B;
  const int bn0 = (d.N == 160 || d.N == 192)
                      ? d.N
                      : ((d.N % 256 == 0) ? 256
                                          : ((d.N % 128 == 0) ? 128 : ((d.N % 64 == 0) ? 64 : ((d.N % 32 == 0) ? 32 : 16))));
  const int budget = 200 * 1024;
  const int taps_src = d.ntaps / d.nmaps;
  int bn = bn0, b_total;
  int b_all = d.ntaps * d.Cin * bn0 * 2;
  // A weight slice that does not fit at the natural N tile but fits at half of it (e.g. conv4x4-s2 64 -> 128: 262 KB vs
  // 131 KB): the ring mode re-streams the whole slice for every pixel-tile unit (420 KB of TMA per unit against ~8k
  // cycles of MMAs: L2 -> SMEM bound), the half-width resident form loads it once per CTA. Off by default (SG2_RES_HALF=1).
  static const int res_half = [] {
    const char* e = getenv("SG2_RES_HALF");
    return e ? atoi(e) : 0;   // measured (r02): 8.09 ms/step with, 7.96 without — N = 64 MMAs run at the 45-cycle floor
  }();
  if (res_half && b_all + 2 * p.a_box_bytes > budget && bn0 >= 128 && (bn0 % 2) == 0 && d.N % (bn0 / 2) == 0 &&
      b_all / 2 + 2 * p.a_box_bytes <= budget) {
    bn = bn0 / 2;
    b_all /= 2;
  }
  if (b_all + 2 * p.a_box_bytes <= budget && tile_mode() != 2) {
    p.b_resident = 1;  // weight-stationary: this CTA's weight slice is loaded once
    p.mt = 1;
    p.tps = taps_src;
    p.stages = 1;
    p.na = (budget - b_all) / p.a_box_bytes;
    b_total = b_all;
  } else {
    p.b_resident = 0;
    p.mt = 1;
    if (tile_mode() != 3) {
      // two pixel tiles per unit halve the weight bytes per MMA; needs 2 x 2 x BN TMEM columns and enough units per CTA
      const int bn2 = (d.N % 128 == 0) ? 128 : (d.N == 192 ? 96 : (d.N == 160 ? 80 : (bn0 <= 128 ? bn0 : 0)));
      if (bn2) {
        const int combos2 = d.ngroups * (d.N / bn2);
        int lanes2 = num_sms() / combos2;
        lanes2 = lanes2 < 1 ? 1 : lanes2;
        if ((pix_tiles + 1) / 2 >= 2 * lanes2) {
          p.mt = 2;
          bn = bn2;
        }
      }
    }
    const int kb = bn * row_b;
    int tps = 1;
    for (int c = 1; c <= taps_src; ++c)
      if (taps_src % c == 0 && c * kb <= 16 * 1024) tps = c;
    p.tps = tps;
    p.na = 2;
    int stages = (budget - p.na * p.mt * p.a_box_bytes) / (tps * kb);
    if (stages < 3) return 1;
    p.stages = stages > 16 ? 16 : stages;
    b_total = p.stages * tps * kb;
    if (p.stages >= 5 && budget - p.na * p.mt * p.a_box_bytes - b_total >= p.mt * p.a_box_bytes) p.na = 3;
  }
  if (p.na > 4) p.na = 4;
  for (int i = 0; i < taps_src; ++i) {
    if (i % p.tps == 0) p.stage_start_mask |= 1u << i;
    if ((i + 1) % p.tps == 0) p.stage_end_mask |= 1u << i;
  }
  p.n_tiles = d.N / bn;
  const int combos = p.ngroups * p.n_tiles;
  const int units = (pix_tiles + p.mt - 1) / p.mt;
  int lanes = num_sms() / combos;
  if (lanes < 1) lanes = 1;
  if (lanes > units) lanes = units;
  p.lanes = lanes;
  pl.bn = bn;
  pl.bk = bk;
  pl.smem = size_t(p.na) * p.mt * p.a_box_bytes + b_total + 1024 + 512;
  return 0;
}

template <int BN, int BK, int NT>
static int launch_tile_t(const GatherDesc& d, TilePlan& pl, cudaStream_t st) {
  TileParams& p = pl.p;
  int rc;
  for (int s = 0; s < d.nmaps; ++s)
    if ((rc = make_act_map(&p.tmA[s], d.a[s], BK, p.pitch, p.ph, 1))) return rc;
  if ((rc = make_w_map(&p.tmB, d.w, (long long)d.ngroups * d.N, (long long)d.ntaps * d.Cin, BK, BN))) return rc;
  static bool attr_done[64] = {};
  if (attr_needed(attr_done)) {
    cudaError_t e = cudaFuncSetAttribute(tile_conv_kernel<BN, BK, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 212 * 1024);
    if (e != cudaSuccess) SG2_FAIL((int)e, "cudaFuncSetAttribute(tile_conv<%d,%d>): %s", BN, BK, cudaGetErrorString(e));
  }
  tile_conv_kernel<BN, BK, NT><<<dim3(p.ngroups * p.n_tiles * p.lanes), kTileThreads, pl.smem, st>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) SG2_FAIL((int)e, "tile_conv<%d,%d> launch: %s", BN, BK, cudaGetErrorString(e));
  return 0;
}

// Returns 1 when the layer should run on the gather kernel instead.
static int launch_tile(const GatherDesc& d, cudaStream_t st) {
  TilePlan pl;
  int rc = plan_tile(d, pl);
  if (rc) return rc;
  const int bn = pl.bn, bk = pl.bk;
  const int nt = d.ntaps / d.nmaps;
  if (nt == 1 && bn == 64 && bk == 64) return launch_tile_t<64, 64, 1>(d, pl, st);   // 64 -> 64 GEMM tiles (D stems)
  if (nt != 4 && nt != 9) return 1;
#define SG2_CASE(BN_, BK_)                                                   \
  if (bn == BN_ && bk == BK_)                                                \
    return nt == 9 ? launch_tile_t<BN_, BK_, 9>(d, pl, st) : launch_tile_t<BN_, BK_, 4>(d, pl, st);
  SG2_CASE(256, 64) SG2_CASE(128, 64) SG2_CASE(64, 64) SG2_CASE(32, 64) SG2_CASE(16, 64)
  SG2_CASE(256, 32) SG2_CASE(128, 32) SG2_CASE(64, 32) SG2_CASE(32, 32) SG2_CASE(16, 32)
  SG2_CASE(256, 16) SG2_CASE(128, 16) SG2_CASE(64, 16) SG2_CASE(32, 16) SG2_CASE(16, 16)
  SG2_CASE(160, 64) SG2_CASE(160, 32) SG2_CASE(192, 64) SG2_CASE(192, 32)
  SG2_CASE(96, 64) SG2_CASE(96, 32) SG2_CASE(80, 64) SG2_CASE(80, 32)
#undef SG2_CASE
  return 1;
}

// pixel tiles (128 GEMM rows each) of a gather launch
static int gather_tiles(const GatherDesc& d) {
  int tw, th, nb;
  if (pick_tile(d.Wg, d.Hg, kBlockM, &tw, &th, &nb)) return 0;
  return ((d.Wg + tw - 1) / tw) * ((d.Hg + th - 1) / th) * ((d.B + nb - 1) / nb);
}

// the plain gather kernel (one 128 x bn tile per CTA)
static int launch_fprop_plain(const GatherDesc& d, int bn, int bk, cudaStream_t st) {
#define SG2_CASE(BN_, BK_) \
  if (bn == BN_ && bk == BK_) return launch_fprop_t<BN_, BK_>(d, st);
  SG2_CASE(256, 64) SG2_CASE(128, 64) SG2_CASE(64, 64) SG2_CASE(32, 64)
  SG2_CASE(256, 32) SG2_CASE(128, 32) SG2_CASE(64, 32) SG2_CASE(32, 32)
  SG2_CASE(256, 16) SG2_CASE(128, 16) SG2_CASE(64, 16) SG2_CASE(32, 16)
  SG2_CASE(16, 64) SG2_CASE(16, 32) SG2_CASE(16, 16)
  SG2_CASE(160, 64) SG2_CASE(160, 32) SG2_CASE(192, 64) SG2_CASE(192, 32)
#undef SG2_CASE
  SG2_FAIL(SG2_EINVAL, "no fprop instance for BN=%d BK=%d", bn, bk);
}

static int launch_fprop(const GatherDesc& d, cudaStream_t st) {
  if (d.Cin % 16) SG2_FAIL(SG2_EINVAL, "K per tap (%d) must be a multiple of 16", d.Cin);
  if (d.N % 16) SG2_FAIL(SG2_EINVAL, "N (%d) must be a multiple of 16", d.N);
  const int bk = (d.Cin % 64 == 0) ? 64 : ((d.Cin % 32 == 0) ? 32 : 16);
  const int bn = (d.N == 160 || d.N == 192)
                     ? d.N
                     : ((d.N % 256 == 0) ? 256
                                         : ((d.N % 128 == 0) ? 128 : ((d.N % 64 == 0) ? 64 : ((d.N % 32 == 0) ? 32 : 16))));
  if (tile_eligible(d)) {
    const int rc = launch_tile(d, st);
    if (rc != 1) return rc;
  }
  if (d.bias9) SG2_FAIL(SG2_EINVAL, "conv_fprop: the region bias needs a tile-resident shape (Cin %d, N %d)", d.Cin, d.N);
  if (d.out_mode == OUT_BF16 && bk == 64 && bn == 256 && d.splitk <= 4 && igemm_pair() && gather_tiles(d) >= 2) {
    // CTA pairs (half of the weight tile per SM) unless the phantom tile of an odd tile count costs an extra wave
    const int tiles = gather_tiles(d), sk = d.splitk < 1 ? 1 : d.splitk;
    const long long per = (long long)(d.N / 256) * d.ngroups * sk;
    const long long cap = (long long)num_sms() * (sk == 1 ? 2 : 1);   // CTAs that run at once (ring-only kernels: two per SM)
    const long long w_plain = (tiles * per + cap - 1) / cap, w_pair = (2 * ((tiles + 1) / 2) * per + cap - 1) / cap;
    if (w_pair <= w_plain) return sk == 1 ? launch_fprop_pair_t<256, 64, true>(d, st) : launch_fprop_pair_t<256, 64, false>(d, st);
  }
  if (d.out_mode == OUT_BF16 && d.splitk > 1) {   // split-K with an in-cluster reduction (bf16 out, statistics, epilogue operand)
    if (bk == 64 && bn == 256 && igemm_mt2() && gather_tiles(d) >= 2) return launch_fprop_cluster_t<256, 64, 2>(d, st);
    if (bk == 64 && bn == 256) return launch_fprop_cluster_t<256, 64>(d, st);
    if (bk == 64 && bn == 128) return launch_fprop_cluster_t<128, 64>(d, st);
    if (bk == 64 && bn == 64) return launch_fprop_cluster_t<64, 64>(d, st);
    SG2_FAIL(SG2_ENOFUSE, "cluster split-K: no instance for BN=%d BK=%d", bn, bk);
  }
  if (d.epi_mode) SG2_FAIL(SG2_ENOFUSE, "epilogue operand: this shape runs on the gather kernel (K %d, N %d)", d.Cin, d.N);
  if (bn == 256 && bk == 64 && igemm_mt2() && gather_tiles(d) >= 2) return launch_fprop_t<256, 64, 2>(d, st);
  return launch_fprop_plain(d, bn, bk, st);
}

static inline int fdiv2(int v) { return v >= 0 ? v / 2 : -((-v + 1) / 2); }  // floor(v/2)

// ------------------------------------------------------------------------------------------ wgrad launch
struct WgradDesc {
  View a[4], b[4];
  int namaps, nbmaps;
  JobW jobs[16];
  int njobs;
  int Wg, Hg, B;  // pixel grid of the dy views
  int Cout, Cin;
  float* dw;
  int splitk;
  int lane_cap;     // tile kernel: upper bound on the CTA lanes per output block (0: fill the SMs)
  float* partials;  // deterministic mode: per-split / per-lane slabs (each laid out like dw), summed by the caller
  int* slabs_out;   // plan only: receives the number of slabs this launch would write; nothing is launched
};

template <int BN, int CWA, int CWB>
static int launch_wgrad_t(const WgradDesc& d, cudaStream_t st) {
  using Cfg = WgradCfg<BN, CWA, CWB>;
  WgradParams p;
  memset(&p, 0, sizeof(p));
  int rc;
  if ((rc = pick_tile(d.Wg, d.Hg, kWgradBKP, &p.tw, &p.th, &p.nb))) return rc;
  if (d.slabs_out) {
    const int pt = ((d.Wg + p.tw - 1) / p.tw) * ((d.Hg + p.th - 1) / p.th) * ((d.B + p.nb - 1) / p.nb);
    *d.slabs_out = d.splitk < 1 ? 1 : (d.splitk > pt ? pt : d.splitk);
    return 0;
  }
  for (int i = 0; i < d.namaps; ++i)
    if ((rc = make_act_map(&p.tmA[i], d.a[i], CWA, p.tw, p.th, p.nb))) return rc;
  for (int i = 0; i < d.nbmaps; ++i)
    if ((rc = make_act_map(&p.tmB[i], d.b[i], CWB, p.tw, p.th, p.nb))) return rc;
  memcpy(p.jobs, d.jobs, sizeof(p.jobs));
  p.njobs = d.njobs;
  p.tiles_x = (d.Wg + p.tw - 1) / p.tw;
  p.tiles_y = (d.Hg + p.th - 1) / p.th;
  p.tiles_b = (d.B + p.nb - 1) / p.nb;
  const int PT = p.tiles_x * p.tiles_y * p.tiles_b;
  p.splitk = d.splitk < 1 ? 1 : (d.splitk > PT ? PT : d.splitk);
  p.Cout = d.Cout;
  p.Cin = d.Cin;
  p.dw = d.dw;
  p.partials = d.partials;
  p.slab = (long long)d.Cout * d.njobs * d.Cin;
  const int smax = max_stages(Cfg::kStageBytes);
  int stages = smax;
  if (stages > PT / p.splitk + 1) stages = PT / p.splitk + 1;
  if (stages < 2) stages = 2;
  p.stages = stages;
  static bool attr_done[64] = {};
  if (attr_needed(attr_done)) {
    cudaError_t e = cudaFuncSetAttribute(igemm_wgrad_kernel<BN, CWA, CWB>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::smem_bytes(smax));
    if (e != cudaSuccess) SG2_FAIL((int)e, "cudaFuncSetAttribute(wgrad): %s", cudaGetErrorString(e));
  }
  const int m_tiles = (d.Cout + kBlockM - 1) / kBlockM, n_tiles = (d.Cin + BN - 1) / BN;
  dim3 grid(m_tiles * n_tiles, d.njobs, p.splitk);
  igemm_wgrad_kernel<BN, CWA, CWB><<<grid, kNumThreads, Cfg::smem_bytes(stages), st>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) SG2_FAIL((int)e, "wgrad<%d,%d,%d> launch: %s", BN, CWA, CWB, cudaGetErrorString(e));
  return 0;
}

// ------------------------------------------------------------------------------------------ tile-resident wgrad
static int tile_wgrad_mode() {
  static int m = [] {
    const char* e = getenv("SG2_TILE_WGRAD");
    return e ? atoi(e) : 1;
  }();
  return m;
}

// Returns 1 when the layer should run on the gather-form wgrad kernel instead.
static int launch_tile_wgrad(const WgradDesc& d, cudaStream_t st) {
  if (!tile_wgrad_mode() || d.Wg < kTileW || d.Hg < kTileH) return 1;
  TileWgradParams p;
  memset(&p, 0, sizeof(p));
  // ---- groups = distinct (dy source, x source) pairs; taps of a group = its jobs in order
  int gcount[4] = {0, 0, 0, 0};
  int mny[4], mxy[4], mnx[4], mxx[4];
  for (int s = 0; s < 4; ++s) mny[s] = mnx[s] = 127, mxy[s] = mxx[s] = -127;
  for (int j = 0; j < d.njobs; ++j) {
    const JobW& jb = d.jobs[j];
    mny[jb.bmap] = jb.dy < mny[jb.bmap] ? jb.dy : mny[jb.bmap];
    mxy[jb.bmap] = jb.dy > mxy[jb.bmap] ? jb.dy : mxy[jb.bmap];
    mnx[jb.bmap] = jb.dx < mnx[jb.bmap] ? jb.dx : mnx[jb.bmap];
    mxx[jb.bmap] = jb.dx > mxx[jb.bmap] ? jb.dx : mxx[jb.bmap];
  }
  int ex = 0, ey = 0;
  for (int s = 0; s < d.nbmaps; ++s) {
    if (mny[s] > mxy[s]) return 1;
    ex = (mxx[s] - mnx[s]) > ex ? (mxx[s] - mnx[s]) : ex;
    ey = (mxy[s] - mny[s]) > ey ? (mxy[s] - mny[s]) : ey;
    p.org_x[s] = mnx[s];
    p.org_y[s] = mny[s];
  }
  p.pitch = kTileW + ex;
  p.ph = kTileH + ey;
  // Small pixel grids with wide channels amortise neither the pipeline ramp nor the 128 x (taps x BN) fp32 epilogue.
  if (d.Cout > 128 && (long long)d.B * d.Wg * d.Hg < 128LL * 16 * num_sms()) return 1;
  // Cin tile = UMMA N: pick the candidate with the least tensor time per pixel tile; an MMA of N columns costs
  // max(N/2, 32 + N/4) cycles (tensor floor vs. the SMEM read of its 128-row dy operand), times taps x Cin/N of them.
  int bn = 0;
  long long best = -1;
  const int cands[] = {256, 192, 160, 128, 96, 64, 32, 16};
  for (int c : cands) {
    if (c > d.Cin || d.Cin % c) continue;
    const int floor_c = c / 2 > 32 + c / 4 ? c / 2 : 32 + c / 4;
    int tc = 1;
    for (int k = 1; k <= 16 && k <= 512 / c; ++k) tc = k;   // taps per CTA cap (refined below)
    const long long cost = (long long)(d.Cin / c) * floor_c + (tc < 3 ? 100000 : 0);  // < 3 taps per CTA reloads dy too often
    if (best < 0 || cost < best) best = cost, bn = c;
  }
  if (!bn) return 1;
  const int cwb = bn % 64 == 0 ? 64 : (bn % 32 == 0 ? 32 : 16);
  const int co_tile = d.Cout < kBlockM ? d.Cout : kBlockM;
  const int cwa = co_tile % 64 == 0 ? 64 : (co_tile % 32 == 0 ? 32 : (co_tile % 16 == 0 ? 16 : 0));
  if (!cwa) return 1;
  const int row_b = cwb * 2;
  for (int j = 0; j < d.njobs; ++j) {
    const JobW& jb = d.jobs[j];
    int g = -1;
    for (int k = 0; k < p.ngroups; ++k)
      if (p.a_src[k] == jb.amap && p.b_src[k] == jb.bmap) g = k;
    if (g < 0) {
      if (p.ngroups == 4) return 1;
      g = p.ngroups++;
      p.a_src[g] = jb.amap;
      p.b_src[g] = jb.bmap;
    }
    const int t = gcount[g]++;
    if (t >= 16) return 1;
    p.tap_off16[g][t] = (uint32_t)(((jb.dy - p.org_y[jb.bmap]) * p.pitch + (jb.dx - p.org_x[jb.bmap])) * row_b) >> 4;
    p.tap_job[g][t] = j;
  }
  for (int g = 1; g < p.ngroups; ++g)
    if (gcount[g] != gcount[0]) return 1;
  p.ntaps = gcount[0];
  const int cap = 512 / bn;
  int taps_cta = 1;
  for (int c = 1; c <= p.ntaps && c <= cap; ++c)
    if (p.ntaps % c == 0) taps_cta = c;
  p.taps_cta = taps_cta;
  p.tap_sets = p.ntaps / taps_cta;
  p.njobs = d.njobs;
  p.cwa = cwa;
  p.cwb = cwb;
  p.a_chunks = co_tile / cwa;
  p.b_chunks = bn / cwb;
  p.a_box_bytes = kTileW * kTileH * cwa * 2;
  p.a_chunk_bytes = p.a_box_bytes;  // 128 rows x >= 32 B: already a multiple of 1024
  p.b_box_bytes = p.pitch * p.ph * row_b;
  p.b_chunk_bytes = (p.b_box_bytes + 1023) & ~1023;
  p.bn = bn;
  p.m_tiles = (d.Cout + kBlockM - 1) / kBlockM;
  p.n_tiles = d.Cin / bn;
  p.tiles_x = (d.Wg + kTileW - 1) / kTileW;
  p.tiles_y = (d.Hg + kTileH - 1) / kTileH;
  p.B = d.B;
  p.magic_img = (uint32_t)((0x100000000ULL + (unsigned)(p.tiles_x * p.tiles_y) - 1) / (unsigned)(p.tiles_x * p.tiles_y));
  p.magic_x = (uint32_t)((0x100000000ULL + (unsigned)p.tiles_x - 1) / (unsigned)p.tiles_x);
  p.Cout = d.Cout;
  p.Cin = d.Cin;
  p.dw = d.dw;
  const int pix_tiles = p.tiles_x * p.tiles_y * p.B;
  const int base = p.ngroups * p.tap_sets * p.m_tiles * p.n_tiles;
  int lanes = (num_sms() + base - 1) / base;
  if (lanes > pix_tiles) lanes = pix_tiles;
  if (d.lane_cap > 0 && lanes > d.lane_cap) lanes = d.lane_cap;   // fewer CTA lanes = fewer partial slabs to reduce
  if (lanes < 1) lanes = 1;
  p.lanes = lanes;
  p.partials = d.partials;
  p.slab = (long long)d.Cout * d.njobs * d.Cin;
  const int stage_bytes = (kBlockM / cwa) * p.a_chunk_bytes + p.b_chunks * p.b_chunk_bytes;
  int stages = (200 * 1024) / stage_bytes;
  if (stages < 2) return 1;
  if (d.slabs_out) {
    *d.slabs_out = lanes;
    return 0;
  }
  if (stages > 4) stages = 4;
  p.stages = stages;
  {
    static int merge_on = [] {
      const char* e = getenv("SG2_WGRAD_MERGE");
      return e ? atoi(e) : 1;
    }();
    bool ok = merge_on && p.ntaps == 9 && p.b_chunks == 1 && taps_cta % 3 == 0 && 3 * bn <= 256;
    const uint32_t px16 = (uint32_t)row_b >> 4;
    for (int g = 0; ok && g < p.ngroups; ++g)
      for (int r = 0; r < 3; ++r)
        ok = ok && p.tap_off16[g][3 * r + 1] == p.tap_off16[g][3 * r] + px16 &&
             p.tap_off16[g][3 * r + 2] == p.tap_off16[g][3 * r] + 2 * px16;
    p.merge3 = ok ? 1 : 0;
  }
  int rc;
  for (int i = 0; i < d.namaps; ++i)
    if ((rc = make_act_map(&p.tmA[i], d.a[i], cwa, kTileW, kTileH, 1))) return rc;
  for (int i = 0; i < d.nbmaps; ++i)
    if ((rc = make_act_map(&p.tmB[i], d.b[i], cwb, p.pitch, p.ph, 1))) return rc;
  static bool attr_done[64] = {};
  if (attr_needed(attr_done)) {
    cudaError_t e = cudaFuncSetAttribute(tile_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 212 * 1024);
    if (e != cudaSuccess) SG2_FAIL((int)e, "cudaFuncSetAttribute(tile_wgrad): %s", cudaGetErrorString(e));
  }
  const size_t smem = size_t(stages) * stage_bytes + 1024 + 256;
  tile_wgrad_kernel<<<dim3(base * lanes), kNumThreads, smem, st>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) SG2_FAIL((int)e, "tile_wgrad launch: %s", cudaGetErrorString(e));
  return 0;
}

// igemm_wgrad_kernel<256, 64, 64> on CTA pairs (igemm_pair.cuh): 256 x 256 channels per pair, half of the activation tile per SM
static int launch_wgrad_pair(const WgradDesc& d, cudaStream_t st) {
  using Cfg = WgradPairCfg;
  WgradParams p;
  memset(&p, 0, sizeof(p));
  int rc;
  if ((rc = pick_tile(d.Wg, d.Hg, kWgradBKP, &p.tw, &p.th, &p.nb))) return rc;
  if (d.slabs_out) {
    const int pt = ((d.Wg + p.tw - 1) / p.tw) * ((d.Hg + p.th - 1) / p.th) * ((d.B + p.nb - 1) / p.nb);
    *d.slabs_out = d.splitk < 1 ? 1 : (d.splitk > pt ? pt : d.splitk);
    return 0;
  }
  for (int i = 0; i < d.namaps; ++i)
    if ((rc = make_act_map(&p.tmA[i], d.a[i], Cfg::kCW, p.tw, p.th, p.nb))) return rc;
  for (int i = 0; i < d.nbmaps; ++i)
    if ((rc = make_act_map(&p.tmB[i], d.b[i], Cfg::kCW, p.tw, p.th, p.nb))) return rc;
  memcpy(p.jobs, d.jobs, sizeof(p.jobs));
  p.njobs = d.njobs;
  p.tiles_x = (d.Wg + p.tw - 1) / p.tw;
  p.tiles_y = (d.Hg + p.th - 1) / p.th;
  p.tiles_b = (d.B + p.nb - 1) / p.nb;
  const int PT = p.tiles_x * p.tiles_y * p.tiles_b;
  p.splitk = d.splitk < 1 ? 1 : (d.splitk > PT ? PT : d.splitk);
  p.Cout = d.Cout;
  p.Cin = d.Cin;
  p.dw = d.dw;
  p.partials = d.partials;
  p.slab = (long long)d.Cout * d.njobs * d.Cin;
  int stages = Cfg::kStages;
  if (stages > PT / p.splitk + 1) stages = PT / p.splitk + 1;
  if (stages < 2) stages = 2;
  p.stages = stages;
  static bool attr_done[64] = {};
  if (attr_needed(attr_done)) {
    cudaError_t e = cudaFuncSetAttribute(igemm_wgrad_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)pair_exclusive_smem(Cfg::smem_bytes(Cfg::kStages)));
    if (e != cudaSuccess) SG2_FAIL((int)e, "cudaFuncSetAttribute(wgrad_pair): %s", cudaGetErrorString(e));
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((d.Cout / kBlockM) * (d.Cin / Cfg::kBN), d.njobs, p.splitk);
  cfg.blockDim = dim3(kNumThreads);
  cfg.dynamicSmemBytes = pair_exclusive_smem(Cfg::smem_bytes(stages));
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, igemm_wgrad_pair_kernel, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    SG2_FAIL((int)e, "wgrad_pair launch: %s", cudaGetErrorString(e));
  }
  return 0;
}

static int launch_wgrad(const WgradDesc& d, cudaStream_t st) {
  {
    const int rc = launch_tile_wgrad(d, st);
    if (rc != 1) return rc;
  }
  if (d.Cout % 32 || d.Cin % 16) SG2_FAIL(SG2_EINVAL, "wgrad needs Cout %% 32 == 0 and Cin %% 16 == 0 (%d, %d)", d.Cout, d.Cin);
  const int cwa = (d.Cout % 64 == 0) ? 64 : 32;
  const int cwb = (d.Cin % 64 == 0) ? 64 : ((d.Cin % 32 == 0) ? 32 : 16);
  const int bn = d.Cin <= 16 ? 16 : (d.Cin <= 32 ? 32 : (d.Cin <= 64 ? 64 : (d.Cin <= 128 ? 128 : 256)));
  if (igemm_pair_wgrad() && d.Cout % 256 == 0 && d.Cin % 256 == 0) return launch_wgrad_pair(d, st);
#define SG2_CASE(BN_, A_, B_) \
  if (bn == BN_ && cwa == A_ && cwb == B_) return launch_wgrad_t<BN_, A_, B_>(d, st);
  SG2_CASE(256, 64, 64) SG2_CASE(128, 64, 64) SG2_CASE(64, 64, 64)
  SG2_CASE(256, 64, 32) SG2_CASE(128, 64, 32) SG2_CASE(64, 64, 32) SG2_CASE(32, 64, 32)
  SG2_CASE(256, 32, 64) SG2_CASE(128, 32, 64) SG2_CASE(64, 32, 64)
  SG2_CASE(256, 32, 32) SG2_CASE(128, 32, 32) SG2_CASE(64, 32, 32) SG2_CASE(32, 32, 32)
  SG2_CASE(16, 64, 16) SG2_CASE(16, 32, 16)
#undef SG2_CASE
  SG2_FAIL(SG2_EINVAL, "no wgrad instance for BN=%d CWA=%d CWB=%d", bn, cwa, cwb);
}

// kh of the 4x4-s2 filter that connects input parity p (row 2i+p) with output row i + d:  see dgrad below.
static const int kS2_kh[2][2] = {{1, 3}, {2, 0}};   // [parity][a]
static const int kS2_dy[2][2] = {{0, -1}, {0, 1}};  // [parity][a] : output row = i + dy

// ------------------------------------------------------------------------------------------ general convolution
// sg2_conv2d_fprop: kh x kw, stride 1 or 2, zero padding, bias + ReLU, channel slices in and out, on the plain gather
// kernel. The pixel tile is the rectangle of at most 128 output pixels that covers the map in the fewest tiles: a partial
// TMA box fills tw*th*nb rows of the 128-row operand, the rest of the MMA rows are issued but never stored. A stride-1
// 1x1 convolution walks the pixels of the whole batch as one row (no waste but the last tile's tail).
struct Conv2dGeo {
  int Ho, Wo, flat, tw, th, nb, bn, bk;
  long long tiles;
};

// output tile width: the smallest gather instance that covers N (weight rows past N are TMA zero fill), else the
// instance with the least padded width
static int conv2d_bn(int N, int bk) {
  static const int wide[] = {16, 32, 64, 128, 160, 192, 256};
  static const int narrow[] = {16, 32, 64, 128, 256};   // BK = 16 has no 160 / 192 instances
  const int* c = bk == 16 ? narrow : wide;
  const int nc = bk == 16 ? 5 : 7;
  for (int i = 0; i < nc; ++i)
    if (c[i] >= N) return c[i];
  int best = 256;
  for (int i = nc - 1; i >= 0 && c[i] >= 128; --i)
    if ((long long)((N + c[i] - 1) / c[i]) * c[i] < (long long)((N + best - 1) / best) * best) best = c[i];
  return best;
}

static int conv2d_geo(int B, int H, int W, int Cin, int Cout, int kh, int kw, int stride, int ph, int pw, Conv2dGeo& g) {
  if (B < 1 || H < 1 || W < 1) SG2_FAIL(SG2_EINVAL, "conv2d: empty input %dx%dx%d", B, H, W);
  if (Cin < 16 || Cin % 16) SG2_FAIL(SG2_EINVAL, "conv2d: Cin %d must be a multiple of 16", Cin);
  if (Cout < 8 || Cout % 8) SG2_FAIL(SG2_EINVAL, "conv2d: Cout %d must be a multiple of 8", Cout);
  if (stride != 1 && stride != 2) SG2_FAIL(SG2_EINVAL, "conv2d: stride %d (1 or 2)", stride);
  if (kh < 1 || kw < 1 || kh * kw > kMaxTaps) SG2_FAIL(SG2_EINVAL, "conv2d: %dx%d kernel (at most %d taps)", kh, kw, kMaxTaps);
  if (ph < 0 || pw < 0 || ph >= kh || pw >= kw) SG2_FAIL(SG2_EINVAL, "conv2d: padding (%d, %d) for a %dx%d kernel", ph, pw, kh, kw);
  if (stride == 2 && (H < 2 || W < 2)) SG2_FAIL(SG2_EINVAL, "conv2d: stride 2 on a %dx%d map", H, W);
  g.Ho = (H + 2 * ph - kh) / stride + 1;
  g.Wo = (W + 2 * pw - kw) / stride + 1;
  if (H + 2 * ph < kh || W + 2 * pw < kw) SG2_FAIL(SG2_EINVAL, "conv2d: %dx%d kernel larger than the padded map", kh, kw);
  g.bk = (Cin % 64 == 0) ? 64 : ((Cin % 32 == 0) ? 32 : 16);
  g.bn = conv2d_bn(Cout, g.bk);
  g.flat = kh == 1 && kw == 1 && stride == 1;
  if (g.flat) {
    const long long P = (long long)B * H * W;
    if (P > 0x7fffffffLL) SG2_FAIL(SG2_EINVAL, "conv2d: %lld pixels", P);
    g.tw = P < kBlockM ? (int)P : kBlockM, g.th = 1, g.nb = 1;
    g.tiles = (P + g.tw - 1) / g.tw;
    return 0;
  }
  if (g.Ho * g.Wo <= kBlockM) {
    g.tw = g.Wo, g.th = g.Ho;
    g.nb = kBlockM / (g.Ho * g.Wo);
    if (g.nb > B) g.nb = B;
  } else {
    long long best = -1;
    for (int tw = 1; tw <= (g.Wo < kBlockM ? g.Wo : kBlockM); ++tw) {
      int th = kBlockM / tw;
      if (th > g.Ho) th = g.Ho;
      const long long t = (long long)((g.Wo + tw - 1) / tw) * ((g.Ho + th - 1) / th);
      if (best < 0 || t <= best) best = t, g.tw = tw, g.th = th;   // ties: the wider tile
    }
    g.nb = 1;
  }
  g.tiles = (long long)((g.Wo + g.tw - 1) / g.tw) * ((g.Ho + g.th - 1) / g.th) * ((B + g.nb - 1) / g.nb);
  return 0;
}

}  // namespace sg2

using namespace sg2;

extern "C" {

int sg2_conv2d_plan(int B, int H, int W, int Cin, int Cout, int kh, int kw, int stride, int ph, int pw,
                    long long* out) {
  Conv2dGeo g;
  const int rc = conv2d_geo(B, H, W, Cin, Cout, kh, kw, stride, ph, pw, g);
  if (rc) return rc;
  const long long v[8] = {g.tiles * kBlockM, (long long)B * g.Ho * g.Wo, (long long)((Cout + g.bn - 1) / g.bn) * g.bn,
                          g.bn, g.bk, g.tw, g.th, g.nb};
  memcpy(out, v, sizeof(v));
  return 0;
}

int sg2_conv2d_fprop(const void* x, int x_ctot, const void* wpk, const float* bias, void* y, int y_ctot, int B, int H,
                     int W, int Cin, int Cout, int kh, int kw, int stride, int ph, int pw, int relu, void* stream) {
  Conv2dGeo g;
  int rc = conv2d_geo(B, H, W, Cin, Cout, kh, kw, stride, ph, pw, g);
  if (rc) return rc;
  if (x_ctot < Cin || (x_ctot % 8) || y_ctot < Cout || (y_ctot % 8))
    SG2_FAIL(SG2_EINVAL, "conv2d: channel strides %d / %d (multiples of 8, >= Cin %d / Cout %d)", x_ctot, y_ctot, Cin, Cout);
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(wpk)) & 15)
    SG2_FAIL(SG2_EINVAL, "conv2d: operands must be 16-byte aligned");
  if (relu != 0 && relu != 1) SG2_FAIL(SG2_EINVAL, "conv2d: relu %d", relu);
  GatherDesc d;
  memset(&d, 0, sizeof(d));
  d.Cin = Cin;
  d.w = wpk;
  d.N = Cout;
  d.out = y;
  d.out_mode = OUT_BF16;
  d.splitk = 1;
  d.bias = bias;
  d.act = relu ? 3 : 0;
  d.ngroups = 1;
  d.tw = g.tw, d.th = g.th, d.nb = g.nb;
  const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(x);
  if (g.flat) {
    const int P = B * H * W;
    d.a[0] = View{xb, Cin, P, 1, 1, (long long)x_ctot, (long long)P * x_ctot, (long long)P * x_ctot};
    d.nmaps = 1;
    d.ntaps = 1;
    d.taps[0][0] = TapF{0, 0, 0, 0};
    d.Wg = P, d.Hg = 1, d.B = 1;
    d.osx = y_ctot, d.osy = (long long)P * y_ctot, d.osb = d.osy;
  } else {
    const View xv{xb, Cin, W, H, B, (long long)x_ctot, (long long)W * x_ctot, (long long)H * W * x_ctot};
    if (stride == 1) {
      d.a[0] = xv;
      d.nmaps = 1;
    } else {   // parity plane (py, px): input pixels (2i + py, 2j + px)
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) {
          View v = xv;
          v.base = xv.base + py * xv.sy + px * xv.sx;
          v.H = (H - py + 1) / 2, v.W = (W - px + 1) / 2;
          v.sy = 2 * xv.sy, v.sx = 2 * xv.sx;
          d.a[py * 2 + px] = v;
        }
      d.nmaps = 4;
    }
    d.ntaps = kh * kw;
    for (int ky = 0; ky < kh; ++ky)
      for (int kx = 0; kx < kw; ++kx) {
        const int ry = ky - ph, rx = kx - pw;   // input row = stride * oy + ry
        d.taps[0][ky * kw + kx] = stride == 1 ? TapF{0, (int8_t)ry, (int8_t)rx, 0}
                                              : TapF{(int8_t)((ry & 1) * 2 + (rx & 1)), (int8_t)fdiv2(ry), (int8_t)fdiv2(rx), 0};
      }
    d.Wg = g.Wo, d.Hg = g.Ho, d.B = B;
    d.osx = y_ctot, d.osy = (long long)g.Wo * y_ctot, d.osb = (long long)g.Ho * g.Wo * y_ctot;
  }
  return launch_fprop_plain(d, g.bn, g.bk, (cudaStream_t)stream);
}

int sg2_version(void) { return 2; }
int sg2_set_sm_reserve(int n_sms) {
  if (n_sms < 0 || n_sms > 64) SG2_FAIL(SG2_EINVAL, "set_sm_reserve: %d", n_sms);
  g_sm_reserve = n_sms;
  return 0;
}
int sg2_set_pair_kernels(int on) {
  if (on < -1 || on > 1) SG2_FAIL(SG2_EINVAL, "set_pair_kernels: %d", on);
  g_pair_override = on;
  return 0;
}
const char* sg2_last_error(void) { return g_err; }

int sg2_conv_fprop(int kind, const void* x, const void* wpk, void* y, int out_mode, int B, int H, int W, int Cin,
                   int Cout, int splitk, double* stats, int stats_groups, int act, const float* bias9, void* stream) {
  GatherDesc d;
  memset(&d, 0, sizeof(d));
  d.stats = stats;
  if (bias9 && (kind != SG2_CONV3x3 || out_mode != SG2_OUT_BF16 || splitk > 1 || (Cout % 4)))
    SG2_FAIL(SG2_EINVAL, "conv_fprop: the region bias applies to a plain bf16 3x3 convolution");
  d.bias9 = bias9;
  if (act != 0 && act != SG2_ACT_LRELU) SG2_FAIL(SG2_EINVAL, "conv_fprop: epilogue activation %d", act);
  if (act && (stats || out_mode != SG2_OUT_BF16)) SG2_FAIL(SG2_EINVAL, "conv_fprop: fused activation needs a bf16 epilogue");
  d.act = act;
  if (stats && stats_groups > 1) {
    if (B % stats_groups) SG2_FAIL(SG2_EINVAL, "conv_fprop: batch %d in %d statistics groups", B, stats_groups);
    d.stats_bg = B / stats_groups;
  }
  if (stats && out_mode != SG2_OUT_BF16) SG2_FAIL(SG2_EINVAL, "fused BN statistics need SG2_OUT_BF16");
  d.Cin = Cin;
  d.w = wpk;
  d.N = Cout;
  d.B = B;
  d.out = y;
  d.out_mode = out_mode;
  d.splitk = splitk;
  const View xv = dense_view(x, B, H, W, Cin);
  switch (kind) {
    case SG2_CONV3x3:
    case SG2_GEMM: {
      d.a[0] = xv;
      d.nmaps = 1;
      d.ngroups = 1;
      if (kind == SG2_GEMM) {
        d.ntaps = 1;
        d.taps[0][0] = TapF{0, 0, 0, 0};
      } else {
        d.ntaps = 9;
        for (int kh = 0; kh < 3; ++kh)
          for (int kw = 0; kw < 3; ++kw) d.taps[0][kh * 3 + kw] = TapF{0, (int8_t)(kh - 1), (int8_t)(kw - 1), 0};
      }
      d.Wg = W;
      d.Hg = H;
      d.osx = Cout;
      d.osy = (long long)W * Cout;
      d.osb = (long long)H * W * Cout;
      break;
    }
    case SG2_UPCONV3x3: {
      // y[2i+py, 2j+px] = sum_{a,b in {0,1}} Wc[py,px][a,b] . x[i+py-1+a, j+px-1+b]
      d.a[0] = xv;
      d.nmaps = 1;
      d.ngroups = 4;
      d.ntaps = 4;
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) {
          const int g = py * 2 + px;
          for (int a = 0; a < 2; ++a)
            for (int b = 0; b < 2; ++b) d.taps[g][a * 2 + b] = TapF{0, (int8_t)(py - 1 + a), (int8_t)(px - 1 + b), 0};
          d.out_off[g] = ((long long)py * 2 * W + px) * Cout;
        }
      d.Wg = W;
      d.Hg = H;
      d.osx = 2LL * Cout;
      d.osy = 2LL * (2 * W) * Cout;
      d.osb = 4LL * H * W * Cout;
      break;
    }
    case SG2_CONV4x4S2: {
      if ((H | W) & 1) SG2_FAIL(SG2_EINVAL, "conv4x4s2 needs even H, W");
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) d.a[py * 2 + px] = plane_view(xv, py, px);
      d.nmaps = 4;
      d.ngroups = 1;
      d.ntaps = 16;
      for (int kh = 0; kh < 4; ++kh)
        for (int kw = 0; kw < 4; ++kw) {
          const int ry = kh - 1, rx = kw - 1;  // input row = 2*oy + ry
          d.taps[0][kh * 4 + kw] = TapF{(int8_t)((ry & 1) * 2 + (rx & 1)), (int8_t)fdiv2(ry), (int8_t)fdiv2(rx), 0};
        }
      d.Wg = W / 2;
      d.Hg = H / 2;
      d.osx = Cout;
      d.osy = (long long)(W / 2) * Cout;
      d.osb = (long long)(H / 2) * (W / 2) * Cout;
      break;
    }
    default:
      SG2_FAIL(SG2_EINVAL, "unknown conv kind %d", kind);
  }
  d.split_stride = (long long)B * d.Hg * d.Wg * d.ngroups * Cout;   // one dense output tensor per split-K slab
  return launch_fprop(d, (cudaStream_t)stream);
}

int sg2_conv_dgrad(int kind, const void* dy, const void* wpkT, void* dx, int out_mode, int B, int H, int W, int Cin,
                   int Cout, int splitk, const void* epi_src, int epi_mode, void* stream) {
  GatherDesc d;
  memset(&d, 0, sizeof(d));
  if (epi_mode != 0 && epi_mode != SG2_EPI_ADD && epi_mode != SG2_EPI_LRELU_MASK)
    SG2_FAIL(SG2_EINVAL, "conv_dgrad: epilogue mode %d", epi_mode);
  if (epi_mode && (!epi_src || (Cin % 8))) SG2_FAIL(SG2_EINVAL, "conv_dgrad: epilogue operand missing / Cin %% 8");
  if (epi_mode && out_mode != SG2_OUT_BF16) SG2_FAIL(SG2_ENOFUSE, "conv_dgrad: the epilogue operand needs a bf16 epilogue");
  d.epi_src = epi_src;
  d.epi_mode = epi_mode;
  d.Cin = Cout;  // contraction runs over the forward output channels
  d.w = wpkT;
  d.N = Cin;
  d.B = B;
  d.out = dx;
  d.out_mode = out_mode;
  d.splitk = splitk;
  switch (kind) {
    case SG2_CONV3x3:
    case SG2_GEMM: {
      d.a[0] = dense_view(dy, B, H, W, Cout);
      d.nmaps = 1;
      d.ngroups = 1;
      if (kind == SG2_GEMM) {
        d.ntaps = 1;
        d.taps[0][0] = TapF{0, 0, 0, 0};
      } else {
        // dx[y,x] = sum_{kh,kw} W[:, :, kh, kw]^T . dy[y-(kh-1), x-(kw-1)]
        d.ntaps = 9;
        for (int kh = 0; kh < 3; ++kh)
          for (int kw = 0; kw < 3; ++kw) d.taps[0][kh * 3 + kw] = TapF{0, (int8_t)(1 - kh), (int8_t)(1 - kw), 0};
      }
      d.Wg = W;
      d.Hg = H;
      d.osx = Cin;
      d.osy = (long long)W * Cin;
      d.osb = (long long)H * W * Cin;
      break;
    }
    case SG2_UPCONV3x3: {
      // dx[u,v] = sum_{py,px,a,b} Wc[py,px][a,b]^T . P_{py,px}[u+1-py-a, v+1-px-b],  P = parity planes of dy (2H x 2W)
      const View dv = dense_view(dy, B, 2 * H, 2 * W, Cout);
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) d.a[py * 2 + px] = plane_view(dv, py, px);
      d.nmaps = 4;
      d.ngroups = 1;
      d.ntaps = 16;
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px)
          for (int a = 0; a < 2; ++a)
            for (int b = 0; b < 2; ++b)
              d.taps[0][(py * 2 + px) * 4 + a * 2 + b] =
                  TapF{(int8_t)(py * 2 + px), (int8_t)(1 - py - a), (int8_t)(1 - px - b), 0};
      d.Wg = W;
      d.Hg = H;
      d.osx = Cin;
      d.osy = (long long)W * Cin;
      d.osb = (long long)H * W * Cin;
      break;
    }
    case SG2_CONV4x4S2: {
      // dx[2i+py, 2j+px] = sum_{a,b} W[:, :, kh(py,a), kw(px,b)]^T . dy[i+dy(py,a), j+dx(px,b)]
      if ((H | W) & 1) SG2_FAIL(SG2_EINVAL, "conv4x4s2 needs even H, W");
      d.a[0] = dense_view(dy, B, H / 2, W / 2, Cout);
      d.nmaps = 1;
      d.ngroups = 4;
      d.ntaps = 4;
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) {
          const int g = py * 2 + px;
          for (int a = 0; a < 2; ++a)
            for (int b = 0; b < 2; ++b)
              d.taps[g][a * 2 + b] = TapF{0, (int8_t)kS2_dy[py][a], (int8_t)kS2_dy[px][b], 0};
          d.out_off[g] = ((long long)py * W + px) * Cin;
        }
      d.Wg = W / 2;
      d.Hg = H / 2;
      d.osx = 2LL * Cin;
      d.osy = 2LL * W * Cin;
      d.osb = (long long)H * W * Cin;
      break;
    }
    default:
      SG2_FAIL(SG2_EINVAL, "unknown conv kind %d", kind);
  }
  d.split_stride = (long long)B * H * W * Cin;
  return launch_fprop(d, (cudaStream_t)stream);
}

static int wgrad_entry(int kind, const void* x, const void* dy, float* dwpk, int B, int H, int W, int Cin, int Cout,
                       int splitk, float* partials, int* slabs_out, void* stream);

int sg2_conv_wgrad(int kind, const void* x, const void* dy, float* dwpk, int B, int H, int W, int Cin, int Cout,
                   int splitk, float* partials, void* stream) {
  return wgrad_entry(kind, x, dy, dwpk, B, H, W, Cin, Cout, splitk, partials, nullptr, stream);
}

int sg2_conv_wgrad_slabs(int kind, int B, int H, int W, int Cin, int Cout, int splitk) {
  int n = 0;
  // the plan only looks at extents; any 16-byte aligned non-null pointers will do for the views
  static const uintptr_t dummy = 4096;
  const int rc = wgrad_entry(kind, (const void*)dummy, (const void*)dummy, (float*)dummy, B, H, W, Cin, Cout, splitk,
                             nullptr, &n, nullptr);
  return rc ? (rc < 0 ? rc : -rc) : n;
}

static int wgrad_entry(int kind, const void* x, const void* dy, float* dwpk, int B, int H, int W, int Cin, int Cout,
                       int splitk, float* partials, int* slabs_out, void* stream) {
  WgradDesc d;
  memset(&d, 0, sizeof(d));
  d.partials = partials;
  d.slabs_out = slabs_out;
  {
    static const int cap = [] {
      const char* e = getenv("SG2_WGRAD_LANE_CAP");
      return e ? atoi(e) : 0;
    }();
    d.lane_cap = cap;
  }
  d.B = B;
  d.Cout = Cout;
  d.Cin = Cin;
  d.dw = dwpk;
  d.splitk = splitk;
  const View xv = dense_view(x, B, H, W, Cin);
  switch (kind) {
    case SG2_CONV3x3:
    case SG2_GEMM: {
      d.a[0] = dense_view(dy, B, H, W, Cout);
      d.b[0] = xv;
      d.namaps = d.nbmaps = 1;
      if (kind == SG2_GEMM) {
        d.njobs = 1;
        d.jobs[0] = JobW{0, 0, 0, 0};
      } else {
        d.njobs = 9;
        for (int kh = 0; kh < 3; ++kh)
          for (int kw = 0; kw < 3; ++kw) d.jobs[kh * 3 + kw] = JobW{0, 0, (int8_t)(kh - 1), (int8_t)(kw - 1)};
      }
      d.Wg = W;
      d.Hg = H;
      break;
    }
    case SG2_UPCONV3x3: {
      const View dv = dense_view(dy, B, 2 * H, 2 * W, Cout);
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) d.a[py * 2 + px] = plane_view(dv, py, px);
      d.b[0] = xv;
      d.namaps = 4;
      d.nbmaps = 1;
      d.njobs = 16;
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px)
          for (int a = 0; a < 2; ++a)
            for (int b = 0; b < 2; ++b)
              d.jobs[(py * 2 + px) * 4 + a * 2 + b] =
                  JobW{(int8_t)(py * 2 + px), 0, (int8_t)(py - 1 + a), (int8_t)(px - 1 + b)};
      d.Wg = W;
      d.Hg = H;
      break;
    }
    case SG2_CONV4x4S2: {
      if ((H | W) & 1) SG2_FAIL(SG2_EINVAL, "conv4x4s2 needs even H, W");
      d.a[0] = dense_view(dy, B, H / 2, W / 2, Cout);
      for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) d.b[py * 2 + px] = plane_view(xv, py, px);
      d.namaps = 1;
      d.nbmaps = 4;
      d.njobs = 16;
      for (int kh = 0; kh < 4; ++kh)
        for (int kw = 0; kw < 4; ++kw) {
          const int ry = kh - 1, rx = kw - 1;
          d.jobs[kh * 4 + kw] = JobW{0, (int8_t)((ry & 1) * 2 + (rx & 1)), (int8_t)fdiv2(ry), (int8_t)fdiv2(rx)};
        }
      d.Wg = W / 2;
      d.Hg = H / 2;
      break;
    }
    default:
      SG2_FAIL(SG2_EINVAL, "unknown conv kind %d", kind);
  }
  return launch_wgrad(d, (cudaStream_t)stream);
}

}  // extern "C"

#ifdef SG2_BUILD_PROBES
// EXPERIMENT (tools/probe_halo.py): shifted-window UMMA descriptors over one halo tile; see halo_probe.cuh.
template <int BN, int BK>
static int launch_halo_probe(const void* x, const void* wpk, void* y, int B, int H, int W, int Cin, int Cout, int pitch,
                             int bo_mode, cudaStream_t st) {
  HaloProbeParams p;
  memset(&p, 0, sizeof(p));
  int rc;
  if ((rc = make_act_map(&p.tmA, dense_view(x, B, H, W, Cin), BK, pitch, kHaloTH + 2, 1))) return rc;
  if ((rc = make_w_map(&p.tmB, wpk, Cout, 9LL * Cin, BK, BN))) return rc;
  p.kchunks = Cin / BK;
  p.pitch = pitch;
  p.bo_mode = bo_mode;
  p.tiles_x = (W + kHaloTW - 1) / kHaloTW;
  p.tiles_y = (H + kHaloTH - 1) / kHaloTH;
  p.W = W;
  p.H = H;
  p.B = B;
  p.N = Cout;
  p.out = y;
  p.stages = 4;
  const int a_bytes = ((pitch * (kHaloTH + 2) * BK * 2) + 1023) & ~1023;
  const size_t smem = 2 * a_bytes + p.stages * BN * BK * 2 + 1024 + 256;
  cudaError_t e = cudaFuncSetAttribute(halo_probe_kernel<BN, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) SG2_FAIL((int)e, "cudaFuncSetAttribute(halo_probe): %s", cudaGetErrorString(e));
  dim3 grid(p.tiles_x * p.tiles_y * B, Cout / BN, 1);
  halo_probe_kernel<BN, BK><<<grid, kNumThreads, smem, st>>>(p);
  SG2_LAUNCH_OK("halo_probe");
}

extern "C" {
/* DIAGNOSTICS: copy the tile kernel's wait-cycle counters (SG2_TILE_DBG & 64) of the last launch to the host. */
int sg2_tile_dbg_read(long long* host_out, int n) {
  if (!g_tile_dbg) SG2_FAIL(SG2_EINVAL, "no tile debug buffer");
  cudaDeviceSynchronize();
  cudaMemcpy(host_out, g_tile_dbg, n * sizeof(long long), cudaMemcpyDeviceToHost);
  return 0;
}
int sg2_probe_halo_fprop(const void* x, const void* wpk, void* y, int B, int H, int W, int Cin, int Cout, int pitch,
                         int bo_mode, void* stream) {
  if (pitch < 10 || pitch > 16) SG2_FAIL(SG2_EINVAL, "pitch %d", pitch);
  cudaStream_t st = (cudaStream_t)stream;
  if (Cin % 64 == 0 && Cout % 64 == 0) return launch_halo_probe<64, 64>(x, wpk, y, B, H, W, Cin, Cout, pitch, bo_mode, st);
  if (Cin % 32 == 0 && Cout % 32 == 0) return launch_halo_probe<32, 32>(x, wpk, y, B, H, W, Cin, Cout, pitch, bo_mode, st);
  SG2_FAIL(SG2_EINVAL, "halo probe: unsupported channels %d -> %d", Cin, Cout);
}

}  // extern "C"
#endif  // SG2_BUILD_PROBES
