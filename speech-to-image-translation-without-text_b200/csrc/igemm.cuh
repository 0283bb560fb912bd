// Implicit-GEMM convolution kernels on tcgen05 / TMEM, operands staged by TMA (sm_100a only).
//
// fprop/dgrad kernel ("gather" form):
//   out[pixel, n] = sum_{tap, c} act[pixel + shift(tap), c] * wpk[n, tap, c]
//   A (activations) : NHWC bf16, 4-D TMA boxes {BK channels, tw, th, nb} = 128 pixels x BK, K-major, swizzled;
//                     zero padding = TMA out-of-bounds fill; stride-2 / nearest-2x convs use parity-plane
//                     tensor maps (strided views of the same NHWC tensor), so nothing is materialised.
//   B (weights)     : packed [group][N][taps*Cin] bf16, 2-D TMA boxes {BK, BN}, K-major, swizzled.
//   D (accumulator) : 128 lanes x BN fp32 columns in TMEM; epilogue warps read it with tcgen05.ld.
//
// wgrad kernel ("outer product over pixels" form):
//   dw[m, job, n] += sum_{pixel} dy[pixel, m] * act[pixel + shift(job), n]
//   Both operands are MN-major (channels contiguous, pixels = K), loaded as {CW channels, 64 pixels} boxes.
#pragma once
#include "ptx.cuh"

namespace sg2 {

constexpr int kBlockM = 128;
constexpr int kNumThreads = 192;  // warp0: TMA producer, warp1: MMA issuer + TMEM owner, warps2-5: epilogue

struct TapF {
  int8_t map, dy, dx, pad;
};
constexpr int kMaxTaps = 32;   // per group: up to 5x5 (sg2_conv2d_fprop)

enum OutMode : int { OUT_BF16 = 0, OUT_F32_ATOMIC = 1, OUT_F32_STORE = 2 };

struct FpropParams {
  CUtensorMap tmA[4];
  CUtensorMap tmB;
  TapF taps[4][kMaxTaps];  // [group][tap]
  int ntaps, kchunks;
  int ngroups, splitk;
  int tw, th, nb;
  int tiles_x, tiles_y, tiles_b;
  int Wo, Ho, B;
  int N;
  long long out_off[4];
  long long sb, sy, sx;
  void* out;
  int out_mode;
  int stages;
  double* stats;  // optional [groups][2][N] fp64: per-channel sum / sum of squares of the (bf16-rounded) outputs, += (BN statistics)
  int stats_bg;  // images per statistics group (0: one group); a tile never straddles groups (checked on the host)
  int act;       // epilogue activation: 0 none, 2 LeakyReLU(0.2) (layers without BatchNorm: the D stems), 3 ReLU
  const float* bias;  // optional [N] fp32, added before the activation (igemm_fprop_kernel only)
  // cluster split-K (igemm_fprop_cluster_kernel): bf16 output, the `splitk` CTAs of a tile form a cluster and reduce
  // their partial tiles through distributed shared memory in rank order
  const void* epi_src;     // optional epilogue operand (layout of the output, bf16), see sg2_conv_dgrad
  int epi_mode;
  long long split_stride;  // OUT_F32_STORE with split-K: split s stores its partial tile into slab s (out + s * split_stride);
                           // the slabs are summed in split order by sg2_splitk_finish (deterministic, no atomics)
};

// MT = pixel tiles (of 128 GEMM rows) per CTA. The main loop of these kernels is bound by the bytes TMA can bring into
// one SM (~42 B/cycle): a 128 x 256 tile needs 48 KB per 64-deep K block against 512 tensor cycles (96 B/cycle, so the
// tensor pipe cannot exceed ~44 %). With MT = 2 the two tiles share every weight stage (two accumulators, all 512 TMEM
// columns at BN = 256): 64 KB per 1024 tensor cycles, i.e. two thirds of the operand bytes per output tile.
template <int BN, int BK, int MT = 1>
struct FpropCfg {
  static constexpr int kSw = BK * 2;  // swizzle span in bytes (128/64/32)
  static constexpr int kABytes = kBlockM * BK * 2;   // one pixel tile
  static constexpr int kBBytes = BN * BK * 2;
  static constexpr int kStageBytes = MT * kABytes + kBBytes;
  static constexpr int kCols = MT * BN;
  static constexpr int kTmemCols = kCols <= 32 ? 32 : (kCols <= 64 ? 64 : (kCols <= 128 ? 128 : (kCols <= 256 ? 256 : 512)));
  static size_t smem_bytes(int stages) { return size_t(stages) * kStageBytes + 1024 + 256; }
};

template <int BN, int BK, int MT = 1>
__global__ void __launch_bounds__(kNumThreads) igemm_fprop_kernel(const __grid_constant__ FpropParams p) {
  using Cfg = FpropCfg<BN, BK, MT>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int S = p.stages;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + size_t(S) * Cfg::kStageBytes);
  uint64_t* empty = full + S;
  uint64_t* tmem_full = empty + S;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);
  __shared__ float s_stats[4 * 2 * (BN < 32 ? 32 : BN)];   // [TMEM lane quarter][2][SN]: one writer warp per slot

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // ---- tile coordinates: blockIdx.x = unit of MT consecutive pixel tiles. A unit's tile past the last one decodes to
  // an image index >= B: its TMA boxes are zero filled, its MMAs are skipped and none of its rows is stored
  int x0[MT], y0[MT], b0[MT];
#pragma unroll
  for (int m = 0; m < MT; ++m) {
    int t = blockIdx.x * MT + m;
    const int tx = t % p.tiles_x;
    t /= p.tiles_x;
    const int ty = t % p.tiles_y;
    const int tb = t / p.tiles_y;
    x0[m] = tx * p.tw, y0[m] = ty * p.th, b0[m] = tb * p.nb;
  }
  const int ntile = (MT == 2 && b0[MT - 1] >= p.B) ? 1 : MT;   // tiles of this unit that exist
  const int n0 = blockIdx.y * BN;
  const int g = blockIdx.z / p.splitk;
  const int split = blockIdx.z % p.splitk;
  const int KB = p.ntaps * p.kchunks;
  const int kb_begin = (int)((long long)KB * split / p.splitk);
  const int kb_end = (int)((long long)KB * (split + 1) / p.splitk);
  const int nkb = kb_end - kb_begin;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmB);
    tma_prefetch_desc(&p.tmA[0]);
    for (int s = 0; s < S; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Issue loops run with the WHOLE warp convergent and one elected lane issuing (elect.sync): the compiler then keeps
  // descriptors in uniform registers and emits back-to-back UTCHMMA/UTMALDG. A divergent `if (lane == 0)` body costs
  // ~146 cycles per tcgen05.mma (tools/probe_mma.py) against a 64-cycle tensor floor at N = 128.
  if (warp == 0) {
    // a pixel tile may be a partial box (tw * th * nb < 128 rows, sg2_conv2d_fprop): only its bytes arrive
    const uint32_t tx_bytes = uint32_t(MT * p.tw * p.th * p.nb * BK * 2 + Cfg::kBBytes);
    int s = 0;
    uint32_t ph = 0;
    for (int it = 0; it < nkb; ++it) {
      mbar_wait(&empty[s], ph ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&full[s], tx_bytes);
        const int kb = kb_begin + it;
        const int tap = kb / p.kchunks;
        const int ch = kb - tap * p.kchunks;
        const TapF tp = p.taps[g][tap];
        uint8_t* sa = smem + size_t(s) * Cfg::kStageBytes;
        uint8_t* sb = sa + MT * Cfg::kABytes;
#pragma unroll
        for (int m = 0; m < MT; ++m)
          tma_load_4d(&p.tmA[tp.map], &full[s], sa + m * Cfg::kABytes, ch * BK, x0[m] + tp.dx, y0[m] + tp.dy, b0[m]);
        tma_load_2d(&p.tmB, &full[s], sb, kb * BK, n0 + g * p.N);
      }
      __syncwarp();
      if (++s == S) {
        s = 0;
        ph ^= 1;
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc_bf16(kBlockM, BN, 0, 0);
    constexpr uint32_t swc = swizzle_code(Cfg::kSw);
    const uint64_t adesc0 = make_smem_desc(smem_u32(smem), 16, 8 * Cfg::kSw, swc);
    const uint64_t bdesc0 = make_smem_desc(smem_u32(smem) + MT * Cfg::kABytes, 16, 8 * Cfg::kSw, swc);
    int s = 0;
    uint32_t ph = 0;
    for (int it = 0; it < nkb; ++it) {
      mbar_wait(&full[s], ph);
      tc_fence_after();
      if (elect_one()) {
        const uint64_t so = uint64_t((uint32_t(s) * uint32_t(Cfg::kStageBytes)) >> 4);
        const uint64_t adesc = adesc0 + so, bdesc = bdesc0 + so;
#pragma unroll
        for (int k = 0; k < BK / 16; ++k)
          umma_f16(tmem_base, adesc + uint64_t(k * 2), bdesc + uint64_t(k * 2), idesc, (it > 0 || k > 0) ? 1u : 0u);
        if (MT == 2 && ntile == 2) {
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)
            umma_f16(tmem_base + uint32_t(BN), adesc + uint64_t((Cfg::kABytes >> 4) + k * 2), bdesc + uint64_t(k * 2), idesc,
                     (it > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(&empty[s]);
      }
      __syncwarp();
      if (++s == S) {
        s = 0;
        ph ^= 1;
      }
    }
    if (elect_one()) umma_commit(tmem_full);
    __syncwarp();
  } else {
    // ---- epilogue: warp w may only touch TMEM lanes [32*(w%4), 32*(w%4)+32)
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int xi = row % p.tw;
    const int yi = (row / p.tw) % p.th;
    const int bi = row / (p.tw * p.th);
    // the rows past a partial box hold stale shared memory: their accumulators are never stored
    const bool in_box = row < p.tw * p.th * p.nb;
    const int ncols = p.N - n0;   // < BN: the weight box ran past N (zero filled); those columns are not stored
    const bool do_stats = (p.stats != nullptr) && (p.out_mode == OUT_BF16);
    const int et = threadIdx.x - 64;  // 0..127 within the epilogue warps
    constexpr int SN = BN < 32 ? 32 : BN;
    mbar_wait(tmem_full, 0);
    tc_fence_after();
#pragma unroll 1
    for (int m = 0; m < ntile; ++m) {
    const bool second = MT == 2 && m == 1;
    const int x0m = second ? x0[MT - 1] : x0[0], y0m = second ? y0[MT - 1] : y0[0], b0m = second ? b0[MT - 1] : b0[0];
    const int x = x0m + xi, y = y0m + yi, b = b0m + bi;
    const bool valid = in_box && (x < p.Wo) && (y < p.Ho) && (b < p.B);
    const long long off = p.out_off[g] + (long long)b * p.sb + (long long)y * p.sy + (long long)x * p.sx + n0 +
                          (p.out_mode == OUT_F32_STORE ? (long long)split * p.split_stride : 0);
    const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(m * BN);
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t v[32];
      tmem_ld_32x32(taddr + c0, v);
      tmem_ld_wait();
      if (nkb <= 0) {   // no K block in this split: the accumulator was never written
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 0u;
      }
      if (p.bias) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (c0 + j < ncols) v[j] = __float_as_uint(__uint_as_float(v[j]) + __ldg(p.bias + n0 + c0 + j));
      }
      if (p.act == 2) {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float f = __uint_as_float(v[j]);
          v[j] = __float_as_uint(f > 0.f ? f : 0.2f * f);
        }
      } else if (p.act == 3) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(fmaxf(__uint_as_float(v[j]), 0.f));
      }
      if (do_stats) {
        // statistics of what BatchNorm will read back: the bf16-rounded outputs of the valid rows
        float a[32], qq[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float r = __bfloat162float(__float2bfloat16_rn(__uint_as_float(v[j])));
          a[j] = (valid && (c0 + j < BN)) ? r : 0.f;
          qq[j] = a[j] * a[j];
        }
        const float cs = warp_transpose_sum(a, lane);
        const float cq = warp_transpose_sum(qq, lane);
        if (c0 + lane < BN) {
          s_stats[q * 2 * SN + c0 + lane] = cs;
          s_stats[q * 2 * SN + SN + c0 + lane] = cq;
        }
      }
      if (valid) {
        if (p.out_mode == OUT_BF16) {
          uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + off + c0);
#pragma unroll
          for (int j = 0; j < (BN < 32 ? BN / 8 : 4); ++j) {
            if (c0 + 8 * j >= ncols) break;
            uint4 o;
            o.x = pack_bf16x2(__uint_as_float(v[8 * j + 0]), __uint_as_float(v[8 * j + 1]));
            o.y = pack_bf16x2(__uint_as_float(v[8 * j + 2]), __uint_as_float(v[8 * j + 3]));
            o.z = pack_bf16x2(__uint_as_float(v[8 * j + 4]), __uint_as_float(v[8 * j + 5]));
            o.w = pack_bf16x2(__uint_as_float(v[8 * j + 6]), __uint_as_float(v[8 * j + 7]));
            dst[j] = o;
          }
        } else if (p.out_mode == OUT_F32_ATOMIC) {
          float* dst = reinterpret_cast<float*>(p.out) + off + c0;
#pragma unroll
          for (int j = 0; j < (BN < 32 ? BN : 32); j += 4)
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + j), "f"(__uint_as_float(v[j])),
                         "f"(__uint_as_float(v[j + 1])), "f"(__uint_as_float(v[j + 2])), "f"(__uint_as_float(v[j + 3]))
                         : "memory");
        } else {
          float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + off + c0);
#pragma unroll
          for (int j = 0; j < (BN < 32 ? BN / 4 : 8); ++j)
            dst[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                 __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        }
      }
    }
    if (do_stats) {
      asm volatile("bar.sync 1, 128;" ::: "memory");
      double* st = p.stats + (p.stats_bg > 0 ? (long long)(b0m / p.stats_bg) * 2 * p.N : 0);
      for (int i = et; i < BN; i += 128) {
        float cs = 0.f, cq = 0.f;
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) {
          cs += s_stats[qq * 2 * SN + i];
          cq += s_stats[qq * 2 * SN + SN + i];
        }
        atomicAdd(&st[n0 + i], (double)cs);
        atomicAdd(&st[p.N + n0 + i], (double)cq);
      }
      if (MT == 2) asm volatile("bar.sync 1, 128;" ::: "memory");   // the next tile overwrites the partial sums
    }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------ cluster split-K
// Same main loop as igemm_fprop_kernel, for layers whose 128 x BN tiles cannot fill the GPU (D's 4x4 / 8x8 maps, the
// generator's first upBlocks). The `splitk` CTAs that share an output tile are ONE thread-block cluster (cluster dims
// (1, 1, splitk)): each accumulates its K range in TMEM, parks the fp32 partial tile in its own shared memory (over the
// operand ring, which is idle by then), and after a cluster barrier CTA r reduces the column units [r*U/S, (r+1)*U/S) of
// the tile over all peers' shared memory in RANK ORDER (deterministic), applies the epilogue (dgrad operand, bf16
// rounding, BatchNorm statistics) and stores bf16. No fp32 slab round trip through HBM, no separate finish launch.
constexpr int kPartPad = 4;   // floats of padding per partial-tile row (bank spread for the 128-bit reads)
template <int BN, int BK, int MT = 1>
struct ClusterCfg {
  static constexpr int kPartRow = BN + kPartPad;
  static constexpr size_t kPartBytes = size_t(kBlockM) * kPartRow * sizeof(float);
  static size_t smem_bytes(int stages) {
    const size_t ring = size_t(stages) * FpropCfg<BN, BK, MT>::kStageBytes;
    return (ring > kPartBytes ? ring : kPartBytes) + 1024 + 512 + 8192 + 256;   // align slack, barriers, statistics partials
  }
};

// MT = 2: two pixel tiles per CTA share every weight stage (see FpropCfg); their partial tiles are exchanged one after
// the other through the same shared-memory buffer.
template <int BN, int BK, int MT = 1>
__global__ void __launch_bounds__(kNumThreads, 1) igemm_fprop_cluster_kernel(const __grid_constant__ FpropParams p) {
  using Cfg = FpropCfg<BN, BK, MT>;
  using CC = ClusterCfg<BN, BK, MT>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int S = p.stages;
  const size_t ring = size_t(S) * Cfg::kStageBytes;
  const size_t data_bytes = ring > CC::kPartBytes ? ring : CC::kPartBytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + data_bytes);
  uint64_t* empty = full + S;
  uint64_t* tmem_full = empty + S;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);
  float* s_red = reinterpret_cast<float*>(smem + data_bytes + 512);   // [128 slots][16] statistics partials (8 KB max use 4 KB)
  float* part = reinterpret_cast<float*>(smem);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  int x0[MT], y0[MT], b0[MT];
#pragma unroll
  for (int m = 0; m < MT; ++m) {
    int t = blockIdx.x * MT + m;
    const int tx = t % p.tiles_x;
    t /= p.tiles_x;
    const int ty = t % p.tiles_y;
    const int tb = t / p.tiles_y;
    x0[m] = tx * p.tw, y0[m] = ty * p.th, b0[m] = tb * p.nb;
  }
  const int ntile = (MT == 2 && b0[MT - 1] >= p.B) ? 1 : MT;   // same for every CTA of the cluster (same blockIdx.x)
  const int n0 = blockIdx.y * BN;
  const int g = blockIdx.z / p.splitk;
  const int split = blockIdx.z % p.splitk;       // == rank in the cluster (cluster dims (1, 1, splitk))
  const int KB = p.ntaps * p.kchunks;
  const int kb_begin = (int)((long long)KB * split / p.splitk);
  const int kb_end = (int)((long long)KB * (split + 1) / p.splitk);
  const int nkb = kb_end - kb_begin;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmB);
    tma_prefetch_desc(&p.tmA[0]);
    for (int s = 0; s < S; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    int s = 0;
    uint32_t ph = 0;
    for (int it = 0; it < nkb; ++it) {
      mbar_wait(&empty[s], ph ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&full[s], Cfg::kStageBytes);
        const int kb = kb_begin + it;
        const int tap = kb / p.kchunks;
        const int ch = kb - tap * p.kchunks;
        const TapF tp = p.taps[g][tap];
        uint8_t* sa = smem + size_t(s) * Cfg::kStageBytes;
        uint8_t* sb = sa + MT * Cfg::kABytes;
#pragma unroll
        for (int m = 0; m < MT; ++m)
          tma_load_4d(&p.tmA[tp.map], &full[s], sa + m * Cfg::kABytes, ch * BK, x0[m] + tp.dx, y0[m] + tp.dy, b0[m]);
        tma_load_2d(&p.tmB, &full[s], sb, kb * BK, n0 + g * p.N);
      }
      __syncwarp();
      if (++s == S) {
        s = 0;
        ph ^= 1;
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc_bf16(kBlockM, BN, 0, 0);
    constexpr uint32_t swc = swizzle_code(Cfg::kSw);
    const uint64_t adesc0 = make_smem_desc(smem_u32(smem), 16, 8 * Cfg::kSw, swc);
    const uint64_t bdesc0 = make_smem_desc(smem_u32(smem) + MT * Cfg::kABytes, 16, 8 * Cfg::kSw, swc);
    int s = 0;
    uint32_t ph = 0;
    for (int it = 0; it < nkb; ++it) {
      mbar_wait(&full[s], ph);
      tc_fence_after();
      if (elect_one()) {
        const uint64_t so = uint64_t((uint32_t(s) * uint32_t(Cfg::kStageBytes)) >> 4);
        const uint64_t adesc = adesc0 + so, bdesc = bdesc0 + so;
#pragma unroll
        for (int k = 0; k < BK / 16; ++k)
          umma_f16(tmem_base, adesc + uint64_t(k * 2), bdesc + uint64_t(k * 2), idesc, (it > 0 || k > 0) ? 1u : 0u);
        if (MT == 2 && ntile == 2) {
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)
            umma_f16(tmem_base + uint32_t(BN), adesc + uint64_t((Cfg::kABytes >> 4) + k * 2), bdesc + uint64_t(k * 2), idesc,
                     (it > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(&empty[s]);
      }
      __syncwarp();
      if (++s == S) {
        s = 0;
        ph ^= 1;
      }
    }
    if (elect_one()) umma_commit(tmem_full);
    __syncwarp();
  }
  if (warp >= 2) {
    mbar_wait(tmem_full, 0);   // every MMA that read the operand ring has completed: the ring is idle from here on
    tc_fence_after();
  }
#pragma unroll 1
  for (int m = 0; m < ntile; ++m) {
    const bool second = MT == 2 && m == 1;
    const int x0m = second ? x0[MT - 1] : x0[0], y0m = second ? y0[MT - 1] : y0[0], b0m = second ? b0[MT - 1] : b0[0];
    if (warp >= 2) {
      // ---- phase 1: my partial tile TMEM -> my shared memory (over the idle operand ring)
      const int q = warp & 3;
      const int row = q * 32 + lane;
      const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(m * BN);
      float* prow = part + (size_t)row * CC::kPartRow;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32(taddr + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          float4 o = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                                 __uint_as_float(v[j + 3]));
          if (nkb <= 0) o = make_float4(0.f, 0.f, 0.f, 0.f);
          if (c0 + j < BN) *reinterpret_cast<float4*>(prow + c0 + j) = o;
        }
      }
      tc_fence_before();
    }
    cluster_sync_all();   // all partial tiles of the cluster are in shared memory

    if (warp >= 2) {
      // ---- phase 2: CTA `split` owns column units [u0, u1) of 8 channels; thread = (row slot, unit): it walks its rows,
      // sums the S partials of its 8 columns in rank order, applies the epilogue and stores 16 bytes of bf16
      constexpr int U = BN / 8;
      const int Sx = p.splitk;
      const int u0 = split * U / Sx, u1 = (split + 1) * U / Sx;
      const int nu = u1 - u0;
      const int et = threadIdx.x - 64;
      const bool do_stats = p.stats != nullptr;
      float cs[8], cq[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) cs[j] = cq[j] = 0.f;
      int slots = 0, slot = 0, uu = 0;
      if (nu > 0) {
        slots = 128 / nu;
        slot = et / nu;
        uu = et - slot * nu;
      }
      const bool active = nu > 0 && slot < slots;
      if (active) {
        const int col = (u0 + uu) * 8;
        const uint32_t my_off = smem_u32(part) + uint32_t(col) * 4u;
        for (int r = slot; r < kBlockM; r += slots) {
          const int xi = r % p.tw, yi = (r / p.tw) % p.th, bi = r / (p.tw * p.th);
          const int x = x0m + xi, y = y0m + yi, b = b0m + bi;
          if (!((x < p.Wo) && (y < p.Ho) && (b < p.B))) continue;
          float a[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) a[j] = 0.f;
          const uint32_t roff = my_off + uint32_t(r) * uint32_t(CC::kPartRow * 4);
          for (int s2 = 0; s2 < Sx; ++s2) {
            const uint32_t ra = dsmem_addr(roff, (uint32_t)s2);
            const float4 lo = dsmem_ld_f4(ra), hi = dsmem_ld_f4(ra + 16);
            a[0] += lo.x; a[1] += lo.y; a[2] += lo.z; a[3] += lo.w;
            a[4] += hi.x; a[5] += hi.y; a[6] += hi.z; a[7] += hi.w;
          }
          const long long off = p.out_off[g] + (long long)b * p.sb + (long long)y * p.sy + (long long)x * p.sx + n0 + col;
          if (p.epi_mode != 0) {
            const uint4 sv = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.epi_src) + off));
            const uint32_t w4[4] = {sv.x, sv.y, sv.z, sv.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float elo = bf16_lo(w4[k]), ehi = bf16_hi(w4[k]);
              if (p.epi_mode == 1) { a[2 * k] += elo; a[2 * k + 1] += ehi; }
              else { a[2 * k] = elo > 0.f ? a[2 * k] : 0.2f * a[2 * k]; a[2 * k + 1] = ehi > 0.f ? a[2 * k + 1] : 0.2f * a[2 * k + 1]; }
            }
          }
          if (p.act == 2) {
#pragma unroll
            for (int j = 0; j < 8; ++j) a[j] = a[j] > 0.f ? a[j] : 0.2f * a[j];
          }
          uint4 o;
          o.x = pack_bf16x2(a[0], a[1]); o.y = pack_bf16x2(a[2], a[3]);
          o.z = pack_bf16x2(a[4], a[5]); o.w = pack_bf16x2(a[6], a[7]);
          *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + off) = o;
          if (do_stats) {
            const uint32_t w4[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float f0 = bf16_lo(w4[k]), f1 = bf16_hi(w4[k]);
              cs[2 * k] += f0; cq[2 * k] = fmaf(f0, f0, cq[2 * k]);
              cs[2 * k + 1] += f1; cq[2 * k + 1] = fmaf(f1, f1, cq[2 * k + 1]);
            }
          }
        }
      }
      if (do_stats) {
        // ordered combine of the row slots: s_red[et][16]; thread (uu, j) of slot 0 sums the slots in order
        float* mine = s_red + et * 16;
#pragma unroll
        for (int j = 0; j < 8; ++j) { mine[j] = cs[j]; mine[8 + j] = cq[j]; }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        for (int task = et; task < nu * 16; task += 128) {     // nu can exceed 8 units for clusters of 2 or 3
          const int u2 = task / 16, k = task % 16;
          float tsum = 0.f;
          for (int sl = 0; sl < slots; ++sl) tsum += s_red[(sl * nu + u2) * 16 + k];
          double* st = p.stats + (p.stats_bg > 0 ? (long long)(b0m / p.stats_bg) * 2 * p.N : 0);
          const int c = n0 + (u0 + u2) * 8 + (k & 7);
          atomicAdd(&st[(k < 8 ? 0 : p.N) + c], (double)tsum);
        }
      }
    }
    cluster_sync_all();   // nobody overwrites its partial tile (or leaves and frees its shared memory) while a peer reads it
  }
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------ wgrad
struct JobW {
  int8_t amap, bmap, dy, dx;
};

struct WgradParams {
  CUtensorMap tmA[4];  // dy maps: {CWA channels, tw, th, nb} boxes
  CUtensorMap tmB[4];  // activation maps: {CWB channels, tw, th, nb} boxes
  JobW jobs[16];
  int njobs;
  int tw, th, nb;  // tw*th*nb == 64 pixels per K block
  int tiles_x, tiles_y, tiles_b;
  int splitk;
  int Cout, Cin;
  float* dw;  // [Cout][njobs][Cin]
  int stages;
  // deterministic mode: split s STORES its partial tile into slab s (partials + s * slab elements, each slab laid out
  // like dw); the caller sums the slabs in order (sg2_reduce_slabs). NULL: red.global.add into dw.
  float* partials;
  long long slab;
};

constexpr int kWgradBKP = 64;  // pixels per K block

template <int BN, int CWA, int CWB>
struct WgradCfg {
  static constexpr int kAChunkBytes = kWgradBKP * CWA * 2;
  static constexpr int kBChunkBytes = kWgradBKP * CWB * 2;
  static constexpr int kAChunks = kBlockM / CWA;
  static constexpr int kBChunks = BN / CWB;
  static constexpr int kABytes = kAChunks * kAChunkBytes;  // 16 KB
  static constexpr int kBBytes = kBChunks * kBChunkBytes;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kTmemCols = BN < 32 ? 32 : BN;
  static size_t smem_bytes(int stages) { return size_t(stages) * kStageBytes + 1024 + 256; }
};

template <int BN, int CWA, int CWB>
__global__ void __launch_bounds__(kNumThreads) igemm_wgrad_kernel(const __grid_constant__ WgradParams p) {
  using Cfg = WgradCfg<BN, CWA, CWB>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int S = p.stages;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + size_t(S) * Cfg::kStageBytes);
  uint64_t* empty = full + S;
  uint64_t* tmem_full = empty + S;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const int n_tiles = (p.Cin + BN - 1) / BN;
  const int m0 = (blockIdx.x / n_tiles) * kBlockM;
  const int n0 = (blockIdx.x % n_tiles) * BN;
  const int job = blockIdx.y;
  const int split = blockIdx.z;
  const int PT = p.tiles_x * p.tiles_y * p.tiles_b;  // pixel tiles = K blocks
  const int kb_begin = (int)((long long)PT * split / p.splitk);
  const int kb_end = (int)((long long)PT * (split + 1) / p.splitk);
  const int nkb = kb_end - kb_begin;
  const int a_chunks = min(Cfg::kAChunks, (p.Cout - m0 + CWA - 1) / CWA);
  const int b_chunks = min(Cfg::kBChunks, (p.Cin - n0 + CWB - 1) / CWB);

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    const JobW jb = p.jobs[job];
    const uint32_t tx_bytes = a_chunks * Cfg::kAChunkBytes + b_chunks * Cfg::kBChunkBytes;
    int s = 0;
    uint32_t ph = 0;
    for (int it = 0; it < nkb; ++it) {
      mbar_wait(&empty[s], ph ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&full[s], tx_bytes);
        int t = kb_begin + it;
        const int tx = t % p.tiles_x;
        t /= p.tiles_x;
        const int ty = t % p.tiles_y;
        const int tb = t / p.tiles_y;
        const int x0 = tx * p.tw, y0 = ty * p.th, b0 = tb * p.nb;
        uint8_t* sa = smem + size_t(s) * Cfg::kStageBytes;
        uint8_t* sb = sa + Cfg::kABytes;
        for (int c = 0; c < a_chunks; ++c)
          tma_load_4d(&p.tmA[jb.amap], &full[s], sa + c * Cfg::kAChunkBytes, m0 + c * CWA, x0, y0, b0);
        for (int c = 0; c < b_chunks; ++c)
          tma_load_4d(&p.tmB[jb.bmap], &full[s], sb + c * Cfg::kBChunkBytes, n0 + c * CWB, x0 + jb.dx, y0 + jb.dy, b0);
      }
      __syncwarp();
      if (++s == S) {
        s = 0;
        ph ^= 1;
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc_bf16(kBlockM, BN, 1, 1);
    constexpr uint32_t swa = swizzle_code(CWA * 2), swb = swizzle_code(CWB * 2);
    // MN-major: LBO = bytes between consecutive channel chunks, SBO = bytes between 8-pixel groups.
    const uint64_t adesc0 = make_smem_desc(smem_u32(smem), Cfg::kAChunkBytes, 8 * CWA * 2, swa);
    const uint64_t bdesc0 = make_smem_desc(smem_u32(smem) + Cfg::kABytes, Cfg::kBChunkBytes, 8 * CWB * 2, swb);
    int s = 0;
    uint32_t ph = 0;
    for (int it = 0; it < nkb; ++it) {
      mbar_wait(&full[s], ph);
      tc_fence_after();
      if (elect_one()) {
        const uint64_t so = uint64_t((uint32_t(s) * uint32_t(Cfg::kStageBytes)) >> 4);
        const uint64_t adesc = adesc0 + so, bdesc = bdesc0 + so;
#pragma unroll
        for (int k = 0; k < kWgradBKP / 16; ++k) {
          const uint64_t ka = uint64_t((k * 16 * CWA * 2) >> 4);
          const uint64_t kbo = uint64_t((k * 16 * CWB * 2) >> 4);
          umma_f16(tmem_base, adesc + ka, bdesc + kbo, idesc, (it > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(&empty[s]);
      }
      __syncwarp();
      if (++s == S) {
        s = 0;
        ph ^= 1;
      }
    }
    if (elect_one()) umma_commit(tmem_full);
    __syncwarp();
  } else {
    const int q = warp & 3;
    const int m = m0 + q * 32 + lane;
    const bool valid = m < p.Cout;
    const bool slabs = p.partials != nullptr;
    float* rowp = (slabs ? p.partials + (long long)split * p.slab : p.dw) + ((long long)m * p.njobs + job) * p.Cin + n0;
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16);
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t v[32];
      tmem_ld_32x32(taddr + c0, v);
      tmem_ld_wait();
      if (slabs) {
        if (valid) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            if (n0 + c0 + j < p.Cin) {
              float4 o = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                                     __uint_as_float(v[j + 3]));
              if (nkb <= 0) o = make_float4(0.f, 0.f, 0.f, 0.f);
              *reinterpret_cast<float4*>(rowp + c0 + j) = o;
            }
          }
        }
      } else if (valid && nkb > 0) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          if (n0 + c0 + j < p.Cin) {
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(rowp + c0 + j),
                         "f"(__uint_as_float(v[j])), "f"(__uint_as_float(v[j + 1])), "f"(__uint_as_float(v[j + 2])),
                         "f"(__uint_as_float(v[j + 3]))
                         : "memory");
          }
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

}  // namespace sg2
