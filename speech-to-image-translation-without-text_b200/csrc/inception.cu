// Bandwidth-bound kernels of the Inception-v3 scorer (model.py:17-109): the preprocessing + resize + im2col stem of
// Conv2d_1a_3x3, the 3x3 pools, the global 8x8 average (pool3) and the softmax. The convolutions run on the gather
// kernel (sg2_conv2d_fprop); the 2048 -> 1000 fc on sg2_linear_fwd.
#include <cuda_bf16.h>

#include "../../include/sg2b200.h"
#include "common.cuh"

namespace sg2 {

constexpr int kIncS = 299;    // Inception's input size
constexpr int kIncS1 = 149;   // Conv2d_1a_3x3 output (3x3 s2 p0)

__device__ __forceinline__ uint32_t pack2(float a, float b) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// One thread per Conv2d_1a output pixel: its 27 taps of the preprocessed, resized image, as F.interpolate(bilinear,
// align_corners=False) computes them (fp32 source index scale*(dst+0.5)-0.5 clamped at 0), each source pixel normalised
// before the interpolation (the reference normalises, then resizes).
__global__ void __launch_bounds__(256) inception_stem_kernel(const float* __restrict__ img, uint4* __restrict__ col, int B,
                                                             int S) {
  const long long n = (long long)B * kIncS1 * kIncS1;
  const float scale = (float)S / (float)kIncS;
  const float mean[3] = {0.485f, 0.456f, 0.406f}, stdv[3] = {0.229f, 0.224f, 0.225f};
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int ox = (int)(i % kIncS1), oy = (int)((i / kIncS1) % kIncS1), b = (int)(i / (kIncS1 * kIncS1));
    float v[32];
#pragma unroll
    for (int k = 27; k < 32; ++k) v[k] = 0.f;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      float sy = scale * ((float)(2 * oy + ky) + 0.5f) - 0.5f;
      sy = sy < 0.f ? 0.f : sy;
      const int y0 = (int)sy, y1 = y0 < S - 1 ? y0 + 1 : y0;
      const float ly = sy - (float)y0;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        float sx = scale * ((float)(2 * ox + kx) + 0.5f) - 0.5f;
        sx = sx < 0.f ? 0.f : sx;
        const int x0 = (int)sx, x1 = x0 < S - 1 ? x0 + 1 : x0;
        const float lx = sx - (float)x0;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float* p = img + ((long long)b * 3 + c) * S * S;
          const float is = 1.f / stdv[c];
          auto f = [&](int yy, int xx) { return ((__ldg(p + (long long)yy * S + xx) * 0.5f + 0.5f) - mean[c]) * is; };
          v[(ky * 3 + kx) * 3 + c] = (1.f - ly) * ((1.f - lx) * f(y0, x0) + lx * f(y0, x1)) +
                                     ly * ((1.f - lx) * f(y1, x0) + lx * f(y1, x1));
        }
      }
    }
    uint4* dst = col + i * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      dst[j] = make_uint4(pack2(v[8 * j], v[8 * j + 1]), pack2(v[8 * j + 2], v[8 * j + 3]), pack2(v[8 * j + 4], v[8 * j + 5]),
                          pack2(v[8 * j + 6], v[8 * j + 7]));
  }
}

// 8 channels (16 bytes) per thread; POOL 0: max 3x3 s2 p0, 1: average 3x3 s1 p1 over 9 (count_include_pad)
template <int POOL>
__global__ void __launch_bounds__(256) pool3_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int y_ctot, int B,
                                                    int H, int W, int C, int Ho, int Wo) {
  const int cv = C / 8;
  const long long n = (long long)B * Ho * Wo * cv;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c8 = (int)(i % cv);
    long long t = i / cv;
    const int ox = (int)(t % Wo);
    t /= Wo;
    const int oy = (int)(t % Ho);
    const int b = (int)(t / Ho);
    float a[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = POOL == 0 ? -INFINITY : 0.f;
#pragma unroll
    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        const int yy = POOL == 0 ? 2 * oy + dy : oy + dy - 1, xx = POOL == 0 ? 2 * ox + dx : ox + dx - 1;
        if (POOL == 1 && (yy < 0 || yy >= H || xx < 0 || xx >= W)) continue;
        const uint4 q = __ldg(x + (((long long)b * H + yy) * W + xx) * cv + c8);
        const uint32_t w4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w4[k]);
          const float lo = __low2float(h), hi = __high2float(h);
          if (POOL == 0) {
            a[2 * k] = fmaxf(a[2 * k], lo);
            a[2 * k + 1] = fmaxf(a[2 * k + 1], hi);
          } else {
            a[2 * k] += lo;
            a[2 * k + 1] += hi;
          }
        }
      }
    if (POOL == 1) {
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] *= (1.f / 9.f);
    }
    y[(((long long)b * Ho + oy) * Wo + ox) * (y_ctot / 8) + c8] =
        make_uint4(pack2(a[0], a[1]), pack2(a[2], a[3]), pack2(a[4], a[5]), pack2(a[6], a[7]));
  }
}

// out[b][c] = mean over the pixels, one thread per (b, c), pixels summed in order (reproducible)
__global__ void __launch_bounds__(256) global_avg_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ out, int B,
                                                         int HW, int C) {
  const long long n = (long long)B * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C), b = (int)(i / C);
    const __nv_bfloat16* p = x + (long long)b * HW * C + c;
    float s = 0.f;
    for (int k = 0; k < HW; ++k) s += __bfloat162float(p[(long long)k * C]);
    out[i] = s / (float)HW;
  }
}

// one block per row: max, sum of exp (block tree reductions in a fixed order), then the quotients
__global__ void __launch_bounds__(256) softmax_rows_kernel(const float* __restrict__ x, float* __restrict__ y, int N) {
  __shared__ float red[256];
  const float* r = x + (long long)blockIdx.x * N;
  float* o = y + (long long)blockIdx.x * N;
  float m = -INFINITY;
  for (int j = threadIdx.x; j < N; j += blockDim.x) m = fmaxf(m, r[j]);
  red[threadIdx.x] = m;
  __syncthreads();
  for (int s = blockDim.x / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] = fmaxf(red[threadIdx.x], red[threadIdx.x + s]);
    __syncthreads();
  }
  m = red[0];
  __syncthreads();
  float sum = 0.f;
  for (int j = threadIdx.x; j < N; j += blockDim.x) sum += expf(r[j] - m);
  red[threadIdx.x] = sum;
  __syncthreads();
  for (int s = blockDim.x / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  const float inv = 1.f / red[0];
  for (int j = threadIdx.x; j < N; j += blockDim.x) o[j] = expf(r[j] - m) * inv;
}

static inline unsigned grid_for(long long n) {
  const long long g = (n + 255) / 256, cap = 148LL * 16;
  return (unsigned)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace sg2

using namespace sg2;

extern "C" {

int sg2_inception_stem(const float* img, void* col, int B, int S, void* stream) {
  if (B < 1 || S < 2) SG2_FAIL(SG2_EINVAL, "inception_stem: B %d, S %d", B, S);
  const long long n = (long long)B * kIncS1 * kIncS1;
  inception_stem_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(img, reinterpret_cast<uint4*>(col), B, S);
  SG2_LAUNCH_OK("inception_stem");
}

int sg2_maxpool3s2(const void* x, void* y, int y_ctot, int B, int H, int W, int C, void* stream) {
  if (B < 1 || H < 3 || W < 3 || C < 8 || (C % 8) || y_ctot < C || (y_ctot % 8))
    SG2_FAIL(SG2_EINVAL, "maxpool3s2: B %d H %d W %d C %d y_ctot %d", B, H, W, C, y_ctot);
  const int Ho = (H - 3) / 2 + 1, Wo = (W - 3) / 2 + 1;
  pool3_kernel<0><<<grid_for((long long)B * Ho * Wo * (C / 8)), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint4*>(x), reinterpret_cast<uint4*>(y), y_ctot, B, H, W, C, Ho, Wo);
  SG2_LAUNCH_OK("maxpool3s2");
}

int sg2_avgpool3s1(const void* x, void* y, int B, int H, int W, int C, void* stream) {
  if (B < 1 || H < 1 || W < 1 || C < 8 || (C % 8)) SG2_FAIL(SG2_EINVAL, "avgpool3s1: B %d H %d W %d C %d", B, H, W, C);
  pool3_kernel<1><<<grid_for((long long)B * H * W * (C / 8)), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint4*>(x), reinterpret_cast<uint4*>(y), C, B, H, W, C, H, W);
  SG2_LAUNCH_OK("avgpool3s1");
}

int sg2_global_avg(const void* x, float* out, int B, int HW, int C, void* stream) {
  if (B < 1 || HW < 1 || C < 1) SG2_FAIL(SG2_EINVAL, "global_avg: B %d HW %d C %d", B, HW, C);
  global_avg_kernel<<<grid_for((long long)B * C), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(x), out, B, HW, C);
  SG2_LAUNCH_OK("global_avg");
}

int sg2_softmax_rows(const float* x, float* y, int M, int N, void* stream) {
  if (M < 1 || N < 1) SG2_FAIL(SG2_EINVAL, "softmax_rows: M %d N %d", M, N);
  softmax_rows_kernel<<<M, 256, 0, (cudaStream_t)stream>>>(x, y, N);
  SG2_LAUNCH_OK("softmax_rows");
}

}  // extern "C"
