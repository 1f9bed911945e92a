// Per-frame quality metrics of the reference's test loop, on the device ("next" row 3 of the scope table).
// Reference: BasicVSR.evaluate (mmedit/models/restorers/basicvsr.py:119-153) calls, per frame,
//   tensor2img (mmedit/core/misc.py:9-74): clamp to [0,1], x255, round half to even -> uint8
//   psnr       (mmedit/core/evaluation/metrics.py:170-215): mean squared error of the uint8 images
//   ssim/_ssim (metrics.py:262-355): float64, 11x11 Gaussian window (sigma 1.5), valid part, mean of the map
// on the host, after a device->host copy of every frame.  Here the frames never leave HBM: one kernel
// accumulates the EXACT integer sum of squared uint8 differences per frame, one the float64 sum of the SSIM map
// per frame and channel (separable 11-tap passes in shared memory).  Both are HBM-bound reads of 2 x 12 B/px (fp32
// frames) or 2 x 3 B/px (uint8 frames); each operand may be either, the kernels see the same uint8 values.
#include <cstdint>

#include "pnp_ops.cuh"

namespace pnp {

namespace {

// One sample of an operand as tensor2img's uint8 value: fp32 frames are quantised (quant_u8), uint8 frames already hold
// that value.  Either way the kernels below see the same float, so the results do not depend on the operand types.
__device__ __forceinline__ float sample_u8(const float* p) { return quant_u8(__ldg(p)); }
__device__ __forceinline__ float sample_u8(const uint8_t* p) { return (float)__ldg(p); }

struct Gauss11 {
  double g[11];
};

constexpr int kTileX = 32, kTileY = 8, kWinX = kTileX + 10, kWinY = kTileY + 10;

template <typename TA, typename TB>
__global__ void __launch_bounds__(256)
sse_u8_kernel(const TA* __restrict__ a, long long a_sf, long long a_sc, long long a_sy,
              const TB* __restrict__ b, long long b_sf, long long b_sc, long long b_sy, int H, int W, int crop,
              unsigned long long* __restrict__ sse) {
  const int f = blockIdx.y;
  const int hc = H - 2 * crop, wc = W - 2 * crop;
  const long long total = 3LL * hc * wc;
  unsigned long long acc = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % wc);
    const long long r = i / wc;
    const int y = (int)(r % hc), c = (int)(r / hc);
    const float va = sample_u8(a + f * a_sf + c * a_sc + (long long)(y + crop) * a_sy + x + crop);
    const float vb = sample_u8(b + f * b_sf + c * b_sc + (long long)(y + crop) * b_sy + x + crop);
    const int d = (int)va - (int)vb;
    acc += (unsigned long long)(d * d);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  __shared__ unsigned long long part[8];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long s = 0;
    for (int i = 0; i < 8; ++i) s += part[i];
    atomicAdd(sse + f, s);
  }
}

// grid (tiles_x, tiles_y, F * n_ch); ssim_sum[f * 3 + k] accumulates channel ch_first + k
template <typename TA, typename TB>
__global__ void __launch_bounds__(256)
ssim_sum_kernel(const TA* __restrict__ a, long long a_sf, long long a_sc, long long a_sy,
                const TB* __restrict__ b, long long b_sf, long long b_sc, long long b_sy, int H, int W, int crop,
                int ch_first, int n_ch, const Gauss11 gk, double* __restrict__ ssim_sum) {
  __shared__ float sa[kWinY][kWinX], sb[kWinY][kWinX];
  __shared__ double hs[5][kWinY][kTileX];
  __shared__ double part[8];
  const int f = blockIdx.z / n_ch, k = blockIdx.z % n_ch, c = ch_first + k;
  const int hc = H - 2 * crop, wc = W - 2 * crop;          // cropped image
  const int hv = hc - 10, wv = wc - 10;                    // valid window positions
  const int x0 = blockIdx.x * kTileX, y0 = blockIdx.y * kTileY;
  const TA* pa = a + f * a_sf + c * a_sc;
  const TB* pb = b + f * b_sf + c * b_sc;
  for (int i = threadIdx.x; i < kWinY * kWinX; i += 256) {
    const int wy = i / kWinX, wx = i % kWinX;
    const int y = y0 + wy, x = x0 + wx;
    float va = 0.f, vb = 0.f;
    if (y < hc && x < wc) {
      va = sample_u8(pa + (long long)(y + crop) * a_sy + x + crop);
      vb = sample_u8(pb + (long long)(y + crop) * b_sy + x + crop);
    }
    sa[wy][wx] = va;
    sb[wy][wx] = vb;
  }
  __syncthreads();
  // horizontal 11-tap pass of the five maps (x, y, x^2, y^2, xy), float64 like the reference
  for (int i = threadIdx.x; i < kWinY * kTileX; i += 256) {
    const int wy = i / kTileX, tx = i % kTileX;
    double s1 = 0, s2 = 0, s11 = 0, s22 = 0, s12 = 0;
#pragma unroll
    for (int t = 0; t < 11; ++t) {
      const double g = gk.g[t], va = (double)sa[wy][tx + t], vb = (double)sb[wy][tx + t];
      s1 += g * va;
      s2 += g * vb;
      s11 += g * (va * va);
      s22 += g * (vb * vb);
      s12 += g * (va * vb);
    }
    hs[0][wy][tx] = s1;
    hs[1][wy][tx] = s2;
    hs[2][wy][tx] = s11;
    hs[3][wy][tx] = s22;
    hs[4][wy][tx] = s12;
  }
  __syncthreads();
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  double val = 0.0;
  if (x0 + tx < wv && y0 + ty < hv) {
    double m[5] = {0, 0, 0, 0, 0};
#pragma unroll
    for (int t = 0; t < 11; ++t) {
      const double g = gk.g[t];
#pragma unroll
      for (int q = 0; q < 5; ++q) m[q] += g * hs[q][ty + t][tx];
    }
    const double C1 = (0.01 * 255) * (0.01 * 255), C2 = (0.03 * 255) * (0.03 * 255);
    const double mu1_sq = m[0] * m[0], mu2_sq = m[1] * m[1], mu12 = m[0] * m[1];
    const double v1 = m[2] - mu1_sq, v2 = m[3] - mu2_sq, v12 = m[4] - mu12;
    val = ((2 * mu12 + C1) * (2 * v12 + C2)) / ((mu1_sq + mu2_sq + C1) * (v1 + v2 + C2));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) val += __shfl_down_sync(0xffffffffu, val, o);
  if (tx == 0) part[ty] = val;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0;
    for (int i = 0; i < 8; ++i) s += part[i];
    atomicAdd(ssim_sum + f * 3 + k, s);
  }
}

template <typename TA, typename TB>
void launch_quality_kernels(const void* a, long long a_sf, long long a_sc, long long a_sy, const void* b, long long b_sf,
                            long long b_sc, long long b_sy, int F, int H, int W, int crop, int ch_first, int n_ch,
                            const Gauss11& gk, unsigned long long* sse, double* ssim_sum, int num_sms,
                            cudaStream_t stream) {
  const TA* pa = static_cast<const TA*>(a);
  const TB* pb = static_cast<const TB*>(b);
  const int hc = H - 2 * crop, wc = W - 2 * crop;
  const long long total = 3LL * hc * wc;
  int blocks = (int)((total + 256 * 8 - 1) / (256 * 8));
  if (blocks > 4 * num_sms) blocks = 4 * num_sms;
  if (blocks < 1) blocks = 1;
  sse_u8_kernel<TA, TB><<<dim3(blocks, F), 256, 0, stream>>>(pa, a_sf, a_sc, a_sy, pb, b_sf, b_sc, b_sy, H, W, crop, sse);
  const int hv = hc - 10, wv = wc - 10;
  dim3 grid((wv + kTileX - 1) / kTileX, (hv + kTileY - 1) / kTileY, F * n_ch);
  ssim_sum_kernel<TA, TB><<<grid, 256, 0, stream>>>(pa, a_sf, a_sc, a_sy, pb, b_sf, b_sc, b_sy, H, W, crop, ch_first,
                                                    n_ch, gk, ssim_sum);
}

}  // namespace

cudaError_t launch_frame_quality(const void* a, bool a_u8, long long a_sf, long long a_sc, long long a_sy,
                                 const void* b, bool b_u8, long long b_sf, long long b_sc, long long b_sy, int F, int H,
                                 int W, int crop, int ch_first, int n_ch, const double* gauss11,
                                 unsigned long long* sse, double* ssim_sum, int num_sms, cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(sse, 0, sizeof(unsigned long long) * F, stream);
  if (e != cudaSuccess) return e;
  e = cudaMemsetAsync(ssim_sum, 0, sizeof(double) * 3 * F, stream);
  if (e != cudaSuccess) return e;
  Gauss11 gk;
  for (int i = 0; i < 11; ++i) gk.g[i] = gauss11[i];
  auto run = a_u8 ? (b_u8 ? launch_quality_kernels<uint8_t, uint8_t> : launch_quality_kernels<uint8_t, float>)
                  : (b_u8 ? launch_quality_kernels<float, uint8_t> : launch_quality_kernels<float, float>);
  run(a, a_sf, a_sc, a_sy, b, b_sf, b_sc, b_sy, F, H, W, crop, ch_first, n_ch, gk, sse, ssim_sum, num_sms, stream);
  return cudaGetLastError();
}

}  // namespace pnp
