// Eval-image metrics on the device (sm_100a): per image of a batch, PSNR (data_range 1) and SSIM (torchmetrics defaults:
// 11x11 gaussian window, sigma 1.5, k1 0.01, k2 0.03, data_range = max(range(pred), range(target)) of that image), i.e.
// what utils/image_metrics.py computes one [1,3,H,W] image at a time (NS/models/kplanes.py:454-515).
//
// Inputs are the renderer's / image cache's layout, fp32 [B,H,W,3], not permuted.  image_metrics.ssim reflect-pads by 5
// and crops 5 from every side of the map, so every value it averages comes from a window lying wholly inside the image:
// the mean here runs over the (H-10)*(W-10)*3 interior windows and needs no padding.
//
// Three launches, no host synchronisation, no allocation (graph-capturable):
//   1. stats:    per (image, block) min / max of pred and target and the sum of squared errors (double);
//   2. ssim:     per (image, tile) the sum of the SSIM map over a 32x16 tile of window positions: the tile plus a 10-pixel
//                halo sits in shared memory, the gaussian is applied separably (rows, then columns) to the five moments
//                mu_p, mu_t, E[p^2], E[t^2], E[pt] of each channel; C1 / C2 come from the image's stats partials;
//   3. finalize: one block per image reduces both sets of partials in a fixed order.
// No float atomics: two calls give bitwise-equal results.
//
// kp_image_metrics_masked runs the same three launches with a uint8 [B,H,W] mask (non-zero: the dynamic region) and
// reports (psnr, ssim) of the masked region and of its complement.  The stats pass splits its sum of squared errors by
// the mask of each value's pixel and counts the masked values; the SSIM pass splits its sum by the mask of each window's
// centre pixel (y+5, x+5) and counts the masked windows.  Every value is added to exactly one of the two sums in the
// order the unmasked kernels add it, and C1 / C2 still come from the whole image, so an all-true (all-false) mask gives
// the dynamic (static) pair bit for bit equal to kp_image_metrics.  A region without a value has NaN metrics.
#include <float.h>
#include <math.h>
#include <math_constants.h>

#include <algorithm>

#include "common.cuh"

namespace kp {

constexpr int kMetricsThreads = 256;
constexpr int kStatsMaxBlocks = 128;  // per image
constexpr int kStatsPerThread = 16;
constexpr int kWin = 11, kHalf = 5;
constexpr int kTileX = 32, kTileY = 16;  // window positions per SSIM block
constexpr int kInX = kTileX + kWin - 1, kInY = kTileY + kWin - 1;

struct MetricsLayout {
  int stats_blocks, tiles_x, tiles_y;
  int64_t minmax_off, sse_off, ssim_off, bytes;
  int64_t sse_static_off, count_off, ssim_static_off, windows_off;  // masked only
};

static MetricsLayout metrics_layout(int B, int H, int W, bool masked = false) {
  MetricsLayout l;
  const int64_t n = (int64_t)H * W * 3;
  l.stats_blocks = (int)std::min<int64_t>(kStatsMaxBlocks, std::max<int64_t>(1, ceil_div(n, (int64_t)kMetricsThreads * kStatsPerThread)));
  l.tiles_x = (int)ceil_div(std::max(W - 10, 0), kTileX);
  l.tiles_y = (int)ceil_div(std::max(H - 10, 0), kTileY);
  const int64_t nb = (int64_t)B * l.stats_blocks;
  l.minmax_off = 0;                                // float4 [B, stats_blocks]
  l.sse_off = l.minmax_off + nb * 16;              // double [B, stats_blocks]
  l.ssim_off = l.sse_off + nb * 8;                 // double [B, tiles_y * tiles_x]
  l.bytes = l.ssim_off + (int64_t)B * l.tiles_x * l.tiles_y * 8;
  if (masked) {
    const int64_t nt = (int64_t)B * l.tiles_x * l.tiles_y;
    l.sse_static_off = l.bytes;                    // double [B, stats_blocks]
    l.count_off = l.sse_static_off + nb * 8;       // double [B, stats_blocks]: masked values (3 per pixel)
    l.ssim_static_off = l.count_off + nb * 8;      // double [B, tiles_y * tiles_x]
    l.windows_off = l.ssim_static_off + nt * 8;    // double [B, tiles_y * tiles_x]: masked windows (3 per position)
    l.bytes = l.windows_off + nt * 8;
  }
  return l;
}

// The masked stats kernel's extra arguments: the uint8 [B,H,W] mask and the partials of the static region and of the
// count.  They are a trailing parameter pack, empty for kp_image_metrics, whose kernel thereby keeps its parameters and
// code.
struct MaskedStats {
  const unsigned char* mask;
  double* sse_static;  // [B, stats_blocks]
  double* count;       // [B, stats_blocks]: masked values, 3 per pixel
};

// The one argument of the masked kernel's pack (named only where the pack is not empty: a local copy of it in the
// unmasked kernel changes that kernel's register assignment).
template <typename T>
__device__ __forceinline__ const T& only(const T& t) { return t; }

// min(pred), max(pred), min(target), max(target) and sum (pred - target)^2 over this block's share of one image.
// Masked: the sum runs over the values whose pixel has a non-zero mask byte, sse_static gets the rest and count the
// number of masked values.
template <bool kMasked, typename... Masked>
__global__ void __launch_bounds__(kMetricsThreads) metrics_stats_kernel(const float* __restrict__ pred, const float* __restrict__ target,
                                                                       int64_t n, float4* __restrict__ minmax, double* __restrict__ sse,
                                                                       Masked... masked) {
  const int b = blockIdx.y, nblk = gridDim.x;
  const float* p = pred + (int64_t)b * n;
  const float* t = target + (int64_t)b * n;
  float pmin = FLT_MAX, pmax = -FLT_MAX, tmin = FLT_MAX, tmax = -FLT_MAX;
  double s = 0.0, s_static = 0.0, c = 0.0;
  int64_t cnt = 0;
  const int64_t stride = (int64_t)nblk * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float pv = __ldg(p + i), tv = __ldg(t + i);
    pmin = fminf(pmin, pv);
    pmax = fmaxf(pmax, pv);
    tmin = fminf(tmin, tv);
    tmax = fmaxf(tmax, tv);
    const double d = (double)pv - (double)tv;
    if constexpr (kMasked) {
      if (__ldg(only(masked...).mask + (int64_t)b * (n / 3) + i / 3)) {
        s = fma(d, d, s);
        ++cnt;
      } else {
        s_static = fma(d, d, s_static);
      }
    } else {
      s = fma(d, d, s);
    }
  }
  __shared__ float4 sm[kMetricsThreads / 32];
  __shared__ double ss[kMasked ? 3 : 1][kMetricsThreads / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    pmin = fminf(pmin, __shfl_xor_sync(0xffffffffu, pmin, o));
    pmax = fmaxf(pmax, __shfl_xor_sync(0xffffffffu, pmax, o));
    tmin = fminf(tmin, __shfl_xor_sync(0xffffffffu, tmin, o));
    tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, o));
  }
  s = warp_sum_d(s);
  if constexpr (kMasked) {
    s_static = warp_sum_d(s_static);
    c = warp_sum_d((double)cnt);  // integers: exact in any order
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    sm[warp] = make_float4(pmin, pmax, tmin, tmax);
    ss[0][warp] = s;
    if constexpr (kMasked) ss[1][warp] = s_static, ss[2][warp] = c;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float4 m = sm[0];
    double tot = ss[0][0], tot_static = 0.0, tot_c = 0.0;
    if constexpr (kMasked) tot_static = ss[1][0], tot_c = ss[2][0];
    for (int w = 1; w < kMetricsThreads / 32; ++w) {
      m = make_float4(fminf(m.x, sm[w].x), fmaxf(m.y, sm[w].y), fminf(m.z, sm[w].z), fmaxf(m.w, sm[w].w));
      tot += ss[0][w];
      if constexpr (kMasked) tot_static += ss[1][w], tot_c += ss[2][w];
    }
    minmax[(int64_t)b * nblk + blockIdx.x] = m;
    sse[(int64_t)b * nblk + blockIdx.x] = tot;
    if constexpr (kMasked) {
      only(masked...).sse_static[(int64_t)b * nblk + blockIdx.x] = tot_static;
      only(masked...).count[(int64_t)b * nblk + blockIdx.x] = tot_c;
    }
  }
}

// One block = kTileY x kTileX window positions (top-left corners) of one image, all three channels.
__global__ void __launch_bounds__(kMetricsThreads) metrics_ssim_kernel(const float* __restrict__ pred, const float* __restrict__ target,
                                                                      int H, int W, const float4* __restrict__ minmax, int stats_blocks,
                                                                      double* __restrict__ ssim_part) {
  __shared__ float s_in[2][3][kInY][kInX];         // pred / target, channel-major
  __shared__ float s_h[5][kInY][kTileX];           // row-filtered moments of one channel
  __shared__ float s_c[2];
  __shared__ float s_g[kWin];
  __shared__ double s_red[kMetricsThreads / 32];
  const int b = blockIdx.z;
  const int x0 = blockIdx.x * kTileX, y0 = blockIdx.y * kTileY;
  const int tid = threadIdx.x;
  const int64_t img_off = (int64_t)b * H * W * 3;

  if (tid < 32) {  // data_range of this image from its stats partials (min / max: exact in any order)
    float pmin = FLT_MAX, pmax = -FLT_MAX, tmin = FLT_MAX, tmax = -FLT_MAX;
    for (int i = tid; i < stats_blocks; i += 32) {
      const float4 m = minmax[(int64_t)b * stats_blocks + i];
      pmin = fminf(pmin, m.x), pmax = fmaxf(pmax, m.y), tmin = fminf(tmin, m.z), tmax = fmaxf(tmax, m.w);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      pmin = fminf(pmin, __shfl_xor_sync(0xffffffffu, pmin, o));
      pmax = fmaxf(pmax, __shfl_xor_sync(0xffffffffu, pmax, o));
      tmin = fminf(tmin, __shfl_xor_sync(0xffffffffu, tmin, o));
      tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, o));
    }
    if (tid == 0) {
      // image_metrics.ssim: python floats from max(pred range, target range); C = (k * data_range)^2 in double
      const double range = fmax((double)(pmax - pmin), (double)(tmax - tmin));
      s_c[0] = (float)((0.01 * range) * (0.01 * range));
      s_c[1] = (float)((0.03 * range) * (0.03 * range));
    }
    if (tid < kWin) {  // exp(-(d / 1.5)^2 / 2), d = -5..5, normalised by its sum
      double sum = 0.0;
      for (int k = 0; k < kWin; ++k) {
        const double d = (k - kHalf) / 1.5;
        sum += exp(-d * d / 2.0);
      }
      const double d = (tid - kHalf) / 1.5;
      s_g[tid] = (float)(exp(-d * d / 2.0) / sum);
    }
  }
  // tile + halo, clamped at the right / bottom edge (clamped pixels only feed window positions outside the map)
  for (int i = tid; i < kInY * kInX * 3; i += kMetricsThreads) {
    const int r = i / (kInX * 3), rem = i - r * (kInX * 3);
    const int col = rem / 3, c = rem - col * 3;
    const int y = min(y0 + r, H - 1), x = min(x0 + col, W - 1);
    const int64_t g = img_off + ((int64_t)y * W + x) * 3 + c;
    s_in[0][c][r][col] = __ldg(pred + g);
    s_in[1][c][r][col] = __ldg(target + g);
  }
  __syncthreads();
  const float c1 = s_c[0], c2 = s_c[1];
  const int n_y = min(kTileY, H - 10 - y0), n_x = min(kTileX, W - 10 - x0);
  double acc = 0.0;
  for (int c = 0; c < 3; ++c) {
    for (int i = tid; i < kInY * kTileX; i += kMetricsThreads) {  // rows
      const int r = i / kTileX, x = i - r * kTileX;
      const float* pr = &s_in[0][c][r][x];
      const float* tr = &s_in[1][c][r][x];
      float mp = 0.f, mt = 0.f, pp = 0.f, tt = 0.f, pt = 0.f;
#pragma unroll
      for (int k = 0; k < kWin; ++k) {
        const float g = s_g[k], pv = pr[k], tv = tr[k];
        mp = fmaf(g, pv, mp);
        mt = fmaf(g, tv, mt);
        pp = fmaf(g, pv * pv, pp);
        tt = fmaf(g, tv * tv, tt);
        pt = fmaf(g, pv * tv, pt);
      }
      s_h[0][r][x] = mp, s_h[1][r][x] = mt, s_h[2][r][x] = pp, s_h[3][r][x] = tt, s_h[4][r][x] = pt;
    }
    __syncthreads();
    for (int i = tid; i < kTileY * kTileX; i += kMetricsThreads) {  // columns, then the SSIM formula of image_metrics.ssim
      const int y = i / kTileX, x = i - y * kTileX;
      if (y >= n_y || x >= n_x) continue;
      float m[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int k = 0; k < kWin; ++k) {
        const float g = s_g[k];
#pragma unroll
        for (int j = 0; j < 5; ++j) m[j] = fmaf(g, s_h[j][y + k][x], m[j]);
      }
      const float mu_p = m[0], mu_t = m[1];
      const float sig_p = m[2] - mu_p * mu_p, sig_t = m[3] - mu_t * mu_t, sig_pt = m[4] - mu_p * mu_t;
      const float num = (2.f * mu_p * mu_t + c1) * (2.f * sig_pt + c2);
      const float den = (mu_p * mu_p + mu_t * mu_t + c1) * (sig_p + sig_t + c2);
      acc += (double)(num / den);
    }
    __syncthreads();
  }
  acc = warp_sum_d(acc);
  if ((tid & 31) == 0) s_red[tid >> 5] = acc;
  __syncthreads();
  if (tid == 0) {
    double tot = 0.0;
    for (int w = 0; w < kMetricsThreads / 32; ++w) tot += s_red[w];
    ssim_part[((int64_t)b * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x] = tot;
  }
}

// metrics_ssim_kernel with the mask: ssim_part sums the windows whose centre pixel (y+5, x+5) has a non-zero mask byte,
// ssim_static the others, and windows counts the masked windows (one per channel).  Only those sums differ from
// metrics_ssim_kernel.  It is a kernel of its own because a template shared with metrics_ssim_kernel changed that
// kernel's register assignment.
__global__ void __launch_bounds__(kMetricsThreads)
    metrics_ssim_masked_kernel(const float* __restrict__ pred, const float* __restrict__ target, int H, int W,
                               const float4* __restrict__ minmax, int stats_blocks, const unsigned char* __restrict__ mask,
                               double* __restrict__ ssim_part, double* __restrict__ ssim_static, double* __restrict__ windows) {
  __shared__ float s_in[2][3][kInY][kInX];         // pred / target, channel-major
  __shared__ float s_h[5][kInY][kTileX];           // row-filtered moments of one channel
  __shared__ float s_c[2];
  __shared__ float s_g[kWin];
  __shared__ double s_red[3][kMetricsThreads / 32];
  const int b = blockIdx.z;
  const int x0 = blockIdx.x * kTileX, y0 = blockIdx.y * kTileY;
  const int tid = threadIdx.x;
  const int64_t img_off = (int64_t)b * H * W * 3;

  if (tid < 32) {  // data_range of this image from its stats partials (min / max: exact in any order)
    float pmin = FLT_MAX, pmax = -FLT_MAX, tmin = FLT_MAX, tmax = -FLT_MAX;
    for (int i = tid; i < stats_blocks; i += 32) {
      const float4 m = minmax[(int64_t)b * stats_blocks + i];
      pmin = fminf(pmin, m.x), pmax = fmaxf(pmax, m.y), tmin = fminf(tmin, m.z), tmax = fmaxf(tmax, m.w);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      pmin = fminf(pmin, __shfl_xor_sync(0xffffffffu, pmin, o));
      pmax = fmaxf(pmax, __shfl_xor_sync(0xffffffffu, pmax, o));
      tmin = fminf(tmin, __shfl_xor_sync(0xffffffffu, tmin, o));
      tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, o));
    }
    if (tid == 0) {
      // image_metrics.ssim: python floats from max(pred range, target range); C = (k * data_range)^2 in double
      const double range = fmax((double)(pmax - pmin), (double)(tmax - tmin));
      s_c[0] = (float)((0.01 * range) * (0.01 * range));
      s_c[1] = (float)((0.03 * range) * (0.03 * range));
    }
    if (tid < kWin) {  // exp(-(d / 1.5)^2 / 2), d = -5..5, normalised by its sum
      double sum = 0.0;
      for (int k = 0; k < kWin; ++k) {
        const double d = (k - kHalf) / 1.5;
        sum += exp(-d * d / 2.0);
      }
      const double d = (tid - kHalf) / 1.5;
      s_g[tid] = (float)(exp(-d * d / 2.0) / sum);
    }
  }
  // tile + halo, clamped at the right / bottom edge (clamped pixels only feed window positions outside the map)
  for (int i = tid; i < kInY * kInX * 3; i += kMetricsThreads) {
    const int r = i / (kInX * 3), rem = i - r * (kInX * 3);
    const int col = rem / 3, c = rem - col * 3;
    const int y = min(y0 + r, H - 1), x = min(x0 + col, W - 1);
    const int64_t g = img_off + ((int64_t)y * W + x) * 3 + c;
    s_in[0][c][r][col] = __ldg(pred + g);
    s_in[1][c][r][col] = __ldg(target + g);
  }
  __syncthreads();
  const float c1 = s_c[0], c2 = s_c[1];
  const int n_y = min(kTileY, H - 10 - y0), n_x = min(kTileX, W - 10 - x0);
  const unsigned char* mk = mask + (int64_t)b * H * W + (int64_t)(y0 + kHalf) * W + x0 + kHalf;
  double acc[3] = {0.0, 0.0, 0.0};  // masked sum, static sum, masked windows
  for (int c = 0; c < 3; ++c) {
    for (int i = tid; i < kInY * kTileX; i += kMetricsThreads) {  // rows
      const int r = i / kTileX, x = i - r * kTileX;
      const float* pr = &s_in[0][c][r][x];
      const float* tr = &s_in[1][c][r][x];
      float mp = 0.f, mt = 0.f, pp = 0.f, tt = 0.f, pt = 0.f;
#pragma unroll
      for (int k = 0; k < kWin; ++k) {
        const float g = s_g[k], pv = pr[k], tv = tr[k];
        mp = fmaf(g, pv, mp);
        mt = fmaf(g, tv, mt);
        pp = fmaf(g, pv * pv, pp);
        tt = fmaf(g, tv * tv, tt);
        pt = fmaf(g, pv * tv, pt);
      }
      s_h[0][r][x] = mp, s_h[1][r][x] = mt, s_h[2][r][x] = pp, s_h[3][r][x] = tt, s_h[4][r][x] = pt;
    }
    __syncthreads();
    for (int i = tid; i < kTileY * kTileX; i += kMetricsThreads) {  // columns, then the SSIM formula of image_metrics.ssim
      const int y = i / kTileX, x = i - y * kTileX;
      if (y >= n_y || x >= n_x) continue;
      float m[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int k = 0; k < kWin; ++k) {
        const float g = s_g[k];
#pragma unroll
        for (int j = 0; j < 5; ++j) m[j] = fmaf(g, s_h[j][y + k][x], m[j]);
      }
      const float mu_p = m[0], mu_t = m[1];
      const float sig_p = m[2] - mu_p * mu_p, sig_t = m[3] - mu_t * mu_t, sig_pt = m[4] - mu_p * mu_t;
      const float num = (2.f * mu_p * mu_t + c1) * (2.f * sig_pt + c2);
      const float den = (mu_p * mu_p + mu_t * mu_t + c1) * (sig_p + sig_t + c2);
      if (__ldg(mk + (int64_t)y * W + x)) {
        acc[0] += (double)(num / den);
        acc[2] += 1.0;
      } else {
        acc[1] += (double)(num / den);
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    acc[r] = warp_sum_d(acc[r]);  // the window count is an integer: exact in any order
    if ((tid & 31) == 0) s_red[r][tid >> 5] = acc[r];
  }
  __syncthreads();
  if (tid == 0) {
    double* parts[3] = {ssim_part, ssim_static, windows};
    for (int r = 0; r < 3; ++r) {
      double tot = 0.0;
      for (int w = 0; w < kMetricsThreads / 32; ++w) tot += s_red[r][w];
      parts[r][((int64_t)b * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x] = tot;
    }
  }
}


// Fixed-order block sum of n doubles (every thread strides, then a fixed tree): the same bits on every call.
__device__ double block_sum_fixed(const double* v, int n, double* s_red) {
  double a = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) a += v[i];
  a = warp_sum_d(a);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = a;
  __syncthreads();
  double tot = 0.0;
  for (int w = 0; w < kMetricsThreads / 32; ++w) tot += s_red[w];
  __syncthreads();
  return tot;
}

__global__ void __launch_bounds__(kMetricsThreads) metrics_finalize_kernel(const double* __restrict__ sse, int stats_blocks,
                                                                          const double* __restrict__ ssim_part, int n_tiles,
                                                                          int64_t n_values, int64_t n_windows, float* __restrict__ out) {
  __shared__ double s_red[kMetricsThreads / 32];
  const int b = blockIdx.x;
  const double e = block_sum_fixed(sse + (int64_t)b * stats_blocks, stats_blocks, s_red);
  const double s = block_sum_fixed(ssim_part + (int64_t)b * n_tiles, n_tiles, s_red);
  if (threadIdx.x == 0) {
    const float mse = (float)(e / (double)n_values);
    out[2 * b] = 10.f * log10f(1.f / mse);
    out[2 * b + 1] = (float)(s / (double)n_windows);
  }
}

// out[b] = (psnr, ssim) of the masked region, then of its complement; the complement's counts are the totals minus the
// masked counts.  A region without a value (no pixel; no window centre for the SSIM) gets NaN.
__global__ void __launch_bounds__(kMetricsThreads)
    metrics_finalize_masked_kernel(const double* __restrict__ sse, const double* __restrict__ sse_static, const double* __restrict__ count,
                                   int stats_blocks, const double* __restrict__ ssim_part, const double* __restrict__ ssim_static,
                                   const double* __restrict__ windows, int n_tiles, int64_t n_values, int64_t n_windows,
                                   float* __restrict__ out) {
  __shared__ double s_red[kMetricsThreads / 32];
  const int b = blockIdx.x;
  const int64_t so = (int64_t)b * stats_blocks, to = (int64_t)b * n_tiles;
  const double e[2] = {block_sum_fixed(sse + so, stats_blocks, s_red), block_sum_fixed(sse_static + so, stats_blocks, s_red)};
  const double s[2] = {block_sum_fixed(ssim_part + to, n_tiles, s_red), block_sum_fixed(ssim_static + to, n_tiles, s_red)};
  const double n_dyn = block_sum_fixed(count + so, stats_blocks, s_red);
  const double w_dyn = block_sum_fixed(windows + to, n_tiles, s_red);
  if (threadIdx.x == 0) {
    const double n[2] = {n_dyn, (double)n_values - n_dyn}, w[2] = {w_dyn, (double)n_windows - w_dyn};
    for (int r = 0; r < 2; ++r) {
      const float mse = (float)(e[r] / n[r]);
      out[4 * b + 2 * r] = n[r] > 0.0 ? 10.f * log10f(1.f / mse) : CUDART_NAN_F;
      out[4 * b + 2 * r + 1] = w[r] > 0.0 ? (float)(s[r] / w[r]) : CUDART_NAN_F;
    }
  }
}

}  // namespace kp

using namespace kp;

extern "C" int64_t kp_image_metrics_scratch_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  return metrics_layout(B, H, W).bytes;
}

extern "C" int kp_image_metrics(const float* pred, const float* target, int B, int H, int W, void* scratch, float* out,
                                void* stream) {
  if (B == 0) return 0;
  KP_CHECK(pred && target && scratch && out, "image_metrics: NULL argument");
  KP_CHECK(B > 0 && H > 0 && W > 0, "image_metrics: B=%d H=%d W=%d", B, H, W);
  KP_CHECK(H >= kWin && W >= kWin, "image_metrics: %dx%d image is smaller than the %dx%d SSIM window (the map would be empty)",
           H, W, kWin, kWin);
  KP_CHECK(B <= 65535, "image_metrics: B=%d images in one call (at most 65535)", B);
  const MetricsLayout l = metrics_layout(B, H, W);
  char* base = static_cast<char*>(scratch);
  double* sse = reinterpret_cast<double*>(base + l.sse_off);
  double* ssim_part = reinterpret_cast<double*>(base + l.ssim_off);
  float4* minmax = reinterpret_cast<float4*>(base + l.minmax_off);
  cudaStream_t st = as_stream(stream);
  const int64_t n = (int64_t)H * W * 3;
  metrics_stats_kernel<false><<<dim3(l.stats_blocks, B), kMetricsThreads, 0, st>>>(pred, target, n, minmax, sse);
  KP_LAUNCH_CHECK("image_metrics(stats)");
  metrics_ssim_kernel<<<dim3(l.tiles_x, l.tiles_y, B), kMetricsThreads, 0, st>>>(pred, target, H, W, minmax, l.stats_blocks, ssim_part);
  KP_LAUNCH_CHECK("image_metrics(ssim)");
  metrics_finalize_kernel<<<B, kMetricsThreads, 0, st>>>(sse, l.stats_blocks, ssim_part, l.tiles_x * l.tiles_y, n,
                                                         (int64_t)(H - 10) * (W - 10) * 3, out);
  KP_LAUNCH_CHECK("image_metrics(finalize)");
  return 0;
}

extern "C" int64_t kp_image_metrics_masked_scratch_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  return metrics_layout(B, H, W, true).bytes;
}

extern "C" int kp_image_metrics_masked(const float* pred, const float* target, const uint8_t* mask, int B, int H, int W,
                                       void* scratch, float* out, void* stream) {
  if (B == 0) return 0;
  KP_CHECK(pred && target && mask && scratch && out, "image_metrics_masked: NULL argument");
  KP_CHECK(B > 0 && H > 0 && W > 0, "image_metrics_masked: B=%d H=%d W=%d", B, H, W);
  KP_CHECK(H >= kWin && W >= kWin,
           "image_metrics_masked: %dx%d image is smaller than the %dx%d SSIM window (the map would be empty)", H, W, kWin, kWin);
  KP_CHECK(B <= 65535, "image_metrics_masked: B=%d images in one call (at most 65535)", B);
  const MetricsLayout l = metrics_layout(B, H, W, true);
  char* base = static_cast<char*>(scratch);
  float4* minmax = reinterpret_cast<float4*>(base + l.minmax_off);
  double* sse = reinterpret_cast<double*>(base + l.sse_off);
  double* sse_static = reinterpret_cast<double*>(base + l.sse_static_off);
  double* count = reinterpret_cast<double*>(base + l.count_off);
  double* ssim_part = reinterpret_cast<double*>(base + l.ssim_off);
  double* ssim_static = reinterpret_cast<double*>(base + l.ssim_static_off);
  double* windows = reinterpret_cast<double*>(base + l.windows_off);
  cudaStream_t st = as_stream(stream);
  const int64_t n = (int64_t)H * W * 3;
  metrics_stats_kernel<true><<<dim3(l.stats_blocks, B), kMetricsThreads, 0, st>>>(pred, target, n, minmax, sse,
                                                                             MaskedStats{mask, sse_static, count});
  KP_LAUNCH_CHECK("image_metrics_masked(stats)");
  metrics_ssim_masked_kernel<<<dim3(l.tiles_x, l.tiles_y, B), kMetricsThreads, 0, st>>>(pred, target, H, W, minmax, l.stats_blocks,
                                                                                        mask, ssim_part, ssim_static, windows);
  KP_LAUNCH_CHECK("image_metrics_masked(ssim)");
  metrics_finalize_masked_kernel<<<B, kMetricsThreads, 0, st>>>(sse, sse_static, count, l.stats_blocks, ssim_part, ssim_static,
                                                                windows, l.tiles_x * l.tiles_y, n, (int64_t)(H - 10) * (W - 10) * 3,
                                                                out);
  KP_LAUNCH_CHECK("image_metrics_masked(finalize)");
  return 0;
}
