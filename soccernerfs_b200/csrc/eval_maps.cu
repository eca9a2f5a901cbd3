// Per-pixel error maps of eval renders on the device (sm_100a): where the quantities kp_image_metrics and
// kp_depth_metrics average come from, one value per pixel, for viewing beside the render and its ground truth.
//
//   err[b,y,x]       = mean over the 3 channels of |pred - gt|;
//   ssim[b,y,x]      = the channel mean of the SSIM window centred on pixel (y, x): the window, constants and per-image
//                      data_range = max(range(pred), range(gt)) of kp_image_metrics, i.e. utils.image_metrics.ssim_map(...)
//                      [b, :, y-5, x-5] averaged over channels; NaN on the 5-pixel border, where no window lies inside;
//   depth_err[b,y,x] = |max(pred, 1e-6) - g| / g (double, rounded once to fp32), g = __fmul_rn(gt, dir_norm) or gt; NaN
//                      where g is not finite or not > 0: the clamp, product and validity rule of kp_depth_metrics.
//
// Two launches, no host synchronisation, no allocation (graph-capturable), no atomics (bitwise reproducible):
//   1. minmax: per (image, block) min / max of pred and gt, for C1 / C2;
//   2. map:    per (image, 32x16 pixel tile) the tile plus a 5-pixel halo on every side sits in shared memory; the gaussian
//              is applied separably to the five moments of each channel with the operations, in the order, of
//              image_metrics.cu's metrics_ssim_kernel, so each channel's value is the one kp_image_metrics adds to its
//              mean; err and depth_err come from the same pass.
// The map kernel is a kernel of its own rather than a variant of metrics_ssim_kernel, so that kernel's code is untouched.
#include <float.h>
#include <math.h>
#include <math_constants.h>

#include <algorithm>

#include "common.cuh"

namespace kp {

constexpr int kMapThreads = 256;
constexpr int kMapStatsMaxBlocks = 128;  // per image
constexpr int kMapStatsPerThread = 16;
constexpr int kMapWin = 11, kMapHalf = 5;
constexpr int kMapTileX = 32, kMapTileY = 16;  // pixels per map block
constexpr int kMapInX = kMapTileX + kMapWin - 1, kMapInY = kMapTileY + kMapWin - 1;

static int map_stats_blocks(int H, int W) {
  const int64_t n = (int64_t)H * W * 3;
  return (int)std::min<int64_t>(kMapStatsMaxBlocks, std::max<int64_t>(1, ceil_div(n, (int64_t)kMapThreads * kMapStatsPerThread)));
}

// min(pred), max(pred), min(gt), max(gt) over this block's share of one image (exact in any order).
__global__ void __launch_bounds__(kMapThreads) eval_maps_minmax_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                                      int64_t n, float4* __restrict__ minmax) {
  const int b = blockIdx.y, nblk = gridDim.x;
  const float* p = pred + (int64_t)b * n;
  const float* t = gt + (int64_t)b * n;
  float pmin = FLT_MAX, pmax = -FLT_MAX, tmin = FLT_MAX, tmax = -FLT_MAX;
  const int64_t stride = (int64_t)nblk * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float pv = __ldg(p + i), tv = __ldg(t + i);
    pmin = fminf(pmin, pv), pmax = fmaxf(pmax, pv), tmin = fminf(tmin, tv), tmax = fmaxf(tmax, tv);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    pmin = fminf(pmin, __shfl_xor_sync(0xffffffffu, pmin, o));
    pmax = fmaxf(pmax, __shfl_xor_sync(0xffffffffu, pmax, o));
    tmin = fminf(tmin, __shfl_xor_sync(0xffffffffu, tmin, o));
    tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, o));
  }
  __shared__ float4 sm[kMapThreads / 32];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = make_float4(pmin, pmax, tmin, tmax);
  __syncthreads();
  if (threadIdx.x == 0) {
    float4 m = sm[0];
    for (int w = 1; w < kMapThreads / 32; ++w)
      m = make_float4(fminf(m.x, sm[w].x), fmaxf(m.y, sm[w].y), fminf(m.z, sm[w].z), fmaxf(m.w, sm[w].w));
    minmax[(int64_t)b * nblk + blockIdx.x] = m;
  }
}

// One block = kMapTileY x kMapTileX pixels of one image; each thread owns two of them.
__global__ void __launch_bounds__(kMapThreads)
    eval_maps_kernel(const float* __restrict__ pred, const float* __restrict__ gt, const float* __restrict__ depth,
                     const float* __restrict__ gt_depth, const float* __restrict__ dir_norm, int H, int W,
                     const float4* __restrict__ minmax, int stats_blocks, float* __restrict__ err, float* __restrict__ ssim,
                     float* __restrict__ depth_err) {
  __shared__ float s_in[2][3][kMapInY][kMapInX];  // pred / gt, channel-major
  __shared__ float s_h[5][kMapInY][kMapTileX];    // row-filtered moments of one channel
  __shared__ float s_c[2];
  __shared__ float s_g[kMapWin];
  const int b = blockIdx.z;
  const int x0 = blockIdx.x * kMapTileX, y0 = blockIdx.y * kMapTileY;
  const int tid = threadIdx.x;
  const int64_t img_off = (int64_t)b * H * W * 3;

  if (tid < 32) {  // data_range of this image from its minmax partials, as metrics_ssim_kernel derives it
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
      const double range = fmax((double)(pmax - pmin), (double)(tmax - tmin));
      s_c[0] = (float)((0.01 * range) * (0.01 * range));
      s_c[1] = (float)((0.03 * range) * (0.03 * range));
    }
    if (tid < kMapWin) {  // exp(-(d / 1.5)^2 / 2), d = -5..5, normalised by its sum
      double sum = 0.0;
      for (int k = 0; k < kMapWin; ++k) {
        const double d = (k - kMapHalf) / 1.5;
        sum += exp(-d * d / 2.0);
      }
      const double d = (tid - kMapHalf) / 1.5;
      s_g[tid] = (float)(exp(-d * d / 2.0) / sum);
    }
  }
  // tile + halo, clamped to the image (clamped pixels only feed border windows, whose value is NaN)
  for (int i = tid; i < kMapInY * kMapInX * 3; i += kMapThreads) {
    const int r = i / (kMapInX * 3), rem = i - r * (kMapInX * 3);
    const int col = rem / 3, c = rem - col * 3;
    const int y = min(max(y0 - kMapHalf + r, 0), H - 1), x = min(max(x0 - kMapHalf + col, 0), W - 1);
    const int64_t g = img_off + ((int64_t)y * W + x) * 3 + c;
    s_in[0][c][r][col] = __ldg(pred + g);
    s_in[1][c][r][col] = __ldg(gt + g);
  }
  __syncthreads();
  const float c1 = s_c[0], c2 = s_c[1];
  constexpr int kPer = kMapTileY * kMapTileX / kMapThreads;
  float acc[kPer];
#pragma unroll
  for (int k = 0; k < kPer; ++k) acc[k] = 0.f;
  for (int c = 0; c < 3; ++c) {
    for (int i = tid; i < kMapInY * kMapTileX; i += kMapThreads) {  // rows
      const int r = i / kMapTileX, x = i - r * kMapTileX;
      const float* pr = &s_in[0][c][r][x];
      const float* tr = &s_in[1][c][r][x];
      float mp = 0.f, mt = 0.f, pp = 0.f, tt = 0.f, pt = 0.f;
#pragma unroll
      for (int k = 0; k < kMapWin; ++k) {
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
#pragma unroll
    for (int k = 0; k < kPer; ++k) {  // columns, then the SSIM formula of image_metrics.ssim
      const int i = tid + k * kMapThreads;
      const int y = i / kMapTileX, x = i - y * kMapTileX;
      float m[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int q = 0; q < kMapWin; ++q) {
        const float g = s_g[q];
#pragma unroll
        for (int j = 0; j < 5; ++j) m[j] = fmaf(g, s_h[j][y + q][x], m[j]);
      }
      const float mu_p = m[0], mu_t = m[1];
      const float sig_p = m[2] - mu_p * mu_p, sig_t = m[3] - mu_t * mu_t, sig_pt = m[4] - mu_p * mu_t;
      const float num = (2.f * mu_p * mu_t + c1) * (2.f * sig_pt + c2);
      const float den = (mu_p * mu_p + mu_t * mu_t + c1) * (sig_p + sig_t + c2);
      acc[k] = __fadd_rn(acc[k], __fdiv_rn(num, den));
    }
    __syncthreads();
  }
#pragma unroll
  for (int k = 0; k < kPer; ++k) {
    const int i = tid + k * kMapThreads;
    const int ty = i / kMapTileX, tx = i - ty * kMapTileX;
    const int y = y0 + ty, x = x0 + tx;
    if (y >= H || x >= W) continue;
    const int64_t pix = (int64_t)b * H * W + (int64_t)y * W + x;
    const bool inside = y >= kMapHalf && y < H - kMapHalf && x >= kMapHalf && x < W - kMapHalf;
    ssim[pix] = inside ? __fdiv_rn(acc[k], 3.f) : CUDART_NAN_F;
    float e = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c)
      e = __fadd_rn(e, fabsf(__fsub_rn(s_in[0][c][ty + kMapHalf][tx + kMapHalf], s_in[1][c][ty + kMapHalf][tx + kMapHalf])));
    err[pix] = __fdiv_rn(e, 3.f);
    if (depth_err != nullptr) {
      const float gv = dir_norm != nullptr ? __fmul_rn(__ldg(gt_depth + pix), __ldg(dir_norm + pix)) : __ldg(gt_depth + pix);
      float out = CUDART_NAN_F;
      if (isfinite(gv) && gv > 0.f) {
        const double pd = (double)__ldg(depth + pix), g = (double)gv;
        const double p = pd < 1e-6 ? 1e-6 : pd;  // max(pred, 1e-6); a NaN prediction stays NaN, as in kp_depth_metrics
        out = (float)__ddiv_rn(fabs(__dsub_rn(p, g)), g);
      }
      depth_err[pix] = out;
    }
  }
}

}  // namespace kp

using namespace kp;

extern "C" int64_t kp_eval_maps_scratch_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  return (int64_t)B * map_stats_blocks(H, W) * (int64_t)sizeof(float4);
}

extern "C" int kp_eval_maps(const float* pred, const float* gt, const float* depth, const float* gt_depth, const float* dir_norm,
                            int B, int H, int W, void* scratch, float* err, float* ssim, float* depth_err, void* stream) {
  KP_CHECK(B >= 0 && H > 0 && W > 0, "eval_maps: B=%d H=%d W=%d", B, H, W);
  if (B == 0) return 0;
  KP_CHECK(pred && gt && scratch && err && ssim, "eval_maps: NULL argument");
  KP_CHECK(H >= kMapWin && W >= kMapWin, "eval_maps: %dx%d image is smaller than the %dx%d SSIM window (the map would be empty)",
           H, W, kMapWin, kMapWin);
  KP_CHECK(B <= 65535, "eval_maps: B=%d images in one call (at most 65535)", B);
  KP_CHECK((depth == nullptr) == (gt_depth == nullptr) && (depth == nullptr) == (depth_err == nullptr),
           "eval_maps: depth, gt_depth and depth_err must be given together");
  KP_CHECK(dir_norm == nullptr || depth != nullptr, "eval_maps: dir_norm needs depth");
  const int nblk = map_stats_blocks(H, W);
  float4* minmax = static_cast<float4*>(scratch);
  cudaStream_t st = as_stream(stream);
  eval_maps_minmax_kernel<<<dim3(nblk, B), kMapThreads, 0, st>>>(pred, gt, (int64_t)H * W * 3, minmax);
  KP_LAUNCH_CHECK("eval_maps(minmax)");
  eval_maps_kernel<<<dim3((unsigned)ceil_div(W, kMapTileX), (unsigned)ceil_div(H, kMapTileY), B), kMapThreads, 0, st>>>(
      pred, gt, depth, gt_depth, dir_norm, H, W, minmax, nblk, err, ssim, depth_err);
  KP_LAUNCH_CHECK("eval_maps(map)");
  return 0;
}
