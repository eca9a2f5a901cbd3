// Depth error of rendered eval frames against ground-truth depth on the device (sm_100a): per image and region the
// standard monocular-depth metrics (abs_rel, sq_rel, rmse, rmse_log, delta < 1.25^k) over the pixels with a valid
// ground truth, i.e. what utils/image_metrics.depth_metrics states in torch.  The definitions are in the header.
//
// Two launches, no host synchronisation, no allocation (graph-capturable):
//   1. stats:    per (image, block) a grid-stride pass over the image's pixels; each valid pixel's four terms are added
//                (in double, __dadd_rn) to the sums of every region it belongs to, and its threshold tests to integer
//                counts; the block reduces them in a fixed order into one partial per region;
//   2. finalize: one warp per image adds the partials of its blocks in block order and writes the [R,8] rows.
// No float atomics: two calls give bitwise-equal results.  The masked kernel keeps the whole image's sums next to the
// dynamic and static ones and adds every pixel to them in the order the unmasked kernel does, so an all-true (all-false)
// mask gives the dynamic (static) row bit for bit equal to the whole row and to the unmasked call.
#include <math.h>
#include <math_constants.h>

#include <algorithm>

#include "common.cuh"

namespace kp {

constexpr int kDepthThreads = 256;
constexpr int kDepthMaxBlocks = 128;  // per image
constexpr int kDepthPerThread = 16;

// One region's partial of one block: the sums of |e|/g, e^2/g, e^2, (log p - log g)^2 and the counts of valid pixels
// and of pixels within 1.25, 1.25^2, 1.25^3.
struct DepthPartial {
  double sum[4];
  unsigned long long count[4];
};

static int depth_blocks(int64_t HW) {
  return (int)std::min<int64_t>(kDepthMaxBlocks, std::max<int64_t>(1, ceil_div(HW, (int64_t)kDepthThreads * kDepthPerThread)));
}

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// R = 1: the whole image; R = 3: whole, dynamic (mask != 0), static.
template <int R>
__global__ void __launch_bounds__(kDepthThreads)
    depth_stats_kernel(const float* __restrict__ pred, const float* __restrict__ gt, const float* __restrict__ dir_norm,
                       const unsigned char* __restrict__ mask, int64_t HW, DepthPartial* __restrict__ partials) {
  const int b = blockIdx.y, nblk = gridDim.x;
  const int64_t off = (int64_t)b * HW;
  double s[R][4];
  unsigned int c[R][4];
#pragma unroll
  for (int r = 0; r < R; ++r)
#pragma unroll
    for (int k = 0; k < 4; ++k) s[r][k] = 0.0, c[r][k] = 0u;
  const int64_t stride = (int64_t)nblk * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += stride) {
    const float gv = dir_norm != nullptr ? __fmul_rn(__ldg(gt + off + i), __ldg(dir_norm + off + i)) : __ldg(gt + off + i);
    if (!(isfinite(gv) && gv > 0.f)) continue;
    const double pd = (double)__ldg(pred + off + i), g = (double)gv;
    const double p = pd < 1e-6 ? 1e-6 : pd;  // max(pred, 1e-6); a NaN prediction stays NaN, as torch.clamp_min keeps it
    const double e = __dsub_rn(p, g), ee = __dmul_rn(e, e);
    const double lg = __dsub_rn(log(p), log(g));
    const double t[4] = {__ddiv_rn(fabs(e), g), __ddiv_rn(ee, g), ee, __dmul_rn(lg, lg)};
    const double ratio = fmax(__ddiv_rn(p, g), __ddiv_rn(g, p));
    const unsigned int hit[4] = {1u, ratio < 1.25 ? 1u : 0u, ratio < 1.5625 ? 1u : 0u, ratio < 1.953125 ? 1u : 0u};
    const bool dyn = R == 3 && __ldg(mask + off + i) != 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (r == 1 && !dyn) continue;
      if (r == 2 && dyn) continue;
#pragma unroll
      for (int k = 0; k < 4; ++k) s[r][k] = __dadd_rn(s[r][k], t[k]), c[r][k] += hit[k];
    }
  }
  __shared__ double ss[R][4][kDepthThreads / 32];
  __shared__ unsigned long long sc[R][4][kDepthThreads / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int r = 0; r < R; ++r)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const double vs = warp_sum_d(s[r][k]);
      const unsigned long long vc = warp_sum_u64(c[r][k]);  // integers: exact in any order
      if (lane == 0) ss[r][k][warp] = vs, sc[r][k][warp] = vc;
    }
  __syncthreads();
  if (threadIdx.x < R * 4) {
    const int r = threadIdx.x / 4, k = threadIdx.x % 4;
    double tot = 0.0;
    unsigned long long cnt = 0;
    for (int w = 0; w < kDepthThreads / 32; ++w) tot += ss[r][k][w], cnt += sc[r][k][w];
    DepthPartial& part = partials[((int64_t)b * nblk + blockIdx.x) * R + r];
    part.sum[k] = tot;
    part.count[k] = cnt;
  }
}

// One warp per image: lane r * 8 + q reduces quantity q (sums 0-3, counts 4-7) of region r over the blocks in block
// order; lane r writes row r = (n_valid, abs_rel, sq_rel, rmse, rmse_log, delta1, delta2, delta3), NaN without a pixel.
__global__ void __launch_bounds__(32) depth_finalize_kernel(const DepthPartial* __restrict__ partials, int nblk, int R,
                                                           double* __restrict__ out) {
  __shared__ double s_sum[3][4];
  __shared__ unsigned long long s_cnt[3][4];
  const int b = blockIdx.x, lane = threadIdx.x;
  if (lane < R * 8) {
    const int r = lane / 8, q = lane % 8;
    const DepthPartial* p = partials + (int64_t)b * nblk * R + r;
    if (q < 4) {
      double tot = 0.0;
      for (int i = 0; i < nblk; ++i) tot += p[(int64_t)i * R].sum[q];
      s_sum[r][q] = tot;
    } else {
      unsigned long long cnt = 0;
      for (int i = 0; i < nblk; ++i) cnt += p[(int64_t)i * R].count[q - 4];
      s_cnt[r][q - 4] = cnt;
    }
  }
  __syncwarp();
  if (lane < R) {
    const int r = lane;
    double* row = out + ((int64_t)b * R + r) * 8;
    const unsigned long long n = s_cnt[r][0];
    const double nd = (double)n;
    row[0] = nd;
    if (n == 0) {
      for (int k = 1; k < 8; ++k) row[k] = CUDART_NAN;
    } else {
      row[1] = s_sum[r][0] / nd;
      row[2] = s_sum[r][1] / nd;
      row[3] = sqrt(s_sum[r][2] / nd);
      row[4] = sqrt(s_sum[r][3] / nd);
      for (int k = 1; k < 4; ++k) row[4 + k] = (double)s_cnt[r][k] / nd;
    }
  }
}

}  // namespace kp

using namespace kp;

extern "C" int64_t kp_depth_metrics_scratch_bytes(int B, int64_t HW, int masked) {
  if (B <= 0 || HW <= 0) return 0;
  return (int64_t)B * depth_blocks(HW) * (masked ? 3 : 1) * (int64_t)sizeof(DepthPartial);
}

extern "C" int kp_depth_metrics(const float* pred, const float* gt, const float* dir_norm, const uint8_t* mask, int B, int64_t HW,
                                void* scratch, double* out, void* stream) {
  KP_CHECK(B >= 0 && HW > 0, "depth_metrics: B=%d HW=%lld", B, (long long)HW);
  if (B == 0) return 0;
  KP_CHECK(pred && gt && scratch && out, "depth_metrics: NULL argument");
  KP_CHECK(B <= 65535, "depth_metrics: B=%d images in one call (at most 65535)", B);
  const int nblk = depth_blocks(HW);
  DepthPartial* partials = static_cast<DepthPartial*>(scratch);
  cudaStream_t st = as_stream(stream);
  if (mask != nullptr) {
    depth_stats_kernel<3><<<dim3(nblk, B), kDepthThreads, 0, st>>>(pred, gt, dir_norm, mask, HW, partials);
  } else {
    depth_stats_kernel<1><<<dim3(nblk, B), kDepthThreads, 0, st>>>(pred, gt, dir_norm, nullptr, HW, partials);
  }
  KP_LAUNCH_CHECK("depth_metrics(stats)");
  depth_finalize_kernel<<<B, 32, 0, st>>>(partials, nblk, mask != nullptr ? 3 : 1, out);
  KP_LAUNCH_CHECK("depth_metrics(finalize)");
  return 0;
}
