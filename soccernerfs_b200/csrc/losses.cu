// Loss kernels (sm_100a).
//   kp_distortion_*  : lossfun_distortion, NS/model_components/losses.py:125-136 (O(S^2) per ray, one warp per ray)
//   kp_interlevel_*  : outer / lossfun_outer, losses.py:46-95 (two searchsorted(side="right") + cumsum differences)
#include "common.cuh"

namespace kp {

constexpr int kRaysPerBlock = 4;

__global__ void __launch_bounds__(32 * kRaysPerBlock) distortion_kernel(const float* __restrict__ sdist,
                                                                        const float* __restrict__ w, int64_t N, int S,
                                                                        const float* __restrict__ grad_per_ray,
                                                                        float* __restrict__ loss, float* __restrict__ gw) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t n = (int64_t)blockIdx.x * kRaysPerBlock + warp;
  if (n >= N) return;
  float* s_ut = smem + (size_t)warp * 2 * S;
  float* s_w = s_ut + S;
  const float* t = sdist + n * (S + 1);
  for (int i = lane; i < S; i += 32) {
    s_ut[i] = (t[i + 1] + t[i]) * 0.5f;
    s_w[i] = w[n * S + i];
  }
  __syncwarp();
  float acc = 0.f;
  const float gn = grad_per_ray != nullptr ? grad_per_ray[n] : 0.f;
  for (int i = lane; i < S; i += 32) {
    const float ui = s_ut[i], wi = s_w[i];
    float inner = 0.f;
    for (int j = 0; j < S; ++j) inner = fmaf(s_w[j], fabsf(ui - s_ut[j]), inner);
    const float width = t[i + 1] - t[i];
    if (gw != nullptr) gw[n * S + i] = gn * (2.f * inner + 2.f * wi * width / 3.f);
    acc += wi * inner + wi * wi * width / 3.f;
  }
  acc = warp_sum(acc);
  if (loss != nullptr && lane == 0) loss[n] = acc;
}

// upper_bound over a sorted smem row: number of entries <= v  (torch.searchsorted side="right")
__device__ __forceinline__ int upper_bound(const float* a, int n, float v) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] <= v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

template <bool BWD>
__global__ void __launch_bounds__(32 * kRaysPerBlock) interlevel_kernel(const float* __restrict__ c,
                                                                        const float* __restrict__ w,
                                                                        const float* __restrict__ cp,
                                                                        const float* __restrict__ wp,
                                                                        const float* __restrict__ gloss, int64_t N, int S,
                                                                        int Sp, float* __restrict__ loss,
                                                                        float* __restrict__ gwp) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t n = (int64_t)blockIdx.x * kRaysPerBlock + warp;
  if (n >= N) return;
  float* s_cp = smem + (size_t)warp * 3 * (Sp + 1);  // [Sp+1]
  float* s_cy = s_cp + (Sp + 1);                     // [Sp+1] = [0, cumsum(wp)]
  float* s_e = s_cy + (Sp + 1);                      // [Sp+1] scatter buffer (bwd)
  for (int i = lane; i <= Sp; i += 32) {
    s_cp[i] = cp[n * (Sp + 1) + i];
    s_e[i] = 0.f;
  }
  // cumsum(wp): double accumulate, fp32 per element (losses.py:64)
  const int epl = (Sp + 31) / 32;
  const int i0 = lane * epl, i1 = min(Sp, i0 + epl);
  double part = 0.0;
  for (int i = i0; i < i1; ++i) part += (double)wp[n * Sp + i];
  double run = warp_excl_scan_d(part, lane);
  for (int i = i0; i < i1; ++i) {
    run += (double)wp[n * Sp + i];
    s_cy[i + 1] = (float)run;
  }
  if (lane == 0) s_cy[0] = 0.f;
  __syncwarp();
  for (int i = lane; i < S; i += 32) {
    const float c0 = c[n * (S + 1) + i], c1 = c[n * (S + 1) + i + 1], wi = w[n * S + i];
    int lo = upper_bound(s_cp, Sp, c0) - 1;      // t1_starts = cp[:-1]
    lo = min(max(lo, 0), Sp - 1);
    int hi = upper_bound(s_cp + 1, Sp, c1);      // t1_ends = cp[1:]
    hi = min(max(hi, 0), Sp - 1);
    const float w_outer = s_cy[hi + 1] - s_cy[lo];
    const float diff = fmaxf(wi - w_outer, 0.f);
    if (!BWD) {
      loss[n * S + i] = diff * diff / (wi + 1e-7f);
    } else {
      // d loss / d w_outer = -2 diff / (w + eps); d w_outer / d wp_k = [k <= hi] - [k < lo]
      const float G = gloss[n * S + i] * (-2.f * diff / (wi + 1e-7f));
      if (G != 0.f) {
        atomicAdd(&s_e[hi + 1], G);
        atomicAdd(&s_e[lo], -G);
      }
    }
  }
  if (BWD) {
    __syncwarp();
    // grad_wp[k] = sum_{j > k} E[j]: suffix scan over Sp+1 entries
    double p2 = 0.0;
    for (int i = i0; i < i1; ++i) p2 += (double)s_e[i + 1];
    const double incl = warp_incl_scan_d(p2, lane);
    const double total = __shfl_sync(0xffffffffu, incl, 31);
    double suffix = total - (incl - p2);  // sum over j >= i0+1
    for (int i = i0; i < i1; ++i) {
      gwp[n * Sp + i] = (float)suffix;
      suffix -= (double)s_e[i + 1];
    }
  }
}

__global__ void repack_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int H, int W, int to_hwc) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)C * H * W;
  if (idx >= total) return;
  // idx enumerates the destination
  if (to_hwc) {
    const int c = (int)(idx % C);
    const int64_t hw = idx / C;
    dst[idx] = src[(int64_t)c * H * W + hw];
  } else {
    const int64_t hw = idx % ((int64_t)H * W);
    const int c = (int)(idx / ((int64_t)H * W));
    dst[idx] = src[hw * C + c];
  }
}

}  // namespace kp

using namespace kp;

extern "C" int kp_distortion_fwd(const float* sdist, const float* w, int64_t N, int S, float* loss_per_ray, void* stream) {
  if (N == 0) return 0;
  KP_CHECK(sdist && w && loss_per_ray && S >= 1, "distortion_fwd: bad arguments");
  const size_t smem = (size_t)kRaysPerBlock * 2 * S * sizeof(float);
  KP_CHECK(smem <= 48 * 1024, "distortion_fwd: S=%d too large", S);
  distortion_kernel<<<(unsigned)ceil_div(N, kRaysPerBlock), 32 * kRaysPerBlock, smem, as_stream(stream)>>>(
      sdist, w, N, S, nullptr, loss_per_ray, nullptr);
  KP_LAUNCH_CHECK("distortion_fwd");
  return 0;
}

extern "C" int kp_distortion_bwd(const float* sdist, const float* w, const float* grad_per_ray, int64_t N, int S,
                                 float* grad_w, void* stream) {
  if (N == 0) return 0;
  KP_CHECK(sdist && w && grad_per_ray && grad_w && S >= 1, "distortion_bwd: bad arguments");
  const size_t smem = (size_t)kRaysPerBlock * 2 * S * sizeof(float);
  KP_CHECK(smem <= 48 * 1024, "distortion_bwd: S=%d too large", S);
  distortion_kernel<<<(unsigned)ceil_div(N, kRaysPerBlock), 32 * kRaysPerBlock, smem, as_stream(stream)>>>(
      sdist, w, N, S, grad_per_ray, nullptr, grad_w);
  KP_LAUNCH_CHECK("distortion_bwd");
  return 0;
}

extern "C" int kp_interlevel_fwd(const float* c, const float* w, const float* cp, const float* wp, int64_t N, int S,
                                 int Sp, float* loss, void* stream) {
  if (N == 0) return 0;
  KP_CHECK(c && w && cp && wp && loss && S >= 1 && Sp >= 1, "interlevel_fwd: bad arguments");
  const size_t smem = (size_t)kRaysPerBlock * 3 * (Sp + 1) * sizeof(float);
  KP_CHECK(smem <= 48 * 1024, "interlevel_fwd: Sp=%d too large", Sp);
  interlevel_kernel<false><<<(unsigned)ceil_div(N, kRaysPerBlock), 32 * kRaysPerBlock, smem, as_stream(stream)>>>(
      c, w, cp, wp, nullptr, N, S, Sp, loss, nullptr);
  KP_LAUNCH_CHECK("interlevel_fwd");
  return 0;
}

extern "C" int kp_interlevel_bwd(const float* c, const float* w, const float* cp, const float* wp, const float* grad_loss,
                                 int64_t N, int S, int Sp, float* grad_wp, void* stream) {
  if (N == 0) return 0;
  KP_CHECK(c && w && cp && wp && grad_loss && grad_wp && S >= 1 && Sp >= 1, "interlevel_bwd: bad arguments");
  const size_t smem = (size_t)kRaysPerBlock * 3 * (Sp + 1) * sizeof(float);
  KP_CHECK(smem <= 48 * 1024, "interlevel_bwd: Sp=%d too large", Sp);
  interlevel_kernel<true><<<(unsigned)ceil_div(N, kRaysPerBlock), 32 * kRaysPerBlock, smem, as_stream(stream)>>>(
      c, w, cp, wp, grad_loss, N, S, Sp, nullptr, grad_wp);
  KP_LAUNCH_CHECK("interlevel_bwd");
  return 0;
}

extern "C" int kp_repack_nchw_to_hwc(const float* src, float* dst, int C, int H, int W, void* stream) {
  KP_CHECK(src && dst, "repack: NULL argument");
  const int64_t total = (int64_t)C * H * W;
  repack_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, as_stream(stream)>>>(src, dst, C, H, W, 1);
  KP_LAUNCH_CHECK("repack_nchw_to_hwc");
  return 0;
}

extern "C" int kp_repack_hwc_to_nchw(const float* src, float* dst, int C, int H, int W, void* stream) {
  KP_CHECK(src && dst, "repack: NULL argument");
  const int64_t total = (int64_t)C * H * W;
  repack_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, as_stream(stream)>>>(src, dst, C, H, W, 0);
  KP_LAUNCH_CHECK("repack_hwc_to_nchw");
  return 0;
}
