// Frame composition on the device (sm_100a): P float panels of one rendered frame -> one uint8 [H, W*P, 3] image, the
// panels side by side in the given order (what ns-render's np.concatenate(..., axis=1) builds), each mapped exactly as
// the model's eval visualisations map it (KPlanesModel.get_image_metrics_and_images, utils/colormaps.py):
//   colour panels (rgb, median_rgb)   the value itself;
//   accumulation                      viridis[(int64)(nan_to_num(a) * 255)]                       (apply_colormap);
//   depth panels (depth, prop_depth_i) near / far = min / max of the frame's panel, d' = clip((d - near) / den, 0, 1),
//                                     den = fp32(double(far) - double(near) + 1e-10), c = turbo[(int64)(d' * 255)],
//                                     c * acc + (1 - acc)                                          (apply_depth_colormap);
// then every channel q = floor(clamp(x, 0, 1) * 255 + 0.5) (NaN -> 0).
//
// Every fp32 operation is the torch restatement's, in its order and rounding, with no FMA contraction.  torch divides a
// CUDA tensor by a Python float as a multiplication by the fp32 reciprocal of the float (BinaryDivTrueKernel.cu, CPU
// scalar operand), so the depth normalisation is (d - near) * rn(1 / den) here too.  A colour-map index outside [0, 255]
// (an accumulation above 1 + 1/255, say) makes apply_colormap assert; the kernel clamps it to the table instead.
//
// Two launches, no host synchronisation, no allocation (graph-capturable):
//   1. minmax:  per (depth panel, block) min / max of the panel (NaN-propagating like torch.min / max), skipped without
//               depth panels;
//   2. compose: per (block of 4-pixel groups, panel) the block reduces its panel's partials (min / max are exact in any
//               order), then every thread maps 4 pixels and stores 12 bytes.
#include <float.h>
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace kp {

constexpr int kComposeThreads = 256;
constexpr int kMinMaxMaxBlocks = 128;  // per depth panel
constexpr int kMinMaxPerThread = 16;

struct ComposeArgs {
  const float* panel[KP_COMPOSE_MAX_PANELS];
  const float* acc[KP_COMPOSE_MAX_PANELS];  // the accumulation a depth panel is blended with, NULL for other kinds
  int kind[KP_COMPOSE_MAX_PANELS];
  int depth_slot[KP_COMPOSE_MAX_PANELS];  // index into the min / max partials, -1 for other kinds
};

static int minmax_blocks(int64_t n) {
  return (int)std::min<int64_t>(kMinMaxMaxBlocks, std::max<int64_t>(1, ceil_div(n, (int64_t)kComposeThreads * kMinMaxPerThread)));
}

// torch.min / max: a NaN anywhere makes the result NaN
__device__ __forceinline__ float nan_min(float a, float b) { return (isnan(a) || isnan(b)) ? __int_as_float(0x7fc00000) : fminf(a, b); }
__device__ __forceinline__ float nan_max(float a, float b) { return (isnan(a) || isnan(b)) ? __int_as_float(0x7fc00000) : fmaxf(a, b); }

__global__ void __launch_bounds__(kComposeThreads) compose_minmax_kernel(const __grid_constant__ ComposeArgs args, int64_t n, int vec, float2* __restrict__ part) {
  const int p = blockIdx.y;
  const int slot = args.depth_slot[p];
  if (slot < 0) return;
  const float* d = args.panel[p];
  float lo = FLT_MAX, hi = -FLT_MAX;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t first = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (vec) {
    for (int64_t i = first; i < n / 4; i += stride) {
      const float4 v = ldg4(d + 4 * i);
      lo = nan_min(nan_min(lo, v.x), nan_min(v.y, nan_min(v.z, v.w)));
      hi = nan_max(nan_max(hi, v.x), nan_max(v.y, nan_max(v.z, v.w)));
    }
    for (int64_t i = (n / 4) * 4 + first; i < n; i += stride) {
      const float v = __ldg(d + i);
      lo = nan_min(lo, v), hi = nan_max(hi, v);
    }
  } else {
    for (int64_t i = first; i < n; i += stride) {
      const float v = __ldg(d + i);
      lo = nan_min(lo, v), hi = nan_max(hi, v);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = nan_min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = nan_max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  __shared__ float2 s[kComposeThreads / 32];
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = make_float2(lo, hi);
  __syncthreads();
  if (threadIdx.x == 0) {
    float2 m = s[0];
    for (int w = 1; w < kComposeThreads / 32; ++w) m = make_float2(nan_min(m.x, s[w].x), nan_max(m.y, s[w].y));
    part[(int64_t)slot * gridDim.x + blockIdx.x] = m;
  }
}

__device__ __forceinline__ uint32_t quantise(float x) {  // floor(clamp(x, 0, 1) * 255 + 0.5); fmaxf drops a NaN
  const float c = fminf(fmaxf(x, 0.f), 1.f);
  return (uint32_t)floorf(__fadd_rn(__fmul_rn(c, 255.f), 0.5f));
}

__device__ __forceinline__ int cmap_index(float v) {  // (int64)(v * 255), clamped to the table
  const float s = __fmul_rn(v, 255.f);
  return (int)fminf(fmaxf(s, 0.f), 255.f);
}

__global__ void __launch_bounds__(kComposeThreads) compose_frame_kernel(const __grid_constant__ ComposeArgs args, int H, int W,
                                                                        int P, int vec, const float* __restrict__ turbo,
                                                                        const float* __restrict__ viridis, const float2* __restrict__ part,
                                                                        int part_blocks, uint8_t* __restrict__ out) {
  __shared__ float s_tab[256 * 3];
  __shared__ float s_near, s_inv;
  const int p = blockIdx.y;
  const int kind = args.kind[p];
  const float* src = args.panel[p];
  const float* __restrict__ acc = args.acc[p];
  if (kind != KP_PANEL_COLOR) {
    const float* tab = kind == KP_PANEL_DEPTH ? turbo : viridis;
    for (int i = threadIdx.x; i < 256 * 3; i += kComposeThreads) s_tab[i] = __ldg(tab + i);
  }
  if (kind == KP_PANEL_DEPTH && threadIdx.x < 32) {
    const float2* mp = part + (int64_t)args.depth_slot[p] * part_blocks;
    float lo = FLT_MAX, hi = -FLT_MAX;
    for (int i = threadIdx.x; i < part_blocks; i += 32) lo = nan_min(lo, mp[i].x), hi = nan_max(hi, mp[i].y);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo = nan_min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
      hi = nan_max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (threadIdx.x == 0) {
      // apply_depth_colormap: python floats near, far; far - near + 1e-10 in double, then torch's fp32 reciprocal
      const float den = (float)((double)hi - (double)lo + 1e-10);
      s_near = lo;
      s_inv = __fdiv_rn(1.f, den);
    }
  }
  __syncthreads();
  const int64_t n = (int64_t)H * W;
  const int64_t g = (int64_t)blockIdx.x * kComposeThreads + threadIdx.x;  // group of 4 flat pixels
  const int64_t pix0 = 4 * g;
  if (pix0 >= n) return;
  const int cnt = n - pix0 < 4 ? (int)(n - pix0) : 4;
  const bool full = vec && cnt == 4;
  float in[12], a[4];
  if (kind == KP_PANEL_COLOR) {
    if (full) {
      const float4 v0 = ldg4(src + 3 * pix0), v1 = ldg4(src + 3 * pix0 + 4), v2 = ldg4(src + 3 * pix0 + 8);
      in[0] = v0.x, in[1] = v0.y, in[2] = v0.z, in[3] = v0.w, in[4] = v1.x, in[5] = v1.y;
      in[6] = v1.z, in[7] = v1.w, in[8] = v2.x, in[9] = v2.y, in[10] = v2.z, in[11] = v2.w;
    } else {
#pragma unroll
      for (int k = 0; k < 12; ++k) in[k] = k < 3 * cnt ? __ldg(src + 3 * pix0 + k) : 0.f;
    }
  } else {
    float v[4];
    if (full) {
      const float4 t = ldg4(src + pix0);
      v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k) v[k] = k < cnt ? __ldg(src + pix0 + k) : 0.f;
    }
    if (kind == KP_PANEL_DEPTH) {
      if (full) {
        const float4 t = ldg4(acc + pix0);
        a[0] = t.x, a[1] = t.y, a[2] = t.z, a[3] = t.w;
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) a[k] = k < cnt ? __ldg(acc + pix0 + k) : 0.f;
      }
    }
    const float near = s_near, inv = s_inv;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      int idx;
      if (kind == KP_PANEL_DEPTH) {
        const float dn = __fmul_rn(__fsub_rn(v[k], near), inv);
        idx = cmap_index(isnan(dn) ? 0.f : fminf(fmaxf(dn, 0.f), 1.f));  // clip keeps a NaN, nan_to_num makes it 0
      } else {
        idx = cmap_index(nan_to_num(v[k]));
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float t = s_tab[3 * idx + c];
        in[3 * k + c] = kind == KP_PANEL_DEPTH ? __fadd_rn(__fmul_rn(t, a[k]), __fsub_rn(1.f, a[k])) : t;
      }
    }
  }
  uint32_t q[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) q[k] = quantise(in[k]);
  const int64_t y = pix0 / W, x = pix0 - y * W;
  if (full && (W & 3) == 0) {  // 4 pixels of one row, 4-byte aligned: three word stores
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + ((y * P + p) * W + x) * 3);
    dst[0] = q[0] | q[1] << 8 | q[2] << 16 | q[3] << 24;
    dst[1] = q[4] | q[5] << 8 | q[6] << 16 | q[7] << 24;
    dst[2] = q[8] | q[9] << 8 | q[10] << 16 | q[11] << 24;
    return;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (k >= cnt) break;
    const int64_t pk = pix0 + k, yk = pk / W, xk = pk - yk * W;
    uint8_t* dst = out + ((yk * P + p) * W + xk) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) dst[c] = (uint8_t)q[3 * k + c];
  }
}

// accumulations: HOST array [P]; entry p is read for a depth panel p only
static int compose_frame(const float* const* panels, const int* kinds, const float* const* accumulations, int P, int H, int W,
                         const float* turbo, const float* viridis, void* scratch, uint8_t* out, void* stream) {
  KP_CHECK(panels && kinds && accumulations && turbo && viridis && scratch && out, "compose_frame: NULL argument");
  KP_CHECK(P >= 1 && P <= KP_COMPOSE_MAX_PANELS, "compose_frame: P=%d panels (1..%d)", P, KP_COMPOSE_MAX_PANELS);
  KP_CHECK(H > 0 && W > 0, "compose_frame: H=%d W=%d", H, W);
  const int64_t n = (int64_t)H * W;
  KP_CHECK(ceil_div(n, 4 * (int64_t)kComposeThreads) <= 0x7fffffff, "compose_frame: %dx%d frame is too large", H, W);
  ComposeArgs args;
  int n_depth = 0;
  bool vec = ((uintptr_t)out & 3) == 0;
  for (int p = 0; p < KP_COMPOSE_MAX_PANELS; ++p) {
    args.panel[p] = nullptr, args.acc[p] = nullptr, args.kind[p] = KP_PANEL_COLOR, args.depth_slot[p] = -1;
    if (p >= P) continue;
    KP_CHECK(panels[p], "compose_frame: panel %d is NULL", p);
    KP_CHECK(kinds[p] == KP_PANEL_COLOR || kinds[p] == KP_PANEL_ACCUMULATION || kinds[p] == KP_PANEL_DEPTH,
             "compose_frame: panel %d has kind %d (0 colour, 1 accumulation, 2 depth)", p, kinds[p]);
    args.panel[p] = panels[p], args.kind[p] = kinds[p];
    if (kinds[p] == KP_PANEL_DEPTH) {
      KP_CHECK(accumulations[p], "compose_frame: depth panel %d needs an accumulation", p);
      args.depth_slot[p] = n_depth++;
      args.acc[p] = accumulations[p];
      vec = vec && ((uintptr_t)accumulations[p] & 15) == 0;
    }
    vec = vec && ((uintptr_t)panels[p] & 15) == 0;
  }
  const int mm_blocks = minmax_blocks(n);
  float2* part = static_cast<float2*>(scratch);
  cudaStream_t st = as_stream(stream);
  if (n_depth > 0) {
    compose_minmax_kernel<<<dim3(mm_blocks, P), kComposeThreads, 0, st>>>(args, n, vec ? 1 : 0, part);
    KP_LAUNCH_CHECK("compose_frame(minmax)");
  }
  const int blocks = (int)ceil_div(n, 4 * (int64_t)kComposeThreads);
  compose_frame_kernel<<<dim3(blocks, P), kComposeThreads, 0, st>>>(args, H, W, P, vec ? 1 : 0, turbo, viridis, part, mm_blocks,
                                                                     out);
  KP_LAUNCH_CHECK("compose_frame");
  return 0;
}

}  // namespace kp

using namespace kp;

extern "C" int64_t kp_compose_frame_scratch_bytes(int H, int W, int P) {
  if (H <= 0 || W <= 0 || P <= 0) return 0;
  return (int64_t)P * minmax_blocks((int64_t)H * W) * (int64_t)sizeof(float2);
}

extern "C" int kp_compose_frame(const float* const* panels, const int* kinds, int P, int H, int W, const float* accumulation,
                                const float* turbo, const float* viridis, void* scratch, uint8_t* out, void* stream) {
  const float* accs[KP_COMPOSE_MAX_PANELS];
  for (int p = 0; p < KP_COMPOSE_MAX_PANELS; ++p) accs[p] = accumulation;
  return compose_frame(panels, kinds, accs, P, H, W, turbo, viridis, scratch, out, stream);
}

extern "C" int kp_compose_frame_accs(const float* const* panels, const int* kinds, const float* const* accumulations, int P,
                                     int H, int W, const float* turbo, const float* viridis, void* scratch, uint8_t* out,
                                     void* stream) {
  return compose_frame(panels, kinds, accumulations, P, H, W, turbo, viridis, scratch, out, stream);
}
