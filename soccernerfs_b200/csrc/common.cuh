// Shared device/host helpers for libkplanes_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/kplanes_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libkplanes_b200 targets sm_100a (B200) only"
#endif

namespace kp {

void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;  // kernels launched through the C-ABI (kp_launch_count); the autograd
                                            // thread and the main thread both launch

#define KP_CHECK(cond, ...)          \
  do {                               \
    if (!(cond)) {                   \
      kp::set_error(__VA_ARGS__);    \
      return 1;                      \
    }                                \
  } while (0)

#define KP_LAUNCH_CHECK(name)                                                      \
  do {                                                                             \
    kp::g_launches += 1;                                                           \
    cudaError_t e__ = cudaGetLastError();                                          \
    if (e__ != cudaSuccess) {                                                      \
      kp::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));       \
      return 2;                                                                    \
    }                                                                              \
  } while (0)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---- device helpers -------------------------------------------------------------------------
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// 256-bit read-only load (sm_100: LDG.E.ENL2.256): a whole 8-channel texel in one request instead of two
struct __align__(32) float8 { float4 a, b; };
__device__ __forceinline__ float8 ldg8(const float* p) {
  float8 r;
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(r.a.x), "=f"(r.a.y), "=f"(r.a.z), "=f"(r.a.w), "=f"(r.b.x), "=f"(r.b.y), "=f"(r.b.z), "=f"(r.b.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ void stg8(float* p, float4 a, float4 b) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w), "f"(b.x),
               "f"(b.y), "f"(b.z), "f"(b.w)
               : "memory");
}

// Vector reduction (no return value) into global memory: one 16-byte L2 atomic instead of four.
__device__ __forceinline__ void red_add_v4(float* addr, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}
__device__ __forceinline__ void red_add_f32(float* addr, float v) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(addr), "f"(v) : "memory");
}

__device__ __forceinline__ float4 mul4(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
__device__ __forceinline__ float4 scale4(float4 a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }
__device__ __forceinline__ float4 fma4(float4 a, float s, float4 c) {
  return make_float4(fmaf(a.x, s, c.x), fmaf(a.y, s, c.y), fmaf(a.z, s, c.z), fmaf(a.w, s, c.w));
}

// Packed fp32 pairs (sm_100 FFMA2 / FMUL2: one issue slot for two IEEE fp32 operations -- the 3-register scalar FFMA issues
// every other cycle per scheduler, so instruction-bound fp32 code doubles its FMA rate; each half rounds exactly like the
// scalar instruction, so results are bit-identical).
__device__ __forceinline__ float2 dup2(float s) { return make_float2(s, s); }
__device__ __forceinline__ float2 lo2(float4 a) { return make_float2(a.x, a.y); }
__device__ __forceinline__ float2 hi2(float4 a) { return make_float2(a.z, a.w); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// inclusive warp scan (double): used to reproduce torch's CPU cumsum, which accumulates fp32 in double
__device__ __forceinline__ double warp_incl_scan_d(double v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    double t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}

// exclusive warp scan (double).  NOT "inclusive - own value": with an infinite element that would be inf - inf = NaN
// for the lane holding it, while torch's cumsum gives the finite prefix (e.g. an infinite density in get_weights).
__device__ __forceinline__ double warp_excl_scan_d(double v, int lane) {
  const double incl = warp_incl_scan_d(v, lane);
  const double up = __shfl_up_sync(0xffffffffu, incl, 1);
  return lane == 0 ? 0.0 : up;
}

// Spherical-harmonics basis (degree 4, 16 terms) of a view direction, the first half of the colour net's input:
// get_normalized_directions (kplanes_field.py:39-44) then tcnn SH maps [0,1] -> [-1,1]; basis NS/utils/math.py:25-86.
__device__ __forceinline__ void sh16(float dx, float dy, float dz, float* out) {
  const float x = ((dx + 1.f) / 2.f) * 2.f - 1.f, y = ((dy + 1.f) / 2.f) * 2.f - 1.f, z = ((dz + 1.f) / 2.f) * 2.f - 1.f;
  const float xx = x * x, yy = y * y, zz = z * z;
  out[0] = 0.28209479177387814f;
  out[1] = 0.4886025119029199f * y;
  out[2] = 0.4886025119029199f * z;
  out[3] = 0.4886025119029199f * x;
  out[4] = 1.0925484305920792f * x * y;
  out[5] = 1.0925484305920792f * y * z;
  out[6] = 0.9461746957575601f * zz - 0.31539156525251999f;
  out[7] = 1.0925484305920792f * x * z;
  out[8] = 0.5462742152960396f * (xx - yy);
  out[9] = 0.5900435899266435f * y * (3.f * xx - yy);
  out[10] = 2.890611442640554f * x * y * z;
  out[11] = 0.4570457994644658f * y * (5.f * zz - 1.f);
  out[12] = 0.3731763325901154f * z * (5.f * zz - 3.f);
  out[13] = 0.4570457994644658f * x * (5.f * zz - 1.f);
  out[14] = 1.445305721320277f * z * (xx - yy);
  out[15] = 0.5900435899266435f * x * (xx - 3.f * yy);
}

// torch.nan_to_num defaults: nan -> 0, +inf -> FLT_MAX, -inf -> -FLT_MAX
__device__ __forceinline__ float nan_to_num(float x) {
  if (isnan(x)) return 0.f;
  if (isinf(x)) return x > 0 ? 3.4028234663852886e38f : -3.4028234663852886e38f;
  return x;
}

// ---- torch.optim.Adam (NS/engine/optimizers.py:74-160), the one update rule of every optimizer kernel ----------------
struct AdamScalars {
  float lr_over_bc1, inv_sqrt_bc2, beta1, beta2, eps, wd, grad_scale;
};

// Bias corrections of a 1-based step, in double as torch computes them.
static inline AdamScalars adam_scalars(float lr, float beta1, float beta2, float eps, float weight_decay, int64_t step,
                                       float grad_scale) {
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  return AdamScalars{(float)(lr / bc1), (float)(1.0 / sqrt(bc2)), beta1, beta2, eps, weight_decay, grad_scale};
}

// hyper_dev (optional, DEVICE float[3] = lr/bias_corr1, 1/sqrt(bias_corr2), grad_scale) overrides the host scalars, so a
// captured CUDA graph can be replayed with fresh per-step values (kp_step_scalars writes them).
__device__ __forceinline__ AdamScalars with_hyper_dev(AdamScalars s, const float* hyper_dev) {
  if (hyper_dev != nullptr) {
    s.lr_over_bc1 = hyper_dev[0];
    s.inv_sqrt_bc2 = hyper_dev[1];
    s.grad_scale = hyper_dev[2];
  }
  return s;
}

// One element; g is the gradient with grad_scale already applied.  Every rounding is spelled out (fmaf, __fmul_rn) so
// that all callers compute the same bits: left to the compiler, `v * beta2 + (1 - beta2) * gr * gr` was contracted one way
// in one kernel and the other way in another.
__device__ __forceinline__ void adam_update(float g, float& p, float& m, float& v, const AdamScalars& s) {
  const float gr = fmaf(s.wd, p, g);
  m = fmaf(gr - m, 1.f - s.beta1, m);
  v = fmaf(v, s.beta2, __fmul_rn(__fmul_rn((1.f - s.beta2), gr), gr));
  p -= s.lr_over_bc1 * m / fmaf(sqrtf(v), s.inv_sqrt_bc2, s.eps);
}
__device__ __forceinline__ void adam_update4(float4 g, float4& p, float4& m, float4& v, const AdamScalars& s) {
  adam_update(g.x, p.x, m.x, v.x, s);
  adam_update(g.y, p.y, m.y, v.y, s);
  adam_update(g.z, p.z, m.z, v.z, s);
  adam_update(g.w, p.w, m.w, v.w, s);
}

}  // namespace kp
