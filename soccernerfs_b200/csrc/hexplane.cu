// Multiscale hexplane field kernels (sm_100a).
//
// Replaces NS/fields/kplanes_field.py:77-126 (interpolate_kplanes: 6*K F.grid_sample launches + Hadamard +
// cat) and the ATen grid_sampler_2d fwd/bwd underneath it (NS/utils/interpolation.py:24-30) with ONE gather
// kernel and ONE scatter kernel over channel-last planes:
//   * a sample is owned by C/4 adjacent lanes, each lane moving 16-byte float4 slices, so the C/4 lanes of a
//     texel read/reduce one contiguous 4*C-byte run (C=32: exactly one 128-byte line);
//   * all plane corners of a scale are issued before first use (24 independent 16-B loads per lane);
//   * the Hadamard product across planes and the concat across scales happen in registers and the
//     features are written once;
//   * the backward re-gathers the six interpolants (product rule needs the other five) instead of saving
//     6*K [M,C] tensors, and scatter-adds with red.global.add.v4.f32 (16-byte L2 reductions).
// Also here: the fused proposal density field (kplanes_field.py:434-460): gather (C=8) -> Hadamard ->
// 8->64->1 MLP -> trunc_exp in one kernel, and its backward.
#include <algorithm>

#include "common.cuh"

namespace kp {

struct PlaneRef {
  const float* p;
  float* g;
  uint8_t* f;  // scatter only, optional: one "touched" byte per texel (set to 1 for every texel that receives a reduction)
  int H, W, ca, cb;
  int stream;  // 1: the plane is far larger than L2 -- its lines are loaded / reduced with the L2 evict_first policy so that
               // they do not push the coarse scales and the (heavily re-used) space-time planes out of the 126 MB L2
};
struct FieldRef {
  PlaneRef pl[KP_MAX_SCALES * KP_MAX_PLANES];
  int reso[KP_MAX_SCALES][4];  // per-scale resolution of coordinates x,y,z,(t): plane (a,b) is [reso[b]][reso[a]][C]
  int n_scales, n_planes;
  uint32_t use_mask;
  int concat;
};

__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ float4 ldg4_stream(const float* p, uint64_t pol) {
  float4 v;
  asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ float8 ldg8_stream(const float* p, uint64_t pol) {
  float8 r;
  asm volatile("ld.global.nc.L2::cache_hint.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
               : "=f"(r.a.x), "=f"(r.a.y), "=f"(r.a.z), "=f"(r.a.w), "=f"(r.b.x), "=f"(r.b.y), "=f"(r.b.z), "=f"(r.b.w)
               : "l"(p), "l"(pol));
  return r;
}
__device__ __forceinline__ void red_add_v4_stream(float* addr, float4 v, uint64_t pol) {
  asm volatile("red.global.add.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w),
               "l"(pol)
               : "memory");
}

static int fill_field(FieldRef& F, const float* const* plane_ptrs, float* const* grad_ptrs, const int32_t* plane_hw,
                      int n_scales, int n_planes, int D, uint32_t use_mask, int concat, int feature_dim = 32) {
  KP_CHECK(n_scales >= 1 && n_scales <= KP_MAX_SCALES, "n_scales=%d out of range [1,%d]", n_scales, KP_MAX_SCALES);
  KP_CHECK((n_planes == 3 && D == 3) || (n_planes == 6 && D == 4), "n_planes=%d / D=%d must be 3/3 or 6/4", n_planes, D);
  static const int comb4[6][2] = {{0, 1}, {0, 2}, {0, 3}, {1, 2}, {1, 3}, {2, 3}};
  static const int comb3[3][2] = {{0, 1}, {0, 2}, {1, 2}};
  for (int k = 0; k < n_scales; ++k)
    for (int p = 0; p < n_planes; ++p) {
      PlaneRef& r = F.pl[k * KP_MAX_PLANES + p];
      r.p = plane_ptrs[k * n_planes + p];
      r.g = grad_ptrs ? grad_ptrs[k * n_planes + p] : nullptr;
      r.f = nullptr;
      r.stream = 0;
      r.H = plane_hw[(k * n_planes + p) * 2 + 0];
      r.W = plane_hw[(k * n_planes + p) * 2 + 1];
      r.ca = (D == 4) ? comb4[p][0] : comb3[p][0];
      r.cb = (D == 4) ? comb4[p][1] : comb3[p][1];
      KP_CHECK(r.p != nullptr && r.H >= 1 && r.W >= 1, "plane (%d,%d) invalid", k, p);
    }
  // K-Planes structure (kplanes_field.py:61-67): within a scale every plane's W / H is the resolution of the
  // coordinate it is indexed by, so the bilinear set-up is done once per coordinate, not once per plane.
  for (int k = 0; k < n_scales; ++k) {
    int* reso = F.reso[k];
    reso[0] = reso[1] = reso[2] = reso[3] = 0;
    for (int p = 0; p < n_planes; ++p) {
      const PlaneRef& r = F.pl[k * KP_MAX_PLANES + p];
      KP_CHECK(reso[r.ca] == 0 || reso[r.ca] == r.W, "scale %d: plane %d has W=%d but coordinate %d has resolution %d", k, p,
               r.W, r.ca, reso[r.ca]);
      reso[r.ca] = r.W;
      KP_CHECK(reso[r.cb] == 0 || reso[r.cb] == r.H, "scale %d: plane %d has H=%d but coordinate %d has resolution %d", k, p,
               r.H, r.cb, reso[r.cb]);
      reso[r.cb] = r.H;
    }
    if (reso[3] == 0) reso[3] = 1;
  }
  F.n_scales = n_scales;
  F.n_planes = n_planes;
  F.use_mask = use_mask;
  F.concat = concat;
  // L2 policy (ncu, 32x preset: the gather read 1.74 GB and the scatter moved 6.1 GB of DRAM for ~0.5 / ~1.4 GB of distinct
  // lines -- the once-per-step lines of the big space planes kept evicting the re-used coarse scales): planes of at least
  // stream_bytes are streamed with evict_first.
  constexpr long long stream_bytes = 16ll << 20;  // (sweep on B200, 32x preset: off 1.35 ms, 96 MB 1.28, 32 MB 1.25, 16 MB 1.19, 4 MB 1.22 ms scatter)
  // only when the field as a whole is far beyond L2 (>= 512 MB): a 152 MB field keeps a 75 % L2 hit rate without any
  // policy, and streaming its largest scale costs more misses than it saves (ncu: gather DRAM reads 193 -> 269 MB)
  long long total_bytes = 0;
  for (int k = 0; k < n_scales; ++k)
    for (int p = 0; p < n_planes; ++p) total_bytes += (long long)F.pl[k * KP_MAX_PLANES + p].H * F.pl[k * KP_MAX_PLANES + p].W * feature_dim * 4;
  if (total_bytes >= (512ll << 20))
    for (int k = 0; k < n_scales; ++k)
      for (int p = 0; p < n_planes; ++p) {
        PlaneRef& r = F.pl[k * KP_MAX_PLANES + p];
        r.stream = ((long long)r.H * r.W * feature_dim * 4 >= stream_bytes) ? 1 : 0;
      }
  return 0;
}

// Sample coordinate in grid_sample's [-1,1] convention.  Ray form follows the reference's op order with
// non-contracted IEEE ops so that coordinates (hence floor() decisions) equal the torch CPU path bit for bit:
//   pos = o + d*(start+end)/2 (rays.py:54);  (pos-aabb0)/(aabb1-aabb0) (scene_box.py:64-65);  [*2-1];  t*2-1.
__device__ __forceinline__ void load_point(const KpPoints& P, int64_t m, float pt[4]) {
  if (P.pts != nullptr) {
#pragma unroll
    for (int d = 0; d < 4; ++d) pt[d] = d < P.D ? P.pts[m * P.D + d] : 0.f;
    return;
  }
  const int64_t n = m / P.S;
  const float t = __fadd_rn(P.starts[m], P.ends[m]);
  if (P.norm_mode == 2) {
    // unbounded scene: SceneContraction(order=inf)(pos) / 2  (kplanes_field.py:278-280 / :436-438,
    // NS/field_components/spatial_distortions.py:66-71): x if |x|_inf < 1 else (2 - 1/|x|) (x/|x|), then [-2,2] -> [-1,1]
    float pos[3];
#pragma unroll
    for (int d = 0; d < 3; ++d)
      pos[d] = __fadd_rn(P.origins[n * 3 + d], __fmul_rn(__fmul_rn(P.directions[n * 3 + d], t), 0.5f));
    const float mag = fmaxf(fabsf(pos[0]), fmaxf(fabsf(pos[1]), fabsf(pos[2])));
    const float k = __fsub_rn(2.f, __fdiv_rn(1.f, mag));
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      const float c = mag < 1.f ? pos[d] : __fmul_rn(k, __fdiv_rn(pos[d], mag));
      pt[d] = __fmul_rn(c, 0.5f);
    }
    pt[3] = (P.D == 4 && P.times != nullptr) ? __fsub_rn(__fmul_rn(P.times[n], 2.f), 1.f) : 0.f;
    return;
  }
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    float v = __fmul_rn(__fmul_rn(P.directions[n * 3 + d], t), 0.5f);  // x/2 == x*0.5 exactly
    float pos = __fadd_rn(P.origins[n * 3 + d], v);
    float q = __fdiv_rn(__fsub_rn(pos, P.aabb[d]), __fsub_rn(P.aabb[3 + d], P.aabb[d]));
    pt[d] = P.norm_mode ? __fsub_rn(__fmul_rn(q, 2.f), 1.f) : q;
  }
  pt[3] = (P.D == 4 && P.times != nullptr) ? __fsub_rn(__fmul_rn(P.times[n], 2.f), 1.f) : 0.f;
}

// ATen grid_sampler_2d, bilinear / padding border / align_corners=True, factored per coordinate axis:
//   i = ((x+1)/2)*(R-1) clamped to [0,R-1]; i0 = floor(i); weights (i0+1-i), (i-i0); corner i0+1 == R is dropped.
struct Axis {
  int i0, i1;
  float w0, w1;
};
__device__ __forceinline__ Axis axis_setup(float x, int R) {
  float ix = __fmul_rn(__fmul_rn(__fadd_rn(x, 1.f), 0.5f), (float)(R - 1));
  ix = fminf((float)(R - 1), fmaxf(ix, 0.f));
  const float fx = floorf(ix);
  Axis a;
  a.i0 = (int)fx;
  a.i1 = a.i0 + 1;
  a.w1 = ix - fx;
  a.w0 = (fx + 1.f) - ix;
  if (a.i1 > R - 1) { a.i1 = R - 1; a.w1 = 0.f; }  // out-of-range corner contributes nothing
  return a;
}
struct Bilerp {
  int o00, o01, o10, o11;  // texel indices (y*W+x)
  float w00, w01, w10, w11;
};
__device__ __forceinline__ Bilerp bilerp_from_axes(const Axis& ax, const Axis& ay, int W) {
  Bilerp b;
  b.o00 = ay.i0 * W + ax.i0; b.o01 = ay.i0 * W + ax.i1; b.o10 = ay.i1 * W + ax.i0; b.o11 = ay.i1 * W + ax.i1;
  b.w00 = ax.w0 * ay.w0; b.w01 = ax.w1 * ay.w0; b.w10 = ax.w0 * ay.w1; b.w11 = ax.w1 * ay.w1;
  return b;
}
// plane p of combinations(range(D),2) samples coordinate CA (-> W) and CB (-> H); compile-time so that the per-axis
// set-up stays in registers
template <int NP>
__host__ __device__ constexpr int plane_ca(int p) {
  return NP == 6 ? (p < 3 ? 0 : (p < 5 ? 1 : 2)) : (p < 2 ? 0 : 1);
}
template <int NP>
__host__ __device__ constexpr int plane_cb(int p) {
  return NP == 6 ? (p < 3 ? p + 1 : (p < 5 ? p - 1 : 3)) : (p < 1 ? 1 : 2);
}
__device__ __forceinline__ void axes_setup(const FieldRef& F, int k, const float pt[4], Axis ax[4]) {
#pragma unroll
  for (int d = 0; d < 4; ++d) ax[d] = axis_setup(pt[d], F.reso[k][d]);
}

__device__ __forceinline__ float4 bilerp_combine(const Bilerp& b, float4 v00, float4 v01, float4 v10, float4 v11) {
  float4 r = scale4(v00, b.w00);
  r = fma4(v01, b.w01, r);
  r = fma4(v10, b.w10, r);
  r = fma4(v11, b.w11, r);
  return r;
}

// ---------------------------------------------------------------------------------------------------
// Forward gather.  C/4 lanes per sample, float4 per lane.
// ---------------------------------------------------------------------------------------------------
template <int C, int NP, bool STREAM>
__global__ void __launch_bounds__(128, 4) hexplane_fwd_kernel(const __grid_constant__ FieldRef F,
                                                            const __grid_constant__ KpPoints P, int64_t M,
                                                            float* __restrict__ out) {
  constexpr int LPS = C / 4;
  const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t m = gt / LPS;
  const int c4 = (int)(gt % LPS) * 4;
  if (m >= M) return;
  if (P.ray_tile > 1 && P.pts == nullptr) {
    // coherent rays (neighbouring pixels of a frame): slot m -> sample s of ray (tile * T + j), j fastest, so the 32 / LPS
    // samples of a warp are the SAME sample index of neighbouring rays.  At every scale whose texels are wider than the
    // pixel footprint they read the same texel lines, which coalesce inside the request (one L2 line request per warp
    // instead of one per sample).  The last tile may hold fewer rays.
    const int64_t n_rays = M / P.S, tile_sz = (int64_t)P.ray_tile * P.S;
    const int64_t tile = m / tile_sz;
    const int r = (int)(m - tile * tile_sz);
    const int t_here = (int)min((int64_t)P.ray_tile, n_rays - tile * P.ray_tile);
    m = (tile * P.ray_tile + r % t_here) * P.S + r / t_here;
  }
  float pt[4];
  load_point(P, m, pt);
  const int out_stride = F.concat ? F.n_scales * C : C;
  const uint64_t pol = STREAM ? l2_policy_evict_first() : 0ull;
  float4 total = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int k = 0; k < F.n_scales; ++k) {
    Axis ax[4];
    axes_setup(F, k, pt, ax);
    Bilerp b[NP];
    float4 v[NP][4];
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      const PlaneRef& pr = F.pl[k * KP_MAX_PLANES + p];
      b[p] = bilerp_from_axes(ax[plane_ca<NP>(p)], ax[plane_cb<NP>(p)], pr.W);
      if ((F.use_mask >> p) & 1u) {
        const float* base = pr.p + c4;
        if (STREAM && pr.stream) {  // (uniform: a property of the plane; STREAM = false compiles the policy code out)
          v[p][0] = ldg4_stream(base + (int64_t)b[p].o00 * C, pol);
          v[p][1] = ldg4_stream(base + (int64_t)b[p].o01 * C, pol);
          v[p][2] = ldg4_stream(base + (int64_t)b[p].o10 * C, pol);
          v[p][3] = ldg4_stream(base + (int64_t)b[p].o11 * C, pol);
        } else {
          v[p][0] = ldg4(base + (int64_t)b[p].o00 * C);
          v[p][1] = ldg4(base + (int64_t)b[p].o01 * C);
          v[p][2] = ldg4(base + (int64_t)b[p].o10 * C);
          v[p][3] = ldg4(base + (int64_t)b[p].o11 * C);
        }
      }
    }
    float4 acc = make_float4(1.f, 1.f, 1.f, 1.f);
#pragma unroll
    for (int p = 0; p < NP; ++p)
      if ((F.use_mask >> p) & 1u) acc = mul4(acc, bilerp_combine(b[p], v[p][0], v[p][1], v[p][2], v[p][3]));
    if (F.concat) {
      *reinterpret_cast<float4*>(out + m * out_stride + k * C + c4) = acc;
    } else {
      total.x += acc.x; total.y += acc.y; total.z += acc.z; total.w += acc.w;
    }
  }
  if (!F.concat) *reinterpret_cast<float4*>(out + m * out_stride + c4) = total;
}

// ---------------------------------------------------------------------------------------------------
// Forward gather, WIDE mapping (C = 32): 4 lanes per sample, 8 channels per lane -- one 256-bit load per corner and packed
// FMUL2 / FFMA2 interpolation.  Per sample the coordinate set-up (identical on every lane of the sample) is done 4x instead
// of 8x and every load / math instruction covers twice the channels: about half the warp instructions of the float4
// kernel above.  Same arithmetic per channel, bit-identical output; where it is used is decided (from measurements) in
// launch_hexplane.
// The planes of a scale are gathered in two groups of NP/2 so that 12 (not 24) 32-byte loads are in flight per lane.
// ---------------------------------------------------------------------------------------------------
template <int NP, bool STREAM>
__global__ void __launch_bounds__(128, 3) hexplane_fwd_wide_kernel(const __grid_constant__ FieldRef F,
                                                                 const __grid_constant__ KpPoints P, int64_t M,
                                                                 float* __restrict__ out) {
  constexpr int C = 32, LPS = 4, G = NP / 2 > 0 ? (NP + 1) / 2 : 1;
  const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t m = gt / LPS;
  const int c8 = (int)(gt % LPS) * 8;
  if (m >= M) return;
  if (P.ray_tile > 1 && P.pts == nullptr) {
    const int64_t n_rays = M / P.S, tile_sz = (int64_t)P.ray_tile * P.S;
    const int64_t tile = m / tile_sz;
    const int r = (int)(m - tile * tile_sz);
    const int t_here = (int)min((int64_t)P.ray_tile, n_rays - tile * P.ray_tile);
    m = (tile * P.ray_tile + r % t_here) * P.S + r / t_here;
  }
  float pt[4];
  load_point(P, m, pt);
  const int out_stride = F.concat ? F.n_scales * C : C;
  const uint64_t pol = STREAM ? l2_policy_evict_first() : 0ull;
  float2 total[4] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
  for (int k = 0; k < F.n_scales; ++k) {
    Axis ax[4];
    axes_setup(F, k, pt, ax);
    float2 acc[4] = {make_float2(1.f, 1.f), make_float2(1.f, 1.f), make_float2(1.f, 1.f), make_float2(1.f, 1.f)};
#pragma unroll
    for (int g0 = 0; g0 < NP; g0 += G) {
      Bilerp b[G];
      float8 v[G][4];
#pragma unroll
      for (int i = 0; i < G; ++i) {
        const int p = g0 + i;
        if (p >= NP) continue;
        const PlaneRef& pr = F.pl[k * KP_MAX_PLANES + p];
        b[i] = bilerp_from_axes(ax[plane_ca<NP>(p)], ax[plane_cb<NP>(p)], pr.W);
        if ((F.use_mask >> p) & 1u) {
          const float* base = pr.p + c8;
          if (STREAM && pr.stream) {
            v[i][0] = ldg8_stream(base + (int64_t)b[i].o00 * C, pol);
            v[i][1] = ldg8_stream(base + (int64_t)b[i].o01 * C, pol);
            v[i][2] = ldg8_stream(base + (int64_t)b[i].o10 * C, pol);
            v[i][3] = ldg8_stream(base + (int64_t)b[i].o11 * C, pol);
          } else {
            v[i][0] = ldg8(base + (int64_t)b[i].o00 * C);
            v[i][1] = ldg8(base + (int64_t)b[i].o01 * C);
            v[i][2] = ldg8(base + (int64_t)b[i].o10 * C);
            v[i][3] = ldg8(base + (int64_t)b[i].o11 * C);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < G; ++i) {
        const int p = g0 + i;
        if (p >= NP || !((F.use_mask >> p) & 1u)) continue;
        const float2 w00 = dup2(b[i].w00), w01 = dup2(b[i].w01), w10 = dup2(b[i].w10), w11 = dup2(b[i].w11);
        // bilerp_combine per channel pair: v00*w00, then fma(v01,w01,.), fma(v10,w10,.), fma(v11,w11,.)
        auto pair = [&](float2 x00, float2 x01, float2 x10, float2 x11) {
          float2 r = __fmul2_rn(x00, w00);
          r = __ffma2_rn(x01, w01, r);
          r = __ffma2_rn(x10, w10, r);
          return __ffma2_rn(x11, w11, r);
        };
        acc[0] = __fmul2_rn(acc[0], pair(lo2(v[i][0].a), lo2(v[i][1].a), lo2(v[i][2].a), lo2(v[i][3].a)));
        acc[1] = __fmul2_rn(acc[1], pair(hi2(v[i][0].a), hi2(v[i][1].a), hi2(v[i][2].a), hi2(v[i][3].a)));
        acc[2] = __fmul2_rn(acc[2], pair(lo2(v[i][0].b), lo2(v[i][1].b), lo2(v[i][2].b), lo2(v[i][3].b)));
        acc[3] = __fmul2_rn(acc[3], pair(hi2(v[i][0].b), hi2(v[i][1].b), hi2(v[i][2].b), hi2(v[i][3].b)));
      }
    }
    if (F.concat) {
      stg8(out + m * out_stride + k * C + c8, make_float4(acc[0].x, acc[0].y, acc[1].x, acc[1].y),
           make_float4(acc[2].x, acc[2].y, acc[3].x, acc[3].y));
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) total[q] = __fadd2_rn(total[q], acc[q]);
    }
  }
  if (!F.concat)
    stg8(out + m * out_stride + c8, make_float4(total[0].x, total[0].y, total[1].x, total[1].y),
         make_float4(total[2].x, total[2].y, total[3].x, total[3].y));
}

// ---------------------------------------------------------------------------------------------------
// Forward gather with the dynamics score (kp_hexplane_fwd_dyn), six planes: the two kernels above with, beside the feature
// product, T = the product of the time planes' interpolants (the same values, multiplied in the same plane order; the
// feature product's operations and bits are unchanged) and delta[m] = mean over scales and channels of |1 - T|.  Kept
// apart from the kernels above so that their code stays exactly what it was.
// ---------------------------------------------------------------------------------------------------
__host__ __device__ constexpr bool is_time_plane(int p) { return p == 2 || p == 4 || p == 5; }  // XT, YT, ZT

// delta = (sum of the LPS lanes' partial sums) / (K * C), written by the sample's first lane.  The lanes of a sample are
// adjacent and leave the kernel together, so the shuffle's group is complete.
template <int LPS>
__device__ __forceinline__ void store_delta(float part, int lane_in_sample, int64_t m, int n_scales, int C, float* delta) {
  static_assert(LPS >= 1 && LPS <= 16 && (LPS & (LPS - 1)) == 0, "lanes per sample: a power of two below the warp");
  const unsigned group = ((1u << LPS) - 1u) << ((threadIdx.x & 31) & ~(LPS - 1));
#pragma unroll
  for (int o = LPS / 2; o > 0; o >>= 1) part += __shfl_xor_sync(group, part, o, LPS);
  if (lane_in_sample == 0) delta[m] = __fdiv_rn(part, (float)(n_scales * C));
}

template <int C, bool STREAM>
__global__ void __launch_bounds__(128, 4) hexplane_fwd_dyn_kernel(const __grid_constant__ FieldRef F,
                                                                const __grid_constant__ KpPoints P, int64_t M,
                                                                float* __restrict__ out, float* __restrict__ delta) {
  constexpr int NP = 6, LPS = C / 4;
  const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t m = gt / LPS;
  const int c4 = (int)(gt % LPS) * 4;
  if (m >= M) return;
  if (P.ray_tile > 1 && P.pts == nullptr) {
    const int64_t n_rays = M / P.S, tile_sz = (int64_t)P.ray_tile * P.S;
    const int64_t tile = m / tile_sz;
    const int r = (int)(m - tile * tile_sz);
    const int t_here = (int)min((int64_t)P.ray_tile, n_rays - tile * P.ray_tile);
    m = (tile * P.ray_tile + r % t_here) * P.S + r / t_here;
  }
  float pt[4];
  load_point(P, m, pt);
  const int out_stride = F.concat ? F.n_scales * C : C;
  const uint64_t pol = STREAM ? l2_policy_evict_first() : 0ull;
  float4 total = make_float4(0.f, 0.f, 0.f, 0.f);
  float dsum = 0.f;  // this lane's sum of |1 - T| over its channels and the scales
  for (int k = 0; k < F.n_scales; ++k) {
    Axis ax[4];
    axes_setup(F, k, pt, ax);
    Bilerp b[NP];
    float4 v[NP][4];
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      const PlaneRef& pr = F.pl[k * KP_MAX_PLANES + p];
      b[p] = bilerp_from_axes(ax[plane_ca<NP>(p)], ax[plane_cb<NP>(p)], pr.W);
      if ((F.use_mask >> p) & 1u) {
        const float* base = pr.p + c4;
        if (STREAM && pr.stream) {
          v[p][0] = ldg4_stream(base + (int64_t)b[p].o00 * C, pol);
          v[p][1] = ldg4_stream(base + (int64_t)b[p].o01 * C, pol);
          v[p][2] = ldg4_stream(base + (int64_t)b[p].o10 * C, pol);
          v[p][3] = ldg4_stream(base + (int64_t)b[p].o11 * C, pol);
        } else {
          v[p][0] = ldg4(base + (int64_t)b[p].o00 * C);
          v[p][1] = ldg4(base + (int64_t)b[p].o01 * C);
          v[p][2] = ldg4(base + (int64_t)b[p].o10 * C);
          v[p][3] = ldg4(base + (int64_t)b[p].o11 * C);
        }
      }
    }
    float4 acc = make_float4(1.f, 1.f, 1.f, 1.f), tp = acc;
#pragma unroll
    for (int p = 0; p < NP; ++p)
      if ((F.use_mask >> p) & 1u) {
        const float4 f = bilerp_combine(b[p], v[p][0], v[p][1], v[p][2], v[p][3]);
        acc = mul4(acc, f);
        if (is_time_plane(p)) tp = mul4(tp, f);
      }
    dsum += fabsf(1.f - tp.x) + fabsf(1.f - tp.y) + fabsf(1.f - tp.z) + fabsf(1.f - tp.w);
    if (F.concat) {
      *reinterpret_cast<float4*>(out + m * out_stride + k * C + c4) = acc;
    } else {
      total.x += acc.x; total.y += acc.y; total.z += acc.z; total.w += acc.w;
    }
  }
  if (!F.concat) *reinterpret_cast<float4*>(out + m * out_stride + c4) = total;
  store_delta<LPS>(dsum, c4 / 4, m, F.n_scales, C, delta);
}

template <bool STREAM>
__global__ void __launch_bounds__(128, 3) hexplane_fwd_wide_dyn_kernel(const __grid_constant__ FieldRef F,
                                                                     const __grid_constant__ KpPoints P, int64_t M,
                                                                     float* __restrict__ out, float* __restrict__ delta) {
  constexpr int NP = 6, C = 32, LPS = 4, G = 3;
  const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t m = gt / LPS;
  const int c8 = (int)(gt % LPS) * 8;
  if (m >= M) return;
  if (P.ray_tile > 1 && P.pts == nullptr) {
    const int64_t n_rays = M / P.S, tile_sz = (int64_t)P.ray_tile * P.S;
    const int64_t tile = m / tile_sz;
    const int r = (int)(m - tile * tile_sz);
    const int t_here = (int)min((int64_t)P.ray_tile, n_rays - tile * P.ray_tile);
    m = (tile * P.ray_tile + r % t_here) * P.S + r / t_here;
  }
  float pt[4];
  load_point(P, m, pt);
  const int out_stride = F.concat ? F.n_scales * C : C;
  const uint64_t pol = STREAM ? l2_policy_evict_first() : 0ull;
  float2 total[4] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
  float dsum = 0.f;
  for (int k = 0; k < F.n_scales; ++k) {
    Axis ax[4];
    axes_setup(F, k, pt, ax);
    float2 acc[4] = {make_float2(1.f, 1.f), make_float2(1.f, 1.f), make_float2(1.f, 1.f), make_float2(1.f, 1.f)};
    float2 tp[4] = {make_float2(1.f, 1.f), make_float2(1.f, 1.f), make_float2(1.f, 1.f), make_float2(1.f, 1.f)};
#pragma unroll
    for (int g0 = 0; g0 < NP; g0 += G) {
      Bilerp b[G];
      float8 v[G][4];
#pragma unroll
      for (int i = 0; i < G; ++i) {
        const int p = g0 + i;
        const PlaneRef& pr = F.pl[k * KP_MAX_PLANES + p];
        b[i] = bilerp_from_axes(ax[plane_ca<NP>(p)], ax[plane_cb<NP>(p)], pr.W);
        if ((F.use_mask >> p) & 1u) {
          const float* base = pr.p + c8;
          if (STREAM && pr.stream) {
            v[i][0] = ldg8_stream(base + (int64_t)b[i].o00 * C, pol);
            v[i][1] = ldg8_stream(base + (int64_t)b[i].o01 * C, pol);
            v[i][2] = ldg8_stream(base + (int64_t)b[i].o10 * C, pol);
            v[i][3] = ldg8_stream(base + (int64_t)b[i].o11 * C, pol);
          } else {
            v[i][0] = ldg8(base + (int64_t)b[i].o00 * C);
            v[i][1] = ldg8(base + (int64_t)b[i].o01 * C);
            v[i][2] = ldg8(base + (int64_t)b[i].o10 * C);
            v[i][3] = ldg8(base + (int64_t)b[i].o11 * C);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < G; ++i) {
        const int p = g0 + i;
        if (!((F.use_mask >> p) & 1u)) continue;
        const float2 w00 = dup2(b[i].w00), w01 = dup2(b[i].w01), w10 = dup2(b[i].w10), w11 = dup2(b[i].w11);
        auto pair = [&](float2 x00, float2 x01, float2 x10, float2 x11) {  // bilerp_combine per channel pair
          float2 r = __fmul2_rn(x00, w00);
          r = __ffma2_rn(x01, w01, r);
          r = __ffma2_rn(x10, w10, r);
          return __ffma2_rn(x11, w11, r);
        };
        const float2 f[4] = {pair(lo2(v[i][0].a), lo2(v[i][1].a), lo2(v[i][2].a), lo2(v[i][3].a)),
                             pair(hi2(v[i][0].a), hi2(v[i][1].a), hi2(v[i][2].a), hi2(v[i][3].a)),
                             pair(lo2(v[i][0].b), lo2(v[i][1].b), lo2(v[i][2].b), lo2(v[i][3].b)),
                             pair(hi2(v[i][0].b), hi2(v[i][1].b), hi2(v[i][2].b), hi2(v[i][3].b))};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          acc[q] = __fmul2_rn(acc[q], f[q]);
          if (is_time_plane(p)) tp[q] = __fmul2_rn(tp[q], f[q]);
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) dsum += fabsf(1.f - tp[q].x) + fabsf(1.f - tp[q].y);
    if (F.concat) {
      stg8(out + m * out_stride + k * C + c8, make_float4(acc[0].x, acc[0].y, acc[1].x, acc[1].y),
           make_float4(acc[2].x, acc[2].y, acc[3].x, acc[3].y));
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) total[q] = __fadd2_rn(total[q], acc[q]);
    }
  }
  if (!F.concat)
    stg8(out + m * out_stride + c8, make_float4(total[0].x, total[0].y, total[1].x, total[1].y),
         make_float4(total[2].x, total[2].y, total[3].x, total[3].y));
  store_delta<LPS>(dsum, c8 / 8, m, F.n_scales, C, delta);
}

// ---------------------------------------------------------------------------------------------------
// Backward scatter: d plane_p[corner] += w_corner * g * prod_{q != p} interp_q.
// ---------------------------------------------------------------------------------------------------
template <int C, int NP, bool STREAM>
__global__ void __launch_bounds__(128, 4) hexplane_bwd_kernel(const __grid_constant__ FieldRef F,
                                                            const __grid_constant__ KpPoints P, int64_t M,
                                                            const float* __restrict__ grad_out) {
  constexpr int LPS = C / 4;
  const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t m = gt / LPS;
  const int c4 = (int)(gt % LPS) * 4;
  if (m >= M) return;
  float pt[4];
  load_point(P, m, pt);
  const int out_stride = F.concat ? F.n_scales * C : C;
  const uint64_t pol = STREAM ? l2_policy_evict_first() : 0ull;
  for (int k = 0; k < F.n_scales; ++k) {
    // a scale without any gradient target is skipped whole (per-scale launches: the caller scatters one scale at a
    // time so that a finished scale can be all-reduced while the next one is scattered)
    bool any_target = false;
#pragma unroll
    for (int p = 0; p < NP; ++p) any_target |= (((F.use_mask >> p) & 1u) != 0) && F.pl[k * KP_MAX_PLANES + p].g != nullptr;
    if (!any_target) continue;
    const float4 g = ldg4(grad_out + m * out_stride + (F.concat ? k * C : 0) + c4);
    Axis ax[4];
    axes_setup(F, k, pt, ax);
    Bilerp b[NP];
    float4 val[NP];
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      const PlaneRef& pr = F.pl[k * KP_MAX_PLANES + p];
      b[p] = bilerp_from_axes(ax[plane_ca<NP>(p)], ax[plane_cb<NP>(p)], pr.W);
      val[p] = make_float4(1.f, 1.f, 1.f, 1.f);
      if ((F.use_mask >> p) & 1u) {
        const float* base = pr.p + c4;
        if (STREAM && pr.stream)
          val[p] = bilerp_combine(b[p], ldg4_stream(base + (int64_t)b[p].o00 * C, pol), ldg4_stream(base + (int64_t)b[p].o01 * C, pol),
                                  ldg4_stream(base + (int64_t)b[p].o10 * C, pol), ldg4_stream(base + (int64_t)b[p].o11 * C, pol));
        else
          val[p] = bilerp_combine(b[p], ldg4(base + (int64_t)b[p].o00 * C), ldg4(base + (int64_t)b[p].o01 * C),
                                  ldg4(base + (int64_t)b[p].o10 * C), ldg4(base + (int64_t)b[p].o11 * C));
      }
    }
    // prefix/suffix products: others[p] = prod_{q != p} val[q]
    float4 pre[NP], suf[NP];
    pre[0] = make_float4(1.f, 1.f, 1.f, 1.f);
#pragma unroll
    for (int p = 1; p < NP; ++p) pre[p] = mul4(pre[p - 1], val[p - 1]);
    suf[NP - 1] = make_float4(1.f, 1.f, 1.f, 1.f);
#pragma unroll
    for (int p = NP - 2; p >= 0; --p) suf[p] = mul4(suf[p + 1], val[p + 1]);
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      const PlaneRef& pr = F.pl[k * KP_MAX_PLANES + p];
      if (!((F.use_mask >> p) & 1u) || pr.g == nullptr) continue;
      const float4 gp = mul4(g, mul4(pre[p], suf[p]));
      float* gb = pr.g + c4;
      if (STREAM && pr.stream) {
        if (b[p].w00 != 0.f) red_add_v4_stream(gb + (int64_t)b[p].o00 * C, scale4(gp, b[p].w00), pol);
        if (b[p].w01 != 0.f) red_add_v4_stream(gb + (int64_t)b[p].o01 * C, scale4(gp, b[p].w01), pol);
        if (b[p].w10 != 0.f) red_add_v4_stream(gb + (int64_t)b[p].o10 * C, scale4(gp, b[p].w10), pol);
        if (b[p].w11 != 0.f) red_add_v4_stream(gb + (int64_t)b[p].o11 * C, scale4(gp, b[p].w11), pol);
      } else {
        if (b[p].w00 != 0.f) red_add_v4(gb + (int64_t)b[p].o00 * C, scale4(gp, b[p].w00));
        if (b[p].w01 != 0.f) red_add_v4(gb + (int64_t)b[p].o01 * C, scale4(gp, b[p].w01));
        if (b[p].w10 != 0.f) red_add_v4(gb + (int64_t)b[p].o10 * C, scale4(gp, b[p].w10));
        if (b[p].w11 != 0.f) red_add_v4(gb + (int64_t)b[p].o11 * C, scale4(gp, b[p].w11));
      }
      // sparse gradient exchange: mark the texels this sample reduced into (one lane of the sample's C/4; plain byte
      // stores of the same value, so no ordering between writers is needed)
      if (pr.f != nullptr && c4 == 0) {
        if (b[p].w00 != 0.f) pr.f[b[p].o00] = 1;
        if (b[p].w01 != 0.f) pr.f[b[p].o01] = 1;
        if (b[p].w10 != 0.f) pr.f[b[p].o10] = 1;
        if (b[p].w11 != 0.f) pr.f[b[p].o11] = 1;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Fused proposal density field (single scale, small C): one thread per sample.
// ---------------------------------------------------------------------------------------------------
template <int C, int NP>
__device__ __forceinline__ void density_features(const FieldRef& F, const float pt[4], float val[NP][C], Axis ax[4]) {
  axes_setup(F, 0, pt, ax);
#pragma unroll
  for (int p = 0; p < NP; ++p) {
    const PlaneRef& pr = F.pl[p];
    const Bilerp b = bilerp_from_axes(ax[plane_ca<NP>(p)], ax[plane_cb<NP>(p)], pr.W);
    if ((F.use_mask >> p) & 1u) {
#pragma unroll
      for (int q = 0; q < C / 4; ++q) {
        const float* base = pr.p + q * 4;
        float4 r = bilerp_combine(b, ldg4(base + (int64_t)b.o00 * C), ldg4(base + (int64_t)b.o01 * C),
                                  ldg4(base + (int64_t)b.o10 * C), ldg4(base + (int64_t)b.o11 * C));
        val[p][q * 4 + 0] = r.x; val[p][q * 4 + 1] = r.y; val[p][q * 4 + 2] = r.z; val[p][q * 4 + 3] = r.w;
      }
    } else {
#pragma unroll
      for (int c = 0; c < C; ++c) val[p][c] = 1.f;
    }
  }
}

// Packed variant: val2[p][c/2] = (feature 2c', feature 2c'+1) of plane p; every product is an FMUL2 / FFMA2 whose halves round
// exactly like bilerp_combine's scalar operations.
template <int C, int NP, bool WIDE>
__device__ __forceinline__ void density_features2(const FieldRef& F, const float pt[4], float2 val2[NP][C / 2], Axis ax[4]) {
  axes_setup(F, 0, pt, ax);
#pragma unroll
  for (int p = 0; p < NP; ++p) {
    const PlaneRef& pr = F.pl[p];
    const Bilerp b = bilerp_from_axes(ax[plane_ca<NP>(p)], ax[plane_cb<NP>(p)], pr.W);
    if ((F.use_mask >> p) & 1u) {
      const float2 w00 = dup2(b.w00), w01 = dup2(b.w01), w10 = dup2(b.w10), w11 = dup2(b.w11);
      if constexpr (C == 8 && WIDE) {
        // one texel = 32 bytes = ONE 256-bit load per corner: half the load instructions and L1 wavefronts of the kernel
        // (it is L1-bound: 69 % l1tex in ncu, every lane of a request on a different line)
        const float8 t00 = ldg8(pr.p + (int64_t)b.o00 * 8), t01 = ldg8(pr.p + (int64_t)b.o01 * 8);
        const float8 t10 = ldg8(pr.p + (int64_t)b.o10 * 8), t11 = ldg8(pr.p + (int64_t)b.o11 * 8);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const float4 v00 = q ? t00.b : t00.a, v01 = q ? t01.b : t01.a, v10 = q ? t10.b : t10.a, v11 = q ? t11.b : t11.a;
          float2 lo = __fmul2_rn(lo2(v00), w00), hi = __fmul2_rn(hi2(v00), w00);
          lo = __ffma2_rn(lo2(v01), w01, lo); hi = __ffma2_rn(hi2(v01), w01, hi);
          lo = __ffma2_rn(lo2(v10), w10, lo); hi = __ffma2_rn(hi2(v10), w10, hi);
          lo = __ffma2_rn(lo2(v11), w11, lo); hi = __ffma2_rn(hi2(v11), w11, hi);
          val2[p][q * 2] = lo;
          val2[p][q * 2 + 1] = hi;
        }
        continue;
      }
#pragma unroll
      for (int q = 0; q < C / 4; ++q) {
        const float* base = pr.p + q * 4;
        const float4 v00 = ldg4(base + (int64_t)b.o00 * C), v01 = ldg4(base + (int64_t)b.o01 * C);
        const float4 v10 = ldg4(base + (int64_t)b.o10 * C), v11 = ldg4(base + (int64_t)b.o11 * C);
        float2 lo = __fmul2_rn(lo2(v00), w00), hi = __fmul2_rn(hi2(v00), w00);
        lo = __ffma2_rn(lo2(v01), w01, lo); hi = __ffma2_rn(hi2(v01), w01, hi);
        lo = __ffma2_rn(lo2(v10), w10, lo); hi = __ffma2_rn(hi2(v10), w10, hi);
        lo = __ffma2_rn(lo2(v11), w11, lo); hi = __ffma2_rn(hi2(v11), w11, hi);
        val2[p][q * 2] = lo;
        val2[p][q * 2 + 1] = hi;
      }
    } else {
#pragma unroll
      for (int c = 0; c < C / 2; ++c) val2[p][c] = make_float2(1.f, 1.f);
    }
  }
}

// Shared-memory weights of the 8 -> hidden -> 1 network in the layout the packed MLP reads: hidden units in PAIRS,
// s_w1p[jp][c] = (w1[2jp][c], w1[2jp+1][c]), s_w2p[jp] = (w2[2jp], w2[2jp+1]); an odd last unit is paired with zeros (its
// partner adds fma(0, 0, raw) = raw).
template <int C>
__device__ __forceinline__ void stage_paired_weights(const float* __restrict__ w1, const float* __restrict__ w2, int hidden,
                                                     float2* s_w1p, float2* s_w2p) {
  const int hp = (hidden + 1) / 2;
  for (int i = threadIdx.x; i < hp * C; i += blockDim.x) {
    const int jp = i / C, c = i % C;
    s_w1p[i] = make_float2(w1[(2 * jp) * C + c], 2 * jp + 1 < hidden ? w1[(2 * jp + 1) * C + c] : 0.f);
  }
  for (int i = threadIdx.x; i < hp; i += blockDim.x) s_w2p[i] = make_float2(w2[2 * i], 2 * i + 1 < hidden ? w2[2 * i + 1] : 0.f);
}

// pre-activations of hidden units (2jp, 2jp+1): the same fma chain over c as the scalar loop, two units per FFMA2
template <int C>
__device__ __forceinline__ float2 paired_preact(const float2* __restrict__ wrow, const float2 f2[C]) {
  float2 pre = make_float2(0.f, 0.f);
  const float4* w4 = reinterpret_cast<const float4*>(wrow);
#pragma unroll
  for (int c = 0; c < C; c += 2) {
    const float4 w = w4[c / 2];
    pre = __ffma2_rn(lo2(w), f2[c], pre);
    pre = __ffma2_rn(hi2(w), f2[c + 1], pre);
  }
  return pre;
}

template <int C, int NP, bool WIDE>
__global__ void __launch_bounds__(128) density_field_fwd_kernel(const __grid_constant__ FieldRef F,
                                                                 const __grid_constant__ KpPoints P, int64_t M,
                                                                 const float* __restrict__ w1, const float* __restrict__ w2,
                                                                 int hidden, int relu, float* __restrict__ density) {
  extern __shared__ __align__(16) float smem[];
  const int hp = (hidden + 1) / 2;
  float2* s_w1p = reinterpret_cast<float2*>(smem);  // [hp][C]
  float2* s_w2p = s_w1p + hp * C;                   // [hp]
  stage_paired_weights<C>(w1, w2, hidden, s_w1p, s_w2p);
  __syncthreads();
  for (int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; m < M; m += (int64_t)gridDim.x * blockDim.x) {
    float pt[4];
    load_point(P, m, pt);
    float2 val2[NP][C / 2];
    Axis ax[4];
    density_features2<C, NP, WIDE>(F, pt, val2, ax);
    float2 f2[C];  // (f[c], f[c]): the multiplicand of both units of a pair
#pragma unroll
    for (int c = 0; c < C / 2; ++c) {
      float2 a = make_float2(1.f, 1.f);
#pragma unroll
      for (int p = 0; p < NP; ++p) a = __fmul2_rn(a, val2[p][c]);
      f2[2 * c] = dup2(a.x);
      f2[2 * c + 1] = dup2(a.y);
    }
    float raw = 0.f;
#pragma unroll 2
    for (int jp = 0; jp < hp; ++jp) {
      float2 pre = paired_preact<C>(s_w1p + jp * C, f2);
      if (relu) {
        pre.x = fmaxf(pre.x, 0.f);
        pre.y = fmaxf(pre.y, 0.f);
      }
      const float2 w2p = s_w2p[jp];
      raw = fmaf(w2p.x, pre.x, raw);
      raw = fmaf(w2p.y, pre.y, raw);
    }
    density[m] = expf(raw);
  }
}

// Backward.  Weight gradients: each warp stages its 32 samples' pre-activations / features / upstream
// gradients in shared memory, then lane l owns hidden units {2l, 2l+1} (for hidden=64) and reduces over the
// 32 samples into registers; registers are flushed with one atomicAdd per weight per block at the end.
// All three fp32 products (forward recompute, d_features, d_weights) run as packed FFMA2 -- the kernel is FMA-issue
// bound (83 M warp instructions per launch in round 1's ncu capture), every half rounds like the scalar fma it replaces.
template <int C, int NP, int HIDDEN, bool WIDE>
__global__ void __launch_bounds__(128, 4) density_field_bwd_kernel(const __grid_constant__ FieldRef F,
                                                                 const __grid_constant__ KpPoints P, int64_t M,
                                                                 const float* __restrict__ w1, const float* __restrict__ w2,
                                                                 int relu, const float* __restrict__ grad_density,
                                                                 float* __restrict__ grad_w1, float* __restrict__ grad_w2) {
  constexpr int WARPS = 4;
  constexpr int HP = HIDDEN / 2;
  static_assert(HIDDEN == 64, "lane l owns the unit pair (2l, 2l+1)");
  extern __shared__ __align__(16) float smem[];
  float* s_w1 = smem;                                      // [HIDDEN][C]   (rows: the d_features product pairs over c)
  float2* s_w1p = reinterpret_cast<float2*>(s_w1 + HIDDEN * C);  // [HP][C]  unit pairs (forward recompute)
  float2* s_w2p = s_w1p + HP * C;                          // [HP]
  float* s_pre = reinterpret_cast<float*>(s_w2p + HP);     // [WARPS][32][HIDDEN+2]  (even row stride: float2 accesses)
  float* s_f = s_pre + WARPS * 32 * (HIDDEN + 2);          // [WARPS][32][C]
  float* s_g = s_f + WARPS * 32 * C;                       // [WARPS][32]
  float* s_acc = s_g + WARPS * 32;                         // [HIDDEN*C + HIDDEN] block accumulators
  for (int i = threadIdx.x; i < HIDDEN * C; i += blockDim.x) s_w1[i] = w1[i];
  stage_paired_weights<C>(w1, w2, HIDDEN, s_w1p, s_w2p);
  for (int i = threadIdx.x; i < HIDDEN * C + HIDDEN; i += blockDim.x) s_acc[i] = 0.f;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int PS = HIDDEN + 2;  // row stride of the staged pre-activations
  float* my_pre = s_pre + warp * 32 * PS;
  float* my_f = s_f + warp * 32 * C;
  float* my_g = s_g + warp * 32;
  float2 acc_w1[C];                       // (d w1[2l][c], d w1[2l+1][c])
  float2 acc_w2 = make_float2(0.f, 0.f);  // (d w2[2l], d w2[2l+1])
#pragma unroll
  for (int c = 0; c < C; ++c) acc_w1[c] = make_float2(0.f, 0.f);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t M_pad = (M + 31) / 32 * 32;
  for (int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; m < M_pad; m += stride) {
    // The gradient reaching a proposal field comes from the interlevel loss, clip(w - w_outer, 0)^2 / (w + eps)
    // (NS/model_components/losses.py:95), which is EXACTLY zero wherever the proposal histogram already bounds the
    // field's: typically 70-90 % of the samples.  A sample with zero upstream gradient contributes nothing to any
    // plane or weight gradient, so a warp whose 32 samples are all zero skips the gather and the MLP altogether.
    const float g_up = (m < M) ? grad_density[m] : 0.f;
    if (__all_sync(0xffffffffu, g_up == 0.f)) continue;
    const bool valid = (m < M) && (g_up != 0.f);
    float pt[4] = {0.f, 0.f, 0.f, 0.f};
    float2 val2[NP][C / 2];
    Axis ax[4];
    float2 fpair[C / 2];  // (f[2c'], f[2c'+1])
    float2 df2[C / 2];    // d loss / d f, same pairing
    float graw = 0.f;
    float2* pre_row = reinterpret_cast<float2*>(my_pre + lane * PS);
    if (valid) {
      load_point(P, m, pt);
      density_features2<C, NP, WIDE>(F, pt, val2, ax);
      float2 f2[C];
#pragma unroll
      for (int c = 0; c < C / 2; ++c) {
        float2 a = make_float2(1.f, 1.f);
#pragma unroll
        for (int p = 0; p < NP; ++p) a = __fmul2_rn(a, val2[p][c]);
        fpair[c] = a;
        f2[2 * c] = dup2(a.x);
        f2[2 * c + 1] = dup2(a.y);
        df2[c] = make_float2(0.f, 0.f);
      }
      float raw = 0.f;
#pragma unroll 2
      for (int jp = 0; jp < HP; ++jp) {
        const float2 pre = paired_preact<C>(s_w1p + jp * C, f2);
        pre_row[jp] = pre;
        const float2 w2p = s_w2p[jp];
        raw = fmaf(w2p.x, relu ? fmaxf(pre.x, 0.f) : pre.x, raw);
        raw = fmaf(w2p.y, relu ? fmaxf(pre.y, 0.f) : pre.y, raw);
      }
      // trunc_exp backward (activations.py:37-39)
      graw = g_up * expf(fminf(fmaxf(raw, -15.f), 15.f));
#pragma unroll 2
      for (int jp = 0; jp < HP; ++jp) {
        const float2 pre = pre_row[jp];
        const float2 w2p = s_w2p[jp];
        const float dpre0 = (relu && !(pre.x > 0.f)) ? 0.f : graw * w2p.x;
        const float dpre1 = (relu && !(pre.y > 0.f)) ? 0.f : graw * w2p.y;
        const float4* r0 = reinterpret_cast<const float4*>(s_w1 + (2 * jp) * C);
        const float4* r1 = reinterpret_cast<const float4*>(s_w1 + (2 * jp + 1) * C);
        // df[c] = fma(dpre_j, w1[j][c], df[c]) in unit order j = 2jp, 2jp+1 (the scalar loop's order), two c per FFMA2
#pragma unroll
        for (int q = 0; q < C / 4; ++q) {
          const float4 w = r0[q];
          df2[2 * q] = __ffma2_rn(dup2(dpre0), lo2(w), df2[2 * q]);
          df2[2 * q + 1] = __ffma2_rn(dup2(dpre0), hi2(w), df2[2 * q + 1]);
        }
#pragma unroll
        for (int q = 0; q < C / 4; ++q) {
          const float4 w = r1[q];
          df2[2 * q] = __ffma2_rn(dup2(dpre1), lo2(w), df2[2 * q]);
          df2[2 * q + 1] = __ffma2_rn(dup2(dpre1), hi2(w), df2[2 * q + 1]);
        }
      }
    } else {
      for (int jp = 0; jp < HP; ++jp) pre_row[jp] = make_float2(0.f, 0.f);
#pragma unroll
      for (int c = 0; c < C / 2; ++c) fpair[c] = make_float2(0.f, 0.f);
    }
#pragma unroll
    for (int c = 0; c < C / 2; ++c) reinterpret_cast<float2*>(my_f + lane * C)[c] = fpair[c];
    my_g[lane] = graw;
    __syncwarp();
    // weight-gradient reduction over the warp's 32 samples: lane l accumulates units (2l, 2l+1)
    const float2 w2l = s_w2p[lane];
#pragma unroll 2
    for (int s = 0; s < 32; ++s) {
      const float gs = my_g[s];
      const float2 pre = reinterpret_cast<const float2*>(my_pre + s * PS)[lane];
      const float2 h = make_float2(relu ? fmaxf(pre.x, 0.f) : pre.x, relu ? fmaxf(pre.y, 0.f) : pre.y);
      const float2 dpre = make_float2((relu && !(pre.x > 0.f)) ? 0.f : gs * w2l.x, (relu && !(pre.y > 0.f)) ? 0.f : gs * w2l.y);
      acc_w2 = __ffma2_rn(dup2(gs), h, acc_w2);
      const float* fs = my_f + s * C;
#pragma unroll
      for (int c = 0; c < C; ++c) acc_w1[c] = __ffma2_rn(dpre, dup2(fs[c]), acc_w1[c]);
    }
    __syncwarp();
    // plane gradients
    if (valid) {
#pragma unroll
      for (int p = 0; p < NP; ++p) {
        const PlaneRef& pr = F.pl[p];
        if (!((F.use_mask >> p) & 1u) || pr.g == nullptr) continue;
        const Bilerp bp = bilerp_from_axes(ax[plane_ca<NP>(p)], ax[plane_cb<NP>(p)], pr.W);
        float2 gp[C / 2];
#pragma unroll
        for (int c = 0; c < C / 2; ++c) {
          float2 a = df2[c];
#pragma unroll
          for (int q = 0; q < NP; ++q)
            if (q != p) a = __fmul2_rn(a, val2[q][c]);
          gp[c] = a;
        }
#pragma unroll
        for (int q = 0; q < C / 4; ++q) {
          const float2 glo = gp[2 * q], ghi = gp[2 * q + 1];
          float* gb = pr.g + q * 4;
          auto red = [&](int32_t off, float w) {
            const float2 a = __fmul2_rn(glo, dup2(w)), b2 = __fmul2_rn(ghi, dup2(w));
            red_add_v4(gb + (int64_t)off * C, make_float4(a.x, a.y, b2.x, b2.y));
          };
          if (bp.w00 != 0.f) red(bp.o00, bp.w00);
          if (bp.w01 != 0.f) red(bp.o01, bp.w01);
          if (bp.w10 != 0.f) red(bp.o10, bp.w10);
          if (bp.w11 != 0.f) red(bp.o11, bp.w11);
        }
      }
    }
  }
  // flush register accumulators: warps -> block smem -> global
  atomicAdd(&s_acc[HIDDEN * C + 2 * lane], acc_w2.x);
  atomicAdd(&s_acc[HIDDEN * C + 2 * lane + 1], acc_w2.y);
#pragma unroll
  for (int c = 0; c < C; ++c) {
    atomicAdd(&s_acc[(2 * lane) * C + c], acc_w1[c].x);
    atomicAdd(&s_acc[(2 * lane + 1) * C + c], acc_w1[c].y);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < HIDDEN * C; i += blockDim.x) red_add_f32(grad_w1 + i, s_acc[i]);
  for (int i = threadIdx.x; i < HIDDEN; i += blockDim.x) red_add_f32(grad_w2 + i, s_acc[HIDDEN * C + i]);
}

// delta != NULL (forward of a six-plane field): the dynamics-score kernels, chosen exactly as the plain forward kernels are
template <int C>
static int launch_hexplane(bool bwd, const FieldRef& F, const KpPoints& P, int64_t M, const float* grad_out, float* out,
                           float* delta, cudaStream_t st) {
  constexpr int LPS = C / 4;
  const int64_t blocks = ceil_div(M * LPS, 128);
  if (blocks == 0) return 0;
  KP_CHECK(blocks < (1ll << 31), "hexplane: M too large");
  bool any_stream = false;  // the L2-policy variant only where a plane asks for it (it costs registers: 0.162 -> 0.181 ms at cfg2)
  for (int k = 0; k < F.n_scales; ++k)
    for (int p = 0; p < F.n_planes; ++p) any_stream |= F.pl[k * KP_MAX_PLANES + p].stream != 0;
  if constexpr (C == 32) {
    // wide mapping (4 lanes x 8 channels per sample).  Measured on B200 (gpurun_out/s3k_bench*): L2-resident field (cfg2
    // training) 0.165 -> 0.150 ms; coherent rays of full-frame inference 361.9 -> 352.3 ms per frame; HBM-resident field with
    // random rays (cfg3 training) 0.359 -> 0.405 ms -- there the float4 kernel keeps more requests in flight.  Hence: wide
    // unless the field streams from HBM (any_stream) with incoherent rays.  Needs 32-byte aligned planes and output rows.
    const bool coherent = P.ray_tile > 1 && P.pts == nullptr;
    bool wide = !bwd && (coherent || !any_stream) && P.ray_tile >= 0;  // (< 0: float4 kernel, tests)
    wide = wide && (reinterpret_cast<uintptr_t>(out) & 31) == 0;
    for (int k = 0; k < F.n_scales && wide; ++k)
      for (int p = 0; p < F.n_planes; ++p) wide = wide && (reinterpret_cast<uintptr_t>(F.pl[k * KP_MAX_PLANES + p].p) & 31) == 0;
    if (wide) {
      const int64_t wb = ceil_div(M * 4, 128);
      if (delta != nullptr) {
        if (any_stream) hexplane_fwd_wide_dyn_kernel<true><<<(unsigned)wb, 128, 0, st>>>(F, P, M, out, delta);
        else hexplane_fwd_wide_dyn_kernel<false><<<(unsigned)wb, 128, 0, st>>>(F, P, M, out, delta);
      } else if (F.n_planes == 6) {
        if (any_stream) hexplane_fwd_wide_kernel<6, true><<<(unsigned)wb, 128, 0, st>>>(F, P, M, out);
        else hexplane_fwd_wide_kernel<6, false><<<(unsigned)wb, 128, 0, st>>>(F, P, M, out);
      } else {
        hexplane_fwd_wide_kernel<3, false><<<(unsigned)wb, 128, 0, st>>>(F, P, M, out);
      }
      KP_LAUNCH_CHECK("hexplane (wide)");
      return 0;
    }
  }
  if (delta != nullptr) {
    if (any_stream) hexplane_fwd_dyn_kernel<C, true><<<(unsigned)blocks, 128, 0, st>>>(F, P, M, out, delta);
    else hexplane_fwd_dyn_kernel<C, false><<<(unsigned)blocks, 128, 0, st>>>(F, P, M, out, delta);
  } else if (F.n_planes == 6) {
    if (any_stream) {
      if (!bwd) hexplane_fwd_kernel<C, 6, true><<<(unsigned)blocks, 128, 0, st>>>(F, P, M, out);
      else hexplane_bwd_kernel<C, 6, true><<<(unsigned)blocks, 128, 0, st>>>(F, P, M, grad_out);
    } else {
      if (!bwd) hexplane_fwd_kernel<C, 6, false><<<(unsigned)blocks, 128, 0, st>>>(F, P, M, out);
      else hexplane_bwd_kernel<C, 6, false><<<(unsigned)blocks, 128, 0, st>>>(F, P, M, grad_out);
    }
  } else {
    if (!bwd) hexplane_fwd_kernel<C, 3, false><<<(unsigned)blocks, 128, 0, st>>>(F, P, M, out);
    else hexplane_bwd_kernel<C, 3, false><<<(unsigned)blocks, 128, 0, st>>>(F, P, M, grad_out);
  }
  KP_LAUNCH_CHECK("hexplane");
  return 0;
}

static int dispatch_hexplane(bool bwd, int C, const FieldRef& F, const KpPoints& P, int64_t M, const float* grad_out,
                             float* out, float* delta, cudaStream_t st) {
  switch (C) {
    case 4: return launch_hexplane<4>(bwd, F, P, M, grad_out, out, delta, st);
    case 8: return launch_hexplane<8>(bwd, F, P, M, grad_out, out, delta, st);
    case 16: return launch_hexplane<16>(bwd, F, P, M, grad_out, out, delta, st);
    case 32: return launch_hexplane<32>(bwd, F, P, M, grad_out, out, delta, st);
    case 64: return launch_hexplane<64>(bwd, F, P, M, grad_out, out, delta, st);
    default: set_error("hexplane: feature dim C=%d unsupported (4,8,16,32,64)", C); return 1;
  }
}

static int check_points(const KpPoints* P, int64_t M) {
  KP_CHECK(P != nullptr, "points is NULL");
  KP_CHECK(P->D == 3 || P->D == 4, "points.D=%d must be 3 or 4", P->D);
  if (M == 0) return 0;
  if (P->pts == nullptr) {
    KP_CHECK(P->origins && P->directions && P->starts && P->ends, "ray-form points need origins/directions/starts/ends");
    KP_CHECK(P->S >= 1 && M % P->S == 0, "M=%lld not a multiple of S=%d", (long long)M, P->S);
    KP_CHECK(P->D == 3 || P->times != nullptr, "dynamic field (D=4) needs times");
  }
  return 0;
}

}  // namespace kp

using namespace kp;

extern "C" int kp_hexplane_fwd(const float* const* plane_ptrs, const int32_t* plane_hw, int n_scales, int n_planes,
                               int C, const KpPoints* points, int64_t M, int concat, uint32_t use_mask, float* out,
                               void* stream) {
  if (check_points(points, M)) return 1;
  KP_CHECK(out != nullptr || M == 0, "hexplane_fwd: out is NULL");
  FieldRef F;
  if (fill_field(F, plane_ptrs, nullptr, plane_hw, n_scales, n_planes, points->D, use_mask, concat, C)) return 1;
  return dispatch_hexplane(false, C, F, *points, M, nullptr, out, nullptr, as_stream(stream));
}

extern "C" int kp_hexplane_fwd_dyn(const float* const* plane_ptrs, const int32_t* plane_hw, int n_scales, int n_planes,
                                   int C, const KpPoints* points, int64_t M, int concat, uint32_t use_mask, float* out,
                                   float* delta, void* stream) {
  KP_CHECK(n_planes == 6, "hexplane_fwd_dyn: a static field (n_planes=%d) has no time planes", n_planes);
  if (check_points(points, M)) return 1;
  KP_CHECK((out != nullptr && delta != nullptr) || M == 0, "hexplane_fwd_dyn: out or delta is NULL");
  FieldRef F;
  if (fill_field(F, plane_ptrs, nullptr, plane_hw, n_scales, n_planes, points->D, use_mask, concat, C)) return 1;
  return dispatch_hexplane(false, C, F, *points, M, nullptr, out, delta, as_stream(stream));
}

extern "C" int kp_hexplane_bwd_flags(const float* const* plane_ptrs, float* const* grad_plane_ptrs, uint8_t* const* touched_ptrs,
                                     const int32_t* plane_hw, int n_scales, int n_planes, int C, const KpPoints* points, int64_t M,
                                     int concat, uint32_t use_mask, const float* grad_out, void* stream) {
  if (check_points(points, M)) return 1;
  KP_CHECK(grad_out != nullptr || M == 0, "hexplane_bwd: grad_out is NULL");
  KP_CHECK(grad_plane_ptrs != nullptr, "hexplane_bwd: grad_plane_ptrs is NULL");
  FieldRef F;
  if (fill_field(F, plane_ptrs, grad_plane_ptrs, plane_hw, n_scales, n_planes, points->D, use_mask, concat, C)) return 1;
  if (touched_ptrs != nullptr)
    for (int k = 0; k < n_scales; ++k)
      for (int p = 0; p < n_planes; ++p) F.pl[k * KP_MAX_PLANES + p].f = touched_ptrs[k * n_planes + p];
  return dispatch_hexplane(true, C, F, *points, M, grad_out, nullptr, nullptr, as_stream(stream));
}

extern "C" int kp_hexplane_bwd(const float* const* plane_ptrs, float* const* grad_plane_ptrs, const int32_t* plane_hw,
                               int n_scales, int n_planes, int C, const KpPoints* points, int64_t M, int concat,
                               uint32_t use_mask, const float* grad_out, void* stream) {
  return kp_hexplane_bwd_flags(plane_ptrs, grad_plane_ptrs, nullptr, plane_hw, n_scales, n_planes, C, points, M, concat, use_mask,
                               grad_out, stream);
}

template <int C>
static int launch_density(bool bwd, const FieldRef& F, const KpPoints& P, int64_t M, const float* w1, const float* w2,
                          int hidden, int relu, float* density, const float* grad_density, float* gw1, float* gw2,
                          cudaStream_t st) {
  if (M == 0) return 0;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  // 8-channel texels are read with one 256-bit load each when every plane is 32-byte aligned (torch allocations and the
  // gradient / parameter buckets are; a view at an odd offset falls back to two 128-bit loads)
  bool wide = C == 8;
  for (int p = 0; p < F.n_planes; ++p) wide = wide && (reinterpret_cast<uintptr_t>(F.pl[p].p) & 31) == 0;
  if (!bwd) {
    const size_t smem = (size_t)((hidden + 1) / 2) * (C + 1) * sizeof(float2);  // unit pairs (stage_paired_weights)
    const int64_t blocks = std::min<int64_t>(ceil_div(M, 128), (int64_t)sms * 16);
    auto launch = [&](auto kern) { kern<<<(unsigned)blocks, 128, smem, st>>>(F, P, M, w1, w2, hidden, relu, density); };
    if (F.n_planes == 6) {
      if (wide) launch(density_field_fwd_kernel<C, 6, true>);
      else launch(density_field_fwd_kernel<C, 6, false>);
    } else {
      if (wide) launch(density_field_fwd_kernel<C, 3, true>);
      else launch(density_field_fwd_kernel<C, 3, false>);
    }
  } else {
    KP_CHECK(hidden == 64, "density_field_bwd: hidden=%d unsupported (64)", hidden);
    constexpr int HIDDEN = 64;
    const size_t smem =  // w1 rows + w1 unit pairs + w2 pairs + staged pre-activations / features / gradients + accumulators
        (size_t)(HIDDEN * C + HIDDEN * C + HIDDEN + 4 * 32 * (HIDDEN + 2) + 4 * 32 * C + 4 * 32 + HIDDEN * C + HIDDEN) * sizeof(float);
    const int64_t blocks = std::min<int64_t>(ceil_div(M, 128), (int64_t)sms * 4);
    auto launch = [&](auto kern) {
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      kern<<<(unsigned)blocks, 128, smem, st>>>(F, P, M, w1, w2, relu, grad_density, gw1, gw2);
    };
    if (F.n_planes == 6) {
      if (wide) launch(density_field_bwd_kernel<C, 6, HIDDEN, true>);
      else launch(density_field_bwd_kernel<C, 6, HIDDEN, false>);
    } else {
      if (wide) launch(density_field_bwd_kernel<C, 3, HIDDEN, true>);
      else launch(density_field_bwd_kernel<C, 3, HIDDEN, false>);
    }
  }
  KP_LAUNCH_CHECK("density_field");
  return 0;
}

static int dispatch_density(bool bwd, int C, const FieldRef& F, const KpPoints& P, int64_t M, const float* w1,
                            const float* w2, int hidden, int relu, float* density, const float* grad_density, float* gw1,
                            float* gw2, cudaStream_t st) {
  switch (C) {
    case 4: return launch_density<4>(bwd, F, P, M, w1, w2, hidden, relu, density, grad_density, gw1, gw2, st);
    case 8: return launch_density<8>(bwd, F, P, M, w1, w2, hidden, relu, density, grad_density, gw1, gw2, st);
    case 16: return launch_density<16>(bwd, F, P, M, w1, w2, hidden, relu, density, grad_density, gw1, gw2, st);
    default: set_error("density_field: feature dim C=%d unsupported (4,8,16)", C); return 1;
  }
}

extern "C" int kp_density_field_fwd(const float* const* plane_ptrs, const int32_t* plane_hw, int n_planes, int C,
                                    const float* w1, const float* w2, int hidden, int relu, const KpPoints* points,
                                    int64_t M, uint32_t use_mask, float* density, void* stream) {
  if (check_points(points, M)) return 1;
  KP_CHECK(w1 && w2 && hidden >= 1 && hidden <= 256, "density_field_fwd: bad MLP arguments");
  FieldRef F;
  if (fill_field(F, plane_ptrs, nullptr, plane_hw, 1, n_planes, points->D, use_mask, 0, C)) return 1;
  return dispatch_density(false, C, F, *points, M, w1, w2, hidden, relu, density, nullptr, nullptr, nullptr,
                          as_stream(stream));
}

extern "C" int kp_density_field_bwd(const float* const* plane_ptrs, float* const* grad_plane_ptrs,
                                    const int32_t* plane_hw, int n_planes, int C, const float* w1, const float* w2,
                                    int hidden, int relu, const KpPoints* points, int64_t M, uint32_t use_mask,
                                    const float* grad_density, float* grad_w1, float* grad_w2, void* stream) {
  if (check_points(points, M)) return 1;
  KP_CHECK(w1 && w2 && grad_w1 && grad_w2 && grad_density, "density_field_bwd: NULL argument");
  KP_CHECK(grad_plane_ptrs != nullptr, "density_field_bwd: grad_plane_ptrs is NULL");
  FieldRef F;
  if (fill_field(F, plane_ptrs, grad_plane_ptrs, plane_hw, 1, n_planes, points->D, use_mask, 0, C)) return 1;
  return dispatch_density(true, C, F, *points, M, w1, w2, hidden, relu, nullptr, grad_density, grad_w1, grad_w2,
                          as_stream(stream));
}
