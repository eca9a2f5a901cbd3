// Decoder MLPs (sigma_net / color_net) -- fp32, bias-free (tcnn FullyFusedMLP semantics in fp32).
// Reference: NS/fields/kplanes_field.py:249-273 (networks), :302-311 (density), :314-358 (colour),
// NS/utils/math.py:25-86 (SH basis), NS/field_components/activations.py:25-41 (trunc_exp).
//
// Implementation: one shared-memory tiled SGEMM kernel (64x64x16 tiles, 4x4 register micro-tiles, operands
// staged reduction-major so both micro-tile operands are 16-byte LDS) instantiated for the three products a
// dense layer needs -- Y = X W^T, dX = dY W, dW += dY^T X (split over the M reduction, atomically
// accumulated) -- with the activations / masks fused in the epilogues.
#include <algorithm>

#include "common.cuh"

int kp_color_fwd_fused_launch(const float* directions, int S, const float* o, int ldo, const float* w3, const float* w4,
                              const float* w5, int64_t M, float* cin, float* h2, float* h3, float* rgb, cudaStream_t st);

namespace kp {

enum { EPI_NONE = 0, EPI_RELU = 1, EPI_SIGMOID = 2, EPI_RELU_MASK = 3, EPI_ATOMIC = 4 };

constexpr int TI = 64, TJ = 64, TR = 16, PAD = 4;

// C[i][j] (+)= sum_r A(i,r) * B(j,r)
//   A_RED_MAJOR == 0: A(i,r) = A[i*lda + r]    (reduction index contiguous)
//   A_RED_MAJOR == 1: A(i,r) = A[r*lda + i]    (output index contiguous)
// R range handled by this block: [blockIdx.z * r_chunk, +r_chunk).
template <int A_RED_MAJOR, int B_RED_MAJOR, int EPI>
__global__ void __launch_bounds__(256) sgemm_kernel(const float* __restrict__ A, int lda, const float* __restrict__ B,
                                                    int ldb, float* __restrict__ Cm, int ldc, int64_t I, int J, int64_t R,
                                                    int64_t r_chunk, const float* __restrict__ aux, int ldaux) {
  __shared__ __align__(16) float As[TR][TI + PAD];
  __shared__ __align__(16) float Bs[TR][TJ + PAD];
  const int tid = threadIdx.x;
  const int64_t i0 = (int64_t)blockIdx.x * TI;
  const int j0 = blockIdx.y * TJ;
  const int64_t r_begin = (int64_t)blockIdx.z * r_chunk;
  const int64_t r_end = r_begin + r_chunk < R ? r_begin + r_chunk : R;
  const int ty = tid / 16, tx = tid % 16;
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;

  for (int64_t r0 = r_begin; r0 < r_end; r0 += TR) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int idx = tid + 256 * e;
      if (A_RED_MAJOR == 0) {
        const int r = idx % TR, i = idx / TR;
        const int64_t gi = i0 + i, gr = r0 + r;
        As[r][i] = (gi < I && gr < r_end) ? __ldg(A + gi * lda + gr) : 0.f;
      } else {
        const int i = idx % TI, r = idx / TI;
        const int64_t gi = i0 + i, gr = r0 + r;
        As[r][i] = (gi < I && gr < r_end) ? __ldg(A + gr * lda + gi) : 0.f;
      }
      if (B_RED_MAJOR == 0) {
        const int r = idx % TR, j = idx / TR;
        const int gj = j0 + j;
        const int64_t gr = r0 + r;
        Bs[r][j] = (gj < J && gr < r_end) ? __ldg(B + (int64_t)gj * ldb + gr) : 0.f;
      } else {
        const int j = idx % TJ, r = idx / TJ;
        const int gj = j0 + j;
        const int64_t gr = r0 + r;
        Bs[r][j] = (gj < J && gr < r_end) ? __ldg(B + gr * ldb + gj) : 0.f;
      }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < TR; ++r) {
      const float4 a = *reinterpret_cast<const float4*>(&As[r][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[r][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) acc[x][y] = fmaf(av[x], bv[y], acc[x][y]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int x = 0; x < 4; ++x) {
    const int64_t gi = i0 + ty * 4 + x;
    if (gi >= I) continue;
#pragma unroll
    for (int y = 0; y < 4; ++y) {
      const int gj = j0 + tx * 4 + y;
      if (gj >= J) continue;
      float v = acc[x][y];
      float* dst = Cm + gi * ldc + gj;
      if (EPI == EPI_RELU) v = fmaxf(v, 0.f);
      if (EPI == EPI_SIGMOID) v = 1.f / (1.f + expf(-v));
      if (EPI == EPI_RELU_MASK) v = (aux[gi * ldaux + gj] > 0.f) ? v : 0.f;
      if (EPI == EPI_ATOMIC) red_add_f32(dst, v); else *dst = v;
    }
  }
}

// The three products of a dense layer.  Shapes covered by the tcgen05 kernels (tc_linear.cu) run on the tensor cores
// (4-term TF32 split, fp32-accurate) -- including the 192->128 first layer of the 32x config, which is cut into
// sub-matrix launches there; anything wider than 256 falls back to the SIMT SGEMM above.
// Y[M,N] = act(X[M,K] W[N,K]^T)
static int g_tc_status = 0;  // first non-zero status of a tensor-core entry point called from this file (checked by the callers)

template <int EPI>
static void gemm_fwd(const float* X, int ldx, const float* W, int ldw, float* Y, int ldy, int64_t M, int N, int K,
                     cudaStream_t st) {
  if (kp_tc_supported(N, K)) {
    const int rc = kp_tc_linear_fwd(X, ldx, W, ldw, Y, ldy, M, N, K, EPI == EPI_RELU ? 1 : (EPI == EPI_SIGMOID ? 2 : 0), st);
    if (rc != 0 && g_tc_status == 0) g_tc_status = rc;
    return;
  }
  dim3 grid((unsigned)ceil_div(M, TI), (unsigned)ceil_div(N, TJ), 1);
  sgemm_kernel<0, 0, EPI><<<grid, 256, 0, st>>>(X, ldx, W, ldw, Y, ldy, M, N, K, K, nullptr, 0);
  kp::g_launches += 1;
}
// dX[M,K] = (dY[M,N] W[N,K]) (* mask(aux > 0))
template <int EPI>
static void gemm_dx(const float* dY, int lddy, const float* W, int ldw, float* dX, int lddx, int64_t M, int N, int K,
                    const float* aux, int ldaux, cudaStream_t st) {
  if (kp_tc_supported(N, K)) {
    const int rc = kp_tc_linear_bwd_data(dY, lddy, W, ldw, dX, lddx, M, N, K, EPI == EPI_RELU_MASK ? aux : nullptr, ldaux, st);
    if (rc != 0 && g_tc_status == 0) g_tc_status = rc;
    return;
  }
  dim3 grid((unsigned)ceil_div(M, TI), (unsigned)ceil_div(K, TJ), 1);
  sgemm_kernel<0, 1, EPI><<<grid, 256, 0, st>>>(dY, lddy, W, ldw, dX, lddx, M, K, N, N, aux, ldaux);
  kp::g_launches += 1;
}
// dW[N,K] += dY[M,N]^T X[M,K]   (reduction over M split across blockIdx.z)
static void gemm_dw(const float* dY, int lddy, const float* X, int ldx, float* dW, int lddw, int64_t M, int N, int K,
                    cudaStream_t st) {
  if (N <= 1024 && K <= 1024) {  // (layers wider than one launch's operand tiles are cut into blocks of dW there)
    const int rc = kp_tc_linear_bwd_weight(dY, lddy, X, ldx, dW, lddw, M, N, K, st);
    if (rc != 0 && g_tc_status == 0) g_tc_status = rc;
    return;
  }
  const int64_t chunk = 1024;
  dim3 grid((unsigned)ceil_div(N, TI), (unsigned)ceil_div(K, TJ), (unsigned)ceil_div(M, chunk));
  sgemm_kernel<1, 1, EPI_ATOMIC><<<grid, 256, 0, st>>>(dY, lddy, X, ldx, dW, lddw, N, K, M, chunk, nullptr, 0);
  kp::g_launches += 1;
}

__global__ void density_from_o_kernel(const float* __restrict__ o, int64_t M, float* __restrict__ density) {
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m < M) density[m] = expf(o[m * 16 + 15]);
}

// d_o[m, 0:15] = grad_geo (or 0); d_o[m,15] = grad_density * exp(clamp(o15, -15, 15))
__global__ void sigma_dout_kernel(const float* __restrict__ o, const float* __restrict__ gdens,
                                  const float* __restrict__ ggeo, int64_t M, float* __restrict__ d_o) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * 16) return;
  const int64_t m = idx / 16;
  const int c = (int)(idx % 16);
  float v = ggeo != nullptr ? ggeo[idx] : 0.f;
  if (c == 15 && gdens != nullptr) v += gdens[m] * expf(fminf(fmaxf(o[idx], -15.f), 15.f));
  d_o[idx] = v;
}

// cin = [SH4(2*((d+1)/2)-1) | geo(15) | 0] (view dependent, width 32) or [geo(15) | 0] (width 16)
__global__ void color_input_kernel(const float* __restrict__ dirs, int S, const float* __restrict__ o, int ldgeo,
                                   int64_t M, float* __restrict__ cin) {
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const float* geo = o + m * ldgeo;
  if (dirs == nullptr) {
    float* dst = cin + m * 16;
#pragma unroll
    for (int c = 0; c < 15; ++c) dst[c] = geo[c];
    dst[15] = 0.f;
    return;
  }
  const int64_t n = m / S;
  float* dst = cin + m * 32;
  float sh[16];
  sh16(dirs[n * 3 + 0], dirs[n * 3 + 1], dirs[n * 3 + 2], sh);
#pragma unroll
  for (int c = 0; c < 16; ++c) dst[c] = sh[c];
#pragma unroll
  for (int c = 0; c < 15; ++c) dst[16 + c] = geo[c];
  dst[31] = 0.f;
}

// d_pre[m, c] = grad_rgb * rgb * (1 - rgb), stored with leading dimension 4
__global__ void sigmoid_grad_kernel(const float* __restrict__ rgb, const float* __restrict__ grgb, int64_t M,
                                    float* __restrict__ dpre) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * 4) return;
  const int64_t m = idx / 4;
  const int c = (int)(idx % 4);
  float v = 0.f;
  if (c < 3) {
    const float s = rgb[m * 3 + c];
    v = grgb[m * 3 + c] * s * (1.f - s);
  }
  dpre[idx] = v;
}


// ---------------------------------------------------------------------------------------------------------------
// Backward of the colour net's output layer (rgb = sigmoid(h3 W5^T), 3 outputs) in plain fp32 SIMT, one pass:
//   dOut[M,3] = grad_rgb * rgb * (1 - rgb) is formed on the fly (never written),
//   dH[M,K] = (dOut . W) * (H > 0)            (the hidden layer's ReLU mask)
//   dW[3,K] += dOut^T . H
// With 3 outputs the two products are 24 FMAs per 16 bytes of H: far below the memory time of streaming H in and dH
// out, so the tensor-core route (two GEMM launches that each stream H again, plus a kernel that materialises dOut)
// only adds launches and passes over memory.  K/4 lanes own one row (coalesced 16-byte accesses); every lane keeps its
// four columns of W and of the dW accumulator in registers; block-level reduction of dW in shared memory, one red per
// weight per block.
// ---------------------------------------------------------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(128) narrow_layer_bwd_kernel(const float* __restrict__ H, float* __restrict__ dH,
                                                               const float* __restrict__ W, float* __restrict__ dW, int64_t M,
                                                               const float* __restrict__ rgb, const float* __restrict__ grad_rgb) {
  constexpr int NO = 3;
  constexpr int LPR = K / 4;      // lanes per row
  constexpr int RPW = 32 / LPR;   // rows per warp pass
  static_assert(LPR == 16 || LPR == 32, "K must be 64 or 128");
  __shared__ float s_acc[NO * K];
  for (int i = threadIdx.x; i < NO * K; i += blockDim.x) s_acc[i] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = lane % LPR, sub = lane / LPR;
  float4 w[NO], acc[NO];
#pragma unroll
  for (int j = 0; j < NO; ++j) {
    w[j] = ldg4(W + (size_t)j * K + 4 * q);
    acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const int64_t warps_total = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t gw = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
  constexpr int U = 4;  // rows in flight per lane: all loads of U rows are issued before the arithmetic
  for (int64_t base = gw * RPW * U; base < M; base += warps_total * RPW * U) {
    float d[U][NO];
    float4 h[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t s = base + u * RPW + sub;
      h[u] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int j = 0; j < NO; ++j) d[u][j] = 0.f;
      if (s < M) {
#pragma unroll
        for (int j = 0; j < NO; ++j) {
          const float sg = __ldg(rgb + s * NO + j);
          d[u][j] = __ldg(grad_rgb + s * NO + j) * sg * (1.f - sg);
        }
        h[u] = ldg4(H + s * K + 4 * q);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t s = base + u * RPW + sub;
      if (s >= M) continue;
      float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int j = 0; j < NO; ++j) {
        o = fma4(w[j], d[u][j], o);
        acc[j] = fma4(h[u], d[u][j], acc[j]);
      }
      if (!(h[u].x > 0.f)) o.x = 0.f;
      if (!(h[u].y > 0.f)) o.y = 0.f;
      if (!(h[u].z > 0.f)) o.z = 0.f;
      if (!(h[u].w > 0.f)) o.w = 0.f;
      *reinterpret_cast<float4*>(dH + s * K + 4 * q) = o;
    }
  }
#pragma unroll
  for (int j = 0; j < NO; ++j) {
    atomicAdd(&s_acc[j * K + 4 * q + 0], acc[j].x);
    atomicAdd(&s_acc[j * K + 4 * q + 1], acc[j].y);
    atomicAdd(&s_acc[j * K + 4 * q + 2], acc[j].z);
    atomicAdd(&s_acc[j * K + 4 * q + 3], acc[j].w);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < NO * K; i += blockDim.x) red_add_f32(dW + i, s_acc[i]);
}

// false when the shape or the alignment does not fit narrow_layer_bwd_kernel (the caller then takes the GEMM route)
static bool launch_narrow_bwd(int K, const float* H, float* dH, const float* W, float* dW, int64_t M, const float* rgb,
                              const float* grad_rgb, cudaStream_t st) {
  if (K != 64 && K != 128) return false;
  if ((((uintptr_t)H | (uintptr_t)dH | (uintptr_t)W) & 15) != 0) return false;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int rpw = 32 / (K / 4);
  const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div(M, 4 * rpw), (int64_t)sms * 4));
  if (K == 64) narrow_layer_bwd_kernel<64><<<grid, 128, 0, st>>>(H, dH, W, dW, M, rgb, grad_rgb);
  else narrow_layer_bwd_kernel<128><<<grid, 128, 0, st>>>(H, dH, W, dW, M, rgb, grad_rgb);
  kp::g_launches += 1;
  return true;
}

}  // namespace kp

using namespace kp;

extern "C" int kp_sigma_net_fwd(const float* feats, const float* w1, const float* w2, int64_t M, int K, int H, float* h1,
                                float* o, float* density, void* stream) {
  if (M == 0) return 0;
  KP_CHECK(feats && w1 && w2 && h1 && o && density && K >= 1 && H >= 1, "sigma_net_fwd: bad arguments");
  cudaStream_t st = as_stream(stream);
  gemm_fwd<EPI_RELU>(feats, K, w1, K, h1, H, M, H, K, st);
  gemm_fwd<EPI_NONE>(h1, H, w2, H, o, 16, M, 16, H, st);
  density_from_o_kernel<<<(unsigned)ceil_div(M, 256), 256, 0, st>>>(o, M, density);
  KP_LAUNCH_CHECK("sigma_net_fwd");
  if (g_tc_status != 0) { const int rc = g_tc_status; g_tc_status = 0; return rc; }  // (kp_last_error holds the message)
  return 0;
}

extern "C" int kp_sigma_net_bwd(const float* feats, const float* w1, const float* w2, int64_t M, int K, int H,
                                const float* h1, const float* o, const float* grad_density, const float* grad_geo,
                                float* grad_feats, float* grad_w1, float* grad_w2, float* scratch, void* stream) {
  if (M == 0) return 0;
  KP_CHECK(feats && w1 && w2 && h1 && o && grad_w1 && grad_w2 && scratch, "sigma_net_bwd: bad arguments");
  cudaStream_t st = as_stream(stream);
  // d_o = dL/do [M,16] cannot share scratch [M,H], which receives d_h1 while d_o is read; it is kept in grad_feats' first
  // M*16 floats (K >= 16), which only the last GEMM writes.
  KP_CHECK(K >= 16 && grad_feats != nullptr, "sigma_net_bwd: needs grad_feats with K >= 16");
  float* d_o = grad_feats;
  sigma_dout_kernel<<<(unsigned)ceil_div(M * 16, 256), 256, 0, st>>>(o, grad_density, grad_geo, M, d_o);
  gemm_dw(d_o, 16, h1, H, grad_w2, H, M, 16, H, st);
  gemm_dx<EPI_RELU_MASK>(d_o, 16, w2, H, scratch, H, M, 16, H, h1, H, st);   // d_h1
  gemm_dw(scratch, H, feats, K, grad_w1, K, M, H, K, st);
  gemm_dx<EPI_NONE>(scratch, H, w1, K, grad_feats, K, M, H, K, nullptr, 0, st);
  KP_LAUNCH_CHECK("sigma_net_bwd");
  if (g_tc_status != 0) { const int rc = g_tc_status; g_tc_status = 0; return rc; }  // (kp_last_error holds the message)
  return 0;
}

extern "C" int kp_color_net_fwd(const float* directions, int S, const float* o, int ldgeo, const float* w3, const float* w4,
                                const float* w5, int64_t M, int H2, float* cin, float* h2, float* h3, float* rgb,
                                void* stream) {
  if (M == 0) return 0;
  KP_CHECK(o && w3 && w4 && w5 && cin && h2 && h3 && rgb && H2 >= 1 && ldgeo >= 15, "color_net_fwd: bad arguments");
  KP_CHECK(directions == nullptr || (S >= 1 && M % S == 0), "color_net_fwd: M must be a multiple of S");
  cudaStream_t st = as_stream(stream);
  if (H2 == 64) {
    // the whole colour net in one tcgen05 launch (decoder_fused.cu): weights resident, activations chained on chip
    kp_color_fwd_fused_launch(directions, S, o, ldgeo, w3, w4, w5, M, cin, h2, h3, rgb, st);
    KP_LAUNCH_CHECK("color_net_fwd");
    return 0;
  }
  const int ldc = directions ? 32 : 16, kin = directions ? 31 : 15;
  color_input_kernel<<<(unsigned)ceil_div(M, 256), 256, 0, st>>>(directions, S, o, ldgeo, M, cin);
  gemm_fwd<EPI_RELU>(cin, ldc, w3, kin, h2, H2, M, H2, kin, st);
  gemm_fwd<EPI_RELU>(h2, H2, w4, H2, h3, H2, M, H2, H2, st);
  gemm_fwd<EPI_SIGMOID>(h3, H2, w5, H2, rgb, 3, M, 3, H2, st);
  KP_LAUNCH_CHECK("color_net_fwd");
  if (g_tc_status != 0) { const int rc = g_tc_status; g_tc_status = 0; return rc; }  // (kp_last_error holds the message)
  return 0;
}

extern "C" int kp_color_net_bwd(int view_dependent, const float* cin, const float* h2, const float* h3, const float* rgb,
                                const float* w3, const float* w4, const float* w5, int64_t M, int H2,
                                const float* grad_rgb, float* grad_o, float* grad_w3, float* grad_w4, float* grad_w5,
                                float* scratch_a, float* scratch_b, void* stream) {
  if (M == 0) return 0;
  KP_CHECK(cin && h2 && h3 && rgb && w3 && w4 && w5 && grad_rgb && grad_o && grad_w3 && grad_w4 && grad_w5 && scratch_a &&
               scratch_b && H2 >= 4,
           "color_net_bwd: bad arguments");
  cudaStream_t st = as_stream(stream);
  const int ldc = view_dependent ? 32 : 16, kin = view_dependent ? 31 : 15, geo_off = view_dependent ? 16 : 0;
  if (!launch_narrow_bwd(H2, h3, scratch_a, w5, grad_w5, M, rgb, grad_rgb, st)) {  // d_h3 -> a, dW5, one pass
    float* dpre = scratch_b;  // [M,4]
    sigmoid_grad_kernel<<<(unsigned)ceil_div(M * 4, 256), 256, 0, st>>>(rgb, grad_rgb, M, dpre);
    gemm_dw(dpre, 4, h3, H2, grad_w5, H2, M, 3, H2, st);
    gemm_dx<EPI_RELU_MASK>(dpre, 4, w5, H2, scratch_a, H2, M, 3, H2, h3, H2, st);       // d_h3 -> a
  }
  gemm_dw(scratch_a, H2, h2, H2, grad_w4, H2, M, H2, H2, st);
  gemm_dx<EPI_RELU_MASK>(scratch_a, H2, w4, H2, scratch_b, H2, M, H2, H2, h2, H2, st);  // d_h2 -> b
  gemm_dw(scratch_b, H2, cin, ldc, grad_w3, kin, M, H2, kin, st);
  cudaMemsetAsync(grad_o, 0, (size_t)M * 16 * sizeof(float), st);
  gemm_dx<EPI_NONE>(scratch_b, H2, w3 + geo_off, kin, grad_o, 16, M, H2, 15, nullptr, 0, st);  // d_geo
  KP_LAUNCH_CHECK("color_net_bwd");
  if (g_tc_status != 0) { const int rc = g_tc_status; g_tc_status = 0; return rc; }  // (kp_last_error holds the message)
  return 0;
}
