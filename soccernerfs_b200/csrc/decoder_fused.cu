// Fused decoder forward on tcgen05: sigma_net (K0 -> 64 -> 16) and color_net ([SH16 | geo15] -> 64 -> 64 -> 3) of the
// K-Planes field evaluated for a 128-sample tile WITHOUT leaving the SM between layers.
//
// Reference: NS/fields/kplanes_field.py:249-273 (the two tcnn FullyFusedMLPs), :302-311 (density = trunc_exp of the
// last sigma output), :314-358 (colour input = [SH4(dir) | 15 geometry features], sigmoid output).
//
// One persistent CTA (8 warps) per SM:
//   * all five weight matrices live in shared memory as hi/lo TF32 UMMA operands for the whole kernel (128 KB);
//   * the feature tile is staged in two 64-column halves through a 64 KB activation region (its global loads for the
//     next tile are issued into registers a full tile ahead), layer 1 accumulates both halves in TMEM;
//   * each layer's accumulator is read back with tcgen05.ld, the activation applied in registers, and the result
//     written straight back into the activation region as the next layer's A operand (hi/lo split, 128B swizzle);
//     spherical harmonics are evaluated by the idle half of the warps while the other half unloads o;
//   * hidden activations are written to global memory only when the backward pass will need them (training);
//     inference (ns-render, BASELINE config 5) touches global memory for features in and (o, density, rgb) out only.
// Accuracy: four-term TF32 split (see tc_linear.cu), fp32-class.
#include "tc_common.cuh"

namespace kp {

// stage a [ROWS x COLS] row-major fp32 weight matrix (ld, rows_valid, cols_valid) as a K-major hi/lo operand
template <int ROWS, int COLS>
__device__ __forceinline__ void stage_weight(const float* __restrict__ src, int ld, int rows_valid, int cols_valid,
                                             float* __restrict__ s_hi, float* __restrict__ s_lo) {
  for (int idx = threadIdx.x; idx < ROWS * COLS; idx += blockDim.x) {
    const int row = idx / COLS, col = idx % COLS;
    const float v = (row < rows_valid && col < cols_valid) ? __ldg(src + row * ld + col) : 0.f;
    const float hi = to_tf32(v);
    const int ch = col >> 2, kb = ch >> 3, c = ch & 7;
    const int off = kb * (ROWS * 32) + row * 32 + ((c ^ (row & 7)) << 2) + (col & 3);
    s_hi[off] = hi;
    s_lo[off] = v - hi;
  }
}

// write 16 consecutive columns [col0, col0+16) of activation row `row` (values in registers) as hi/lo A-operand chunks
__device__ __forceinline__ void store_act16(const float* x, int row, int col0, float* __restrict__ s_hi, float* __restrict__ s_lo) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int ch = (col0 >> 2) + q, kb = ch >> 3, c = ch & 7;
    const int off = kb * (128 * 32) + row * 32 + ((c ^ (row & 7)) << 2);
    float4 hi, lo;
    hi.x = tf32_hi(x[4 * q]); hi.y = tf32_hi(x[4 * q + 1]); hi.z = tf32_hi(x[4 * q + 2]); hi.w = tf32_hi(x[4 * q + 3]);
    lo.x = x[4 * q] - hi.x; lo.y = x[4 * q + 1] - hi.y; lo.z = x[4 * q + 2] - hi.z; lo.w = x[4 * q + 3] - hi.w;
    *reinterpret_cast<float4*>(s_hi + off) = hi;
    *reinterpret_cast<float4*>(s_lo + off) = lo;
  }
}

// issue the four partial products of  D[128 x N] (+)= A[128 x 8*K8] * B[N x 8*K8]^T  (both K-major, 128B swizzle)
template <int K8>
__device__ __forceinline__ void issue_layer(uint32_t tmem_d, const float* a_hi, const float* a_lo, const float* b_hi,
                                            const float* b_lo, int b_rows, int n, bool accumulate_first) {
  const uint32_t idesc = umma_idesc_tf32(128, n, 0, 0);
  const uint64_t a_d[2] = {desc_kmajor(smem_u32(a_hi), 128, 0, 0), desc_kmajor(smem_u32(a_lo), 128, 0, 0)};
  const uint64_t b_d[2] = {desc_kmajor(smem_u32(b_hi), b_rows, 0, 0), desc_kmajor(smem_u32(b_lo), b_rows, 0, 0)};
  const uint32_t b_blk = (uint32_t)(b_rows * 128) >> 4;
#pragma unroll
  for (int t = 0; t < 4; ++t) {  // lo*lo + lo*hi + hi*lo + hi*hi
    const uint64_t ad0 = a_d[t <= 1], bd0 = b_d[t == 0 || t == 2];
#pragma unroll
    for (int k8 = 0; k8 < K8; ++k8) {
      const uint32_t a_off = (uint32_t)(((k8 >> 2) * 128 * 128 + (k8 & 3) * 32) >> 4);
      const uint32_t b_off = (uint32_t)(k8 >> 2) * b_blk + (uint32_t)(((k8 & 3) * 32) >> 4);
      umma_tf32(tmem_d, ad0 + a_off, bd0 + b_off, idesc, (accumulate_first || (t | k8) != 0) ? 1u : 0u);
    }
  }
}

// Shared-memory carve-up of the colour net's weights (layers 3-5) and the 128 x 64 activation region, behind the sigma
// net's weights in decoder_fwd_fused_kernel and alone in color_fwd_fused_kernel.  All regions are multiples of 1 KB.
struct ColorSmem {
  float *w3_hi, *w3_lo;    // [64 x 32]
  float *w4_hi, *w4_lo;    // [64 x 64]
  float *w5_hi, *w5_lo;    // [16 x 64] (3 valid rows)
  float *act_hi, *act_lo;  // [128 x 64]
};
constexpr int kColorSmemFloats = 2 * 64 * 32 + 2 * 64 * 64 + 2 * 16 * 64 + 2 * 128 * 64;
// the sigma net's weights in front of it in decoder_fwd_fused_kernel: w1 [64 x K0P] and w2 [16 x 64], hi + lo
__host__ __device__ constexpr int sigma_smem_floats(int K0P) { return 2 * 64 * K0P + 2 * 16 * 64; }
// dynamic shared memory of a fused kernel whose colour-net region starts `lead_floats` in (+ 1 KB for align1024)
constexpr size_t fused_smem_bytes(int lead_floats) { return (size_t)(lead_floats + kColorSmemFloats) * sizeof(float) + 1024; }

__device__ __forceinline__ ColorSmem color_smem(float* p) {
  ColorSmem s;
  s.w3_hi = p;
  s.w3_lo = s.w3_hi + 64 * 32;
  s.w4_hi = s.w3_lo + 64 * 32;
  s.w4_lo = s.w4_hi + 64 * 64;
  s.w5_hi = s.w4_lo + 64 * 64;
  s.w5_lo = s.w5_hi + 16 * 64;
  s.act_hi = s.w5_lo + 16 * 64;
  s.act_lo = s.act_hi + 128 * 64;
  return s;
}

// w3 [64 x kin] (colour-input width kin = 31 or 15), w4 [64 x 64], w5 [3 x 64]
__device__ __forceinline__ void stage_color_weights(const float* w3, const float* w4, const float* w5, int kin, const ColorSmem& s) {
  stage_weight<64, 32>(w3, kin, 64, kin, s.w3_hi, s.w3_lo);
  stage_weight<64, 64>(w4, 64, 64, 64, s.w4_hi, s.w4_lo);
  stage_weight<16, 64>(w5, 64, 3, 64, s.w5_hi, s.w5_lo);
}

// The colour input is [SH(16) | geo(15) | 0] (view dependent, cin width 32) or [geo(15) | 0 | zeros(16)] (cin width 16,
// the zero half only in the activation region).  Warps 0-3 write the geometry half from x (x[15] = 0) ...
__device__ __forceinline__ void store_geo_input(const float* x, int row, bool valid, int64_t grow, bool view_dep, float* cin,
                                                const ColorSmem& s) {
  store_act16(x, row, view_dep ? 16 : 0, s.act_hi, s.act_lo);
  if (cin != nullptr && valid) {
#pragma unroll
    for (int q = 0; q < 4; ++q)
      *reinterpret_cast<float4*>(cin + grow * (view_dep ? 32 : 16) + (view_dep ? 16 : 0) + 4 * q) =
          make_float4(x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]);
  }
}
// ... and warps 4-7 the SH basis of the sample's ray direction, or the zero half (x is scratch)
__device__ __forceinline__ void store_sh_input(float* x, int row, bool valid, int64_t grow, const float* dirs, int S, float* cin,
                                               const ColorSmem& s) {
  if (dirs != nullptr) {
    const int64_t ray = valid ? grow / S : 0;
    sh16(dirs[ray * 3 + 0], dirs[ray * 3 + 1], dirs[ray * 3 + 2], x);
    store_act16(x, row, 0, s.act_hi, s.act_lo);
    if (cin != nullptr && valid) {
#pragma unroll
      for (int q = 0; q < 4; ++q)
        *reinterpret_cast<float4*>(cin + grow * 32 + 4 * q) = make_float4(x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) x[j] = 0.f;
    store_act16(x, row, 16, s.act_hi, s.act_lo);  // zero the unused half of the 32-wide colour input
  }
}

// Layers 3-5 on the colour input written to the activation region by every thread: h2 = relu(cin W3^T),
// h3 = relu(h2 W4^T), rgb = sigmoid(h3 W5^T); h2 / h3 go to global memory only when given (training).  Ends with the
// fences after which the next tile's MMAs may reuse the TMEM accumulator.  Every thread of the CTA calls it.
__device__ __forceinline__ void color_layers(const ColorSmem& s, const uint32_t& tmem_slot, uint64_t* mma_bar, uint32_t& parity,
                                             int quad, int half, int row, bool valid, int64_t grow, float* h2, float* h3,
                                             float* rgb) {
  publish_smem_and_sync();
  // ---- layer 3: h2 = relu(cin W3^T) ------------------------------------------------------------------------------
  if (threadIdx.x == 0) {
    issue_layer<4>(tmem_slot, s.act_hi, s.act_lo, s.w3_hi, s.w3_lo, 64, 64, false);
    umma_commit(mma_bar);
  }
  mbar_wait(mma_bar, parity);
  parity ^= 1;
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tbase = tmem_slot + ((uint32_t)(quad * 32) << 16);
  float x[32];
  uint32_t v[16];
#pragma unroll 1
  for (int layer = 0; layer < 2; ++layer) {  // epilogue of h2 then of h3
#pragma unroll
    for (int part = 0; part < 2; ++part) {
      tmem_ld16(tbase + (uint32_t)(half * 32 + part * 16), v);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int j = 0; j < 16; ++j) x[part * 16 + j] = fmaxf(__uint_as_float(v[j]), 0.f);
    }
    store_act16(x, row, half * 32, s.act_hi, s.act_lo);
    store_act16(x + 16, row, half * 32 + 16, s.act_hi, s.act_lo);
    float* hbuf = layer == 0 ? h2 : h3;
    if (hbuf != nullptr && valid) {
#pragma unroll
      for (int q = 0; q < 8; ++q)
        *reinterpret_cast<float4*>(hbuf + grow * 64 + half * 32 + 4 * q) = make_float4(x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]);
    }
    publish_smem_and_sync();
    if (threadIdx.x == 0) {
      if (layer == 0) issue_layer<8>(tmem_slot, s.act_hi, s.act_lo, s.w4_hi, s.w4_lo, 64, 64, false);  // h3 = relu(h2 W4^T)
      else issue_layer<8>(tmem_slot, s.act_hi, s.act_lo, s.w5_hi, s.w5_lo, 16, 16, false);             // rgb = sigmoid(h3 W5^T)
      umma_commit(mma_bar);
    }
    mbar_wait(mma_bar, parity);
    parity ^= 1;
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  }
  // epilogue 5: rgb
  if (half == 0) {
    tmem_ld16(tbase, v);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    if (valid) {
#pragma unroll
      for (int c = 0; c < 3; ++c) rgb[grow * 3 + c] = 1.f / (1.f + expf(-__uint_as_float(v[c])));
    }
  }
  // TMEM reads of this tile complete before the next tile's MMAs reuse the accumulator
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

struct DecoderArgs {
  const float* feats;  // [M, K0]
  const float* dirs;   // [N, 3] or nullptr (disable_viewing_dependent)
  const float *w1, *w2, *w3, *w4, *w5;
  float *h1, *cin, *h2, *h3;  // [M,64], [M,32|16], [M,64], [M,64] or nullptr (inference: not materialised)
  float *o, *density, *rgb;   // [M,16], [M], [M,3]
  int64_t M;
  int K0, S;
};

template <int K0P>  // padded feature width: 64 or 128
__global__ void __launch_bounds__(256, 1) decoder_fwd_fused_kernel(const __grid_constant__ DecoderArgs A) {
  extern __shared__ uint8_t smem_raw[];
  float* w1_hi = align1024(smem_raw);
  float* w1_lo = w1_hi + 64 * K0P;
  float* w2_hi = w1_lo + 64 * K0P;  // [16 x 64]
  float* w2_lo = w2_hi + 16 * 64;
  const ColorSmem cs = color_smem(w1_hi + sigma_smem_floats(K0P));
  __shared__ __align__(8) uint64_t mma_bar;
  __shared__ uint32_t tmem_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool view_dep = A.dirs != nullptr;

  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mma_bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  tmem_alloc(&tmem_slot, warp);
  stage_weight<64, K0P>(A.w1, A.K0, 64, A.K0, w1_hi, w1_lo);
  stage_weight<16, 64>(A.w2, 64, 16, 64, w2_hi, w2_lo);
  stage_color_weights(A.w3, A.w4, A.w5, view_dep ? 31 : 15, cs);

  const int quad = warp & 3, half = warp >> 2;
  const int row = quad * 32 + lane;
  const int64_t n_tiles = (A.M + 127) / 128;
  uint32_t parity = 0;
  constexpr int HALVES = K0P / 64;
  TileRegs<64> pre[HALVES];
  if ((int64_t)blockIdx.x < n_tiles) {
    const int64_t r0 = (int64_t)blockIdx.x * 128;
#pragma unroll
    for (int hh = 0; hh < HALVES; ++hh)
      tile_load<64>(pre[hh], A.feats + r0 * A.K0 + hh * 64, A.K0, (int)min((int64_t)128, A.M - r0), A.K0 - hh * 64);
  }
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t row0 = tile * 128;
    const int rows_valid = (int)min((int64_t)128, A.M - row0);
    const bool valid = row < rows_valid;
    const int64_t grow = row0 + row;
    // ---- layer 1: h1 = relu(X W1^T), X staged in 64-column halves through the activation region -------------
#pragma unroll
    for (int hh = 0; hh < HALVES; ++hh) {
      tile_store<0, 64>(pre[hh], cs.act_hi, cs.act_lo);
      publish_smem_and_sync();
      if (threadIdx.x == 0) {
        issue_layer<8>(tmem_slot, cs.act_hi, cs.act_lo, w1_hi + hh * (2 * 64 * 32), w1_lo + hh * (2 * 64 * 32), 64, 64, hh != 0);
        umma_commit(&mma_bar);
      }
      mbar_wait(&mma_bar, parity);
      parity ^= 1;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    {  // prefetch the next tile's features; they land while layers 2..5 run
      const int64_t nxt = tile + gridDim.x;
      if (nxt < n_tiles) {
#pragma unroll
        for (int hh = 0; hh < HALVES; ++hh)
          tile_load<64>(pre[hh], A.feats + nxt * 128 * A.K0 + hh * 64, A.K0, (int)min((int64_t)128, A.M - nxt * 128),
                        A.K0 - hh * 64);
      }
    }
    const uint32_t tbase = tmem_slot + ((uint32_t)(quad * 32) << 16);
    float x[32];
    uint32_t v[16];
    // epilogue 1: each thread owns 32 of the 64 hidden units of its row
#pragma unroll
    for (int part = 0; part < 2; ++part) {
      tmem_ld16(tbase + (uint32_t)(half * 32 + part * 16), v);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int j = 0; j < 16; ++j) x[part * 16 + j] = fmaxf(__uint_as_float(v[j]), 0.f);
    }
    // all TMEM reads done before layer 2 overwrites the accumulator; all MMAs of layer 1 have completed (waited), so
    // the activation region is free to take h1
    store_act16(x, row, half * 32, cs.act_hi, cs.act_lo);
    store_act16(x + 16, row, half * 32 + 16, cs.act_hi, cs.act_lo);
    if (A.h1 != nullptr && valid) {
#pragma unroll
      for (int q = 0; q < 8; ++q)
        *reinterpret_cast<float4*>(A.h1 + grow * 64 + half * 32 + 4 * q) = make_float4(x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]);
    }
    publish_smem_and_sync();
    // ---- layer 2: o = h1 W2^T (16 outputs: 15 geometry features + sigma_raw) --------------------------------------
    if (threadIdx.x == 0) {
      issue_layer<8>(tmem_slot, cs.act_hi, cs.act_lo, w2_hi, w2_lo, 16, 16, false);
      umma_commit(&mma_bar);
    }
    mbar_wait(&mma_bar, parity);
    parity ^= 1;
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // epilogue 2: warps 0-3 unload o (and write geo into the colour input), warps 4-7 evaluate the SH basis
    if (half == 0) {
      tmem_ld16(tbase, v);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int j = 0; j < 16; ++j) x[j] = __uint_as_float(v[j]);
      if (valid) {
#pragma unroll
        for (int q = 0; q < 4; ++q)
          *reinterpret_cast<float4*>(A.o + grow * 16 + 4 * q) = make_float4(x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]);
        A.density[grow] = expf(x[15]);  // trunc_exp forward (activations.py:31-33)
      }
      x[15] = 0.f;  // colour input = [.. | geo(15) | 0]
      store_geo_input(x, row, valid, grow, view_dep, A.cin, cs);
    } else {
      store_sh_input(x, row, valid, grow, A.dirs, A.S, A.cin, cs);
    }
    color_layers(cs, tmem_slot, &mma_bar, parity, quad, half, row, valid, grow, A.h2, A.h3, A.rgb);
  }
  tmem_free(tmem_slot, warp);
}


// ---------------------------------------------------------------------------------------------------------------
// Colour net alone (layers 3-5 of the chain above) for decoders whose sigma net does not fit the fully fused kernel (the
// 32x preset: 192 -> 128 -> 16): input = the sigma net's output o [M, ldo] (15 geometry features), optional view
// directions; h2 / h3 / cin are written only when given (training).  Same layer chain, same epilogues, one launch instead
// of color_input + three GEMM launches that each stream [M,64] activations through HBM.
// ---------------------------------------------------------------------------------------------------------------
struct ColorArgs {
  const float* o;     // [M, ldo]
  const float* dirs;  // [N, 3] or nullptr
  const float *w3, *w4, *w5;
  float *cin, *h2, *h3, *rgb;
  int64_t M;
  int ldo, S;
};

__global__ void __launch_bounds__(256, 1) color_fwd_fused_kernel(const __grid_constant__ ColorArgs A) {
  extern __shared__ uint8_t smem_raw[];
  const ColorSmem cs = color_smem(align1024(smem_raw));
  __shared__ __align__(8) uint64_t mma_bar;
  __shared__ uint32_t tmem_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool view_dep = A.dirs != nullptr;
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mma_bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  tmem_alloc(&tmem_slot, warp);
  stage_color_weights(A.w3, A.w4, A.w5, view_dep ? 31 : 15, cs);
  const int quad = warp & 3, half = warp >> 2;
  const int row = quad * 32 + lane;
  const int64_t n_tiles = (A.M + 127) / 128;
  uint32_t parity = 0;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t row0 = tile * 128;
    const int rows_valid = (int)min((int64_t)128, A.M - row0);
    const bool valid = row < rows_valid;
    const int64_t grow = row0 + row;
    float x[16];
    if (half == 0) {
#pragma unroll
      for (int j = 0; j < 16; ++j) x[j] = (valid && j < 15) ? __ldg(A.o + grow * A.ldo + j) : 0.f;
      store_geo_input(x, row, valid, grow, view_dep, A.cin, cs);
    } else {
      store_sh_input(x, row, valid, grow, A.dirs, A.S, A.cin, cs);
    }
    color_layers(cs, tmem_slot, &mma_bar, parity, quad, half, row, valid, grow, A.h2, A.h3, A.rgb);
  }
  tmem_free(tmem_slot, warp);
}

}  // namespace kp

using namespace kp;

// 1 if kp_decoder_fwd_fused covers this decoder shape (hidden widths 64, feature width <= 128).
extern "C" int kp_decoder_fused_supported(int K0, int H1, int H2) { return (K0 >= 16 && K0 <= 128 && H1 == 64 && H2 == 64) ? 1 : 0; }

extern "C" int kp_decoder_fwd_fused(const float* feats, int K0, const float* directions, int S, const float* w1,
                                    const float* w2, const float* w3, const float* w4, const float* w5, int64_t M, int H1,
                                    int H2, float* h1, float* cin, float* h2, float* h3, float* o, float* density,
                                    float* rgb, void* stream) {
  if (M == 0) return 0;
  KP_CHECK(kp_decoder_fused_supported(K0, H1, H2), "decoder_fwd_fused: unsupported shape K0=%d H1=%d H2=%d", K0, H1, H2);
  KP_CHECK(feats && w1 && w2 && w3 && w4 && w5 && o && density && rgb, "decoder_fwd_fused: NULL argument");
  KP_CHECK(directions == nullptr || (S >= 1 && M % S == 0), "decoder_fwd_fused: M must be a multiple of S");
  KP_CHECK((K0 & 3) == 0, "decoder_fwd_fused: K0=%d must be a multiple of 4", K0);
  DecoderArgs a;
  a.feats = feats; a.dirs = directions; a.w1 = w1; a.w2 = w2; a.w3 = w3; a.w4 = w4; a.w5 = w5;
  a.h1 = h1; a.cin = cin; a.h2 = h2; a.h3 = h3; a.o = o; a.density = density; a.rgb = rgb;
  a.M = M; a.K0 = K0; a.S = S;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(M, 128), sms);
  cudaStream_t st = as_stream(stream);
  if (K0 <= 64) {
    const size_t smem = fused_smem_bytes(sigma_smem_floats(64));
    cudaFuncSetAttribute(decoder_fwd_fused_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    decoder_fwd_fused_kernel<64><<<grid, 256, smem, st>>>(a);
  } else {
    const size_t smem = fused_smem_bytes(sigma_smem_floats(128));
    cudaFuncSetAttribute(decoder_fwd_fused_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    decoder_fwd_fused_kernel<128><<<grid, 256, smem, st>>>(a);
  }
  KP_LAUNCH_CHECK("decoder_fwd_fused");
  return 0;
}

// Internal (called by kp_color_net_fwd in mlp.cu when the hidden width is 64): the colour net forward in one launch.
int kp_color_fwd_fused_launch(const float* directions, int S, const float* o, int ldo, const float* w3, const float* w4,
                              const float* w5, int64_t M, float* cin, float* h2, float* h3, float* rgb, cudaStream_t st) {
  ColorArgs a;
  a.o = o; a.dirs = directions; a.w3 = w3; a.w4 = w4; a.w5 = w5; a.cin = cin; a.h2 = h2; a.h3 = h3; a.rgb = rgb;
  a.M = M; a.ldo = ldo; a.S = S;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(M, 128), sms);
  const size_t smem = fused_smem_bytes(0);
  cudaFuncSetAttribute(color_fwd_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  color_fwd_fused_kernel<<<grid, 256, smem, st>>>(a);
  kp::g_launches += 1;
  return 0;
}
