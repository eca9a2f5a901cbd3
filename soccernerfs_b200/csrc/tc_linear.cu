// Dense layers of the decoders on the 5th-generation tensor cores (tcgen05 + TMEM), fp32-accurate via a TF32 split.
//
//   forward        Y[M,N]   = act( X[M,K] W[N,K]^T )
//   backward data  dX[M,K]  = ( dY[M,N] W[N,K] ) * (aux > 0)
//   backward wgt   dW[N,K] += dY[M,N]^T X[M,K]
//
// all fp32 row-major, bias-free (tcnn FullyFusedMLP semantics, NS/fields/kplanes_field.py:249-273).  The decoders'
// parity bar is 1e-4 relative in fp32, which a single TF32 pass (10-bit mantissa) cannot meet, so each operand is
// split x = hi + lo (activations: hi = x with the 13 low mantissa bits cleared -- what kind::tf32 reads of an fp32 word
// anyway -- and lo = x - hi exactly; weights: hi = cvt.rna.tf32(x)) and the partial products are accumulated in the fp32
// TMEM accumulator: all four (lo*lo + lo*hi + hi*lo + hi*hi) in the forward, where a pre-activation rounded across zero
// would flip a ReLU and with it a sample's whole gradient; three (lo*lo dropped, 2^-22 relative) in the backward products,
// which feed no branch.  The only other loss is the tensor core's truncation of lo (<= 2^-21 relative): fp32-class.
// The kernels the layers run on are the warp-specialised, TMA-fed pipelines of tc_ws.cuh (tc_ws_gemm_kernel,
// tc_ws_wgrad_kernel below); tc_rowtile_kernel is the single-stage kernel kept for layers wider than those take.
//
// Shared-memory operand tiles: a [ROWS x COLS] fp32 tile is stored as COLS/32 blocks of [ROWS x 32]; each block is
// ROWS/8 atoms of 8 rows x 128 bytes with the 128-byte swizzle (16-byte chunk c of row r at chunk c ^ (r & 7)).
// Two UMMA views of such a tile are used, so no transposed copy of any operand is ever made:
//   K-major  view (SWIZZLE_128B):          MN = tile rows, K = tile cols  (forward A = X tile, B = W)
//   MN-major view (SWIZZLE_128B_BASE32B):  MN = tile cols, K = tile rows  (backward-data B = W "transposed";
//                  weight-gradient A = X tile, B = dY tile with K = the 128 samples of the tile)
// For 32-bit operands the tensor core only accepts the 32-byte-base swizzle in the MN-major view (atoms of 4 rows x
// 128 bytes, 32-byte chunk q of row r at chunk q ^ (r & 3)), so a tile is staged in the swizzle of the view it is
// consumed in.
#include <string.h>

#include "tc_common.cuh"
#include "tc_ws.cuh"

namespace kp {

// ---------------------------------------------------------------------------------------------------------------
// Row-tile GEMM:  OUT[128 rows, N] = A[128, R] * B      (R = reduction depth, padded to 32; N padded to 32 for MN-B)
//   B_MN == 0 (forward):        B = W [N x R]  K-major            ; epilogue act
//   B_MN == 1 (backward data):  B = W [R x N]  MN-major view      ; epilogue (aux > 0) mask
// ---------------------------------------------------------------------------------------------------------------
template <int B_MN, int R_pad>
__global__ void __launch_bounds__(256) tc_rowtile_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ W,
                                                         int64_t ldw, float* __restrict__ OUT, int64_t ldo, int64_t M, int N,
                                                         int N_pad, int R, int act, const float* __restrict__ aux,
                                                         int64_t ldaux, int beta) {
  extern __shared__ uint8_t smem_raw[];
  const int b_rows = B_MN ? R_pad : N_pad, b_cols = B_MN ? N_pad : R_pad;
  float* a_hi = align1024(smem_raw);
  float* a_lo = a_hi + 128 * R_pad;
  float* b_hi = a_lo + 128 * R_pad;
  float* b_lo = b_hi + b_rows * b_cols;
  __shared__ __align__(8) uint64_t mma_bar;
  __shared__ uint32_t tmem_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mma_bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  tmem_alloc(&tmem_slot, warp);
  // weights are staged ONCE per (persistent) CTA
  if (B_MN) stage_tile<1>(W, ldw, b_rows, R, N, b_cols, b_hi, b_lo);
  else stage_tile<0>(W, ldw, b_rows, N, R, b_cols, b_hi, b_lo);
  const uint32_t idesc = umma_idesc_tf32(128, N_pad, 0, B_MN);
  const int quad = warp & 3, half = warp >> 2;
  const int row = quad * 32 + lane;
  const int64_t n_tiles = (M + 127) / 128;
  uint32_t parity = 0;
  TileRegs<R_pad> pre;
  if ((int64_t)blockIdx.x < n_tiles)
    tile_load<R_pad>(pre, A + (int64_t)blockIdx.x * 128 * lda, lda, (int)min((int64_t)128, M - (int64_t)blockIdx.x * 128), R);
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t row0 = tile * 128;
    const int rows_valid = (int)min((int64_t)128, M - row0);
    tile_store<0, R_pad>(pre, a_hi, a_lo);
    publish_smem_and_sync();
    {  // issue the next tile's global loads now; they complete while the MMAs and the epilogue below run
      const int64_t nxt = tile + gridDim.x;
      if (nxt < n_tiles) tile_load<R_pad>(pre, A + nxt * 128 * lda, lda, (int)min((int64_t)128, M - nxt * 128), R);
    }
    const uint32_t tmem_d = tmem_slot;
    if (threadIdx.x == 0) {
      // One thread issues every MMA: keep its instruction stream short -- base descriptors once, then only the
      // 14-bit start-address field advances by compile-time constants (fully unrolled).
      const uint64_t a_d[2] = {desc_kmajor(smem_u32(a_hi), 128, 0, 0), desc_kmajor(smem_u32(a_lo), 128, 0, 0)};
      const uint64_t b_d[2] = {B_MN ? desc_mnmajor(smem_u32(b_hi), b_rows, 0) : desc_kmajor(smem_u32(b_hi), b_rows, 0, 0),
                               B_MN ? desc_mnmajor(smem_u32(b_lo), b_rows, 0) : desc_kmajor(smem_u32(b_lo), b_rows, 0, 0)};
      const uint32_t b_blk = (uint32_t)(b_rows * 128) >> 4;  // K-major B: 16-byte units between 32-col blocks
#pragma unroll
      for (int t = 0; t < 4; ++t) {  // lo*lo + lo*hi + hi*lo + hi*hi (small terms first)
        const uint64_t ad0 = a_d[t <= 1], bd0 = b_d[t == 0 || t == 2];
#pragma unroll
        for (int k8 = 0; k8 < R_pad / 8; ++k8) {
          const uint32_t a_off = (uint32_t)(((k8 >> 2) * 128 * 128 + (k8 & 3) * 32) >> 4);
          const uint32_t b_off = B_MN ? (uint32_t)((k8 * 1024) >> 4) : (uint32_t)(k8 >> 2) * b_blk + (uint32_t)(((k8 & 3) * 32) >> 4);
          umma_tf32(tmem_d, ad0 + a_off, bd0 + b_off, idesc, (t | k8) != 0);
        }
      }
      umma_commit(&mma_bar);
    }
    mbar_wait(&mma_bar, parity);
    parity ^= 1;
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // epilogue: warps w and w+4 share TMEM lane quadrant (w & 3) and split the columns
    const uint32_t taddr = tmem_d + ((uint32_t)(quad * 32) << 16);
    for (int c0 = half * 16; c0 < N_pad; c0 += 32) {
      uint32_t v[16];
      tmem_ld16(taddr + (uint32_t)c0, v);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      if (row < rows_valid && c0 < N) {
        float* dst = OUT + (row0 + row) * ldo + c0;
        const float* ax = aux ? aux + (row0 + row) * ldaux + c0 : nullptr;
        float x[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          x[j] = __uint_as_float(v[j]);
          // beta: OUT already holds the partial product of an earlier K slice (reduction depths > 128 are split over
          // launches; the activation is applied by the launch that adds the last slice)
          if (beta && c0 + j < N) x[j] += dst[j];
          if (!B_MN) {
            if (act == ACT_RELU) x[j] = fmaxf(x[j], 0.f);
            else if (act == ACT_SIGMOID) x[j] = 1.f / (1.f + expf(-x[j]));
          }
        }
        const bool full = (c0 + 16 <= N) && ((ldo & 3) == 0) && ((reinterpret_cast<uintptr_t>(OUT) & 15) == 0);
        if (full && (ax == nullptr || ((ldaux & 3) == 0 && (reinterpret_cast<uintptr_t>(aux) & 15) == 0))) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            float4 o4 = make_float4(x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]);
            if (B_MN && ax != nullptr) {
              const float4 m4 = __ldg(reinterpret_cast<const float4*>(ax + 4 * q));
              if (!(m4.x > 0.f)) o4.x = 0.f;
              if (!(m4.y > 0.f)) o4.y = 0.f;
              if (!(m4.z > 0.f)) o4.z = 0.f;
              if (!(m4.w > 0.f)) o4.w = 0.f;
            }
            *reinterpret_cast<float4*>(dst + 4 * q) = o4;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            if (c0 + j < N) {
              float o1 = x[j];
              if (B_MN && ax != nullptr && !(ax[j] > 0.f)) o1 = 0.f;
              dst[j] = o1;
            }
          }
        }
      }
    }
    // all TMEM reads of this tile done before the next tile's MMAs overwrite the accumulator
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  }
  tmem_free(tmem_slot, warp);
}

// ---------------------------------------------------------------------------------------------------------------
// Arguments of the row-tile GEMM pipelines:  OUT[128 rows, N] = epilogue(A[128, R] * B), R = n_slices slices of KS columns,
// output columns cut into grid.y slices of N_slice <= 128 (rows n0.. of W for the forward, columns k0.. of W for the
// backward-data product, which reads the same row-major W through an MN-major view).
// ---------------------------------------------------------------------------------------------------------------
struct PipeArgs {
  const float* A; int64_t lda;      // [M, R]
  const float* W; int64_t ldw;      // forward: [N_total, R]; backward data: [R, N_total]
  float* OUT; int64_t ldo;          // [M, N_total]
  const float* aux; int64_t ldaux;  // backward data: ReLU mask source [M, N_total] or NULL
  int64_t M;
  int N_total, N_slice, N_pad;      // output columns: total, per blockIdx.y slice, padded slice width (32 | 64 | 128)
  int R, n_slices;                  // reduction depth and its number of KS-column slices
  int act, beta;
};

__device__ __forceinline__ void tmem_alloc_cols(uint32_t* slot, int warp, uint32_t ncols) {
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
}
__device__ __forceinline__ void tmem_free_cols(uint32_t taddr, int warp, uint32_t ncols) {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols));
}

// ---------------------------------------------------------------------------------------------------------------
// Warp-specialised row-tile GEMM (tc_ws.cuh): same operands, layouts and epilogues as tc_rowtile_kernel, but loading,
// MMA issue and unloading run on their own warps and meet only at mbarriers:
//   full[st]  : 256 producer arrivals   -> the MMA warp may read stage st
//   empty[st] : tcgen05.commit          -> the producers may overwrite stage st
//   accf[a]   : tcgen05.commit          -> the epilogue warps may unload accumulator a
//   acce[a]   : 4 epilogue-warp arrivals -> the MMA warp may overwrite accumulator a
// ---------------------------------------------------------------------------------------------------------------
template <int B_MN, int KS, int ACT, bool MASK, bool TMA>
__global__ void __launch_bounds__(TMA ? kTmaThreads : kWsThreads, 1)
    tc_ws_gemm_kernel(const __grid_constant__ PipeArgs P, const __grid_constant__ CUtensorMap tmA, int n_stages) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int kProdWarp0 = TMA ? kWsEpiWarps + 2 : kWsEpiWarps + 1;
  const int R_tot = P.n_slices * KS;
  const int b_rows = B_MN ? R_tot : P.N_pad, b_cols = B_MN ? P.N_pad : R_tot;
  float* b_hi = align1024(smem_raw);
  float* b_lo = b_hi + b_rows * b_cols;
  float* a_st = b_lo + b_rows * b_cols;  // [n_stages][hi | lo][128 x KS]
  __shared__ __align__(8) uint64_t full[kWsMaxStages], empty[kWsMaxStages], tfull[kWsMaxStages], accf[2], acce[2];
  __shared__ uint32_t tmem_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col0 = blockIdx.y * P.N_slice;
  const int N = min(P.N_slice, P.N_total - col0);
  const uint32_t tmem_cols = P.N_pad <= 32 ? 64u : (P.N_pad <= 64 ? 128u : 256u);
  if (threadIdx.x == 0) {
    for (int i = 0; i < n_stages; ++i) {
      mbar_init(&full[i], kWsProdThreads);
      mbar_init(&empty[i], 1);
      mbar_init(&tfull[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&accf[i], 1);
      mbar_init(&acce[i], kWsEpiWarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  tmem_alloc_cols(&tmem_slot, warp, tmem_cols);
  // weights of this column slice, once per CTA (all warps)
  if (B_MN) stage_tile<1>(P.W + col0, P.ldw, b_rows, P.R, N, b_cols, b_hi, b_lo);
  else stage_tile<0>(P.W + (int64_t)col0 * P.ldw, P.ldw, b_rows, N, P.R, b_cols, b_hi, b_lo);
  publish_smem_and_sync();
  const int64_t n_tiles = (P.M + 127) / 128;
  const int my_tiles = (int64_t)blockIdx.x < n_tiles ? (int)((n_tiles - 1 - blockIdx.x) / gridDim.x + 1) : 0;
  const int ns = P.n_slices;
  const uint32_t tmem_base = tmem_slot;

  if (TMA && warp >= kProdWarp0) {
    // ------------------------------------------------ producers (TMA-fed): derive lo from the landed hi tile ----
    const int pt = threadIdx.x - 32 * kProdWarp0;
    const int n_steps = my_tiles * ns;
    int st = 0;
    uint32_t use = 0;
    for (int s = 0; s < n_steps; ++s) {
      mbar_wait_spin(&tfull[st], use & 1);  // the TMA boxes of this step have landed (async-proxy writes visible)
      float* a_hi = a_st + st * (2 * 128 * KS);
      ws_derive_lo<128 * KS / 4>(a_hi, a_hi + 128 * KS, pt);
      fence_async_smem();
      mbar_arrive(&full[st]);
      if (++st == n_stages) { st = 0; ++use; }
    }
  } else if (TMA && warp == kTmaWarp) {
    // ------------------------------------------------ TMA issuer -----------------------------------------------
    if (lane == 0) {
      tma_prefetch_desc(&tmA);
      int st = 0;
      uint32_t use = 0;
      for (int jl = 0; jl < my_tiles; ++jl) {
        const int64_t tile = blockIdx.x + (int64_t)jl * gridDim.x;
        for (int kc = 0; kc < ns; ++kc) {
          if (use > 0) mbar_wait_spin(&empty[st], (use - 1) & 1);  // the MMAs that read this stage have completed
          float* a_hi = a_st + st * (2 * 128 * KS);
          mbar_expect_tx(&tfull[st], 128 * KS * 4);
#pragma unroll
          for (int kb = 0; kb < KS / 32; ++kb)
            tma_load_2d(a_hi + kb * (128 * 32), &tmA, kc * KS + kb * 32, (int)(tile * 128), &tfull[st]);
          if (++st == n_stages) { st = 0; ++use; }
        }
      }
    }
  } else if (!TMA && warp >= kProdWarp0) {
    // ------------------------------------------------ producers (register-fed) ---------------------------------
    const int pt = threadIdx.x - 32 * kProdWarp0;
    const int off0 = ws_store_offset<128, KS, 0>(pt);
    const bool a_vec = ((P.lda & 3) == 0) && ((reinterpret_cast<uintptr_t>(P.A) & 15) == 0);
    const int n_steps = my_tiles * ns;
    int ljl = 0, lkc = 0;  // (tile, K slice) of the next load
    auto issue_load = [&](WsRegs<128, KS>& t) {
      const int64_t tile = blockIdx.x + (int64_t)ljl * gridDim.x;
      const int rows_valid = (int)min((int64_t)128, P.M - tile * 128);
      const int cols_valid = P.R - lkc * KS;
      const float* src = P.A + tile * 128 * P.lda + lkc * KS;
      if (a_vec && rows_valid == 128 && cols_valid >= KS) ws_load<128, KS, true>(t, src, P.lda, pt, 128, KS);
      else ws_load<128, KS, false>(t, src, P.lda, pt, rows_valid, cols_valid);
      if (++lkc == ns) { lkc = 0; ++ljl; }
    };
    int st = 0;
    uint32_t use = 0;
    // register ring of D steps: D x (128 x KS x 4 bytes) of loads in flight per CTA, so the global-memory latency is
    // spread over D steps of conversion work instead of being paid once per step
    constexpr int D = KS == 32 ? 4 : 2;
    WsRegs<128, KS> ring[D];
#pragma unroll
    for (int d = 0; d < D; ++d)
      if (d < n_steps) issue_load(ring[d]);
    for (int s = 0; s < n_steps; s += D) {
#pragma unroll
      for (int d = 0; d < D; ++d) {
        if (s + d < n_steps) {
          if (use > 0) mbar_wait_spin(&empty[st], (use - 1) & 1);
          float* a_hi = a_st + st * (2 * 128 * KS);
          ws_store<128, KS>(ring[d], a_hi, a_hi + 128 * KS, off0);
          fence_async_smem();  // generic-proxy stores -> visible to the tensor core's async proxy
          mbar_arrive(&full[st]);
          if (++st == n_stages) { st = 0; ++use; }
          if (s + d + D < n_steps) issue_load(ring[d]);  // refill this slot: step s + d + D
        }
      }
    }
  } else if (warp == kWsEpiWarps) {
    // ------------------------------------------------ MMA issuer -----------------------------------------------
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_tf32(128, P.N_pad, 0, B_MN);
      const uint64_t b_d[2] = {B_MN ? desc_mnmajor(smem_u32(b_hi), b_rows, 0) : desc_kmajor(smem_u32(b_hi), b_rows, 0, 0),
                               B_MN ? desc_mnmajor(smem_u32(b_lo), b_rows, 0) : desc_kmajor(smem_u32(b_lo), b_rows, 0, 0)};
      const uint32_t b_blk = (uint32_t)(b_rows * 128) >> 4;  // K-major B: 16-byte units between 32-col blocks
      int st = 0;
      uint32_t use = 0;
      for (int jl = 0; jl < my_tiles; ++jl) {
        const int acc = jl & 1;
        const uint32_t ua = (uint32_t)jl >> 1;
        if (ua > 0) mbar_wait_spin(&acce[acc], (ua - 1) & 1);  // the epilogue has unloaded this accumulator's previous tile
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * P.N_pad);
        for (int kc = 0; kc < ns; ++kc) {
          mbar_wait_spin(&full[st], use & 1);
          tc_fence_after();
          const uint32_t a_base = smem_u32(a_st + st * (2 * 128 * KS));
          const uint64_t a_d[2] = {desc_kmajor(a_base, 128, 0, 0), desc_kmajor(a_base + 128 * KS * 4, 128, 0, 0)};
          // forward: lo*lo + lo*hi + hi*lo + hi*hi (small terms first): the pre-activations decide ReLU branches, so all
          // four terms are kept.  Backward products (B_MN) feed no branch: the 2^-22-relative lo*lo term is dropped.
          constexpr int T0 = B_MN ? 1 : 0;
#pragma unroll
          for (int t = T0; t < 4; ++t) {
            const uint64_t ad0 = a_d[t <= 1], bd0 = b_d[t == 0 || t == 2];
#pragma unroll
            for (int k8 = 0; k8 < KS / 8; ++k8) {
              const int kk = kc * (KS / 8) + k8;  // K step within the whole reduction
              const uint32_t a_off = (uint32_t)(((k8 >> 2) * 128 * 128 + (k8 & 3) * 32) >> 4);
              const uint32_t b_off = B_MN ? (uint32_t)((kk * 1024) >> 4) : (uint32_t)(kk >> 2) * b_blk + (uint32_t)(((kk & 3) * 32) >> 4);
              umma_tf32(tmem_d, ad0 + a_off, bd0 + b_off, idesc, (kc | (t - T0) | k8) != 0);
            }
          }
          umma_commit(&empty[st]);  // arrives when the MMAs above have read the stage
          if (++st == n_stages) { st = 0; ++use; }
        }
        umma_commit(&accf[acc]);  // ... and when the tile's accumulator is complete
      }
    }
  } else {
    // ------------------------------------------------ epilogue -------------------------------------------------
    const int quad = warp;  // TMEM lane quadrant this warp may access
    const bool o_vec = ((P.ldo & 3) == 0) && (((reinterpret_cast<uintptr_t>(P.OUT) + (size_t)col0 * 4) & 15) == 0);
    const bool m_vec = !MASK || (((P.ldaux & 3) == 0) && (((reinterpret_cast<uintptr_t>(P.aux) + (size_t)col0 * 4) & 15) == 0));
    const bool fastv = o_vec && m_vec;
    float* epi = a_st + (size_t)n_stages * (2 * 128 * KS) + quad * (32 * 36);  // this warp's transpose buffer
    for (int jl = 0; jl < my_tiles; ++jl) {
      const int acc = jl & 1;
      const uint32_t ua = (uint32_t)jl >> 1;
      const int64_t tile = blockIdx.x + (int64_t)jl * gridDim.x;
      const int64_t row0 = tile * 128;
      const int rows_valid = (int)min((int64_t)128, P.M - row0);
      mbar_wait_sleep(&accf[acc], ua & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)(acc * P.N_pad) + ((uint32_t)(quad * 32) << 16);
      // Accumulator rows arrive one per lane (tcgen05.ld 32x32b).  Storing them like that would touch 32 different 128-byte
      // lines per STG (ncu: the epilogue's uncoalesced LDG/STG kept l1tex at 58 % and bounded the kernel), so each 32 x 32
      // block goes through a padded shared-memory transpose: afterwards a lane owns 16 bytes of a row and a warp-wide
      // LDG / STG covers 4 rows x 128 contiguous bytes.
      const int rows_w = min(32, rows_valid - quad * 32);  // valid rows among this warp's 32 (may be <= 0)
      const int rr = lane >> 3, cc = (lane & 7) * 4;
      float* out_w = P.OUT + (row0 + quad * 32) * P.ldo + col0;
      const float* aux_w = MASK ? P.aux + (row0 + quad * 32) * P.ldaux + col0 : nullptr;
      for (int c0 = 0; c0 < N; c0 += 32) {
        const int c = c0 + cc;
        const bool vec = fastv && (c + 4 <= N);
        float4 m4[8];
        if (MASK && vec) {
#pragma unroll
          for (int it = 0; it < 8; ++it)
            if (it * 4 + rr < rows_w) m4[it] = __ldg(reinterpret_cast<const float4*>(aux_w + (int64_t)(it * 4 + rr) * P.ldaux + c));
        }
        uint32_t v[32];
        tmem_ld16(taddr + (uint32_t)c0, v);
        tmem_ld16(taddr + (uint32_t)c0 + 16u, v + 16);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int q = 0; q < 8; ++q)
          *reinterpret_cast<float4*>(epi + lane * 36 + 4 * q) =
              make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int r = it * 4 + rr;
          if (r < rows_w && c < N) {
            float4 x = *reinterpret_cast<const float4*>(epi + r * 36 + cc);
            if (ACT == ACT_RELU) {
              x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f);
            } else if (ACT == ACT_SIGMOID) {
              x.x = 1.f / (1.f + expf(-x.x)); x.y = 1.f / (1.f + expf(-x.y)); x.z = 1.f / (1.f + expf(-x.z)); x.w = 1.f / (1.f + expf(-x.w));
            }
            float* dst = out_w + (int64_t)r * P.ldo + c;
            if (vec) {
              if (MASK) {
                if (!(m4[it].x > 0.f)) x.x = 0.f;
                if (!(m4[it].y > 0.f)) x.y = 0.f;
                if (!(m4[it].z > 0.f)) x.z = 0.f;
                if (!(m4[it].w > 0.f)) x.w = 0.f;
              }
              *reinterpret_cast<float4*>(dst) = x;
            } else {
              const float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                if (c + j < N) {
                  float o1 = xs[j];
                  if (MASK && !(aux_w[(int64_t)r * P.ldaux + c + j] > 0.f)) o1 = 0.f;
                  dst[j] = o1;
                }
              }
            }
          }
        }
        __syncwarp();
      }
      tc_fence_before();  // this warp's TMEM reads are ordered before the arrival the MMA warp waits on
      __syncwarp();
      if (lane == 0) mbar_arrive(&acce[acc]);
    }
  }
  tmem_free_cols(tmem_base, warp, tmem_cols);
}

// ---------------------------------------------------------------------------------------------------------------
// Warp-specialised weight gradient:  D[k, n] += sum_s X[s, k] * dY[s, n]  (D = dW^T) over this CTA's sub-tiles of ROWS
// samples.  Both operands are activations, so both are staged per step (MN-major views, K = the ROWS samples) by the
// producer warps into an n_stages ring; the MMA warp accumulates every step into ONE TMEM accumulator; after the last
// step the epilogue warps add D into dW with one red per weight.
// ---------------------------------------------------------------------------------------------------------------
template <int K_PAD, int N_PAD, int ROWS, bool TMA>
__global__ void __launch_bounds__(TMA ? kTmaThreads : kWsThreads, 1)
    tc_ws_wgrad_kernel(const float* __restrict__ X, int64_t ldx, const float* __restrict__ dY, int64_t lddy, float* __restrict__ dW,
                       int64_t lddw, int64_t M, int K_in, int N_out, int n_stages, const __grid_constant__ CUtensorMap tmX,
                       const __grid_constant__ CUtensorMap tmY) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int STAGE = 2 * ROWS * (K_PAD + N_PAD);  // floats: [x_hi | x_lo | y_hi | y_lo]
  constexpr int kProdWarp0 = TMA ? kWsEpiWarps + 2 : kWsEpiWarps + 1;
  float* st_base = align1024(smem_raw);
  __shared__ __align__(8) uint64_t full[kWsMaxStages], empty[kWsMaxStages], tfull[kWsMaxStages], done;
  __shared__ uint32_t tmem_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr uint32_t tmem_cols = N_PAD <= 32 ? 32u : (N_PAD <= 64 ? 64u : 128u);
  if (threadIdx.x == 0) {
    for (int i = 0; i < n_stages; ++i) {
      mbar_init(&full[i], kWsProdThreads);
      mbar_init(&empty[i], 1);
      mbar_init(&tfull[i], 1);
    }
    mbar_init(&done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  tmem_alloc_cols(&tmem_slot, warp, tmem_cols);
  publish_smem_and_sync();
  const uint32_t tmem_d = tmem_slot;
  const int64_t n_sub = (M + ROWS - 1) / ROWS;
  const int my_steps = (int64_t)blockIdx.x < n_sub ? (int)((n_sub - 1 - blockIdx.x) / gridDim.x + 1) : 0;

  if (TMA && warp >= kProdWarp0) {
    // producers (TMA-fed): derive both lo operands from the landed hi tiles
    const int pt = threadIdx.x - 32 * kProdWarp0;
    int st = 0;
    uint32_t use = 0;
    for (int s = 0; s < my_steps; ++s) {
      mbar_wait_spin(&tfull[st], use & 1);
      float* b = st_base + (size_t)st * STAGE;
      ws_derive_lo<ROWS * K_PAD / 4>(b, b + ROWS * K_PAD, pt);
      ws_derive_lo<ROWS * N_PAD / 4>(b + 2 * ROWS * K_PAD, b + 2 * ROWS * K_PAD + ROWS * N_PAD, pt);
      fence_async_smem();
      mbar_arrive(&full[st]);
      if (++st == n_stages) { st = 0; ++use; }
    }
  } else if (TMA && warp == kTmaWarp) {
    if (lane == 0) {
      tma_prefetch_desc(&tmX);
      tma_prefetch_desc(&tmY);
      int st = 0;
      uint32_t use = 0;
      for (int s = 0; s < my_steps; ++s) {
        const int64_t sub = blockIdx.x + (int64_t)s * gridDim.x;
        if (use > 0) mbar_wait_spin(&empty[st], (use - 1) & 1);
        float* b = st_base + (size_t)st * STAGE;
        mbar_expect_tx(&tfull[st], ROWS * (K_PAD + N_PAD) * 4);
#pragma unroll
        for (int kb = 0; kb < K_PAD / 32; ++kb) tma_load_2d(b + kb * (ROWS * 32), &tmX, kb * 32, (int)(sub * ROWS), &tfull[st]);
#pragma unroll
        for (int kb = 0; kb < N_PAD / 32; ++kb)
          tma_load_2d(b + 2 * ROWS * K_PAD + kb * (ROWS * 32), &tmY, kb * 32, (int)(sub * ROWS), &tfull[st]);
        if (++st == n_stages) { st = 0; ++use; }
      }
    }
  } else if (!TMA && warp >= kProdWarp0) {
    const int pt = threadIdx.x - 32 * kProdWarp0;
    const int offx = ws_store_offset<ROWS, K_PAD, 1>(pt), offy = ws_store_offset<ROWS, N_PAD, 1>(pt);
    const bool x_vec = ((ldx & 3) == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0) && K_in >= K_PAD;
    const bool y_vec = ((lddy & 3) == 0) && ((reinterpret_cast<uintptr_t>(dY) & 15) == 0) && N_out >= N_PAD;
    int lstep = 0;
    auto issue_load = [&](WsRegs<ROWS, K_PAD>& tx, WsRegs<ROWS, N_PAD>& ty) {
      const int64_t sub = blockIdx.x + (int64_t)lstep * gridDim.x;
      const int rv = (int)min((int64_t)ROWS, M - sub * ROWS);
      if (x_vec && rv == ROWS) ws_load<ROWS, K_PAD, true>(tx, X + sub * ROWS * ldx, ldx, pt, ROWS, K_PAD);
      else ws_load<ROWS, K_PAD, false>(tx, X + sub * ROWS * ldx, ldx, pt, rv, K_in);
      if (y_vec && rv == ROWS) ws_load<ROWS, N_PAD, true>(ty, dY + sub * ROWS * lddy, lddy, pt, ROWS, N_PAD);
      else ws_load<ROWS, N_PAD, false>(ty, dY + sub * ROWS * lddy, lddy, pt, rv, N_out);
      ++lstep;
    };
    int st = 0;
    uint32_t use = 0;
    constexpr int D = 2;  // register ring: two steps of loads in flight
    WsRegs<ROWS, K_PAD> rx[D];
    WsRegs<ROWS, N_PAD> ry[D];
#pragma unroll
    for (int d = 0; d < D; ++d)
      if (d < my_steps) issue_load(rx[d], ry[d]);
    for (int s = 0; s < my_steps; s += D) {
#pragma unroll
      for (int d = 0; d < D; ++d) {
        if (s + d < my_steps) {
          if (use > 0) mbar_wait_spin(&empty[st], (use - 1) & 1);
          float* b = st_base + (size_t)st * STAGE;
          ws_store<ROWS, K_PAD>(rx[d], b, b + ROWS * K_PAD, offx);
          ws_store<ROWS, N_PAD>(ry[d], b + 2 * ROWS * K_PAD, b + 2 * ROWS * K_PAD + ROWS * N_PAD, offy);
          fence_async_smem();
          mbar_arrive(&full[st]);
          if (++st == n_stages) { st = 0; ++use; }
          if (s + d + D < my_steps) issue_load(rx[d], ry[d]);
        }
      }
    }
  } else if (warp == kWsEpiWarps) {
    if (lane == 0) {
      // M = 128 rows of D; when K_PAD < 128 the MN blocks beyond the X tile read whatever follows in shared memory
      // (the allocation keeps ROWS x 128 floats of slack): those D rows (k >= K_in) are never read back.
      const uint32_t idesc = umma_idesc_tf32(128, N_PAD, 1, 1);
      int st = 0;
      uint32_t use = 0;
      for (int s = 0; s < my_steps; ++s) {
        mbar_wait_spin(&full[st], use & 1);
        tc_fence_after();
        const uint32_t b = smem_u32(st_base + (size_t)st * STAGE);
        const uint64_t a_d[2] = {desc_mnmajor(b, ROWS, 0), desc_mnmajor(b + ROWS * K_PAD * 4, ROWS, 0)};
        const uint64_t b_d[2] = {desc_mnmajor(b + 2 * ROWS * K_PAD * 4, ROWS, 0),
                                 desc_mnmajor(b + (2 * ROWS * K_PAD + ROWS * N_PAD) * 4, ROWS, 0)};
#pragma unroll
        for (int t = 1; t < 4; ++t) {  // lo*hi + hi*lo + hi*hi (lo*lo, 2^-22 relative, dropped: the sum feeds no branch)
          const uint64_t ad0 = a_d[t <= 1], bd0 = b_d[t == 0 || t == 2];
#pragma unroll
          for (int r8 = 0; r8 < ROWS / 8; ++r8)  // K-steps of 8 samples (1024 bytes each)
            umma_tf32(tmem_d, ad0 + (uint32_t)(r8 * 64), bd0 + (uint32_t)(r8 * 64), idesc, (uint32_t)((s | (t - 1) | r8) != 0));
        }
        umma_commit(&empty[st]);
        if (++st == n_stages) { st = 0; ++use; }
      }
      umma_commit(&done);
    }
  } else if (my_steps > 0) {
    mbar_wait_sleep(&done, 0);
    tc_fence_after();
    const int quad = warp;
    const int k = quad * 32 + lane;  // D row = input feature index
    const uint32_t taddr = tmem_d + ((uint32_t)(quad * 32) << 16);
    for (int c0 = 0; c0 < N_PAD; c0 += 16) {
      if (c0 >= N_out) break;
      uint32_t v[16];
      tmem_ld16(taddr + (uint32_t)c0, v);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      if (k < K_in) {
#pragma unroll
        for (int j = 0; j < 16; ++j)
          if (c0 + j < N_out) red_add_f32(dW + (int64_t)(c0 + j) * lddw + k, __uint_as_float(v[j]));
      }
    }
  }
  tmem_free_cols(tmem_d, warp, tmem_cols);
}

static int pad_dim(int x) { return x <= 32 ? 32 : (x <= 64 ? 64 : 128); }  // operand tile widths: 32 | 64 | 128

template <typename Kern>
static unsigned persistent_grid(Kern kern, int64_t n_tiles, size_t smem) {
  int dev = 0, sms = 148, per_sm = 1;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  // CTAs per SM from the kernel's own resources.  (cudaOccupancyMaxActiveBlocksPerMultiprocessor answers 1 for these
  // kernels whatever their footprint -- measured on B200, driver 580 -- so it is not used.)
  cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, kern) == cudaSuccess) {
    int smem_sm = 0;
    cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
    const int regs_cta = ((fa.numRegs + 7) / 8 * 8) * 256;
    const size_t smem_cta = smem + fa.sharedSizeBytes + 1024;  // + the per-CTA reservation
    per_sm = std::min<int>(65536 / std::max(1, regs_cta), (int)((size_t)smem_sm / smem_cta));
  }
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 4) per_sm = 4;  // 4 x 128 TMEM columns
  return (unsigned)std::min<int64_t>(n_tiles, (int64_t)sms * per_sm);
}

template <int B_MN, int R_PAD>
static void launch_rowtile(const float* A, int64_t lda, const float* W, int64_t ldw, float* OUT, int64_t ldo, int64_t M, int N,
                           int N_pad, int R, int act, const float* aux, int64_t ldaux, int beta, cudaStream_t st) {
  const size_t smem = (size_t)(2 * 128 * R_PAD + 2 * N_pad * R_PAD) * sizeof(float) + 1024;
  auto kern = tc_rowtile_kernel<B_MN, R_PAD>;
  kern<<<persistent_grid(kern, ceil_div(M, 128), smem), 256, smem, st>>>(A, lda, W, ldw, OUT, ldo, M, N, N_pad, R, act, aux, ldaux,
                                                                         beta);
  kp::g_launches += 1;
}
template <int B_MN>
static void dispatch_rowtile(int R_pad, const float* A, int64_t lda, const float* W, int64_t ldw, float* OUT, int64_t ldo,
                             int64_t M, int N, int N_pad, int R, int act, const float* aux, int64_t ldaux, int beta,
                             cudaStream_t st) {
  if (R_pad == 32) launch_rowtile<B_MN, 32>(A, lda, W, ldw, OUT, ldo, M, N, N_pad, R, act, aux, ldaux, beta, st);
  else if (R_pad == 64) launch_rowtile<B_MN, 64>(A, lda, W, ldw, OUT, ldo, M, N, N_pad, R, act, aux, ldaux, beta, st);
  else launch_rowtile<B_MN, 128>(A, lda, W, ldw, OUT, ldo, M, N, N_pad, R, act, aux, ldaux, beta, st);
}

// One tc_ws_gemm_kernel launch: OUT[M, N_total] = epilogue(A[M, R] * B) with the output columns cut into grid.y slices.
// Returns false when the shape does not fit.
template <int B_MN, int KS, int ACT, bool MASK>
static void launch_ws_inst(const PipeArgs& P, const CUtensorMap* tm, int n_stages, dim3 grid, size_t smem, cudaStream_t st) {
  if (tm != nullptr) {
    auto kern = tc_ws_gemm_kernel<B_MN, KS, ACT, MASK, true>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<grid, kTmaThreads, smem, st>>>(P, *tm, n_stages);
  } else {
    auto kern = tc_ws_gemm_kernel<B_MN, KS, ACT, MASK, false>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    CUtensorMap dummy;
    memset(&dummy, 0, sizeof(dummy));
    kern<<<grid, kWsThreads, smem, st>>>(P, dummy, n_stages);
  }
}
template <int B_MN>
static bool launch_ws(const float* A, int64_t lda, const float* W, int64_t ldw, float* OUT, int64_t ldo, int64_t M, int N_total,
                      int R, int act, const float* aux, int64_t ldaux, cudaStream_t st) {
  const size_t epi_bytes = (size_t)kWsEpiWarps * 32 * 36 * sizeof(float);  // the epilogue warps' transpose buffers
  const size_t budget = 227 * 1024 - 2048 - epi_bytes;  // - 1 KB alignment slack - static shared memory (barriers)
  int KS = 0, n_slices = 0, N_slice = 0, N_pad = 0, n_stages = 0;
  // widest column slice, then the K-slice width that gives the deeper ring (>= 2 stages needed)
  for (int cand = std::min(N_total, 128);; cand = (cand > 64 ? 64 : 32)) {
    const int np = pad_dim(cand);
    for (int ks : {64, 32}) {
      if (ks == 64 && R <= 32) continue;
      const int nsl = (int)ceil_div(R, ks);
      const size_t b_bytes = (size_t)2 * np * nsl * ks * sizeof(float);
      const size_t stage = (size_t)2 * 128 * ks * sizeof(float);
      if (b_bytes + 2 * stage > budget) continue;
      const int stages = (int)std::min<size_t>(kWsMaxStages, (budget - b_bytes) / stage);
      if (KS == 0 || (ks == 32 && n_stages < 3 && stages > n_stages)) { KS = ks; n_slices = nsl; N_slice = cand; N_pad = np; n_stages = stages; }
    }
    if (KS != 0 || cand <= 32) break;
  }
  if (KS == 0) return false;
  PipeArgs P;
  P.A = A; P.lda = lda; P.W = W; P.ldw = ldw; P.OUT = OUT; P.ldo = ldo; P.aux = aux; P.ldaux = ldaux; P.M = M;
  P.N_total = N_total; P.N_slice = N_slice; P.N_pad = N_pad; P.R = R; P.n_slices = n_slices; P.act = act; P.beta = 0;
  const size_t smem = (size_t)2 * N_pad * n_slices * KS * sizeof(float) + (size_t)n_stages * 2 * 128 * KS * sizeof(float) + epi_bytes + 1024;
  const unsigned gy = (unsigned)ceil_div(N_total, N_slice);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int64_t n_tiles = ceil_div(M, 128);
  const unsigned gx = (unsigned)std::max<int64_t>(1, std::min<int64_t>(n_tiles, (int64_t)sms / gy));
  const dim3 grid(gx, gy);
  const bool mask = aux != nullptr;
  // activation tiles through the TMA engine when the matrix can be described by a tensor map (16-byte aligned rows)
  CUtensorMap tmA;
  const bool use_tma = make_tmap_2d(&tmA, A, M, R, lda, 128, false);
  const CUtensorMap* tm = use_tma ? &tmA : nullptr;
  if (B_MN) {
    if (KS == 64) { if (mask) launch_ws_inst<1, 64, 0, true>(P, tm, n_stages, grid, smem, st); else launch_ws_inst<1, 64, 0, false>(P, tm, n_stages, grid, smem, st); }
    else { if (mask) launch_ws_inst<1, 32, 0, true>(P, tm, n_stages, grid, smem, st); else launch_ws_inst<1, 32, 0, false>(P, tm, n_stages, grid, smem, st); }
  } else {
    if (KS == 64) {
      if (act == ACT_RELU) launch_ws_inst<0, 64, ACT_RELU, false>(P, tm, n_stages, grid, smem, st);
      else if (act == ACT_SIGMOID) launch_ws_inst<0, 64, ACT_SIGMOID, false>(P, tm, n_stages, grid, smem, st);
      else launch_ws_inst<0, 64, ACT_NONE, false>(P, tm, n_stages, grid, smem, st);
    } else {
      if (act == ACT_RELU) launch_ws_inst<0, 32, ACT_RELU, false>(P, tm, n_stages, grid, smem, st);
      else if (act == ACT_SIGMOID) launch_ws_inst<0, 32, ACT_SIGMOID, false>(P, tm, n_stages, grid, smem, st);
      else launch_ws_inst<0, 32, ACT_NONE, false>(P, tm, n_stages, grid, smem, st);
    }
  }
  kp::g_launches += 1;
  return true;
}

template <int K_PAD, int N_PAD>
static bool launch_ws_wgrad(const float* X, int64_t ldx, const float* dY, int64_t lddy, float* dW, int64_t lddw, int64_t M, int K,
                            int N, cudaStream_t st) {
  constexpr int ROWS = 64;
  const size_t stage = (size_t)2 * ROWS * (K_PAD + N_PAD) * sizeof(float);
  const size_t slack = (size_t)ROWS * 128 * sizeof(float);  // the A operand always spans 4 MN blocks (M = 128)
  const size_t budget = 227 * 1024 - 2048 - slack;  // - 1 KB alignment slack - static shared memory (barriers)
  const int n_stages = (int)std::min<size_t>(kWsMaxStages, budget / stage);
  if (n_stages < 2) return false;
  const size_t smem = (size_t)n_stages * stage + slack + 1024;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div(M, ROWS), sms));
  CUtensorMap tmX, tmY;
  const bool use_tma = make_tmap_2d(&tmX, X, M, K, ldx, ROWS, true) && make_tmap_2d(&tmY, dY, M, N, lddy, ROWS, true);
  if (use_tma) {
    auto kern = tc_ws_wgrad_kernel<K_PAD, N_PAD, ROWS, true>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<grid, kTmaThreads, smem, st>>>(X, ldx, dY, lddy, dW, lddw, M, K, N, n_stages, tmX, tmY);
  } else {
    memset(&tmX, 0, sizeof(tmX));
    auto kern = tc_ws_wgrad_kernel<K_PAD, N_PAD, ROWS, false>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<grid, kWsThreads, smem, st>>>(X, ldx, dY, lddy, dW, lddw, M, K, N, n_stages, tmX, tmX);
  }
  return true;
}

template <int K_PAD, int N_PAD>
static void launch_wgrad(const float* X, int64_t ldx, const float* dY, int64_t lddy, float* dW, int64_t lddw, int64_t M, int K,
                         int N, cudaStream_t st) {
  if (!launch_ws_wgrad<K_PAD, N_PAD>(X, ldx, dY, lddy, dW, lddw, M, K, N, st))
    set_error("tc_linear_bwd_weight: operand tiles [%d + %d columns] do not fit the pipeline", K_PAD, N_PAD);
}
template <int K_PAD>
static void dispatch_wgrad(int N_pad, const float* X, int64_t ldx, const float* dY, int64_t lddy, float* dW, int64_t lddw,
                           int64_t M, int K, int N, cudaStream_t st) {
  if (N_pad == 32) launch_wgrad<K_PAD, 32>(X, ldx, dY, lddy, dW, lddw, M, K, N, st);
  else if (N_pad == 64) launch_wgrad<K_PAD, 64>(X, ldx, dY, lddy, dW, lddw, M, K, N, st);
  else launch_wgrad<K_PAD, 128>(X, ldx, dY, lddy, dW, lddw, M, K, N, st);
}

}  // namespace kp

using namespace kp;

// Shapes one launch covers: operand tiles must fit shared memory.
static bool tc_single(int N, int K) { return N >= 1 && N <= 128 && K >= 1 && K <= 128 && pad_dim(N) * pad_dim(K) <= 128 * 64; }

// Which layers the tensor-core path covers.  Layers wider than one launch's operand tiles (the 192 -> 128 first layer
// of the 32x config, NS/configs/method_configs.py:523-524) are cut into slices of <= 64 output / input columns and
// <= 128 reduction columns, each slice one launch on a sub-matrix (pointer offset + leading dimension).
extern "C" int kp_tc_supported(int N, int K) {
  return (N >= 1 && N <= 1024 && K >= 1 && K <= 1024 && (tc_single(N, K) || K <= 32 || K % 4 == 0)) ? 1 : 0;
}

extern "C" int kp_tc_linear_fwd(const float* X, int64_t ldx, const float* W, int64_t ldw, float* Y, int64_t ldy, int64_t M,
                                int N, int K, int act, void* stream) {
  if (M == 0) return 0;
  KP_CHECK(X && W && Y && kp_tc_supported(N, K), "tc_linear_fwd: unsupported shape N=%d K=%d", N, K);
  KP_CHECK(act >= 0 && act <= 2, "tc_linear_fwd: act=%d", act);
  cudaStream_t st = as_stream(stream);
  if (K <= 192 && launch_ws<0>(X, ldx, W, ldw, Y, ldy, M, N, K, act, nullptr, 0, st)) {
    // warp-specialised pipeline: K sliced inside the kernel, output columns over grid.y
  } else if (tc_single(N, K)) {
    dispatch_rowtile<0>(pad_dim(K), X, ldx, W, ldw, Y, ldy, M, N, pad_dim(N), K, act, nullptr, 0, 0, st);
  } else {
    // output columns in slices of 64, reduction in slices of 128: Y[:, n0:n1] = act( sum_k X[:, k0:k1] W[n0:n1, k0:k1]^T ),
    // partial sums kept in Y itself (beta) and the activation applied with the last K slice
    for (int n0 = 0; n0 < N; n0 += 64) {
      const int nn = std::min(64, N - n0);
      for (int k0 = 0; k0 < K; k0 += 128) {
        const int kk = std::min(128, K - k0);
        const bool last = k0 + 128 >= K;
        dispatch_rowtile<0>(pad_dim(kk), X + k0, ldx, W + (int64_t)n0 * ldw + k0, ldw, Y + n0, ldy, M, nn, pad_dim(nn), kk,
                            last ? act : 0, nullptr, 0, k0 > 0 ? 1 : 0, st);
      }
    }
  }
  kp::g_launches -= 1;  // every launch was counted; KP_LAUNCH_CHECK counts one more
  KP_LAUNCH_CHECK("tc_linear_fwd");
  return 0;
}

// dX[M,K] = (dY[M,N] W[N,K]) masked by (aux[M,K] > 0) when aux != NULL.
extern "C" int kp_tc_linear_bwd_data(const float* dY, int64_t lddy, const float* W, int64_t ldw, float* dX, int64_t lddx,
                                     int64_t M, int N, int K, const float* aux, int64_t ldaux, void* stream) {
  if (M == 0) return 0;
  KP_CHECK(dY && W && dX && kp_tc_supported(N, K), "tc_linear_bwd_data: unsupported shape N=%d K=%d", N, K);
  cudaStream_t st = as_stream(stream);
  if (N <= 192 && launch_ws<1>(dY, lddy, W, ldw, dX, lddx, M, K, N, 0, aux, ldaux, st)) {
    // warp-specialised pipeline: reduction over N_out sliced inside the kernel, output (K_in) columns over grid.y
  } else if (tc_single(N, K)) {
    // reduction over N_out (R), output width K_in
    dispatch_rowtile<1>(pad_dim(N), dY, lddy, W, ldw, dX, lddx, M, K, pad_dim(K), N, 0, aux, ldaux, 0, st);
  } else {
    // input columns in slices of 64, reduction (N_out) in slices of 128; the ReLU mask is applied with the last slice
    for (int k0 = 0; k0 < K; k0 += 64) {
      const int kk = std::min(64, K - k0);
      for (int n0 = 0; n0 < N; n0 += 128) {
        const int nn = std::min(128, N - n0);
        const bool last = n0 + 128 >= N;
        dispatch_rowtile<1>(pad_dim(nn), dY + n0, lddy, W + (int64_t)n0 * ldw + k0, ldw, dX + k0, lddx, M, kk, pad_dim(kk), nn, 0,
                            (last && aux) ? aux + k0 : nullptr, ldaux, n0 > 0 ? 1 : 0, st);
      }
    }
  }
  kp::g_launches -= 1;
  KP_LAUNCH_CHECK("tc_linear_bwd_data");
  return 0;
}

// dW[N,K] += dY[M,N]^T X[M,K]
extern "C" int kp_tc_linear_bwd_weight(const float* dY, int64_t lddy, const float* X, int64_t ldx, float* dW, int64_t lddw,
                                       int64_t M, int N, int K, void* stream) {
  if (M == 0) return 0;
  KP_CHECK(dY && X && dW && N >= 1 && N <= 1024 && K >= 1 && K <= 1024, "tc_linear_bwd_weight: unsupported shape N=%d K=%d", N, K);
  cudaStream_t st = as_stream(stream);
  // one launch covers pad(N) + pad(K) <= 192 operand columns; wider layers are cut into [<=128 x <=64] blocks of dW
  const bool single = N <= 128 && K <= 128 && pad_dim(N) + pad_dim(K) <= 192;
  const int n_step = single ? N : 128, k_step = single ? K : 64;
  for (int n0 = 0; n0 < N; n0 += n_step) {
    const int nn = std::min(n_step, N - n0);
    for (int k0 = 0; k0 < K; k0 += k_step) {
      const int kk = std::min(k_step, K - k0);
      const int Kp = pad_dim(kk), Np = pad_dim(nn);
      const float* Xs = X + k0;
      const float* dYs = dY + n0;
      float* dWs = dW + (int64_t)n0 * lddw + k0;
      if (Kp == 32) dispatch_wgrad<32>(Np, Xs, ldx, dYs, lddy, dWs, lddw, M, kk, nn, st);
      else if (Kp == 64) dispatch_wgrad<64>(Np, Xs, ldx, dYs, lddy, dWs, lddw, M, kk, nn, st);
      else dispatch_wgrad<128>(Np, Xs, ldx, dYs, lddy, dWs, lddw, M, kk, nn, st);
      kp::g_launches += 1;
    }
  }
  kp::g_launches -= 1;  // KP_LAUNCH_CHECK counts one
  KP_LAUNCH_CHECK("tc_linear_bwd_weight");
  return 0;
}
