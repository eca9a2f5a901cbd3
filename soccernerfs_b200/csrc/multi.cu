// Multi-tensor streaming kernels (sm_100a): one launch covers every plane / parameter of a group.
//   kp_plane_reg_fused(_range, _shard) : values and gradients of the K-Planes regularisers
//                                        (NS/model_components/losses.py:356-452) over a list of channel-last planes in
//                                        one sweep (the default model has 36 planes; per-plane launches were
//                                        launch-latency bound).
//   kp_plane_reg_adam                  : the same regulariser stencil fused with an in-place Adam step.
//   kp_adam_multi                      : torch.optim.Adam over a list of dense fp32 tensors that share one step count
//                                        (NS/engine/optimizers.py:74-160, method_configs.py:546-557); hyper-parameters
//                                        may come from device memory so the step can be replayed from a CUDA graph.
// Both Adam passes apply the update rule of common.cuh (adam_update).
// Work is split into fixed-size chunks or tiles; a block finds its (tensor, chunk) by a short scan of a prefix table
// that travels in the kernel parameters.
#include "common.cuh"

namespace kp {

constexpr int kMaxTensors = 64;
constexpr int kChunk = 2048;  // float4 elements per block of adam_multi_kernel (256 threads x 8)

__device__ __forceinline__ int find_tensor(const int* first_block, int n, int b) {
  int p = 0;
  while (p + 1 < n && first_block[p + 1] <= b) ++p;
  return p;
}

__device__ __forceinline__ float4 sub4m(float4 a, float4 b) { return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); }
__device__ __forceinline__ float sq4m(float4 a) { return a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w; }
__device__ __forceinline__ float sgnm(float x) { return (x > 0.f) ? 1.f : ((x < 0.f) ? -1.f : 0.f); }

// ---------------------------------------------------------------------------------------------------------------
// The regulariser stencil, shared by the sweep and the reg+Adam pass so that both compute the same bits.
// (k.x, k.y, k.z, k.w) = coef[p, 0..3] of the terms selected by bit i of terms, 0 otherwise.
__device__ __forceinline__ float4 reg_coef(const float* coef, int p, uint32_t terms) {
  return make_float4((terms & 1u) ? coef[p * 4 + 0] : 0.f, (terms & 2u) ? coef[p * 4 + 1] : 0.f,
                     (terms & 4u) ? coef[p * 4 + 2] : 0.f, (terms & 8u) ? coef[p * 4 + 3] : 0.f);
}

// One float4 element c = row h of a channel-last plane with H rows.  a, b / d, e are rows h-2, h-1 / h+1, h+2 of the
// same column (zero outside the plane); l() / r() return the W neighbours and are called only where has_l / has_r, so a
// caller can read them where they live.  Adds to s the terms whose first element is c (only when cnt) and returns
// sum_i k_i * d(sums[i]) / dc, sums[i] as in kp_plane_reg_fused (include/kplanes_b200.h).
template <class L, class R>
__device__ __forceinline__ float4 reg_stencil(uint32_t terms, const float4& k, int h, int H, bool has_l, bool has_r, bool cnt,
                                              const float4& a, const float4& b, const float4& c, const float4& d,
                                              const float4& e, const L& l, const R& r, float4& s) {
  float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
  if (terms & 1u) {  // squared first difference along H
    if (h + 1 < H) { const float4 df = sub4m(d, c); if (cnt) s.x += sq4m(df); g = fma4(df, -2.f * k.x, g); }
    if (h >= 1) g = fma4(sub4m(c, b), 2.f * k.x, g);
  }
  if (terms & 2u) {  // squared first difference along W
    if (has_r) { const float4 df = sub4m(r(), c); if (cnt) s.y += sq4m(df); g = fma4(df, -2.f * k.y, g); }
    if (has_l) g = fma4(sub4m(c, l()), 2.f * k.y, g);
  }
  if (terms & 4u) {  // squared second difference along H
    if (h + 2 < H) { const float4 dd = sub4m(sub4m(e, d), sub4m(d, c)); if (cnt) s.z += sq4m(dd); g = fma4(dd, 2.f * k.z, g); }
    if (h >= 1 && h + 1 < H) g = fma4(sub4m(sub4m(d, c), sub4m(c, b)), -4.f * k.z, g);
    if (h >= 2) g = fma4(sub4m(sub4m(c, b), sub4m(b, a)), 2.f * k.z, g);
  }
  if (terms & 8u) {  // |1 - t|
    if (cnt) s.w += fabsf(1.f - c.x) + fabsf(1.f - c.y) + fabsf(1.f - c.z) + fabsf(1.f - c.w);
    g.x -= k.w * sgnm(1.f - c.x); g.y -= k.w * sgnm(1.f - c.y); g.z -= k.w * sgnm(1.f - c.z); g.w -= k.w * sgnm(1.f - c.w);
  }
  return g;
}

// Block reduction (256 threads) of the per-thread sums s: adds the block's totals of the selected terms to
// plane_sums[0..3].  Called by every thread of the block.
__device__ __forceinline__ void add_reg_sums(double* plane_sums, uint32_t terms, const float4& s) {
  __shared__ double red[4][8];
  const double dd[4] = {warp_sum_d((double)s.x), warp_sum_d((double)s.y), warp_sum_d((double)s.z), warp_sum_d((double)s.w)};
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0)
    for (int k = 0; k < 4; ++k) red[k][warp] = dd[k];
  __syncthreads();
  if (threadIdx.x < 4 && ((terms >> threadIdx.x) & 1u)) {
    double acc = 0.0;
    for (int wv = 0; wv < 8; ++wv) acc += red[threadIdx.x][wv];
    atomicAdd(&plane_sums[threadIdx.x], acc);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Fused regulariser pass: values AND gradients of all terms of a plane in ONE sweep.
//   losses.py:356-452 are means of squares of plane differences, so d(coef * term)/d(plane) needs no forward result:
//   the training step streams every plane once, accumulates the four sums (for the reported loss values) and WRITES
//   coef . d(sums)/d(plane) into the gradient bucket -- which also replaces the bucket's memset (the scatter kernels
//   then add the data gradients on top).  Compared with memset + forward sweep + read-modify-write backward sweep this
//   moves 2x instead of 5x the plane bytes.
// Decomposition: a block owns 256 consecutive float4 columns of kRegRows rows and walks down H keeping the rows
// h-2 .. h+2 in registers (each element is loaded once per block + halo); the W neighbours come from L1.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kRegRows = 32;

struct RegPlane {
  const float* t;
  float* g;
  int H, W, C4;
  uint32_t terms;
};
struct RegTable {
  RegPlane pl[kMaxTensors];
  int first_block[kMaxTensors + 1];  // first tile (block) of each plane
  int tiles_x[kMaxTensors];          // tiles across a row of each plane
  int n;
};

// write_range (optional, DEVICE int64 [P,2]): gradients are written only for float4 elements [begin, end) of plane p (the
// sums always cover the whole plane) -- the data-parallel step with the sparse gradient exchange lets every rank write
// the regularisers' gradient for ITS shard of the bucket only.
template <bool ACCUMULATE>
__global__ void __launch_bounds__(256) plane_reg_fused_kernel(const __grid_constant__ RegTable T, const float* __restrict__ coef,
                                                              double* __restrict__ sums, const long long* __restrict__ write_range,
                                                              int sums_in_range) {
  const int p = find_tensor(T.first_block, T.n, blockIdx.x);
  const RegPlane& P = T.pl[p];
  const float* __restrict__ t = P.t;
  const int H = P.H, W = P.W, C4 = P.C4;
  const uint32_t terms = P.terms;
  const float4 coef4 = coef != nullptr ? reg_coef(coef, p, terms) : make_float4(0.f, 0.f, 0.f, 0.f);  // NULL: sums only
  const int local = blockIdx.x - T.first_block[p];
  const int tx = local % T.tiles_x[p], ty = local / T.tiles_x[p];
  const int row4 = W * C4;                      // float4 elements per row
  const int col = tx * 256 + threadIdx.x;       // float4 column of this thread
  const bool active = col < row4;
  const int wcol = active ? col / C4 : 0;
  const int h0 = ty * kRegRows, h1 = min(H, h0 + kRegRows);
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  const bool need2 = (terms & 4u) != 0;
  const long long wr0 = write_range ? write_range[2 * p] : 0, wr1 = write_range ? write_range[2 * p + 1] : 0;
  const bool shard_sums = write_range != nullptr && sums_in_range != 0;
  if (shard_sums) {
    // shard mode: a tile without any element of [wr0, wr1) has nothing to write and nothing to count (block-uniform exit)
    const long long lo = (long long)h0 * row4 + tx * 256;
    const long long hi = (long long)(h1 - 1) * row4 + min(row4, tx * 256 + 256) - 1;
    if (hi < wr0 || lo >= wr1) return;
  }
  float4 s = zero;
  if (active) {
    const float* base = t + (size_t)col * 4;
    const size_t rstride = (size_t)row4 * 4;
    float* __restrict__ gbase = P.g;  // never aliases the planes: lets the loads of later rows move above the stores
    auto row_at = [&](int h) -> float4 { return (h >= 0 && h < H) ? ldg4(base + (size_t)h * rstride) : zero; };
    const bool hasL = wcol >= 1, hasR = wcol + 1 < W, needW = (terms & 2u) != 0;
    // one row: c = row h, b / a = rows h-1 / h-2, d / e = rows h+1 / h+2, l / r = W neighbours of row h
    auto do_row = [&](int h, const float4& a, const float4& b, const float4& c, const float4& d, const float4& e, const float4& l,
                      const float4& r) {
      const long long e4 = (long long)h * row4 + col;
      const bool in_range = write_range == nullptr || (e4 >= wr0 && e4 < wr1);
      const bool cnt = !shard_sums || in_range;  // shard mode: every term is counted by the rank that owns its element
      float4 g = reg_stencil(terms, coef4, h, H, hasL, hasR, cnt, a, b, c, d, e, [&] { return l; }, [&] { return r; }, s);
      if (gbase != nullptr && in_range) {
        float4* gp = reinterpret_cast<float4*>(gbase + (size_t)h * rstride + (size_t)col * 4);
        if (ACCUMULATE) { const float4 cur = *gp; g.x += cur.x; g.y += cur.y; g.z += cur.z; g.w += cur.w; }
        *gp = g;
      }
    };
    float4 a = need2 ? row_at(h0 - 2) : zero, b = row_at(h0 - 1), c = row_at(h0), d = row_at(h0 + 1);
    // four rows per iteration: the four next rows and the eight W neighbours are loaded up front (12 independent 16-byte
    // loads in flight per thread -- the one-row-at-a-time version ran at 1.1 TB/s)
    for (int h = h0; h < h1; h += 4) {
      float4 nr[4], l[4], r[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) nr[i] = row_at(h + 2 + i);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool in = h + i < h1;
        l[i] = (needW && hasL && in) ? ldg4(base + (size_t)(h + i) * rstride - C4 * 4) : zero;
        r[i] = (needW && hasR && in) ? ldg4(base + (size_t)(h + i) * rstride + C4 * 4) : zero;
      }
      do_row(h, a, b, c, d, nr[0], l[0], r[0]);
      if (h + 1 < h1) do_row(h + 1, b, c, d, nr[0], nr[1], l[1], r[1]);
      if (h + 2 < h1) do_row(h + 2, c, d, nr[0], nr[1], nr[2], l[2], r[2]);
      if (h + 3 < h1) do_row(h + 3, d, nr[0], nr[1], nr[2], nr[3], l[3], r[3]);
      a = nr[0]; b = nr[1]; c = nr[2]; d = nr[3];
    }
  }
  if (sums != nullptr) add_reg_sums(sums + p * 4, terms, s);
}

struct AdamTensor {
  float* p;
  const float* g;
  float* m;
  float* v;
  int64_t n;
};
struct AdamTable {
  AdamTensor t[kMaxTensors];
  int first_block[kMaxTensors + 1];
  int n;
};

__global__ void __launch_bounds__(256) adam_multi_kernel(const __grid_constant__ AdamTable T,
                                                         const float* __restrict__ hyper_dev, AdamScalars s) {
  s = with_hyper_dev(s, hyper_dev);
  const int ti = find_tensor(T.first_block, T.n, blockIdx.x);
  const AdamTensor& A = T.t[ti];
  const int64_t base = (int64_t)(blockIdx.x - T.first_block[ti]) * kChunk * 4;
  const bool vec_ok = ((((uintptr_t)A.p | (uintptr_t)A.g | (uintptr_t)A.m | (uintptr_t)A.v) & 15) == 0);
#pragma unroll 2
  for (int it = 0; it < kChunk / 256; ++it) {
    const int64_t i4 = base + ((int64_t)it * 256 + threadIdx.x) * 4;
    if (i4 >= A.n) break;
    if (vec_ok && i4 + 4 <= A.n) {
      float4 pp = *reinterpret_cast<float4*>(A.p + i4);
      const float4 gg = *reinterpret_cast<const float4*>(A.g + i4);
      float4 mm = *reinterpret_cast<float4*>(A.m + i4), vv = *reinterpret_cast<float4*>(A.v + i4);
      adam_update4(scale4(gg, s.grad_scale), pp, mm, vv, s);
      *reinterpret_cast<float4*>(A.p + i4) = pp;
      *reinterpret_cast<float4*>(A.m + i4) = mm;
      *reinterpret_cast<float4*>(A.v + i4) = vv;
    } else {
      for (int64_t i = i4; i < A.n && i < i4 + 4; ++i) adam_update(A.g[i] * s.grad_scale, A.p[i], A.m[i], A.v[i], s);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// (f1) Regulariser stencil + Adam in ONE streaming pass per plane (SURVEY.md 8f rank 1; NS/engine/optimizers.py:74-160
// over NS/model_components/losses.py:356-452).  Per element the pass reads p, g, m, v once and writes p, m, v (and
// g = 0 for the next step): the regularisers' gradient is computed on the fly from the PRE-update plane values and is
// never materialised (the separate sweep wrote 1x and the optimizer re-read 1x the plane bytes for it).
//   total gradient  = g * grad_scale + sum_i coef[p,i] * d(sums[p,i]) / d(plane)
// The stencil needs pre-update neighbours while the planes are updated in place.  Tiles of kFRows rows x 256 float4
// columns are owned by one block each; a block walks down its rows with the rows h-2 .. h+2 in registers (loaded
// before the row is overwritten) and exchanges the W neighbours through shared memory before anyone writes the row.
// Neighbours OUTSIDE the tile (2 rows above / below, one texel left / right) may already have been updated by the
// block that owns them, so a tiny first kernel snapshots every tile's halo (<= 12.5 % of the plane bytes) and the main
// kernel reads halo values from the snapshot only.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kFRows = 64;                            // rows per tile
constexpr int kFMaxC4 = 8;                            // float4 per texel supported (C <= 32)
constexpr int kFHaloRows = 4 * 256;                   // float4: rows h0-2, h0-1, h1, h1+1 of the tile's 256 columns
constexpr int kFHaloF4 = kFHaloRows + kFRows * 2 * kFMaxC4;  // + [row][left | right][C4] texel columns
constexpr int kFMaxTensors = 40;

struct RegAdamPlane {
  float* p;
  float* g;
  float* m;
  float* v;
  int H, W, C4;
  uint32_t terms;
};
struct RegAdamTable {
  RegAdamPlane pl[kFMaxTensors];
  int first_block[kFMaxTensors + 1];
  int tiles_x[kFMaxTensors];
  int n;
};

__global__ void __launch_bounds__(256) plane_halo_snapshot_kernel(const __grid_constant__ RegAdamTable T, float4* __restrict__ halo) {
  const int p = find_tensor(T.first_block, T.n, blockIdx.x);
  const RegAdamPlane& P = T.pl[p];
  const int H = P.H, C4 = P.C4, row4 = P.W * P.C4;
  const int local = blockIdx.x - T.first_block[p];
  const int tx = local % T.tiles_x[p], ty = local / T.tiles_x[p];
  const int col = tx * 256 + threadIdx.x;
  const int h0 = ty * kFRows, h1 = min(H, h0 + kFRows);
  const float4* __restrict__ src = reinterpret_cast<const float4*>(P.p);
  float4* dst = halo + (size_t)blockIdx.x * kFHaloF4;
  if (col < row4) {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int h = r < 2 ? h0 - 2 + r : h1 + (r - 2);
      if (h >= 0 && h < H) dst[r * 256 + threadIdx.x] = src[(size_t)h * row4 + col];
    }
  }
  const int n_side = (h1 - h0) * 2 * C4;
  for (int i = threadIdx.x; i < n_side; i += 256) {
    const int hh = i / (2 * C4), side = (i / C4) & 1, k = i % C4;
    const int c = side ? tx * 256 + 256 + k : tx * 256 - C4 + k;
    if (c >= 0 && c < row4) dst[kFHaloRows + (hh * 2 + side) * kFMaxC4 + k] = src[(size_t)(h0 + hh) * row4 + c];
  }
}

template <bool ZERO_GRAD>
__global__ void __launch_bounds__(256, 3) plane_reg_adam_kernel(const __grid_constant__ RegAdamTable T, const float4* __restrict__ halo,
                                                             const float* __restrict__ coef, double* __restrict__ sums,
                                                             const float* __restrict__ hyper_dev, AdamScalars adam) {
  adam = with_hyper_dev(adam, hyper_dev);
  __shared__ float4 xch[2][256];
  const int p = find_tensor(T.first_block, T.n, blockIdx.x);
  const RegAdamPlane& P = T.pl[p];
  const int H = P.H, W = P.W, C4 = P.C4, row4 = W * C4;
  const uint32_t terms = P.terms;
  const float4 coef4 = reg_coef(coef, p, terms);
  const int local = blockIdx.x - T.first_block[p];
  const int tx = local % T.tiles_x[p], ty = local / T.tiles_x[p];
  const int tid = threadIdx.x;
  const int col = tx * 256 + tid;
  const bool active = col < row4;
  const int wcol = active ? col / C4 : 0;
  const bool hasL = active && wcol >= 1, hasR = active && wcol + 1 < W;
  const bool edgeL = tid < C4, edgeR = tid >= 256 - C4;
  const int h0 = ty * kFRows, h1 = min(H, h0 + kFRows);
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  const bool need2 = (terms & 4u) != 0;
  float4* __restrict__ pp = reinterpret_cast<float4*>(P.p);
  float4* __restrict__ gp = reinterpret_cast<float4*>(P.g);
  float4* __restrict__ mp = reinterpret_cast<float4*>(P.m);
  float4* __restrict__ vp = reinterpret_cast<float4*>(P.v);
  const float4* __restrict__ hl = halo + (size_t)blockIdx.x * kFHaloF4;
  const int kc = tid % C4;
  // pre-update value of row h at this thread's column: own tile rows come from the plane (this block has not written
  // them yet when they are requested), rows of other tiles from the snapshot
  auto old_row = [&](int h) -> float4 {
    if (!active || h < 0 || h >= H) return zero;
    if (h < h0) return hl[(h - (h0 - 2)) * 256 + tid];
    if (h >= h1) return hl[(2 + (h - h1)) * 256 + tid];
    return pp[(size_t)h * row4 + col];
  };
  auto halo_side = [&](int h, int side) -> float4 { return hl[kFHaloRows + ((h - h0) * 2 + side) * kFMaxC4 + kc]; };
  float4 s = zero;
  float4 a = need2 ? old_row(h0 - 2) : zero, b = old_row(h0 - 1), c = old_row(h0), d = old_row(h0 + 1);
  float4 gn = zero, mn = zero, vn = zero, hLn = zero, hRn = zero;
  if (active) {
    const size_t i0 = (size_t)h0 * row4 + col;
    gn = gp[i0]; mn = mp[i0]; vn = vp[i0];
    if (edgeL && hasL) hLn = halo_side(h0, 0);
    if (edgeR && hasR) hRn = halo_side(h0, 1);
  }
  for (int h = h0; h < h1; ++h) {
    const float4 e = old_row(h + 2);
    const float4 gg = gn, mm0 = mn, vv0 = vn, hL = hLn, hR = hRn;
    if (active && h + 1 < h1) {  // next row's streams in flight under this row's arithmetic
      const size_t in = (size_t)(h + 1) * row4 + col;
      gn = gp[in]; mn = mp[in]; vn = vp[in];
      if (edgeL && hasL) hLn = halo_side(h + 1, 0);
      if (edgeR && hasR) hRn = halo_side(h + 1, 1);
    }
    float4* x = xch[h & 1];
    x[tid] = c;
    __syncthreads();  // every thread's pre-update row h is visible before any thread overwrites row h in global memory
    if (active) {
      // W neighbours: the exchanged row inside the tile, the halo snapshot at its edges (where x[tid -/+ C4] would fall
      // outside the exchanged row)
      const float4 g = reg_stencil(terms, coef4, h, H, hasL, hasR, true, a, b, c, d, e,
                                   [&] { return edgeL ? hL : x[tid - C4]; }, [&] { return edgeR ? hR : x[tid + C4]; }, s);
      float4 pn = c, mm = mm0, vv = vv0;
      const float gs = adam.grad_scale;
      adam_update4(make_float4(fmaf(gg.x, gs, g.x), fmaf(gg.y, gs, g.y), fmaf(gg.z, gs, g.z), fmaf(gg.w, gs, g.w)), pn, mm, vv,
                   adam);
      const size_t i = (size_t)h * row4 + col;
      pp[i] = pn; mp[i] = mm; vp[i] = vv;
      // untouched lines (85 % of the 32x scale per step) are still zero: skip the store (same value, less HBM write traffic)
      if (ZERO_GRAD && (gg.x != 0.f || gg.y != 0.f || gg.z != 0.f || gg.w != 0.f)) gp[i] = zero;
    }
    a = b; b = c; c = d; d = e;
  }
  if (sums != nullptr) add_reg_sums(sums + p * 4, terms, s);
}

// Per-step scalars of a graph-replayed training step, from the device-resident step counter: the proposal-weight
// anneal exponent (NS/models/kplanes.py:326-331), the cosine-decayed learning rate (NS/engine/schedulers.py:126-142,
// both tabulated by the host once) and Adam's bias corrections (torch.optim.Adam) -- one single-thread kernel instead
// of ~30 0-d torch ops per step; it also advances the counter.
struct StepScalars {
  float* hyper[4];
  float beta1[4], beta2[4];
  int n_groups;
};
__global__ void step_scalars_kernel(long long* __restrict__ step_counter, const double* __restrict__ lr_table,
                                    const float* __restrict__ anneal_table, long long max_steps, float grad_scale,
                                    float* __restrict__ anneal_out, const __grid_constant__ StepScalars S) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const long long s = *step_counter;
  const long long idx = s < max_steps ? s : max_steps;
  if (anneal_out != nullptr) *anneal_out = anneal_table[idx];
  const double lr = lr_table[idx], t = (double)(s + 1);
  for (int g = 0; g < S.n_groups; ++g) {
    const double bc1 = 1.0 - pow((double)S.beta1[g], t), bc2 = 1.0 - pow((double)S.beta2[g], t);
    S.hyper[g][0] = (float)(lr / bc1);
    S.hyper[g][1] = (float)rsqrt(bc2);
    S.hyper[g][2] = grad_scale;
  }
  *step_counter = s + 1;
}

// Planes [begin, end) of the fused sweep; a plane with a gradient target needs the coefficient table.
static int fill_reg_table(RegTable& T, const float* const* planes, float* const* grads, const int32_t* hwc,
                          const uint32_t* terms, int begin, int end, bool have_coef) {
  int nb = 0, k = 0;
  for (int i = begin; i < end; ++i, ++k) {
    RegPlane& r = T.pl[k];
    r.t = planes[i];
    r.g = grads ? grads[i] : nullptr;
    r.H = hwc[i * 3 + 0];
    r.W = hwc[i * 3 + 1];
    const int C = hwc[i * 3 + 2];
    KP_CHECK(r.t != nullptr && r.H >= 1 && r.W >= 1 && C >= 4 && C % 4 == 0, "plane_reg_fused: plane %d invalid (C %% 4 != 0?)", i);
    KP_CHECK(have_coef || r.g == nullptr, "plane_reg_fused: plane %d has a gradient target but coef_dev is NULL", i);
    r.C4 = C / 4;
    r.terms = terms[i];
    T.first_block[k] = nb;
    T.tiles_x[k] = (int)ceil_div((int64_t)r.W * r.C4, 256);
    nb += T.tiles_x[k] * (int)ceil_div(r.H, kRegRows);
  }
  T.first_block[k] = nb;
  T.n = k;
  return 0;
}

}  // namespace kp

using namespace kp;

extern "C" int kp_step_scalars(int64_t* step_counter, const double* lr_table, const float* anneal_table, int64_t max_steps,
                               int n_groups, const float* betas_host, float grad_scale, float* anneal_out,
                               float* const* hyper_out_host, void* stream) {
  KP_CHECK(step_counter && lr_table && anneal_table && betas_host && hyper_out_host && n_groups >= 1 && n_groups <= 4,
           "step_scalars: bad arguments (1..4 optimizer groups)");
  StepScalars S;
  S.n_groups = n_groups;
  for (int g = 0; g < n_groups; ++g) {
    KP_CHECK(hyper_out_host[g] != nullptr, "step_scalars: hyper_out[%d] is NULL", g);
    S.hyper[g] = hyper_out_host[g];
    S.beta1[g] = betas_host[2 * g];
    S.beta2[g] = betas_host[2 * g + 1];
  }
  step_scalars_kernel<<<1, 32, 0, as_stream(stream)>>>(reinterpret_cast<long long*>(step_counter), lr_table, anneal_table,
                                                      (long long)max_steps, grad_scale, anneal_out, S);
  KP_LAUNCH_CHECK("step_scalars");
  return 0;
}

static int plane_reg_fused_impl(const float* const* planes, float* const* grads, const int32_t* hwc, const uint32_t* terms, int P,
                                const float* coef_dev, int accumulate, double* sums, const int64_t* write_range_dev,
                                int sums_in_range, void* stream);

extern "C" int kp_plane_reg_fused(const float* const* planes, float* const* grads, const int32_t* hwc, const uint32_t* terms,
                                  int P, const float* coef_dev, int accumulate, double* sums, void* stream) {
  return plane_reg_fused_impl(planes, grads, hwc, terms, P, coef_dev, accumulate, sums, nullptr, 0, stream);
}

extern "C" int kp_plane_reg_fused_range(const float* const* planes, float* const* grads, const int32_t* hwc, const uint32_t* terms,
                                        int P, const float* coef_dev, int accumulate, double* sums, const int64_t* write_range_dev,
                                        void* stream) {
  return plane_reg_fused_impl(planes, grads, hwc, terms, P, coef_dev, accumulate, sums, write_range_dev, 0, stream);
}

extern "C" int kp_plane_reg_fused_shard(const float* const* planes, float* const* grads, const int32_t* hwc, const uint32_t* terms,
                                        int P, const float* coef_dev, int accumulate, double* sums, const int64_t* write_range_dev,
                                        void* stream) {
  KP_CHECK(write_range_dev != nullptr, "plane_reg_fused_shard: needs the per-plane ranges");
  return plane_reg_fused_impl(planes, grads, hwc, terms, P, coef_dev, accumulate, sums, write_range_dev, 1, stream);
}

static int plane_reg_fused_impl(const float* const* planes, float* const* grads, const int32_t* hwc, const uint32_t* terms, int P,
                                const float* coef_dev, int accumulate, double* sums, const int64_t* write_range_dev,
                                int sums_in_range, void* stream) {
  KP_CHECK(planes && hwc && terms && P >= 0, "plane_reg_fused: bad arguments");
  for (int begin = 0; begin < P; begin += kMaxTensors) {
    const int end = std::min(P, begin + kMaxTensors);
    RegTable T;
    if (fill_reg_table(T, planes, grads, hwc, terms, begin, end, coef_dev != nullptr)) return 1;
    const int nb = T.first_block[T.n];
    if (nb == 0) continue;
    const float* cf = coef_dev ? coef_dev + (size_t)begin * 4 : nullptr;
    double* s = sums ? sums + (size_t)begin * 4 : nullptr;
    const long long* wr = write_range_dev ? reinterpret_cast<const long long*>(write_range_dev) + (size_t)begin * 2 : nullptr;
    if (accumulate) plane_reg_fused_kernel<true><<<nb, 256, 0, as_stream(stream)>>>(T, cf, s, wr, sums_in_range);
    else plane_reg_fused_kernel<false><<<nb, 256, 0, as_stream(stream)>>>(T, cf, s, wr, sums_in_range);
    KP_LAUNCH_CHECK("plane_reg_fused");
  }
  return 0;
}

extern "C" int kp_adam_multi(float* const* params, const float* const* grads, float* const* exp_avg,
                             float* const* exp_avg_sq, const int64_t* sizes, int P, float lr, float beta1, float beta2,
                             float eps, float weight_decay, int64_t step, float grad_scale, const float* hyper_dev,
                             void* stream) {
  KP_CHECK(params && grads && exp_avg && exp_avg_sq && sizes && P >= 0 && step >= 1, "adam_multi: bad arguments");
  const AdamScalars adam = adam_scalars(lr, beta1, beta2, eps, weight_decay, step, grad_scale);
  for (int begin = 0; begin < P; begin += kMaxTensors) {
    const int end = std::min(P, begin + kMaxTensors);
    AdamTable T;
    int nb = 0, k = 0;
    for (int i = begin; i < end; ++i, ++k) {
      KP_CHECK(params[i] && grads[i] && exp_avg[i] && exp_avg_sq[i], "adam_multi: NULL tensor %d", i);
      T.t[k] = AdamTensor{params[i], grads[i], exp_avg[i], exp_avg_sq[i], sizes[i]};
      T.first_block[k] = nb;
      nb += (int)ceil_div(ceil_div(sizes[i], 4), kChunk);
    }
    T.first_block[k] = nb;
    T.n = k;
    if (nb == 0) continue;
    adam_multi_kernel<<<nb, 256, 0, as_stream(stream)>>>(T, hyper_dev, adam);
    KP_LAUNCH_CHECK("adam_multi");
  }
  return 0;
}

static bool reg_adam_c_ok(int C) { return C == 4 || C == 8 || C == 16 || C == 32; }

extern "C" int kp_plane_reg_adam_supported(int C) { return reg_adam_c_ok(C) ? 1 : 0; }

// Bytes of halo scratch kp_plane_reg_adam needs for these planes (one snapshot slot per tile).
extern "C" int64_t kp_plane_reg_adam_scratch_bytes(const int32_t* hwc, int P) {
  int64_t tiles = 0;
  for (int i = 0; i < P; ++i)
    tiles += ceil_div((int64_t)hwc[i * 3 + 1] * (hwc[i * 3 + 2] / 4), 256) * ceil_div((int64_t)hwc[i * 3 + 0], kFRows);
  return tiles * kFHaloF4 * (int64_t)sizeof(float4);
}

extern "C" int kp_plane_reg_adam(float* const* planes, float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
                                 const int32_t* hwc, const uint32_t* terms, int P, const float* coef_dev, float lr, float beta1,
                                 float beta2, float eps, float weight_decay, int64_t step, float grad_scale,
                                 const float* hyper_dev, double* sums, void* scratch, int64_t scratch_bytes, int zero_grads,
                                 void* stream) {
  KP_CHECK(planes && grads && exp_avg && exp_avg_sq && hwc && terms && coef_dev && P >= 0 && step >= 1 && scratch,
           "plane_reg_adam: bad arguments");
  KP_CHECK(scratch_bytes >= kp_plane_reg_adam_scratch_bytes(hwc, P), "plane_reg_adam: scratch too small (%lld bytes)",
           (long long)scratch_bytes);
  const AdamScalars adam = adam_scalars(lr, beta1, beta2, eps, weight_decay, step, grad_scale);
  float4* halo = reinterpret_cast<float4*>(scratch);
  for (int begin = 0; begin < P; begin += kFMaxTensors) {
    const int end = std::min(P, begin + kFMaxTensors);
    RegAdamTable T;
    int nb = 0, k = 0;
    for (int i = begin; i < end; ++i, ++k) {
      RegAdamPlane& r = T.pl[k];
      r.p = planes[i]; r.g = grads[i]; r.m = exp_avg[i]; r.v = exp_avg_sq[i];
      r.H = hwc[i * 3 + 0]; r.W = hwc[i * 3 + 1];
      const int C = hwc[i * 3 + 2];
      KP_CHECK(r.p && r.g && r.m && r.v && r.H >= 1 && r.W >= 1 && reg_adam_c_ok(C), "plane_reg_adam: plane %d invalid (C in {4,8,16,32})", i);
      KP_CHECK(((((uintptr_t)r.p | (uintptr_t)r.g | (uintptr_t)r.m | (uintptr_t)r.v) & 15) == 0), "plane_reg_adam: plane %d not 16-byte aligned", i);
      r.C4 = C / 4;
      r.terms = terms[i];
      T.first_block[k] = nb;
      T.tiles_x[k] = (int)ceil_div((int64_t)r.W * r.C4, 256);
      nb += T.tiles_x[k] * (int)ceil_div(r.H, kFRows);
    }
    T.first_block[k] = nb;
    T.n = k;
    if (nb == 0) continue;
    cudaStream_t st = as_stream(stream);
    plane_halo_snapshot_kernel<<<nb, 256, 0, st>>>(T, halo);
    kp::g_launches += 1;
    double* s = sums ? sums + (size_t)begin * 4 : nullptr;
    const float* cf = coef_dev + (size_t)begin * 4;
    if (zero_grads) plane_reg_adam_kernel<true><<<nb, 256, 0, st>>>(T, halo, cf, s, hyper_dev, adam);
    else plane_reg_adam_kernel<false><<<nb, 256, 0, st>>>(T, halo, cf, s, hyper_dev, adam);
    KP_LAUNCH_CHECK("plane_reg_adam");
    halo += (size_t)nb * kFHaloF4;
  }
  return 0;
}
