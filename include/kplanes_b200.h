/*
 * kplanes_b200.h -- C-ABI of libkplanes_b200.so: the B200 (sm_100a) K-Planes train/render hot path.
 *
 * Drop-in boundary (SURVEY.md 8b).  Every entry point takes raw DEVICE pointers, plain sizes and a
 * cudaStream_t passed as void*; returns 0 on success, non-zero on failure (message via
 * kp_last_error()).  No torch / C++ types cross this boundary.  The Python host side
 * (soccernerfs_b200/) binds these with ctypes and wraps them in torch.autograd.Functions that mirror
 * the reference's nerfstudio plugin surface.  NS = nerfstudio/nerfstudio in the reference checkout.
 *
 * Layout conventions
 *   planes      channel-last fp32 [H][W][C] (the reference keeps [1,C,H,W]; repacked once on load).
 *               Plane (a,b) of combinations(range(D),2) has W = reso[a], H = reso[b] and is sampled
 *               at (pts[a] -> W, pts[b] -> H)   (NS/fields/kplanes_field.py:61-67, :113).
 *   plane_ptrs  HOST array [n_scales*n_planes] of device pointers, scale-major.
 *   plane_hw    HOST array [n_scales*n_planes*2] of (H, W).
 *   ray form    origins[N,3], directions[N,3], starts[N,S], ends[N,S], times[N] (may be NULL),
 *               aabb HOST float[6] = min xyz, max xyz.  Sample position = o + d*(start+end)/2
 *               (NS/cameras/rays.py:54) normalised by the aabb (NS/data/scene_box.py:56-66) to
 *               [0,1] (norm_mode 0: KPlanesDensityField quirk, kplanes_field.py:439-440) or to
 *               [-1,1] (norm_mode 1: KPlanesField, kplanes_field.py:283-284), or contracted with
 *               SceneContraction(order=inf) and halved (norm_mode 2: bounded=False, kplanes_field.py:278-280,
 *               NS/field_components/spatial_distortions.py:42-88; aabb unused); time -> t*2-1.
 *   point form  pts[M,D] already in grid_sample's [-1,1] convention (D = 3 or 4).
 */
#ifndef KPLANES_B200_H_
#define KPLANES_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KP_ABI_VERSION 4
#define KP_MAX_SCALES 8
#define KP_MAX_PLANES 6

int kp_abi_version(void);
const char* kp_last_error(void);
long long kp_launch_count(void); /* kernels launched through this library since load */

/* Where sample coordinates come from (exactly one of pts / ray form is used). */
typedef struct KpPoints {
  const float* pts;        /* [M,D] or NULL */
  const float* origins;    /* [N,3] */
  const float* directions; /* [N,3] */
  const float* starts;     /* [N,S] */
  const float* ends;       /* [N,S] */
  const float* times;      /* [N] or NULL */
  int32_t D;               /* 3 (static) or 4 (dynamic) */
  int32_t S;               /* samples per ray (ray form) */
  int32_t norm_mode;       /* 0: aabb -> [0,1], 1: aabb -> [-1,1], 2: SceneContraction(L_inf) / 2 (unbounded scenes) */
  float aabb[6];
  int32_t ray_tile;        /* ray form, gather only: > 1 = the threads of a warp take the SAME sample index of ray_tile
                              neighbouring rays instead of consecutive samples of one ray (full-frame inference: neighbouring
                              pixels read the same texels, which then coalesce inside one request).  Results are written
                              at the samples' own rows: only the thread -> sample assignment changes.  0/1 = off; < 0 = off and the
                              4-channels-per-lane kernel forced (tests compare the two mappings). */
} KpPoints;

/* ---- (a1-a3) multiscale hexplane field: replaces interpolate_kplanes, NS/fields/kplanes_field.py:77-126
 *      (6*n_scales F.grid_sample calls + Hadamard + cat, NS/utils/interpolation.py:5-33). ------------- */
int kp_hexplane_fwd(const float* const* plane_ptrs, const int32_t* plane_hw, int n_scales, int n_planes,
                    int C, const KpPoints* points, int64_t M, int concat, uint32_t use_mask,
                    float* out /* [M, n_scales*C] (concat) or [M, C] */, void* stream);
/* Forward only, dynamic fields (n_planes = 6; 3 is an error): out exactly as kp_hexplane_fwd writes it, bit for bit, from
 * the same texel reads, and the dynamics score of every sample
 *   T[k,c] = prod over the time planes XT, YT, ZT kept by use_mask of their bilinear interpolants (scale k, channel c),
 *   delta  = 1/(n_scales*C) * sum_k sum_c |1 - T[k,c]|                                              (fp32 [M]),
 * the per-sample form of sparse_transients_loss (NS/model_components/losses.py, kplanes_field.py:97-100 for the time
 * planes' place in the Hadamard product of interpolate_kplanes, :77-126): 0 where the time planes are the identity. */
int kp_hexplane_fwd_dyn(const float* const* plane_ptrs, const int32_t* plane_hw, int n_scales, int n_planes, int C,
                        const KpPoints* points, int64_t M, int concat, uint32_t use_mask, float* out, float* delta /* [M] */,
                        void* stream);
/* grad_plane_ptrs: HOST array of device pointers (same order); entries may be NULL (frozen plane,
 * kplanes_field.py:102-110).  Gradients are ACCUMULATED (red.global.add) into the buffers. */
int kp_hexplane_bwd(const float* const* plane_ptrs, float* const* grad_plane_ptrs, const int32_t* plane_hw,
                    int n_scales, int n_planes, int C, const KpPoints* points, int64_t M, int concat,
                    uint32_t use_mask, const float* grad_out, void* stream);
/* Same, and additionally marks every texel that received a reduction: touched_ptrs (HOST array of device pointers, same
 * order, entries may be NULL) point to one byte per texel of the plane, set to 1 (never cleared here).  The data-parallel
 * step exchanges only the marked 128-byte lines of the HBM-resident scales (kp_peer_sharded_adam_sparse). */
int kp_hexplane_bwd_flags(const float* const* plane_ptrs, float* const* grad_plane_ptrs, uint8_t* const* touched_ptrs,
                          const int32_t* plane_hw, int n_scales, int n_planes, int C, const KpPoints* points, int64_t M,
                          int concat, uint32_t use_mask, const float* grad_out, void* stream);

/* ---- (a6) proposal density field: KPlanesDensityField.get_density, kplanes_field.py:434-460:
 *      single-scale planes (C = 4|8|16) -> Hadamard -> [hidden x C] ReLU (or linear) -> [1 x hidden] ->
 *      trunc_exp, fused in one kernel.  w1 [hidden,C], w2 [hidden] row-major (torch Linear layout). --- */
int kp_density_field_fwd(const float* const* plane_ptrs, const int32_t* plane_hw, int n_planes, int C,
                         const float* w1, const float* w2, int hidden, int relu, const KpPoints* points,
                         int64_t M, uint32_t use_mask, float* density /* [M] */, void* stream);
int kp_density_field_bwd(const float* const* plane_ptrs, float* const* grad_plane_ptrs, const int32_t* plane_hw,
                         int n_planes, int C, const float* w1, const float* w2, int hidden, int relu,
                         const KpPoints* points, int64_t M, uint32_t use_mask, const float* grad_density /* [M] */,
                         float* grad_w1, float* grad_w2 /* accumulated */, void* stream);

/* ---- (a4,a5) decoders: sigma_net / color_net (tcnn FullyFusedMLP in the reference, kplanes_field.py:249-273;
 *      bias-free, ReLU hidden).  sigma: feats[M,K] -> h1[M,H] -> o[M,16]; density = trunc_exp(o[:,15])
 *      (kplanes_field.py:307-311, NS/field_components/activations.py:25-41).
 *      color: cin = [SH4((d+1)/2 *2-1) (16, if dirs!=NULL) | geo o[:,0:15]] -> H2 -> H2 -> 3, sigmoid
 *      (kplanes_field.py:314-358, NS/utils/math.py:25-86).  Hidden activations are written to caller
 *      buffers and re-read by the backward. -------------------------------------------------------- */
int kp_sigma_net_fwd(const float* feats, const float* w1, const float* w2, int64_t M, int K, int H,
                     float* h1 /* [M,H] */, float* o /* [M,16] */, float* density /* [M] */, void* stream);
int kp_sigma_net_bwd(const float* feats, const float* w1, const float* w2, int64_t M, int K, int H,
                     const float* h1, const float* o, const float* grad_density /* [M] or NULL */,
                     const float* grad_o /* [M,16] upstream grad of o (col 15 added to the density path), or NULL */, float* grad_feats /* [M,K] */,
                     float* grad_w1, float* grad_w2 /* accumulated */, float* scratch /* [M,H] */, void* stream);
int kp_color_net_fwd(const float* directions /* [N,3] or NULL */, int S, const float* geo /* [M,>=15] */,
                     int ldgeo /* row stride of geo: 16 for a view of o, 15 if packed */, const float* w3, const float* w4, const float* w5, int64_t M, int H2,
                     float* cin /* [M,32|16] */, float* h2, float* h3 /* [M,H2] */, float* rgb /* [M,3] */,
                     void* stream);
int kp_color_net_bwd(int view_dependent, const float* cin, const float* h2, const float* h3, const float* rgb,
                     const float* w3, const float* w4, const float* w5, int64_t M, int H2,
                     const float* grad_rgb /* [M,3] */, float* grad_o /* [M,16], cols 0..14 written, col 15 zeroed */,
                     float* grad_w3, float* grad_w4, float* grad_w5 /* accumulated */,
                     float* scratch_a, float* scratch_b /* [M,H2] each */, void* stream);

/* Dense layer on tcgen05 tensor cores, fp32-accurate through the 4-term TF32 split x = hi + lo (building block of the
 * decoders): Y[M,N] = act(X[M,K] W[N,K]^T), act 0 none / 1 ReLU / 2 sigmoid; N, K <= 256 (K a multiple of 4 beyond one
 * launch's tile: layers wider than 64 x 128 are cut into sub-matrix launches, partial sums held in Y). */
int kp_tc_linear_fwd(const float* X, int64_t ldx, const float* W, int64_t ldw, float* Y, int64_t ldy, int64_t M, int N,
                     int K, int act, void* stream);
/* dX[M,K] = (dY[M,N] W[N,K]) masked by (aux[M,K] > 0) when aux != NULL (ReLU backward of the producing layer). */
int kp_tc_linear_bwd_data(const float* dY, int64_t lddy, const float* W, int64_t ldw, float* dX, int64_t lddx, int64_t M,
                          int N, int K, const float* aux, int64_t ldaux, void* stream);
/* dW[N,K] += dY[M,N]^T X[M,K]: persistent CTAs accumulate in TMEM over their sample tiles, one atomic flush each. */
int kp_tc_linear_bwd_weight(const float* dY, int64_t lddy, const float* X, int64_t ldx, float* dW, int64_t lddw, int64_t M,
                            int N, int K, void* stream);
int kp_tc_supported(int N, int K); /* 1 if the tensor-core path covers a layer with N outputs and K inputs */

/* Fused decoder forward (sigma_net + SH + color_net for hidden widths 64, feature width <= 128) in ONE tcgen05 kernel:
 * weights resident in shared memory, activations never leave the SM between layers.  h1/cin/h2/h3 may be NULL
 * (inference): then only o [M,16], density [M] and rgb [M,3] are written.  Replaces kp_sigma_net_fwd + kp_color_net_fwd
 * (NS/fields/kplanes_field.py:302-311, 314-358). */
int kp_decoder_fused_supported(int K0, int H1, int H2);
int kp_decoder_fwd_fused(const float* feats, int K0, const float* directions /* [N,3] or NULL */, int S, const float* w1,
                         const float* w2, const float* w3, const float* w4, const float* w5, int64_t M, int H1, int H2,
                         float* h1, float* cin, float* h2, float* h3, float* o, float* density, float* rgb, void* stream);

/* ---- (a13) AABBBoxCollider._intersect_with_aabb, NS/model_components/scene_colliders.py:57-95 ---- */
int kp_aabb_intersect(const float* origins, const float* directions, int64_t N, const float* aabb_host6,
                      float near_plane, float* nears, float* fars, void* stream);

/* ---- (f2) nerfstudio.utils.math._intersect_aabb, NS/utils/math.py:201-238 (max_bound = invalid_value = 1e10), what
 *      Cameras.generate_rays(aabb_box=...) fills RayBundle.nears / fars with for a crop-box render
 *      (NS/cameras/cameras.py:478-497, scripts/render.py:101-106).  aabb_host6 = x,y,z min then max (HOST).
 *      Bit-identical to the reference's torch ops, NaN propagation of torch.min / max / clamp included. ---- */
int kp_intersect_aabb(const float* origins, const float* directions, int64_t N, const float* aabb_host6,
                      float* t_min, float* t_max, void* stream);

/* ---- (a7) SpacedSampler / UniformSampler, NS/model_components/ray_samplers.py:79-126.
 *      lin_bins [S+1] = torch.linspace(0,1,S+1) (device).  t_rand [N,S+1] or [N,1] (rand_stride 0)
 *      or NULL (eval).  spacing: 0 uniform (x), 1 UniformLinDispPiecewise (ray_samplers.py:236-246).
 *      Outputs spacing bins [N,S+1] and euclidean bins [N,S+1]. ------------------------------------- */
int kp_uniform_bins(const float* lin_bins, const float* t_rand, int rand_stride, const float* nears,
                    const float* fars, int64_t N, int S, int spacing, float* spacing_bins, float* euclid_bins,
                    float* starts, float* ends, float* deltas /* [N,S] each, all three or none */, void* stream);

/* ---- (a8) PDFSampler.generate_ray_samples (include_original=False), ray_samplers.py:274-369:
 *      warp-per-ray inverse-CDF search.  weights [N,S_in] (already annealed), existing spacing bins
 *      [N,S_in+1], u_base [S_out+1] = torch.linspace(0, 1-1/nb, nb) (device), rand [N,S_out+1] | [N,1]
 *      (rand_stride 0) | NULL (eval: u_base + 1/(2 nb)).  Outputs spacing bins, euclidean bins [N,S_out+1]
 *      and the int64 searchsorted(side="right") indices (bit-exact target). ------------------------- */
int kp_pdf_resample(const float* weights, const float* existing_bins, int S_in, const float* u_base,
                    const float* rand, int rand_stride, const float* nears, const float* fars, int64_t N,
                    int S_out, float histogram_padding, float eps, int spacing, float* cdf_out /* [N,S_in+1] or NULL */,
                    float* spacing_bins, float* euclid_bins, int64_t* inds /* [N,S_out+1] or NULL */,
                    const float* anneal_dev /* DEVICE scalar or NULL */, float anneal_host /* used if anneal_dev NULL:
                    weights are raised to this power first, ray_samplers.py:584 */,
                    float* starts, float* ends, float* deltas /* [N,S_out] each or NULL */, void* stream);

/* ---- (a10) RaySamples.get_weights, NS/cameras/rays.py:127-149: warp-per-ray transmittance scan ---- */
int kp_weights_fwd(const float* deltas, const float* densities, int64_t N, int S, float* weights, void* stream);
int kp_weights_bwd(const float* deltas, const float* densities, const float* grad_weights, int64_t N, int S,
                   float* grad_densities, void* stream);

/* ---- (a11,a12) renderers, NS/model_components/renderers.py:58-140, 197-223, 226-287, 290-362.
 *      One pass per ray: comp_rgb = sum w*rgb + bg*(1-sum w), accumulation = sum w,
 *      median_index = clamp(searchsorted(cumsum(w), 0.5, "left")), expected depth numerator/denominator.
 *      bg_mode: 0 tensor bg[N,3], 1 last_sample.  nan_to_num_rgb: eval-mode RGBRenderer (renderers.py:133). */
int kp_render_fwd(const float* weights, const float* rgb /* [N,S,3] or NULL */, const float* steps /* [N,S] or NULL */,
                  const float* bg /* [N,3] or NULL */, int bg_mode, int nan_to_num_rgb, int64_t N, int S,
                  float* comp_rgb /* [N,3] or NULL */, float* accumulation /* [N] or NULL */,
                  int64_t* median_index /* [N] or NULL */, float* expected_depth /* [N] or NULL (unclipped) */,
                  const float* starts, const float* ends /* [N,S], for median_depth */,
                  float* median_depth /* [N] or NULL: (starts+ends)/2 at the median index */, void* stream);
int kp_render_bwd(const float* weights, const float* rgb, const float* bg, int bg_mode, int64_t N, int S,
                  const float* grad_comp /* [N,3] or NULL */, const float* grad_acc /* [N] or NULL */,
                  float* grad_weights /* [N,S] */, float* grad_rgb /* [N,S,3] or NULL */, void* stream);

/* ---- (a14) mip-NeRF-360 losses, NS/model_components/losses.py:46-144 ------------------------------
 *      distortion: per-ray loss [N] (mean taken by caller) and grad wrt w.  interlevel: per-(ray,sample)
 *      loss [N,S] for one proposal level and grad wrt the proposal weights. */
int kp_distortion_fwd(const float* sdist /* [N,S+1] */, const float* w /* [N,S] */, int64_t N, int S,
                      float* loss_per_ray, void* stream);
int kp_distortion_bwd(const float* sdist, const float* w, const float* grad_per_ray, int64_t N, int S,
                      float* grad_w, void* stream);
int kp_interlevel_fwd(const float* c /* [N,S+1] */, const float* w /* [N,S] */, const float* cp /* [N,Sp+1] */,
                      const float* wp /* [N,Sp] */, int64_t N, int S, int Sp, float* loss /* [N,S] */, void* stream);
int kp_interlevel_bwd(const float* c, const float* w, const float* cp, const float* wp, const float* grad_loss /* [N,S] */,
                      int64_t N, int S, int Sp, float* grad_wp /* [N,Sp] */, void* stream);

/* ---- (a15) plane regularisers, losses.py:356-452, values AND gradients in ONE sweep per plane, one launch for a
 *      whole list of channel-last planes [H,W,C].  planes/grads: HOST arrays [P] of device pointers, hwc: HOST int32
 *      [P*3] = (H, W, C) per plane, terms: HOST uint32 [P] (bit i selects sums[p,i]).  For plane p:
 *        sums[p,0] = sum (t[h+1]-t[h])^2, sums[p,1] = sum (t[w+1]-t[w])^2, sums[p,2] = sum (second diff along H)^2,
 *        sums[p,3] = sum |1-t|
 *      (DEVICE double [P,4], ACCUMULATED; may be NULL), and grads[p] (may be NULL) = or += sum_i coef_dev[p,i] *
 *      d(sums[p,i])/d(plane), coef_dev DEVICE float [P,4] so that no host sync is needed.  coef_dev may be NULL only when
 *      every grads[p] is NULL (sums only).  With accumulate = 0 the sweep also stands in for the gradient buffer's
 *      memset: every element of grads[p] is written. */
int kp_plane_reg_fused(const float* const* planes, float* const* grads, const int32_t* hwc, const uint32_t* terms, int P,
                       const float* coef_dev /* [P,4], or NULL */, int accumulate, double* sums /* [P,4] accumulated, or NULL */,
                       void* stream);
/* Same; write_range_dev (DEVICE int64 [P,2], or NULL = everything): the gradient of plane p is written only for its float4
 * elements [begin, end) -- sums still cover the whole plane.  Used by the data-parallel step with the sparse gradient
 * exchange, where every rank contributes the regularisers' gradient for its own shard of the bucket only. */
int kp_plane_reg_fused_range(const float* const* planes, float* const* grads, const int32_t* hwc, const uint32_t* terms, int P,
                             const float* coef_dev, int accumulate, double* sums, const int64_t* write_range_dev, void* stream);
/* Shard form of the same sweep: the SUMS are restricted to [begin, end) as well (every term is counted where its centre
 * element lives), and tiles without an element of the range are skipped -- a rank reads only its shard of the planes
 * (+ halo).  The per-rank sums of a partition of the plane add up to kp_plane_reg_fused's.  Replaces, per rank, 1/world of
 * the regulariser evaluation every DDP replica of the reference repeats in full (NS/models/kplanes.py:430-446). */
int kp_plane_reg_fused_shard(const float* const* planes, float* const* grads, const int32_t* hwc, const uint32_t* terms, int P,
                             const float* coef_dev, int accumulate, double* sums, const int64_t* write_range_dev, void* stream);

/* Adam over a list of dense fp32 tensors in one launch.  hyper_dev (optional, DEVICE float[3] = lr/bias_corr1,
 * 1/sqrt(bias_corr2), grad_scale) overrides the host-computed scalars so a captured CUDA graph can be replayed
 * with fresh per-step values. */
int kp_adam_multi(float* const* params, const float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
                  const int64_t* sizes, int P, float lr, float beta1, float beta2, float eps, float weight_decay,
                  int64_t step, float grad_scale, const float* hyper_dev, void* stream);

/* (f1) Regulariser stencil + Adam in ONE streaming pass per plane (NS/engine/optimizers.py:74-160 applied to
 * NS/model_components/losses.py:356-452 + the data gradient): per element reads plane, grad, exp_avg, exp_avg_sq once and
 * writes plane, exp_avg, exp_avg_sq (and grad = 0 when zero_grads).  Total gradient = grads[p] * grad_scale +
 * sum_i coef_dev[p,i] * d(sums[p,i])/d(plane), the regulariser part computed from the PRE-update plane values and never
 * materialised; sums (may be NULL) accumulates the regulariser sums of the pre-update planes as kp_plane_reg_fused does.
 * hwc = (H, W, C) per plane, C in {4, 8, 16, 32} (kp_plane_reg_adam_supported); all four tensors of a plane share the
 * channel-last layout.  scratch: device buffer of >= kp_plane_reg_adam_scratch_bytes(hwc, P) bytes (halo snapshot of the
 * tiles: neighbours are read from it so that in-place updates of adjacent tiles cannot be observed).  step is 1-based;
 * hyper_dev as in kp_adam_multi. */
int kp_plane_reg_adam_supported(int C);
int64_t kp_plane_reg_adam_scratch_bytes(const int32_t* hwc /* host [P,3] */, int P);
int kp_plane_reg_adam(float* const* planes, float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
                      const int32_t* hwc /* host [P,3] */, const uint32_t* terms /* host [P] */, int P,
                      const float* coef_dev /* [P,4] */, float lr, float beta1, float beta2, float eps, float weight_decay,
                      int64_t step, float grad_scale, const float* hyper_dev, double* sums /* [P,4] accumulated, or NULL */,
                      void* scratch, int64_t scratch_bytes, int zero_grads, void* stream);

/* Per-step scalars of a CUDA-graph-replayed step, computed on the device from *step_counter (then incremented):
 * anneal_out = anneal_table[min(step, max_steps)] (proposal-weight anneal, NS/models/kplanes.py:326-331) and, per
 * optimizer group g, hyper_out[g] = (lr_table[..] / (1 - beta1^t), 1 / sqrt(1 - beta2^t), grad_scale) with t = step + 1
 * -- the hyper_dev triple kp_adam_multi reads.  betas_host: HOST float[2*n_groups]; hyper_out_host: HOST array of DEVICE
 * float[3] pointers; n_groups <= 4. */
int kp_step_scalars(int64_t* step_counter, const double* lr_table, const float* anneal_table, int64_t max_steps, int n_groups,
                    const float* betas_host, float grad_scale, float* anneal_out /* device, or NULL */,
                    float* const* hyper_out_host, void* stream);

/* Repack between the reference's NCHW [1,C,H,W] checkpoint layout and channel-last [H,W,C]. */
int kp_repack_nchw_to_hwc(const float* src, float* dst, int C, int H, int W, void* stream);
int kp_repack_hwc_to_nchw(const float* src, float* dst, int C, int H, int W, void* stream);

/* ---- (f2) pixel -> ray generation: Cameras._generate_rays_from_coords, NS/cameras/cameras.py:505-741,
 *      as driven by RayGenerator.forward (NS/model_components/ray_generators.py:43-59) when
 *      ray_indices [N,3] = (camera,row,col) is given, or by Cameras.generate_rays(camera_indices=cam) for the
 *      row-major pixel range [first_pixel, first_pixel+N) of camera `cam` (image width `width`) when it is NULL.
 *      pixel_offset is get_image_coords' 0.5.  Outputs as in the reference's RayBundle: origins/directions [N,3],
 *      pixel_area [N], directions_norm [N] (metadata), times [N] (cameras.times[cam]).
 *      distortion (ABI 4): OpenCV k1,k2,k3,k4,p1,p2 per camera, undone by radial_and_tangential_undistort's 10 Newton
 *      iterations (NS/cameras/camera_utils.py:298-401) for every non-equirectangular camera (cameras.py:635-654); NULL =
 *      none.  cam_types (ABI 4): CameraType values per camera, 1 perspective / 2 fisheye / 3 equirectangular
 *      (cameras.py:42-47, direction models :665-697); NULL = all perspective.  Both NULL: the undistorted perspective
 *      kernel. ---- */
int kp_generate_rays(const float* c2w /* [n_cams,3,4] */, const float* intrinsics /* [n_cams,4] fx,fy,cx,cy */,
                     const float* cam_times /* [n_cams] or NULL */, const float* distortion /* [n_cams,6] or NULL */,
                     const int32_t* cam_types /* [n_cams] or NULL */, int n_cams, const int64_t* ray_indices /* or NULL */,
                     int cam, int width, int64_t first_pixel, int64_t N, float pixel_offset, float* origins,
                     float* directions, float* pixel_area, float* directions_norm /* or NULL */, float* times /* or NULL */,
                     void* stream);

/* ---- (f4) IST importance map: DynamicDataset.compute_ist, NS/data/datasets/dynamic_dataset.py:328-470.
 *      images [B,H*W,3] fp32; nbr_offsets [B+1] / nbrs: DEVICE int32 CSR lists of each image's temporal neighbours
 *      (same camera, 0.01 < |dt| <= ist_range, built by the host); out [B,H*W] fp16: mean over channels of the max abs
 *      difference to the neighbours, <= alpha zeroed; ones for an image without neighbours. ---- */
int kp_ist_map(const float* images, int B, int64_t HW, const int32_t* nbr_offsets, const int32_t* nbrs, float alpha,
               void* out_fp16, void* stream);
/* ISG map of DynamicDataset.compute_isg (NS/data/datasets/dynamic_dataset.py:215-326) on device images [B,H,W,3] fp32:
 * per camera the per-pixel, per-channel lower median over its frames (cam_offsets int32 [n_cams+1] / cam_images int32:
 * CSR lists of image indices per camera; at most 256 frames per camera), then per image (image_cam int32 [B] = its
 * camera slot) the Geman-McClure residual (1/3) * sum_c d_c^2 / (d_c^2 + gamma_sq), fp16 [B,H,W].  median_scratch: device
 * float [n_cams, H*W, 3].  Bit-identical to the reference's torch ops. */
int kp_isg_map(const float* images, int B, int64_t HW, const int32_t* cam_offsets, const int32_t* cam_images,
               const int32_t* image_cam, int n_cams, int max_frames_per_cam, float gamma_sq, float* median_scratch,
               void* out_fp16, void* stream);

/* ---- (f4) importance pixel sampling: the per-image torch.multinomial calls of DynamicBasedPixelSampler.sample_method
 *      (NS/data/pixel_samplers.py:340-426) for all images of a step at once.  weights_fp16 [B,HW]: the IST / ISG maps
 *      (device).  sel: DEVICE int32 [n_sel,3] = (image, k, first output row) per visited image, as the reference's loop
 *      assigns them (the host walks the shuffled image order and skips all-zero maps, :381-393); k <= k_max.  For each
 *      entry k pixels are drawn proportionally to the image's weights -- without replacement if the map has >= k non-zero
 *      pixels, else with replacement (:396-398) -- and written as int64 (image, row, col) triplets to rows
 *      [first, first + k) of out, without replacement in decreasing order of the race key (torch.multinomial's order).
 *      Exponential race on Philox4x32-10 keyed by `seed` (csrc/pixel_sampler_math.cuh): the reference's DISTRIBUTION, not
 *      its random stream.  An entry whose map is all zero gets rows of -1 (the reference's loop skips such images; so
 *      does the host side here).  scratch: kp_importance_pixels_scratch_bytes(n_sel, k_max) device bytes.  6 launches + 1 memset,
 *      no host synchronisation. ---- */
int64_t kp_importance_pixels_scratch_bytes(int n_sel, int k_max);
int kp_importance_pixels(const void* weights_fp16, int B, int64_t HW, int width, const int32_t* sel, int n_sel, int k_max,
                         uint64_t seed, void* scratch, int64_t* out, void* stream);

/* ---- (a14b) loss head: the reductions, coefficients, total and PSNR that KPlanesModel.get_loss_dict /
 *      get_metrics_dict (NS/models/kplanes.py:392-452) and the trainer's sum(loss_dict.values())
 *      (NS/engine/trainer.py:398-400) apply to the per-ray / per-sample loss kernels' outputs, one launch per
 *      direction.  vals3 = (coef_rgb * mse, coef_dist * mean(dist_per_ray), coef_il * sum_l mean(il_l));
 *      total = vals3[0..2] + sum(extra) (extra: already scaled terms, e.g. the plane regularisers);
 *      psnr = -10 log10(mse).  workspace4: 4 doubles, zero before the FIRST call (the kernel re-zeroes it). ---- */
#define KP_LOSS_HEAD_MAX_LEVELS 4
int kp_loss_head_fwd(const float* pred /* [N,3] */, const float* image /* [N,3] */, int64_t N,
                     const float* dist_per_ray /* [N] or NULL */, const float* const* il_ptrs /* HOST array [n_levels] */,
                     const int64_t* il_counts /* HOST: elements per level */, int n_levels, float coef_rgb, float coef_dist,
                     float coef_il, const float* extra /* device [n_extra] or NULL */, int n_extra, double* workspace4,
                     float* vals3, float* total, float* psnr, void* stream);
int kp_loss_head_bwd(const float* pred, const float* image, int64_t N, const int64_t* il_counts, int n_levels,
                     float coef_rgb, float coef_dist, float coef_il, const float* grad_total /* device scalar or NULL */,
                     const float* grad_vals3 /* device [3] or NULL */, float* grad_pred /* [N,3] or NULL */,
                     float* grad_dist /* [N] or NULL */, float* const* grad_il_ptrs /* HOST array [n_levels] or NULL */,
                     void* stream);

/* ---- eval-image metrics: per image of a batch the PSNR (data_range 1) and SSIM (11x11 gaussian window, sigma 1.5,
 *      k1 0.01, k2 0.03, data_range = max(range(pred), range(target)) of the image) that utils/image_metrics.py computes
 *      one image at a time (NS/models/kplanes.py:454-515).  pred, target: fp32 [B,H,W,3]; out: fp32 [B,2] = (psnr, ssim).
 *      The SSIM mean runs over the (H-10)*(W-10)*3 windows lying wholly inside the image (exactly what image_metrics.ssim
 *      keeps after its reflect-pad + crop); H or W < 11 is an error.  scratch: kp_image_metrics_scratch_bytes(B, H, W)
 *      device bytes, 16-byte aligned.  3 launches, no host synchronisation, no float atomics (bitwise reproducible),
 *      graph-capturable. ---- */
int64_t kp_image_metrics_scratch_bytes(int B, int H, int W);
int kp_image_metrics(const float* pred, const float* target, int B, int H, int W, void* scratch, float* out, void* stream);
/* The same metrics split by a region mask: mask uint8 [B,H,W], non-zero = the dynamic region; out fp32 [B,4] =
 * (psnr_dynamic, ssim_dynamic, psnr_static, ssim_static), the static region being the complement of the mask.  PSNR of
 * a region R: 10 log10(1 / mse_R), mse_R = the squared error summed (in double) over R's pixels and channels / (3 |R|).
 * SSIM of R: the mean of kp_image_metrics' SSIM map over the interior windows whose centre pixel (y+5, x+5) lies in R,
 * all 3 channels, with C1 / C2 from the whole image's data range.  A region without a pixel gets NaN for both, one
 * without a window centre NaN for its SSIM.  An all-true (all-false) mask gives the dynamic (static) pair bit for bit
 * equal to kp_image_metrics.  scratch: kp_image_metrics_masked_scratch_bytes(B, H, W) device bytes, 16-byte aligned.
 * 3 launches, no host synchronisation, no float atomics, graph-capturable. */
int64_t kp_image_metrics_masked_scratch_bytes(int B, int H, int W);
int kp_image_metrics_masked(const float* pred, const float* target, const uint8_t* mask, int B, int H, int W, void* scratch,
                            float* out, void* stream);

/* ---- eval depth metrics: rendered depth against ground-truth depth, per image and region.  pred, gt: fp32 [B,H,W]
 *      (HW = H*W pixels per image); dir_norm: fp32 [B,H,W] or NULL; mask: uint8 [B,H,W] or NULL, non-zero = dynamic.
 *      Ground truth g = __fmul_rn(gt, dir_norm) in fp32 when dir_norm is given (z-depth -> distance along the unit ray,
 *      as depth_loss and get_image_metrics_and_images do for is_euclidean_depth=False), else g = gt.  A pixel is valid
 *      when g is finite and g > 0 (0 / inf: sky and background).  In double: p = max(pred, 1e-6) (a NaN pred stays NaN),
 *      e = p - g; over the valid pixels of a region, with n_valid of them:
 *        abs_rel = mean |e| / g,  sq_rel = mean e^2 / g,  rmse = sqrt(mean e^2),  rmse_log = sqrt(mean (log p - log g)^2),
 *        delta_k = the share with max(p / g, g / p) < 1.25^k, k = 1, 2, 3 (1.25, 1.5625, 1.953125: exact in binary).
 *      out: double [B,R,8], row = (n_valid, abs_rel, sq_rel, rmse, rmse_log, delta1, delta2, delta3); n_valid = 0 gives
 *      NaN for the other seven.  R = 1 (the whole image) without a mask, R = 3 (whole, dynamic, static = the complement)
 *      with one.  Every region adds its pixels in the unmasked pass's order, so an all-true (all-false) mask gives the
 *      dynamic (static) row bit for bit equal to the whole row and to the unmasked call.  Counts are integers, sums
 *      doubles.  scratch: kp_depth_metrics_scratch_bytes(B, HW, mask != NULL) device bytes, 8-byte aligned.  2 launches,
 *      no host synchronisation, no float atomics (bitwise reproducible), graph-capturable. ---- */
int64_t kp_depth_metrics_scratch_bytes(int B, int64_t HW, int masked);
int kp_depth_metrics(const float* pred, const float* gt, const float* dir_norm, const uint8_t* mask, int B, int64_t HW,
                     void* scratch, double* out, void* stream);

/* ---- eval error maps: per pixel the quantities kp_image_metrics and kp_depth_metrics average, for viewing.  pred, gt:
 *      fp32 [B,H,W,3], H and W >= 11; outputs fp32 [B,H,W]:
 *        err       = (|pred_0 - gt_0| + |pred_1 - gt_1| + |pred_2 - gt_2|) / 3;
 *        ssim      = at 5 <= y < H-5, 5 <= x < W-5 the channel mean of the SSIM of the window centred on (y, x), with
 *                    kp_image_metrics' window, constants and per-image data_range (each channel's value is the one
 *                    kp_image_metrics adds to its mean); NaN on the 5-pixel border, where no window lies inside;
 *        depth_err = |max(depth, 1e-6) - g| / g in double, rounded to fp32, g = __fmul_rn(gt_depth, dir_norm) or gt_depth,
 *                    NaN where g is not finite or not > 0 (kp_depth_metrics' clamp, product and validity rule).
 *      depth, gt_depth: fp32 [B,H,W], given together with depth_err or all three NULL; dir_norm: fp32 [B,H,W] or NULL.
 *      scratch: kp_eval_maps_scratch_bytes(B, H, W) device bytes, 16-byte aligned.  2 launches, no host
 *      synchronisation, no atomics (bitwise reproducible), graph-capturable. ---- */
int64_t kp_eval_maps_scratch_bytes(int B, int H, int W);
int kp_eval_maps(const float* pred, const float* gt, const float* depth, const float* gt_depth, const float* dir_norm, int B,
                 int H, int W, void* scratch, float* err, float* ssim, float* depth_err, void* stream);

/* ---- frame composition for a rendered camera path (the per-frame image work of ns-render, REF/nerfstudio/scripts/
 *      render.py: colour-map every requested output and concatenate them along the width): P <= KP_COMPOSE_MAX_PANELS
 *      panels of one frame -> out uint8 [H, W*P, 3], panel p in columns [p*W, (p+1)*W).  panels: HOST array [P] of fp32
 *      device pointers, [H,W,3] for KP_PANEL_COLOR, [H,W,1] otherwise; kinds: HOST array [P].  The mapping is that of
 *      KPlanesModel.get_image_metrics_and_images (utils/colormaps.py): colour as is; accumulation -> viridis[(int64)(a*255)];
 *      depth -> turbo[(int64)(d'*255)] * acc + (1 - acc), d' = clip((d - min) * rn(1/den), 0, 1), den =
 *      fp32(double(max) - double(min) + 1e-10), min / max over the frame's panel; accumulation: fp32 [H,W,1], needed with a
 *      depth panel.  turbo, viridis: fp32 [256,3] device tables (utils/colormaps._table); a colour-map index outside
 *      [0, 255] is clamped.  Every channel is quantised as floor(clamp(x, 0, 1) * 255 + 0.5), NaN -> 0.  Bit-identical to
 *      that torch restatement on the device.  scratch: kp_compose_frame_scratch_bytes(H, W, P) device bytes, 8-byte
 *      aligned.  1 launch (2 with a depth panel), no host synchronisation, graph-capturable. ---- */
#define KP_COMPOSE_MAX_PANELS 8
#define KP_PANEL_COLOR 0
#define KP_PANEL_ACCUMULATION 1
#define KP_PANEL_DEPTH 2
int64_t kp_compose_frame_scratch_bytes(int H, int W, int P);
int kp_compose_frame(const float* const* panels, const int* kinds, int P, int H, int W, const float* accumulation,
                     const float* turbo, const float* viridis, void* scratch, uint8_t* out, void* stream);
/* Same, each depth panel blended with its own accumulation: accumulations is a HOST array [P] of device pointers, entry p
 * read only when kinds[p] is KP_PANEL_DEPTH (e.g. depth_static with accumulation_static beside depth with accumulation).
 * kp_compose_frame is this call with its accumulation in every entry. */
int kp_compose_frame_accs(const float* const* panels, const int* kinds, const float* const* accumulations, int P, int H,
                          int W, const float* turbo, const float* viridis, void* scratch, uint8_t* out, void* stream);

/* ---- baseline JPEG encoding of a composed frame (the image files and Motion-JPEG video of a rendered camera path):
 *      image uint8 [H, W, 3] RGB, 1 <= H, W <= 65535 -> out: one baseline JFIF file (SOF0, YCbCr 4:2:0, the Annex K.1
 *      quantisation tables at the IJG quality scaling, the Annex K.3 Huffman tables, RSTm every KP_JPEG_RESTART_MCUS
 *      MCUs), SOI ... EOI, and *length = its byte count (int64, device).  header: the KP_JPEG_HEADER_BYTES bytes
 *      kp_jpeg_header(H, W, quality) writes (on the HOST; the caller copies them to the device once per key), SOI to SOS;
 *      the kernel quantises with the header's DQT tables.  out: kp_jpeg_encode_capacity(H, W) device bytes, the worst
 *      case (bytes past *length are not written).  scratch: kp_jpeg_encode_scratch_bytes(H, W) device bytes, 256-byte
 *      aligned.  Colour conversion, edge padding and chroma downsampling are libjpeg's integer formulas; the DCT is fp32.
 *      3 launches, no host synchronisation, graph-capturable. ---- */
#define KP_JPEG_RESTART_MCUS 4
#define KP_JPEG_HEADER_BYTES 613
int64_t kp_jpeg_encode_capacity(int H, int W);
int64_t kp_jpeg_encode_scratch_bytes(int H, int W);
int kp_jpeg_header(int H, int W, int quality, uint8_t* header);
int kp_jpeg_encode(const uint8_t* image, int H, int W, const uint8_t* header, void* scratch, uint8_t* out, int64_t* length,
                   void* stream);

/* ---- (e) data-parallel gradient all-reduce over NVLink peer memory (replaces the NCCL all-reduce torch DDP issues
 *      around NS/engine/trainer.py:382-412).  Every rank allocates one ARENA = [KP_PEER_SIGNAL_BYTES of flag words |
 *      data], exports its CUDA-IPC handle, and opens the arenas of the other ranks of the node.  kp_peer_allreduce
 *      sums floats [begin, begin+count) of the data regions of all ranks IN PLACE (every rank ends with the same,
 *      bit-identical sums; addition order is rank 0..N-1).  It must be enqueued by every rank, with the same
 *      (begin, count, blocks), in the same order; cross-GPU synchronisation is inside the kernel, which is
 *      CUDA-graph capturable. ---- */
#define KP_PEER_MAX_WORLD 8
#define KP_PEER_MAX_BLOCKS 160
#define KP_PEER_SIGNAL_BYTES 16384
int kp_peer_alloc(int64_t data_bytes, void** arena, void* ipc_handle64 /* out: 64-byte cudaIpcMemHandle_t */);
int kp_peer_open(const void* ipc_handle64, void** arena /* out: this process' mapping of a peer's arena */);
int kp_peer_close(void* arena /* from kp_peer_open */);
int kp_peer_free(void* arena /* from kp_peer_alloc */);
int kp_peer_error(const void* own_arena, uint32_t* error_word /* host; non-zero: a cross-GPU barrier timed out */);
int kp_peer_allreduce(void* const* arenas /* HOST array [world]: arenas[rank] = own, others = opened */, int rank,
                      int world, int64_t begin /* float index, multiple of 4 */, int64_t count, int blocks /* <=0: 64 */,
                      void* stream);

/* Sharded optimizer step fused with its collectives (reduce-scatter -> Adam -> all-gather in one kernel per rank):
 * gradients at float offset grad_begin and parameters at param_begin of every arena's data region, `count` floats
 * (multiples of 4).  Rank r owns floats [count*r/world, count*(r+1)/world) (at float4 granularity): it sums the world's
 * gradients for them, updates ITS moments (exp_avg_shard / exp_avg_sq_shard, local buffers covering only the shard) with
 * torch.optim.Adam's rule (grad_scale, e.g. 1/world, applied to the sum) and writes the new parameters into every
 * rank's arena.  Same calling discipline as kp_peer_allreduce.  hyper_dev as in kp_adam_multi. */
int kp_peer_sharded_adam(void* const* arenas, int rank, int world, int64_t grad_begin, int64_t param_begin, int64_t count,
                         float* exp_avg_shard, float* exp_avg_sq_shard, float lr, float beta1, float beta2, float eps,
                         float weight_decay, int64_t step, float grad_scale, const float* hyper_dev, int blocks, void* stream);
/* Sparse variant for HBM-resident plane groups: touched_begin (float offset in the data region, like grad_begin) locates
 * one byte per 128-byte line of the gradient region in every arena: 0 = line is all zeros (not read over NVLink), 1 =
 * reduced into this step (kp_hexplane_bwd_flags), 2 = always dense.  The owner reads its own shard's lines unconditionally
 * and, after the end barrier, every rank zeroes its marked lines outside its shard and clears their marks (the bucket needs
 * no memset).  grad_begin and count must be multiples of 32 floats. */
int kp_peer_sharded_adam_sparse(void* const* arenas, int rank, int world, int64_t grad_begin, int64_t param_begin,
                                int64_t touched_begin, int64_t count, float* exp_avg_shard, float* exp_avg_sq_shard, float lr,
                                float beta1, float beta2, float eps, float weight_decay, int64_t step, float grad_scale,
                                const float* hyper_dev, int blocks, void* stream);

/* ---- (d) measurement: memory-hierarchy probe with the field kernels' own access pattern (8 lanes = one 128-byte
 *      line of a pseudo-random texel; mode 0: 16-byte read-only loads, mode 1: red.global.add.v4.f32).  One launch
 *      touches blocks*32*iters lines of buf[0 : n_lines*32] (iters rounded up to a multiple of 8); bench.py times it
 *      over an L2-resident and an HBM-resident buffer to get the achievable L2 / random-line HBM rates the gather
 *      and the scatter are reported against (SURVEY.md 8d). ---- */
int kp_line_probe(float* buf, int64_t n_lines, int mode, int blocks, int iters, uint32_t seed, float* sink /* device [1] */,
                  int64_t* lines_touched /* host, or NULL */, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KPLANES_B200_H_ */
