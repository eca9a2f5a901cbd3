"""float64 reference of the hexplane gather / scatter and the fused proposal density field, with element-wise fp32 error bounds.

The kernels (soccernerfs_b200/csrc/hexplane.cu) are checked element by element rather than per tensor: every output is
compared with this reference against a bound gamma * u * A, where A is the same function evaluated on |planes|, |grad|,
|weights| (bilinear weights are >= 0, so A bounds the magnitude of every term that was rounded) and gamma counts the
roundings on the longest path from an input to that output.  Constants are derived from the kernels' operation order next
to where they are defined; they are upper bounds, not tuned.

Coordinates are computed in fp32 exactly as ``load_point`` / ``axis_setup`` compute them (separate fp32 ops, each rounded
once), so the floor decisions and the zero corner weights are the kernel's own.  Everything after the axis set-up is
float64.  All functions run on whichever device their inputs live on.
"""
from __future__ import annotations

import itertools
from typing import Sequence

import torch

U = 2.0 ** -24  # unit round-off of fp32 (round to nearest)


def gamma(n) -> float:
    """Classic gamma_n = n u / (1 - n u): bounds the relative error of n roundings, second-order terms included."""
    return n * U / (1.0 - n * U)


# ---- per-operation rounding counts (first-order, relative to the magnitude A of the result) -------------------------------
# bilerp_combine: r = v00*w00, then three fma: the first term passes 1 mul + 3 fma; its corner weight w00 = wx0*wy0 is one
# more fp32 product.  Each bilinear interpolant is therefore within 5u of sum_c |v_c| w_c.
BILERP = 5
# Gather of one scale: acc = 1, acc *= interp_p for every active plane (the first multiply by 1 is exact: NP-1 roundings),
# each factor carrying BILERP.  |prod(x_p + e_p) - prod(x_p)| <= NP * 5u * prod(a_p) to first order.
def gamma_gather(n_planes: int, n_scales: int, concat: bool) -> int:
    g = BILERP * n_planes + (n_planes - 1)
    # sum mode: total = 0; total += acc_k (the first add is exact): n_scales - 1 more roundings of terms bounded by sum A_k
    return g if concat else g + n_scales - 1


# Scatter of one (sample, plane, corner): others = pre[p] * suf[p] (prefix / suffix products: NP-2 roundings plus the
# product of the two: NP-1), g * others (1), * corner weight (1), and the fp32 corner weight itself (1): NP+2 roundings,
# plus BILERP on each of the NP-1 other interpolants.  The n reductions into a texel (onto its prior value) add n more
# roundings on the longest path of any summation order -- added per texel by the caller.
def gamma_scatter(n_planes: int) -> int:
    return BILERP * (n_planes - 1) + n_planes + 2


# Density features f_c = prod_p interp_p (NP-1 FMUL2 from 1, plus BILERP per plane); pre_j = fma chain over C channels from 0
# (C roundings); raw = fma chain over H units from 0 (H roundings).  ReLU is 1-Lipschitz and adds nothing.  So
# |raw32 - raw| <= gamma(H + C + 6NP - 1) * R with R = sum_j |w2_j| sum_c |w1_jc| prod_p a_pc.
def gamma_density_raw(n_planes: int, c: int, hidden: int) -> int:
    return hidden + c + gamma_gather(n_planes, 1, True)


# expf is within 2 ulp (CUDA C Programming Guide, single-precision functions), and 1 ulp <= 2u relative: 4u.
EXPF = 4


# Density backward, per (sample, output) term relative to its magnitude, on top of the raw error e_raw (which enters through
# exp: e^(raw + e) = e^raw (1 + e + ...)):  graw = g * expf(.) (EXPF + 1), dpre = graw * w2 (1), df_c = fma chain over H
# units (H), * the NP-1 other interpolants (NP-1 roundings + BILERP each), * corner weight (1) and its rounding (1).
def gamma_density_plane(n_planes: int, hidden: int) -> int:
    return EXPF + 1 + 1 + hidden + (n_planes - 1) * (1 + BILERP) + 2


# grad_w2_j term graw * h_j: graw (EXPF + 1) and h_j = relu(pre_j) (C + 6NP - 1 relative to sum_c |w1_jc| F_c).
# grad_w1_jc term dpre_j * f_c: dpre (EXPF + 2) and f_c (6NP - 1).  The larger of the two covers both.
def gamma_density_weights(n_planes: int, c: int) -> int:
    return EXPF + 2 + c + gamma_gather(n_planes, 1, True)


# ---- coordinates ---------------------------------------------------------------------------------------------------------
def _f32(x, like: torch.Tensor) -> torch.Tensor:
    return torch.as_tensor(x, dtype=torch.float32, device=like.device)


def coords(P) -> torch.Tensor:
    """fp32 [M,4] sample coordinates of an ``ops.Points``-like object, op for op as ``load_point`` (missing axes = 0)."""
    if P.pts is not None:
        pts = P.pts.float().reshape(-1, P.D)
        out = torch.zeros(pts.shape[0], 4, dtype=torch.float32, device=pts.device)
        out[:, : P.D] = pts
        return out
    o, d = P.origins.float().reshape(-1, 3), P.directions.float().reshape(-1, 3)
    t = (P.starts.float().reshape(-1) + P.ends.float().reshape(-1))[:, None]  # one fp32 add
    n = torch.arange(t.shape[0], device=o.device) // P.S
    pos = o[n] + (d[n] * t) * 0.5  # (d*t)*0.5 then + o: three roundings, each a separate op
    out = torch.zeros(t.shape[0], 4, dtype=torch.float32, device=o.device)
    if P.norm_mode == 2:
        # SceneContraction(order=inf), then halved: x if |x|_inf < 1 else (2 - 1/|x|)(x/|x|)
        mag = pos.abs().amax(dim=1, keepdim=True)
        k = 2.0 - torch.div(torch.ones_like(mag), mag)
        out[:, :3] = torch.where(mag < 1.0, pos, k * torch.div(pos, mag)) * 0.5
    else:
        lo = _f32(P.aabb[:3], o)
        q = torch.div(pos - lo, _f32(P.aabb[3:], o) - lo)
        out[:, :3] = q * 2.0 - 1.0 if P.norm_mode else q
    if P.D == 4 and P.times is not None:
        out[:, 3] = (P.times.float().reshape(-1)[n] * 2.0) - 1.0
    return out


def axis(x: torch.Tensor, R: int):
    """``axis_setup`` in fp32: -> (i0, i1) int64, (w0, w1) fp32.  The corner i1 == R is replaced by i1 = R-1, w1 = 0."""
    ix = ((x + 1.0) * 0.5) * float(R - 1)
    ix = ix.clamp(0.0, float(R - 1))
    fx = torch.floor(ix)
    w1, w0 = ix - fx, (fx + 1.0) - ix
    i0 = fx.long()
    i1 = i0 + 1
    over = i1 > R - 1
    return i0, torch.where(over, torch.full_like(i1, R - 1), i1), w0, torch.where(over, torch.zeros_like(w1), w1)


# ---- field layout ---------------------------------------------------------------------------------------------------------
def plane_axes(n_planes: int):
    """(ca, cb) of each plane: combinations(range(D), 2); coordinate ca indexes W, cb indexes H."""
    return list(itertools.combinations(range(3 if n_planes == 3 else 4), 2))


def texels(plane: torch.Tensor, dtype=torch.float64) -> torch.Tensor:
    """[1,C,H,W] (any memory format) -> [H*W, C] in texel order y*W + x."""
    return plane[0].permute(1, 2, 0).reshape(-1, plane.shape[1]).to(dtype)


def corners(pt: torch.Tensor, planes: Sequence[torch.Tensor], dtype=torch.float64):
    """Per plane of one scale: (idx [M,4] texel indices, w [M,4] corner weights) in corner order 00, 01, 10, 11 (y, x).
    The corner weight is the product of the fp32 axis weights, exact in float64.  Axis weights are 0 or >= 2^-25, so their
    fp32 product never underflows: w != 0 here exactly where the kernel's fp32 weight is != 0."""
    reso = [1, 1, 1, 1]
    for (a, b), p in zip(plane_axes(len(planes)), planes):
        reso[a], reso[b] = p.shape[3], p.shape[2]
    ax = [axis(pt[:, d], reso[d]) for d in range(4)]
    out = []
    for (a, b), p in zip(plane_axes(len(planes)), planes):
        W = p.shape[3]
        x0, x1, wx0, wx1 = ax[a]
        y0, y1, wy0, wy1 = ax[b]
        idx = torch.stack([y0 * W + x0, y0 * W + x1, y1 * W + x0, y1 * W + x1], dim=1)
        wx0, wx1, wy0, wy1 = (v.to(dtype) for v in (wx0, wx1, wy0, wy1))
        out.append((idx, torch.stack([wx0 * wy0, wx1 * wy0, wx0 * wy1, wx1 * wy1], dim=1)))
    return out


def _interps(cs, planes, use_mask, absolute, dtype):
    """Per plane: bilinear interpolant [M,C] (None for a plane outside use_mask, whose factor is 1)."""
    out = []
    for p, ((idx, w), plane) in enumerate(zip(cs, planes)):
        if not (use_mask >> p) & 1:
            out.append(None)
            continue
        t = texels(plane, dtype)
        if absolute:
            t = t.abs()
        out.append(sum(w[:, j, None] * t[idx[:, j]] for j in range(4)))
    return out


def _product(vals, skip: int = -1):
    r = None
    for q, v in enumerate(vals):
        if v is not None and q != skip:
            r = v if r is None else r * v
    return r


# ---- gather / scatter -----------------------------------------------------------------------------------------------------
def gather(pt: torch.Tensor, ms_planes: Sequence[Sequence[torch.Tensor]], use_mask: int, concat: bool,
           absolute: bool = False, dtype=torch.float64) -> torch.Tensor:
    """Multiscale features: per scale the product of the active planes' interpolants; scales concatenated or summed."""
    per_scale = []
    for planes in ms_planes:
        c = planes[0].shape[1]
        r = _product(_interps(corners(pt, planes, dtype), planes, use_mask, absolute, dtype))
        per_scale.append(torch.ones(pt.shape[0], c, dtype=dtype, device=pt.device) if r is None else r)
    return torch.cat(per_scale, dim=1) if concat else sum(per_scale)


def scatter(pt: torch.Tensor, ms_planes: Sequence[Sequence[torch.Tensor]], use_mask: int, concat: bool, grad_out: torch.Tensor,
            need: Sequence[bool], absolute: bool = False, dtype=torch.float64):
    """Exact plane gradients of ``gather`` for upstream ``grad_out``: -> (grads, counts, touched), flat over scales x planes.
    grads[i]: [H*W, C] (None where need[i] is False), counts[i]: int64 [H*W] = number of (sample, corner) pairs with a
    non-zero weight that reduce into the texel, touched[i] = counts[i] > 0."""
    n_planes = len(ms_planes[0])
    grads, counts = [], []
    for k, planes in enumerate(ms_planes):
        c = planes[0].shape[1]
        g = grad_out[:, k * c:(k + 1) * c] if concat else grad_out
        g = g.to(dtype).abs() if absolute else g.to(dtype)
        cs = corners(pt, planes, dtype)
        vals = _interps(cs, planes, use_mask, absolute, dtype)
        for p, plane in enumerate(planes):
            i = k * n_planes + p
            if not (need[i] and (use_mask >> p) & 1):
                grads.append(None)
                counts.append(None)
                continue
            others = _product(vals, skip=p)
            gp = g if others is None else g * others
            out, n = _scatter_corners(cs[p], gp, plane, dtype)
            grads.append(out)
            counts.append(n)
    return grads, counts, [None if n is None else n > 0 for n in counts]


def _scatter_corners(cp, gp, plane, dtype):
    idx, w = cp
    hw = plane.shape[2] * plane.shape[3]
    out = torch.zeros(hw, plane.shape[1], dtype=dtype, device=gp.device)
    n = torch.zeros(hw, dtype=torch.int64, device=gp.device)
    for j in range(4):
        live = w[:, j] != 0
        out.index_add_(0, idx[live, j], w[live, j, None] * gp[live])
        n.index_add_(0, idx[live, j], torch.ones_like(idx[live, j]))
    return out, n


# ---- fused proposal density field -------------------------------------------------------------------------------------------
def density(pt: torch.Tensor, planes: Sequence[torch.Tensor], w1: torch.Tensor, w2: torch.Tensor, relu: bool, use_mask: int,
            absolute: bool = False, dtype=torch.float64):
    """-> (raw [M], pre [M,H]): raw = W2 act(W1 f), density = exp(raw).  ``absolute``: |planes|, |W1|, |W2|, no ReLU."""
    f = gather(pt, [planes], use_mask, True, absolute, dtype)
    w1, w2 = w1.to(dtype), w2.to(dtype).reshape(-1)
    if absolute:
        w1, w2 = w1.abs(), w2.abs()
    pre = f @ w1.t()
    h = torch.relu(pre) if relu and not absolute else pre
    return h @ w2, pre


def density_backward(pt: torch.Tensor, planes: Sequence[torch.Tensor], w1: torch.Tensor, w2: torch.Tensor, relu: bool,
                     use_mask: int, grad_density: torch.Tensor, need: Sequence[bool], absolute: bool = False,
                     dtype=torch.float64):
    """Gradients of sum(grad_density * trunc_exp(raw)): -> (plane grads [H*W,C] | None, counts, grad_w1 [H,C], grad_w2 [H]).
    trunc_exp's gradient is exp(clamp(raw, -15, 15)); ReLU's is 0 at pre <= 0.  ``absolute``: every factor replaced by its
    magnitude with the ReLU mask and exp(clamp(raw)) of the real evaluation, which gives the magnitude of each summed term."""
    raw, pre = density(pt, planes, w1, w2, relu, use_mask, False, dtype)
    act = (pre > 0).to(dtype) if relu else torch.ones_like(pre)
    g = grad_density.to(dtype)
    W1, W2 = w1.to(dtype), w2.to(dtype).reshape(-1)
    cs = corners(pt, planes, dtype)
    vals = _interps(cs, planes, use_mask, absolute, dtype)
    if absolute:  # |h_j| <= |pre_j| <= sum_c |w1_jc| F_c: the magnitude the pre-activation's error is relative to
        g, W1, W2 = g.abs(), W1.abs(), W2.abs()
        pre = density(pt, planes, w1, w2, relu, use_mask, True, dtype)[1]
    f = _product(vals)
    if f is None:
        f = torch.ones(pt.shape[0], planes[0].shape[1], dtype=dtype, device=pt.device)
    graw = g * torch.exp(raw.clamp(-15.0, 15.0))
    dpre = graw[:, None] * W2[None, :] * act
    gw2 = (graw[:, None] * pre * act).sum(0)
    gw1 = dpre.t() @ f
    df = dpre @ W1
    grads, counts = [], []
    for p, plane in enumerate(planes):
        if not (need[p] and (use_mask >> p) & 1):
            grads.append(None)
            counts.append(None)
            continue
        others = _product(vals, skip=p)
        out, n = _scatter_corners(cs[p], df if others is None else df * others, plane, dtype)
        grads.append(out)
        counts.append(n)
    return grads, counts, gw1, gw2


def relu_ties(pt: torch.Tensor, planes, w1, w2, use_mask: int, window: float = 2.0) -> torch.Tensor:
    """[M] bool: some hidden unit's float64 pre-activation lies within ``window`` times its fp32 error bound of 0, so the
    kernel's ReLU may take the other branch there (its gradient then differs by O(1), whatever the precision)."""
    _, pre = density(pt, planes, w1, w2, True, use_mask)
    _, mag = density(pt, planes, w1, w2, True, use_mask, absolute=True)
    n_planes, c = len(planes), planes[0].shape[1]
    bound = gamma(c + gamma_gather(n_planes, 1, True)) * mag
    return (pre.abs() <= window * bound).any(dim=1)


def ratio(err: torch.Tensor, bound: torch.Tensor) -> float:
    """max err / bound (0 where both are 0; inf where only the bound is 0)."""
    err, bound = err.double(), bound.double()
    r = torch.where(err == 0, torch.zeros_like(err), err / bound)
    return float(r.max()) if r.numel() else 0.0



# ---- element-wise checks (shared by the GPU tests and the bound's sensitivity tests) ---------------------------------------
def gather_ratio(out: torch.Tensor, pt, ms_planes, use_mask: int, concat: bool) -> float:
    """max over elements of |out - ref| / (gamma * A) for a gather result ``out``."""
    ref = gather(pt, ms_planes, use_mask, concat)
    bound = gamma(gamma_gather(len(ms_planes[0]), len(ms_planes), concat)) * gather(pt, ms_planes, use_mask, concat, True)
    return ratio((out.double() - ref).abs(), bound)


def scatter_ratio(got, prior, pt, ms_planes, use_mask: int, concat: bool, grad_out, need):
    """Scatter results ``got`` (per plane [H*W,C] or None) accumulated onto ``prior`` -> (worst err / bound, touched sets).
    Per texel the bound is gamma(gamma_scatter + n) * (|prior| + sum of the |terms|), n = the texel's reduction count."""
    ref, n, touched = scatter(pt, ms_planes, use_mask, concat, grad_out, need)
    mag, _, _ = scatter(pt, ms_planes, use_mask, concat, grad_out, need, True)
    gs, worst = gamma_scatter(len(ms_planes[0])), 0.0
    for i, r in enumerate(ref):
        if r is None:
            continue
        p0 = prior[i].double()
        bound = gamma(gs + n[i].double())[:, None] * (p0.abs() + mag[i])
        worst = max(worst, ratio((got[i].double() - (p0 + r)).abs(), bound))
    return worst, touched


def density_ratio(dens: torch.Tensor, pt, planes, w1, w2, relu: bool, use_mask: int) -> float:
    """|log(density) - raw| against gamma(H + C + 6NP - 1) R + gamma(EXPF)."""
    raw, _ = density(pt, planes, w1, w2, relu, use_mask)
    mag, _ = density(pt, planes, w1, w2, relu, use_mask, True)
    bound = gamma(gamma_density_raw(len(planes), planes[0].shape[1], w1.shape[0])) * mag + gamma(EXPF)
    return ratio((torch.log(dens.double()) - raw).abs(), bound)


def density_weight_sum_depth(M: int, sms: int) -> int:
    """Longest chain of fp32 additions into one weight gradient in ``density_field_bwd_kernel``: a lane fma-accumulates 32
    samples per grid-stride iteration (blocks = min(ceil(M/128), 4 SMs) of 128 threads), four warps meet in shared-memory
    atomics, then one red per block onto the prior value."""
    blocks = min(-(-M // 128), 4 * sms)
    iters = -(-(-(-M // 32) * 32) // (blocks * 128))
    return 32 * iters + 4 + blocks


def density_backward_ratios(got, prior, pt, planes, w1, w2, relu: bool, use_mask: int, grad_density, need, sms: int):
    """got / prior = (plane grads list, grad_w1 [H,C], grad_w2 [H]) after / before the backward -> {name: err / bound}.
    Per term the error is (e_raw + gamma) times its magnitude, with e_raw the sample's bound on |raw32 - raw| (it reaches
    every gradient through exp); the sums add gamma(depth) on |prior| + sum |terms| (depth: n per texel, the weight sums'
    chain otherwise)."""
    n_planes, c, hidden = len(planes), planes[0].shape[1], w1.shape[0]
    R, _ = density(pt, planes, w1, w2, relu, use_mask, True)
    e_raw = gamma(gamma_density_raw(n_planes, c, hidden)) * R
    ref = density_backward(pt, planes, w1, w2, relu, use_mask, grad_density, need)
    mag = density_backward(pt, planes, w1, w2, relu, use_mask, grad_density, need, True)
    coef = e_raw + gamma(max(gamma_density_plane(n_planes, hidden), gamma_density_weights(n_planes, c)))
    err = density_backward(pt, planes, w1, w2, relu, use_mask, grad_density.double().abs() * coef, need, True)
    out = {}
    for p in range(n_planes):
        if ref[0][p] is None:
            continue
        p0 = prior[0][p].double()
        bound = err[0][p] + gamma(ref[1][p].double())[:, None] * (p0.abs() + mag[0][p])
        out[f"plane{p}"] = ratio((got[0][p].double() - (p0 + ref[0][p])).abs(), bound)
    depth = density_weight_sum_depth(pt.shape[0], sms)
    for name, j in (("w1", 2), ("w2", 3)):
        p0 = prior[j - 1].double().reshape(ref[j].shape)
        bound = err[j] + gamma(depth) * (p0.abs() + mag[j])
        out[name] = ratio((got[j - 1].double().reshape(ref[j].shape) - (p0 + ref[j])).abs(), bound)
    return out
