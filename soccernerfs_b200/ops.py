"""torch.autograd.Function shims over the C-ABI kernels (one Function per fused op).

Planes keep the reference's logical shape ``[1, C, H, W]`` (state-dict compatible with
NS/fields/kplanes_field.py:67) but live in ``torch.channels_last`` memory, i.e. physically ``[H][W][C]`` --
the layout the gather/scatter kernels need for 16-byte feature loads.  All kernels run in fp32 on the
current CUDA stream; under ``torch.autocast`` inputs are promoted to fp32 exactly as the reference's
``_TruncExp`` does with ``custom_fwd(cast_inputs=torch.float32)`` (NS/field_components/activations.py:29).
"""
from __future__ import annotations

from ctypes import c_float, c_int32, c_int64, c_void_p
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import call, f32c, ptr, stream_ptr


# ------------------------------------------------------------------------------------------------
# plane layout helpers
# ------------------------------------------------------------------------------------------------
def new_plane(c: int, h: int, w: int, device=None) -> torch.Tensor:
    """Empty fp32 plane of logical shape [1,C,H,W], physical layout [H][W][C]."""
    return torch.empty((1, h, w, c), dtype=torch.float32, device=device).permute(0, 3, 1, 2)


def is_channel_last(p: torch.Tensor) -> bool:
    return p.dim() == 4 and p.shape[0] == 1 and p.permute(0, 2, 3, 1).is_contiguous()


def as_channel_last(p: torch.Tensor) -> torch.Tensor:
    """Return ``p`` (logical [1,C,H,W]) with physical [H][W][C] memory; copies only if it is not already."""
    if p.dtype != torch.float32:
        p = p.float()
    if is_channel_last(p):
        return p
    return p.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)


def _plane_ptrs(planes: Sequence[Optional[torch.Tensor]]):
    arr = (c_void_p * len(planes))()
    for i, p in enumerate(planes):
        arr[i] = 0 if p is None else p.data_ptr()
    return arr


def _plane_hw(planes: Sequence[torch.Tensor]):
    arr = (c_int32 * (2 * len(planes)))()
    for i, p in enumerate(planes):
        arr[2 * i], arr[2 * i + 1] = p.shape[2], p.shape[3]
    return arr


def grad_sink(p: torch.Tensor) -> Optional[torch.Tensor]:
    """Gradient-accumulation fusion: a parameter may carry ``_kp_grad_sink`` -- a persistent, caller-zeroed buffer
    with the parameter's layout (normally the tensor installed as ``p.grad``, see distributed.GradBucket).  Kernels
    then accumulate their gradient straight into it (all of them are red/+= kernels) and autograd receives ``None``
    for that input: no per-op gradient tensors, no zero fills and no autograd ``add`` passes over the planes."""
    sink = getattr(p, "_kp_grad_sink", None)  # (called inside Function.forward, where grad mode is always off)
    if sink is None or not p.requires_grad:
        return None
    # a sink is only honoured while it still IS the parameter's .grad: after someone else's zero_grad(set_to_none=True)
    # or a new .grad tensor (another trainer / a plain torch optimizer took over the model) autograd gets real gradients
    g = p.grad
    if g is None or g.data_ptr() != sink.data_ptr():
        return None
    return sink


def _targets(tensors, sinks, need):
    """Per input: the buffer a backward kernel accumulates into (the sink or a fresh zero tensor) and what is
    returned to autograd (None when sunk)."""
    fresh_need = [n and s is None for n, s in zip(need, sinks)]
    fresh = zeros_like_planes(tensors, fresh_need)
    targets = [s if (n and s is not None) else f for s, f, n in zip(sinks, fresh, need)]
    returned = [None if (s is not None) else f for s, f in zip(sinks, fresh)]
    return targets, returned


def zeros_like_planes(planes: Sequence[torch.Tensor], need: Sequence[bool]) -> List[Optional[torch.Tensor]]:
    """One flat zero-filled buffer carved into channel-last views (a single memset for all plane gradients)."""
    total = sum(p.numel() for p, n in zip(planes, need) if n)
    if total == 0:
        return [None] * len(planes)
    flat = torch.zeros(total, dtype=torch.float32, device=planes[0].device)
    out, off = [], 0
    for p, n in zip(planes, need):
        if not n:
            out.append(None)
            continue
        _, c, h, w = p.shape
        out.append(flat[off: off + p.numel()].view(1, h, w, c).permute(0, 3, 1, 2))
        off += p.numel()
    return out


@dataclass
class Points:
    """Sample coordinates: explicit ``pts`` [M,D] in [-1,1], or ray form (see include/kplanes_b200.h)."""

    D: int
    pts: Optional[torch.Tensor] = None
    origins: Optional[torch.Tensor] = None  # [N,3]
    directions: Optional[torch.Tensor] = None  # [N,3]
    starts: Optional[torch.Tensor] = None  # [N,S]
    ends: Optional[torch.Tensor] = None  # [N,S]
    times: Optional[torch.Tensor] = None  # [N]
    S: int = 1
    norm_mode: int = 1
    aabb: Tuple[float, ...] = (0.0,) * 6
    ray_tile: int = 0  # gather only (KpPoints.ray_tile): warps take one sample index of this many neighbouring rays

    @property
    def M(self) -> int:
        return self.pts.shape[0] if self.pts is not None else self.starts.numel()

    def tensors(self) -> List[Optional[torch.Tensor]]:
        return [self.pts, self.origins, self.directions, self.starts, self.ends, self.times]

    def struct(self) -> _lib.KpPoints:
        return _lib.make_points(pts=self.pts, origins=self.origins, directions=self.directions, starts=self.starts,
                                ends=self.ends, times=self.times, D=self.D, S=self.S, norm_mode=self.norm_mode,
                                aabb=self.aabb, ray_tile=self.ray_tile)


def points_from_pts(pts: torch.Tensor) -> Points:
    pts = f32c(pts.detach())
    return Points(D=pts.shape[-1], pts=pts.view(-1, pts.shape[-1]))


def points_from_rays(origins, directions, starts, ends, times, aabb, norm_mode: int, dynamic: bool, ray_tile: int = 0) -> Points:
    """origins/directions [N,3], starts/ends [N,S], times [N] or None."""
    return Points(
        D=4 if dynamic else 3, origins=f32c(origins.detach()), directions=f32c(directions.detach()),
        starts=f32c(starts.detach()), ends=f32c(ends.detach()),
        times=None if (times is None or not dynamic) else f32c(times.detach()).view(-1),
        S=starts.shape[-1], norm_mode=norm_mode, aabb=tuple(aabb), ray_tile=ray_tile,
    )


# ------------------------------------------------------------------------------------------------
# (a1-a3) multiscale hexplane features
# ------------------------------------------------------------------------------------------------
class _Hexplane(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points: Points, n_scales: int, concat: bool, use_mask: int, post_backward, *planes):
        ctx.sinks = [grad_sink(p) for p in planes]
        # sparse gradient exchange: per-texel "touched" bytes of the planes whose gradient sink is a marked bucket
        ctx.touched = [getattr(p, "_kp_touched", None) if s is not None else None for p, s in zip(planes, ctx.sinks)]
        ctx.post_backward = post_backward
        planes = [as_channel_last(p.detach()) for p in planes]
        n_planes = len(planes) // n_scales
        c = planes[0].shape[1]
        m = points.M
        out = torch.empty((m, n_scales * c if concat else c), dtype=torch.float32, device=planes[0].device)
        pstruct = points.struct()
        call("kp_hexplane_fwd", _plane_ptrs(planes), _plane_hw(planes), n_scales, n_planes, c, pstruct, m, int(concat),
             use_mask, ptr(out), stream_ptr())
        ctx.points, ctx.cfg, ctx.planes = points, (n_scales, n_planes, c, concat, use_mask), planes
        return out

    @staticmethod
    def backward(ctx, grad_out):
        n_scales, n_planes, c, concat, use_mask = ctx.cfg
        planes, points = ctx.planes, ctx.points
        need = [ctx.needs_input_grad[5 + i] and bool((use_mask >> (i % n_planes)) & 1) for i in range(len(planes))]
        targets, grads = _targets(planes, ctx.sinks, need)
        hook = ctx.post_backward
        marks = _plane_ptrs(ctx.touched) if any(t is not None for t in ctx.touched) else None

        def scatter(tg):
            if marks is not None:
                call("kp_hexplane_bwd_flags", _plane_ptrs(planes), _plane_ptrs(tg), marks, _plane_hw(planes), n_scales, n_planes, c,
                     points.struct(), points.M, int(concat), use_mask, ptr(g), stream_ptr())
            else:
                call("kp_hexplane_bwd", _plane_ptrs(planes), _plane_ptrs(tg), _plane_hw(planes), n_scales, n_planes, c,
                     points.struct(), points.M, int(concat), use_mask, ptr(g), stream_ptr())

        if any(need):
            g = f32c(grad_out)
            if hook is not None and getattr(hook, "per_scale", False) and n_scales > 1:
                # one scatter launch per scale, finest (largest planes) first: hook(k) can start reducing scale k's
                # gradients while the remaining scales are scattered
                for k in reversed(range(n_scales)):
                    scatter([t if i // n_planes == k else None for i, t in enumerate(targets)])
                    hook(k)
                hook = None
            else:
                scatter(targets)
        if hook is not None:
            hook()  # e.g. start the gradient all-reduce of the field bucket while the proposals back-propagate
        return (None, None, None, None, None, *grads)


def hexplane_features(ms_planes: Sequence[Sequence[torch.Tensor]], points: Points, concat: bool,
                      use_mask: int = 0x3F, post_backward=None) -> torch.Tensor:
    """interpolate_kplanes (NS/fields/kplanes_field.py:77-126) -> [M, K*C] (concat) or [M, C] (sum).
    ``post_backward``: optional callable run right after the scatter kernel has been enqueued in the backward."""
    flat = [p for grids in ms_planes for p in grids]
    return _Hexplane.apply(points, len(ms_planes), concat, use_mask, post_backward, *flat)


def hexplane_features_dyn(ms_planes: Sequence[Sequence[torch.Tensor]], points: Points, concat: bool,
                          use_mask: int = 0x3F) -> Tuple[torch.Tensor, torch.Tensor]:
    """Inference only, dynamic fields: ``hexplane_features``' features (the same bits) and the dynamics score [M] of every
    sample, 1/(K*C) * sum_k sum_c |1 - prod of the time planes' interpolants| (kp_hexplane_fwd_dyn).  No backward."""
    if torch.is_grad_enabled() and any(p.requires_grad for grids in ms_planes for p in grids):
        raise RuntimeError("hexplane_features_dyn has no backward: call it under torch.no_grad()")
    planes = [as_channel_last(p.detach()) for grids in ms_planes for p in grids]
    n_scales = len(ms_planes)
    c, m = planes[0].shape[1], points.M
    out = torch.empty((m, n_scales * c if concat else c), dtype=torch.float32, device=planes[0].device)
    delta = torch.empty((m,), dtype=torch.float32, device=planes[0].device)
    call("kp_hexplane_fwd_dyn", _plane_ptrs(planes), _plane_hw(planes), n_scales, len(planes) // n_scales, c, points.struct(), m,
         int(concat), use_mask, ptr(out), ptr(delta), stream_ptr())
    return out, delta


# ------------------------------------------------------------------------------------------------
# (a6) fused proposal density field
# ------------------------------------------------------------------------------------------------
class _DensityField(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points: Points, relu: bool, use_mask: int, w1, w2, *planes):
        ctx.sinks = [grad_sink(p) for p in planes]
        ctx.wsinks = (grad_sink(w1), grad_sink(w2))
        planes = [as_channel_last(p.detach()) for p in planes]
        w1c, w2c = f32c(w1.detach()), f32c(w2.detach()).view(-1)
        c, hidden, m = planes[0].shape[1], w1c.shape[0], points.M
        density = torch.empty((m,), dtype=torch.float32, device=w1c.device)
        call("kp_density_field_fwd", _plane_ptrs(planes), _plane_hw(planes), len(planes), c, ptr(w1c), ptr(w2c), hidden,
             int(relu), points.struct(), m, use_mask, ptr(density), stream_ptr())
        ctx.points, ctx.cfg, ctx.planes, ctx.w = points, (relu, use_mask, c, hidden), planes, (w1c, w2c, w2.shape)
        return density

    @staticmethod
    def backward(ctx, grad_density):
        relu, use_mask, c, hidden = ctx.cfg
        planes, points = ctx.planes, ctx.points
        w1c, w2c, w2_shape = ctx.w
        n_planes = len(planes)
        need = [ctx.needs_input_grad[5 + i] and bool((use_mask >> i) & 1) for i in range(n_planes)]
        targets, grads = _targets(planes, ctx.sinks, need)
        s1, s2 = ctx.wsinks
        if s1 is not None and s2 is not None and s1.is_contiguous() and s2.is_contiguous():
            gw1, gw2, ret1, ret2 = s1, s2.view(-1), None, None
        else:
            gw = torch.zeros(w1c.numel() + w2c.numel(), dtype=torch.float32, device=w1c.device)
            gw1, gw2 = gw[: w1c.numel()].view_as(w1c), gw[w1c.numel():]
            ret1, ret2 = gw1, gw2.view(w2_shape)
        call("kp_density_field_bwd", _plane_ptrs(planes), _plane_ptrs(targets), _plane_hw(planes), n_planes, c, ptr(w1c),
             ptr(w2c), hidden, int(relu), points.struct(), points.M, use_mask, ptr(f32c(grad_density)), ptr(gw1), ptr(gw2),
             stream_ptr())
        return (None, None, None, ret1, ret2, *grads)


def density_field(planes: Sequence[torch.Tensor], w1: torch.Tensor, w2: torch.Tensor, points: Points, relu: bool = True,
                  use_mask: int = 0x3F) -> torch.Tensor:
    """KPlanesDensityField.get_density (kplanes_field.py:434-460) fused: -> density [M]."""
    return _DensityField.apply(points, relu, use_mask, w1, w2, *planes)


# ------------------------------------------------------------------------------------------------
# (a4, a5) decoders
# ------------------------------------------------------------------------------------------------
class _SigmaNet(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, w1, w2):
        ctx.set_materialize_grads(False)
        ctx.wsinks = (grad_sink(w1), grad_sink(w2))
        x, w1c, w2c = f32c(feats.detach()), f32c(w1.detach()), f32c(w2.detach())
        m, k = x.shape
        h = w1c.shape[0]
        assert w1c.shape == (h, k) and w2c.shape == (16, h), "sigma_net: w1 [H,K], w2 [16,H]"
        h1 = torch.empty((m, h), dtype=torch.float32, device=x.device)
        o = torch.empty((m, 16), dtype=torch.float32, device=x.device)
        density = torch.empty((m,), dtype=torch.float32, device=x.device)
        call("kp_sigma_net_fwd", ptr(x), ptr(w1c), ptr(w2c), m, k, h, ptr(h1), ptr(o), ptr(density), stream_ptr())
        ctx.save_for_backward(x, w1c, w2c, h1, o)
        return o, density

    @staticmethod
    def backward(ctx, grad_o, grad_density):
        x, w1c, w2c, h1, o = ctx.saved_tensors
        m, k = x.shape
        h = w1c.shape[0]
        gx = torch.empty_like(x)
        s1, s2 = ctx.wsinks
        if s1 is not None and s2 is not None and s1.is_contiguous() and s2.is_contiguous():
            gw1, gw2, ret = s1, s2, (None, None)
        else:
            gw = torch.zeros(w1c.numel() + w2c.numel(), dtype=torch.float32, device=x.device)
            gw1, gw2 = gw[: w1c.numel()].view_as(w1c), gw[w1c.numel():].view_as(w2c)
            ret = (gw1, gw2)
        scratch = torch.empty_like(h1)
        call("kp_sigma_net_bwd", ptr(x), ptr(w1c), ptr(w2c), m, k, h, ptr(h1), ptr(o),
             ptr(None if grad_density is None else f32c(grad_density)), ptr(None if grad_o is None else f32c(grad_o)),
             ptr(gx), ptr(gw1), ptr(gw2), ptr(scratch), stream_ptr())
        return (gx, *ret)


def sigma_net(feats: torch.Tensor, w1: torch.Tensor, w2: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """-> (o [M,16] = [geo 15 | sigma_raw], density [M] = trunc_exp(sigma_raw)).  kplanes_field.py:302-311."""
    return _SigmaNet.apply(feats, w1, w2)


class _ColorNet(torch.autograd.Function):
    @staticmethod
    def forward(ctx, directions, samples_per_ray: int, geo, w3, w4, w5):
        ctx.wsinks = (grad_sink(w3), grad_sink(w4), grad_sink(w5))
        w3c, w4c, w5c = f32c(w3.detach()), f32c(w4.detach()), f32c(w5.detach())
        g = geo.detach()
        if g.dtype != torch.float32:
            g = g.float()
        # geo may be the [:, :15] view of the sigma net's [M,16] output: pass the row stride instead of copying
        if not (g.dim() == 2 and g.shape[1] == 15 and g.stride(1) == 1 and g.stride(0) in (15, 16)):
            g = g.reshape(-1, 15).contiguous()
        m, ldgeo = g.shape[0], g.stride(0)
        h2d = w3c.shape[0]
        view_dep = directions is not None
        d = f32c(directions.detach()) if view_dep else None
        assert w3c.shape == (h2d, 31 if view_dep else 15) and w4c.shape == (h2d, h2d) and w5c.shape == (3, h2d)
        dev = g.device
        cin = torch.empty((m, 32 if view_dep else 16), dtype=torch.float32, device=dev)
        h2 = torch.empty((m, h2d), dtype=torch.float32, device=dev)
        h3 = torch.empty((m, h2d), dtype=torch.float32, device=dev)
        rgb = torch.empty((m, 3), dtype=torch.float32, device=dev)
        call("kp_color_net_fwd", ptr(d), samples_per_ray, c_void_p(g.data_ptr()), ldgeo, ptr(w3c), ptr(w4c), ptr(w5c), m,
             h2d, ptr(cin), ptr(h2), ptr(h3), ptr(rgb), stream_ptr())
        ctx.save_for_backward(cin, h2, h3, rgb, w3c, w4c, w5c)
        ctx.view_dep = view_dep
        return rgb

    @staticmethod
    def backward(ctx, grad_rgb):
        cin, h2, h3, rgb, w3c, w4c, w5c = ctx.saved_tensors
        m, h2d = h2.shape
        dev = h2.device
        go = torch.empty((m, 16), dtype=torch.float32, device=dev)
        if all(s is not None and s.is_contiguous() for s in ctx.wsinks):
            gw3, gw4, gw5 = ctx.wsinks
            ret = (None, None, None)
        else:
            gw = torch.zeros(w3c.numel() + w4c.numel() + w5c.numel(), dtype=torch.float32, device=dev)
            a, b = w3c.numel(), w3c.numel() + w4c.numel()
            gw3, gw4, gw5 = gw[:a].view_as(w3c), gw[a:b].view_as(w4c), gw[b:].view_as(w5c)
            ret = (gw3, gw4, gw5)
        sa, sb = torch.empty_like(h2), torch.empty_like(h2)
        call("kp_color_net_bwd", int(ctx.view_dep), ptr(cin), ptr(h2), ptr(h3), ptr(rgb), ptr(w3c), ptr(w4c), ptr(w5c), m,
             h2d, ptr(f32c(grad_rgb)), ptr(go), ptr(gw3), ptr(gw4), ptr(gw5), ptr(sa), ptr(sb), stream_ptr())
        return (None, None, go[:, :15], *ret)


def color_net(directions: Optional[torch.Tensor], samples_per_ray: int, geo: torch.Tensor, w3, w4, w5) -> torch.Tensor:
    """[SH4(dir) | geo] -> rgb [M,3] (sigmoid).  directions [N,3] per ray or None (disable_viewing_dependent)."""
    return _ColorNet.apply(directions, samples_per_ray, geo, w3, w4, w5)


class _DecoderFused(torch.autograd.Function):
    """sigma_net + SH + color_net in one tcgen05 kernel (forward); the backward runs the per-layer tensor-core kernels
    on the activations the forward saved (none are saved, and none written, when no gradient is needed)."""

    @staticmethod
    def forward(ctx, feats, directions, samples_per_ray: int, w1, w2, w3, w4, w5):
        ctx.set_materialize_grads(False)  # an unused output (o in training) arrives as None, not as a [M,16] zero fill + add
        ctx.wsinks = tuple(grad_sink(w) for w in (w1, w2, w3, w4, w5))
        x = f32c(feats.detach())
        ws = [f32c(w.detach()) for w in (w1, w2, w3, w4, w5)]
        m, k = x.shape
        view_dep = directions is not None
        d = f32c(directions.detach()) if view_dep else None
        dev = x.device
        need_grad = any(ctx.needs_input_grad)
        h1 = torch.empty((m, 64), dtype=torch.float32, device=dev) if need_grad else None
        h2 = torch.empty((m, 64), dtype=torch.float32, device=dev) if need_grad else None
        h3 = torch.empty((m, 64), dtype=torch.float32, device=dev) if need_grad else None
        cin = torch.empty((m, 32 if view_dep else 16), dtype=torch.float32, device=dev) if need_grad else None
        o = torch.empty((m, 16), dtype=torch.float32, device=dev)
        density = torch.empty((m,), dtype=torch.float32, device=dev)
        rgb = torch.empty((m, 3), dtype=torch.float32, device=dev)
        call("kp_decoder_fwd_fused", ptr(x), k, ptr(d), samples_per_ray, *[ptr(w) for w in ws], m, 64, 64, ptr(h1), ptr(cin),
             ptr(h2), ptr(h3), ptr(o), ptr(density), ptr(rgb), stream_ptr())
        if need_grad:
            ctx.save_for_backward(x, h1, o, cin, h2, h3, rgb, *ws)
        ctx.view_dep = view_dep
        return o, density, rgb

    @staticmethod
    def backward(ctx, grad_o, grad_density, grad_rgb):
        x, h1, o, cin, h2, h3, rgb, w1c, w2c, w3c, w4c, w5c = ctx.saved_tensors
        m, k = x.shape
        dev = x.device
        sinks = ctx.wsinks
        if all(s is not None and s.is_contiguous() for s in sinks):
            gws, ret = list(sinks), (None,) * 5
        else:
            flat = torch.zeros(sum(w.numel() for w in (w1c, w2c, w3c, w4c, w5c)), dtype=torch.float32, device=dev)
            gws, off = [], 0
            for w in (w1c, w2c, w3c, w4c, w5c):
                gws.append(flat[off: off + w.numel()].view_as(w))
                off += w.numel()
            ret = tuple(gws)
        go = torch.empty((m, 16), dtype=torch.float32, device=dev)
        if grad_rgb is not None:
            sa, sb = torch.empty_like(h2), torch.empty_like(h2)
            call("kp_color_net_bwd", int(ctx.view_dep), ptr(cin), ptr(h2), ptr(h3), ptr(rgb), ptr(w3c), ptr(w4c), ptr(w5c), m, 64,
                 ptr(f32c(grad_rgb)), ptr(go), ptr(gws[2]), ptr(gws[3]), ptr(gws[4]), ptr(sa), ptr(sb), stream_ptr())
            if grad_o is not None:
                go = go + f32c(grad_o)
        else:
            go = f32c(grad_o) if grad_o is not None else None
        gx = torch.empty_like(x)
        scratch = torch.empty_like(h1)
        call("kp_sigma_net_bwd", ptr(x), ptr(w1c), ptr(w2c), m, k, 64, ptr(h1), ptr(o),
             ptr(None if grad_density is None else f32c(grad_density)), ptr(go), ptr(gx), ptr(gws[0]), ptr(gws[1]), ptr(scratch),
             stream_ptr())
        return (gx, None, None, *ret)


class _Linear(torch.autograd.Function):
    """y = act(x w^T) on the tensor-core dense-layer kernels (kp_tc_linear_*), any layer shape they cover.  The building
    block of the non-default decoder branches (linear decoder / colour basis, appearance embedding), which are composed
    from it in ``fields/kplanes_field.py``; the default decoders use the fused kernels above."""

    @staticmethod
    def forward(ctx, x, w, act: int):
        xs, wc = f32c(x.detach()), f32c(w.detach())
        m, k = xs.shape
        n = wc.shape[0]
        if wc.shape[1] != k:
            raise RuntimeError(f"linear: x [{m},{k}] vs w {tuple(wc.shape)}")
        y = torch.empty((m, n), dtype=torch.float32, device=xs.device)
        call("kp_tc_linear_fwd", ptr(xs), k, ptr(wc), k, ptr(y), n, m, n, k, int(act), stream_ptr())
        ctx.save_for_backward(xs, wc, y)
        ctx.act, ctx.wsink = int(act), grad_sink(w)
        return y

    @staticmethod
    def backward(ctx, gy):
        xs, wc, y = ctx.saved_tensors
        m, k = xs.shape
        n = wc.shape[0]
        g = f32c(gy)
        if ctx.act == 1:
            g = g * (y > 0)
        elif ctx.act == 2:
            g = g * y * (1 - y)
        g = f32c(g)
        gx = gw = None
        if ctx.needs_input_grad[0]:
            gx = torch.empty_like(xs)
            call("kp_tc_linear_bwd_data", ptr(g), n, ptr(wc), k, ptr(gx), k, m, n, k, ptr(None), 0, stream_ptr())
        if ctx.needs_input_grad[1]:
            sink = ctx.wsink
            if sink is not None and sink.is_contiguous():
                target = sink
            else:
                target = gw = torch.zeros_like(wc)
            call("kp_tc_linear_bwd_weight", ptr(g), n, ptr(xs), k, ptr(target), k, m, n, k, stream_ptr())
        return gx, gw, None


def linear(x: torch.Tensor, w: torch.Tensor, act: str = "none") -> torch.Tensor:
    """act(x [M,K] @ w [N,K]^T); act in {"none", "relu", "sigmoid"} (bias-free: tcnn FullyFusedMLP semantics)."""
    return _Linear.apply(x, w, {"none": 0, "relu": 1, "sigmoid": 2}[act])


class _TruncExp(torch.autograd.Function):
    """NS/field_components/activations.py:25-41: forward exp(x), backward g * exp(clamp(x, -15, 15))."""

    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return torch.exp(x)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return g * torch.exp(x.clamp(-15, 15))


trunc_exp = _TruncExp.apply


def sh4(directions01: torch.Tensor) -> torch.Tensor:
    """Degree-4 spherical harmonics of 2x-1 (tcnn's SphericalHarmonics input convention; basis NS/utils/math.py:25-86)
    as tensor ops -> [..., 16].  Only the non-default decoder branches use this form; the fused decoder kernel evaluates
    the same basis in registers."""
    d = directions01 * 2.0 - 1.0
    x, y, z = d[..., 0], d[..., 1], d[..., 2]
    xx, yy, zz = x * x, y * y, z * z
    comps = [
        torch.full_like(x, 0.28209479177387814), 0.4886025119029199 * y, 0.4886025119029199 * z, 0.4886025119029199 * x,
        1.0925484305920792 * x * y, 1.0925484305920792 * y * z, 0.9461746957575601 * zz - 0.31539156525251999,
        1.0925484305920792 * x * z, 0.5462742152960396 * (xx - yy), 0.5900435899266435 * y * (3 * xx - yy),
        2.890611442640554 * x * y * z, 0.4570457994644658 * y * (5 * zz - 1), 0.3731763325901154 * z * (5 * zz - 3),
        0.4570457994644658 * x * (5 * zz - 1), 1.445305721320277 * z * (xx - yy), 0.5900435899266435 * x * (xx - 3 * yy),
    ]
    return torch.stack(comps, dim=-1)


def decoder_fused_supported(k0: int, h1: int, h2: int) -> bool:
    return bool(_lib.load().kp_decoder_fused_supported(int(k0), int(h1), int(h2)))


def decoder_fused(feats, directions, samples_per_ray: int, w1, w2, w3, w4, w5):
    """-> (o [M,16], density [M], rgb [M,3]).  KPlanesField.get_density + get_outputs in one kernel."""
    return _DecoderFused.apply(feats, directions, samples_per_ray, w1, w2, w3, w4, w5)


# ------------------------------------------------------------------------------------------------
# (a13, a7, a8) ray setup and resampling (no gradients: bins are detached, ray_samplers.py:357)
# ------------------------------------------------------------------------------------------------
def aabb_intersect(origins, directions, aabb6: Sequence[float], near_plane: float):
    o, d = f32c(origins), f32c(directions)
    n = o.shape[0]
    nears = torch.empty((n,), dtype=torch.float32, device=o.device)
    fars = torch.empty_like(nears)
    call("kp_aabb_intersect", ptr(o), ptr(d), n, (c_float * 6)(*[float(v) for v in aabb6]), float(near_plane), ptr(nears),
         ptr(fars), stream_ptr())
    return nears, fars


def intersect_aabb(origins, directions, aabb6: Sequence[float]):
    """nerfstudio.utils.math._intersect_aabb (math.py:201-238) on the device: origins / directions [N,3], aabb6 = min then
    max (host floats) -> t_min [N], t_max [N]; 1e10 twice for a ray that misses the box."""
    o, d = f32c(origins), f32c(directions)
    n = o.shape[0]
    t_min = torch.empty((n,), dtype=torch.float32, device=o.device)
    t_max = torch.empty_like(t_min)
    call("kp_intersect_aabb", ptr(o), ptr(d), n, (c_float * 6)(*[float(v) for v in aabb6]), ptr(t_min), ptr(t_max), stream_ptr())
    return t_min, t_max


_LINSPACE_CACHE = {}


def _cached_linspace(key, start, end, steps, device):
    k = (key, steps, str(device))
    if k not in _LINSPACE_CACHE:
        _LINSPACE_CACHE[k] = torch.linspace(start, end, steps, device="cpu").to(device)
    return _LINSPACE_CACHE[k]


def uniform_bins(nears, fars, num_samples: int, t_rand: Optional[torch.Tensor], spacing: int = 0, want_frustums: bool = False):
    """-> (spacing_bins [N,S+1], euclidean_bins [N,S+1][, starts, ends, deltas [N,S]]).  ray_samplers.py:79-126."""
    nears, fars = f32c(nears).view(-1), f32c(fars).view(-1)
    n = nears.shape[0]
    lin = _cached_linspace("uni", 0.0, 1.0, num_samples + 1, nears.device)
    sb = torch.empty((n, num_samples + 1), dtype=torch.float32, device=nears.device)
    eb = torch.empty_like(sb)
    fr = torch.empty((3, n, num_samples), dtype=torch.float32, device=nears.device) if want_frustums else None
    stride = 0
    if t_rand is not None:
        t_rand = f32c(t_rand)
        stride = 0 if t_rand.shape[-1] == 1 else num_samples + 1
    call("kp_uniform_bins", ptr(lin), ptr(t_rand), stride, ptr(nears), ptr(fars), n, num_samples, spacing, ptr(sb), ptr(eb),
         ptr(fr[0] if want_frustums else None), ptr(fr[1] if want_frustums else None), ptr(fr[2] if want_frustums else None),
         stream_ptr())
    if want_frustums:
        return sb, eb, fr[0], fr[1], fr[2]
    return sb, eb


def pdf_resample(weights, existing_bins, nears, fars, num_samples: int, rand: Optional[torch.Tensor],
                 histogram_padding: float = 0.01, eps: float = 1e-5, spacing: int = 0, want_inds: bool = False,
                 want_cdf: bool = False, anneal=1.0, want_frustums: bool = False):
    """-> (spacing_bins [N,S_out+1], euclidean_bins, inds int64 | None, cdf | None[, starts, ends, deltas]).
    ``anneal``: python float or 0-d device tensor; weights are raised to this power first (ray_samplers.py:584).
    ray_samplers.py:274-369."""
    w, eb_in = f32c(weights.detach()), f32c(existing_bins.detach())
    nears, fars = f32c(nears).view(-1), f32c(fars).view(-1)
    n, s_in = w.shape
    nb = num_samples + 1
    u_base = _cached_linspace("pdf", 0.0, 1.0 - (1.0 / nb), nb, w.device)
    sb = torch.empty((n, nb), dtype=torch.float32, device=w.device)
    eb = torch.empty_like(sb)
    inds = torch.empty((n, nb), dtype=torch.int64, device=w.device) if want_inds else None
    cdf = torch.empty((n, s_in + 1), dtype=torch.float32, device=w.device) if want_cdf else None
    fr = torch.empty((3, n, num_samples), dtype=torch.float32, device=w.device) if want_frustums else None
    stride = 0
    if rand is not None:
        rand = f32c(rand)
        stride = 0 if rand.shape[-1] == 1 else nb
    anneal_dev, anneal_host = (anneal.detach().float().reshape(1), 1.0) if isinstance(anneal, torch.Tensor) else (None, float(anneal))
    call("kp_pdf_resample", ptr(w), ptr(eb_in), s_in, ptr(u_base), ptr(rand), stride, ptr(nears), ptr(fars), n, num_samples,
         float(histogram_padding), float(eps), spacing, ptr(cdf), ptr(sb), ptr(eb), ptr(inds), ptr(anneal_dev), anneal_host,
         ptr(fr[0] if want_frustums else None), ptr(fr[1] if want_frustums else None), ptr(fr[2] if want_frustums else None),
         stream_ptr())
    if want_frustums:
        return sb, eb, inds, cdf, fr[0], fr[1], fr[2]
    return sb, eb, inds, cdf


# ------------------------------------------------------------------------------------------------
# (a10-a12) compositing
# ------------------------------------------------------------------------------------------------
class _Weights(torch.autograd.Function):
    @staticmethod
    def forward(ctx, deltas, densities):
        d, s = f32c(deltas.detach()), f32c(densities.detach())
        n, ns = d.shape
        w = torch.empty_like(d)
        call("kp_weights_fwd", ptr(d), ptr(s), n, ns, ptr(w), stream_ptr())
        ctx.save_for_backward(d, s)
        return w

    @staticmethod
    def backward(ctx, gw):
        d, s = ctx.saved_tensors
        gs = torch.empty_like(s)
        call("kp_weights_bwd", ptr(d), ptr(s), ptr(f32c(gw)), d.shape[0], d.shape[1], ptr(gs), stream_ptr())
        return None, gs


def get_weights(deltas: torch.Tensor, densities: torch.Tensor) -> torch.Tensor:
    """[N,S] x [N,S] -> [N,S].  RaySamples.get_weights, NS/cameras/rays.py:127-149."""
    return _Weights.apply(deltas, densities)


class _CompositeRGB(torch.autograd.Function):
    @staticmethod
    def forward(ctx, weights, rgb, bg, bg_mode: int, nan_to_num: bool):
        w, c = f32c(weights.detach()), f32c(rgb.detach())
        n, s = w.shape
        b = None if bg is None else f32c(bg.detach().expand(n, 3))
        comp = torch.empty((n, 3), dtype=torch.float32, device=w.device)
        call("kp_render_fwd", ptr(w), ptr(c), ptr(None), ptr(b), bg_mode, int(nan_to_num), n, s, ptr(comp), ptr(None), ptr(None),
             ptr(None), ptr(None), ptr(None), ptr(None), stream_ptr())
        ctx.save_for_backward(w, c, b)
        ctx.bg_mode = bg_mode
        return comp

    @staticmethod
    def backward(ctx, gcomp):
        w, c, b = ctx.saved_tensors
        n, s = w.shape
        gw = torch.empty_like(w)
        grgb = torch.empty_like(c) if ctx.needs_input_grad[1] else None
        call("kp_render_bwd", ptr(w), ptr(c), ptr(b), ctx.bg_mode, n, s, ptr(f32c(gcomp)), ptr(None), ptr(gw), ptr(grgb),
             stream_ptr())
        return gw, grgb, None, None, None


def composite_rgb(weights, rgb, background, nan_to_num: bool = False) -> torch.Tensor:
    """weights [N,S], rgb [N,S,3], background: "last_sample" or tensor [N,3]/[3] -> [N,3].  renderers.py:71-116."""
    if isinstance(background, str):
        assert background == "last_sample"
        return _CompositeRGB.apply(weights, rgb, None, 1, nan_to_num)
    return _CompositeRGB.apply(weights, rgb, background, 0, nan_to_num)


class _Accumulate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, weights):
        w = f32c(weights.detach())
        n, s = w.shape
        acc = torch.empty((n,), dtype=torch.float32, device=w.device)
        call("kp_render_fwd", ptr(w), ptr(None), ptr(None), ptr(None), 0, 0, n, s, ptr(None), ptr(acc), ptr(None), ptr(None),
             ptr(None), ptr(None), ptr(None), stream_ptr())
        ctx.shape = (n, s)
        return acc

    @staticmethod
    def backward(ctx, gacc):
        return f32c(gacc).view(-1, 1).expand(*ctx.shape)


def accumulate(weights: torch.Tensor) -> torch.Tensor:
    """sum_s w -> [N].  AccumulationRenderer, renderers.py:197-223."""
    return _Accumulate.apply(weights)


def median_index(weights: torch.Tensor) -> torch.Tensor:
    """clamp(searchsorted(cumsum(w), 0.5, "left"), 0, S-1) -> int64 [N].  renderers.py:260-263."""
    w = f32c(weights.detach())
    n, s = w.shape
    idx = torch.empty((n,), dtype=torch.int64, device=w.device)
    call("kp_render_fwd", ptr(w), ptr(None), ptr(None), ptr(None), 0, 0, n, s, ptr(None), ptr(None), ptr(idx), ptr(None),
         ptr(None), ptr(None), ptr(None), stream_ptr())
    return idx


def median_depth(weights: torch.Tensor, starts: torch.Tensor, ends: torch.Tensor) -> torch.Tensor:
    """(starts + ends)/2 at the median index, one kernel (DepthRenderer "median", renderers.py:256-264) -> [N]."""
    w, st, en = f32c(weights.detach()), f32c(starts.detach()), f32c(ends.detach())
    n, s = w.shape
    out = torch.empty((n,), dtype=torch.float32, device=w.device)
    call("kp_render_fwd", ptr(w), ptr(None), ptr(None), ptr(None), 0, 0, n, s, ptr(None), ptr(None), ptr(None), ptr(None),
         ptr(st), ptr(en), ptr(out), stream_ptr())
    return out


def expected_depth(weights: torch.Tensor, steps: torch.Tensor) -> torch.Tensor:
    """sum w*steps / (sum w + 1e-10), unclipped, no grad -> [N].  renderers.py:266-281."""
    w, st = f32c(weights.detach()), f32c(steps.detach())
    n, s = w.shape
    out = torch.empty((n,), dtype=torch.float32, device=w.device)
    call("kp_render_fwd", ptr(w), ptr(None), ptr(st), ptr(None), 0, 0, n, s, ptr(None), ptr(None), ptr(None), ptr(out),
         ptr(None), ptr(None), ptr(None), stream_ptr())
    return out


# ------------------------------------------------------------------------------------------------
# (a14) distortion / interlevel losses
# ------------------------------------------------------------------------------------------------
class _Distortion(torch.autograd.Function):
    @staticmethod
    def forward(ctx, sdist, w):
        t, wc = f32c(sdist.detach()), f32c(w.detach())
        n, s = wc.shape
        loss = torch.empty((n,), dtype=torch.float32, device=wc.device)
        call("kp_distortion_fwd", ptr(t), ptr(wc), n, s, ptr(loss), stream_ptr())
        ctx.save_for_backward(t, wc)
        return loss

    @staticmethod
    def backward(ctx, g):
        t, wc = ctx.saved_tensors
        gw = torch.empty_like(wc)
        call("kp_distortion_bwd", ptr(t), ptr(wc), ptr(f32c(g)), wc.shape[0], wc.shape[1], ptr(gw), stream_ptr())
        return None, gw


def distortion_per_ray(sdist: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """lossfun_distortion (losses.py:125-136): sdist [N,S+1], w [N,S] -> [N]."""
    return _Distortion.apply(sdist, w)


class _Interlevel(torch.autograd.Function):
    @staticmethod
    def forward(ctx, c, w, cp, wp):
        cc, wc, cpc, wpc = f32c(c.detach()), f32c(w.detach()), f32c(cp.detach()), f32c(wp.detach())
        n, s = wc.shape
        sp = wpc.shape[1]
        loss = torch.empty((n, s), dtype=torch.float32, device=wc.device)
        call("kp_interlevel_fwd", ptr(cc), ptr(wc), ptr(cpc), ptr(wpc), n, s, sp, ptr(loss), stream_ptr())
        ctx.save_for_backward(cc, wc, cpc, wpc)
        return loss

    @staticmethod
    def backward(ctx, g):
        cc, wc, cpc, wpc = ctx.saved_tensors
        gwp = torch.empty_like(wpc)
        call("kp_interlevel_bwd", ptr(cc), ptr(wc), ptr(cpc), ptr(wpc), ptr(f32c(g)), wc.shape[0], wc.shape[1], wpc.shape[1],
             ptr(gwp), stream_ptr())
        return None, None, None, gwp


def lossfun_outer(c, w, cp, wp) -> torch.Tensor:
    """lossfun_outer (losses.py:78-95): final-level (c [N,S+1], w [N,S]) vs proposal (cp [N,Sp+1], wp [N,Sp]) -> [N,S]."""
    return _Interlevel.apply(c, w, cp, wp)


# ------------------------------------------------------------------------------------------------
# (a15) plane regularisers
# ------------------------------------------------------------------------------------------------
PLANE_REG_BACKWARDS = 0  # number of regulariser backward passes run so far (the trainer orders its all-reduce after it)


def _reg_tables(planes, terms):
    from ctypes import c_uint32

    hwc = (c_int32 * (3 * len(planes)))()
    tm = (c_uint32 * len(planes))()
    for i, (p, t) in enumerate(zip(planes, terms)):
        hwc[3 * i], hwc[3 * i + 1], hwc[3 * i + 2] = p.shape[2], p.shape[3], p.shape[1]
        tm[i] = t
    return hwc, tm


def generate_rays(c2w: torch.Tensor, intrinsics: torch.Tensor, cam_times: Optional[torch.Tensor],
                  ray_indices: Optional[torch.Tensor] = None, cam: int = 0, width: int = 1, first_pixel: int = 0,
                  n: Optional[int] = None, pixel_offset: float = 0.5, distortion: Optional[torch.Tensor] = None,
                  cam_types: Optional[torch.Tensor] = None):
    """Pixel -> ray generation (cameras.py:505-741).  Either ``ray_indices`` int64 [N,3] (camera,row,col) or a row-major
    pixel range of camera ``cam``.  ``distortion`` fp32 [n_cams,6] (OpenCV k1..k4,p1,p2) and ``cam_types`` int32 [n_cams]
    (CameraType values) select the lens kernel; both None = undistorted perspective cameras.
    -> origins [N,3], directions [N,3], pixel_area [N], directions_norm [N], times [N] | None."""
    c2w_c, intr = f32c(c2w), f32c(intrinsics)
    if ray_indices is not None:
        if ray_indices.dtype != torch.int64 or not ray_indices.is_contiguous():
            ray_indices = ray_indices.to(torch.int64).contiguous()
        n = ray_indices.shape[0]
    dev = c2w_c.device
    origins = torch.empty((n, 3), dtype=torch.float32, device=dev)
    directions = torch.empty((n, 3), dtype=torch.float32, device=dev)
    pixel_area = torch.empty((n,), dtype=torch.float32, device=dev)
    norm = torch.empty((n,), dtype=torch.float32, device=dev)
    times = None if cam_times is None else torch.empty((n,), dtype=torch.float32, device=dev)
    ct = None if cam_times is None else f32c(cam_times).view(-1)
    n_cams = c2w_c.shape[0]
    if distortion is not None:
        distortion = f32c(distortion)
        if tuple(distortion.shape) != (n_cams, 6) or distortion.device != dev:
            raise ValueError(f"generate_rays: distortion must be [{n_cams}, 6] on {dev}")
    if cam_types is not None:
        if cam_types.dtype != torch.int32 or not cam_types.is_contiguous() or cam_types.numel() != n_cams or cam_types.device != dev:
            raise ValueError(f"generate_rays: cam_types must be contiguous int32 [{n_cams}] on {dev}")
    call("kp_generate_rays", ptr(c2w_c), ptr(intr), ptr(ct), ptr(distortion), ptr(cam_types), n_cams, ptr(ray_indices), int(cam), int(width),
         int(first_pixel), int(n), float(pixel_offset), ptr(origins), ptr(directions), ptr(pixel_area), ptr(norm), ptr(times),
         stream_ptr())
    return origins, directions, pixel_area, norm, times


_SAMPLER_SCRATCH = {}


def importance_pixels(weights: torch.Tensor, sel: torch.Tensor, k_max: int, n_out: int, image_width: int, seed: int) -> torch.Tensor:
    """Importance pixel sampling on the device (kp_importance_pixels): weights fp16 CUDA [B,H,W] or [B,HW]; sel int32
    [n_sel,3] = (image, k, first output row) on the host (uploaded here) or already on the device; -> int64 [n_out,3]
    (image, row, col).  Per entry k pixels proportional to the image's weights, without replacement when the map has
    >= k non-zero pixels, else with replacement -- DynamicBasedPixelSampler's torch.multinomial calls
    (NS/data/pixel_samplers.py:396-398) for the whole step in six launches, no host synchronisation."""
    if weights.dtype != torch.float16 or not weights.is_cuda or not weights.is_contiguous():
        raise RuntimeError("importance_pixels: weights must be a contiguous fp16 CUDA tensor (there is no CPU path)")
    b = weights.shape[0]
    hw = weights.numel() // max(b, 1)
    if sel.dtype != torch.int32 or sel.dim() != 2 or sel.shape[1] != 3:
        raise ValueError("importance_pixels: sel must be int32 [n_sel, 3] = (image, k, first output row)")
    dev = weights.device
    n_sel = sel.shape[0]
    out = torch.empty((n_out, 3), dtype=torch.int64, device=dev)
    if n_sel == 0 or n_out == 0:
        return out
    if not sel.is_cuda:
        # a table that arrives on the host is checked like tensor indexing would be (rows the kernel writes must lie inside
        # `out`); a device-resident table is trusted -- checking it would cost a synchronisation
        img, k, first = sel[:, 0], sel[:, 1], sel[:, 2]
        if int(img.min()) < 0 or int(img.max()) >= b:
            raise IndexError(f"importance_pixels: image index out of range [0, {b})")
        if int(k.min()) < 0 or int(k.max()) > int(k_max) or int(first.min()) < 0 or int((first + k).max()) > n_out:
            raise IndexError("importance_pixels: a table entry's rows [first, first + k) leave the output or k exceeds k_max")
        sel = sel.contiguous().pin_memory().to(dev, non_blocking=True)
    nbytes = int(_lib.load().kp_importance_pixels_scratch_bytes(n_sel, int(k_max)))
    key = (str(dev), torch.cuda.current_stream(dev).cuda_stream)
    scratch = _SAMPLER_SCRATCH.get(key)
    if scratch is None or scratch.numel() < nbytes:
        scratch = _SAMPLER_SCRATCH[key] = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    call("kp_importance_pixels", c_void_p(weights.data_ptr()), b, hw, int(image_width), c_void_p(sel.data_ptr()), n_sel, int(k_max),
         int(seed) & 0xFFFFFFFFFFFFFFFF, c_void_p(scratch.data_ptr()), ptr(out), stream_ptr())
    return out


def isg_map(images: torch.Tensor, cam_ids: torch.Tensor, gamma: float) -> torch.Tensor:
    """ISG weight map on the device (kp_isg_map): images [B,H,W,3] fp32 CUDA, cam_ids [B] -> fp16 [B,H,W]."""
    if images.dim() != 4 or images.shape[-1] != 3:
        raise ValueError("isg_map: images must be [B,H,W,3]")
    img = f32c(images)
    b, h, w = img.shape[:3]
    ids = cam_ids.reshape(-1).cpu()
    uniq = torch.unique(ids)
    slot = {int(c): k for k, c in enumerate(uniq.tolist())}
    groups = [torch.where(ids == c)[0] for c in uniq]
    offsets = torch.tensor([0] + list(torch.cumsum(torch.tensor([len(g) for g in groups]), 0).tolist()), dtype=torch.int32)
    cam_images = torch.cat(groups).to(torch.int32)
    image_cam = torch.tensor([slot[int(c)] for c in ids.tolist()], dtype=torch.int32)
    dev = img.device
    offsets, cam_images, image_cam = offsets.to(dev), cam_images.to(dev), image_cam.to(dev)
    scratch = torch.empty(len(uniq) * h * w * 3, dtype=torch.float32, device=dev)
    out = torch.empty((b, h, w), dtype=torch.float16, device=dev)
    import numpy as np

    gamma_sq = float(np.float32(float(gamma) ** 2))  # python double gamma**2, then cast to fp32 like torch's scalar add
    call("kp_isg_map", ptr(img), b, h * w, c_void_p(offsets.data_ptr()), c_void_p(cam_images.data_ptr()),
         c_void_p(image_cam.data_ptr()), len(uniq), max(len(g) for g in groups), gamma_sq, ptr(scratch), c_void_p(out.data_ptr()),
         stream_ptr())
    return out


def ist_map(images: torch.Tensor, nbr_offsets: torch.Tensor, nbrs: torch.Tensor, alpha: float) -> torch.Tensor:
    """IST importance map (dynamic_dataset.py:328-470): images [B,H,W,3] fp32 (CUDA), CSR neighbour lists int32 (CUDA)
    -> fp16 [B,H,W]."""
    img = f32c(images)
    b, h, w = img.shape[:3]
    if img.shape[-1] != 3:
        raise ValueError("ist_map: images must be [B,H,W,3]")
    off = nbr_offsets.to(device=img.device, dtype=torch.int32).contiguous()
    nb = nbrs.to(device=img.device, dtype=torch.int32).contiguous()
    if off.numel() != b + 1:
        raise ValueError("ist_map: nbr_offsets must have B+1 entries")
    out = torch.empty((b, h, w), dtype=torch.float16, device=img.device)
    call("kp_ist_map", ptr(img), b, h * w, c_void_p(off.data_ptr()), c_void_p(nb.data_ptr() if nb.numel() else 0), float(alpha),
         c_void_p(out.data_ptr()), stream_ptr())
    return out


def image_metrics(pred: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """Per-image (psnr, ssim) of a batch on the device (kp_image_metrics): pred, target fp32 CUDA [B,H,W,3] with
    H, W >= 11 -> fp32 [B,2].  Equal to ``utils.image_metrics.psnr`` / ``ssim`` applied image by image to the
    [1,3,H,W] forms; no host synchronisation, so it can be captured in a CUDA graph."""
    if pred.dim() != 4 or pred.shape[-1] != 3 or target.shape != pred.shape:
        raise ValueError(f"image_metrics: pred and target must both be [B,H,W,3] (got {tuple(pred.shape)}, {tuple(target.shape)})")
    if pred.dtype != torch.float32 or target.dtype != torch.float32:
        raise TypeError("image_metrics: pred and target must be float32")
    if not pred.is_cuda or target.device != pred.device:
        raise RuntimeError("image_metrics: pred and target must be CUDA tensors on one device (there is no CPU path)")
    b, h, w = pred.shape[:3]
    if h < 11 or w < 11:
        raise ValueError(f"image_metrics: {h}x{w} images are smaller than the 11x11 SSIM window")
    pred, target = pred.contiguous(), target.contiguous()
    out = torch.empty((b, 2), dtype=torch.float32, device=pred.device)
    if b == 0:
        return out
    scratch = torch.empty(int(_lib.load().kp_image_metrics_scratch_bytes(b, h, w)), dtype=torch.uint8, device=pred.device)
    call("kp_image_metrics", ptr(pred), ptr(target), b, h, w, c_void_p(scratch.data_ptr()), ptr(out), stream_ptr())
    return out


def image_metrics_masked(pred: torch.Tensor, target: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """Per-image (psnr_dynamic, ssim_dynamic, psnr_static, ssim_static) of a batch on the device
    (kp_image_metrics_masked): pred, target fp32 CUDA [B,H,W,3] with H, W >= 11, mask bool or uint8 [B,H,W] (non-zero:
    the dynamic region; the static region is the rest) -> fp32 [B,4].  Equal to ``utils.image_metrics.region_psnr_ssim``;
    NaN for a region without a pixel (SSIM: without a window centre).  No host synchronisation, so it can be captured in
    a CUDA graph."""
    if pred.dim() != 4 or pred.shape[-1] != 3 or target.shape != pred.shape:
        raise ValueError(f"image_metrics_masked: pred and target must both be [B,H,W,3] (got {tuple(pred.shape)}, "
                         f"{tuple(target.shape)})")
    if mask.shape != pred.shape[:3]:
        raise ValueError(f"image_metrics_masked: mask must be [B,H,W] = {tuple(pred.shape[:3])} (got {tuple(mask.shape)})")
    if pred.dtype != torch.float32 or target.dtype != torch.float32:
        raise TypeError("image_metrics_masked: pred and target must be float32")
    if mask.dtype not in (torch.bool, torch.uint8):
        raise TypeError(f"image_metrics_masked: mask must be bool or uint8 (got {mask.dtype})")
    if not pred.is_cuda or target.device != pred.device or mask.device != pred.device:
        raise RuntimeError("image_metrics_masked: pred, target and mask must be CUDA tensors on one device (there is no CPU path)")
    b, h, w = pred.shape[:3]
    if h < 11 or w < 11:
        raise ValueError(f"image_metrics_masked: {h}x{w} images are smaller than the 11x11 SSIM window")
    pred, target = pred.contiguous(), target.contiguous()
    mask = mask.contiguous()
    if mask.dtype == torch.bool:
        mask = mask.view(torch.uint8)  # one byte, 0 or 1
    out = torch.empty((b, 4), dtype=torch.float32, device=pred.device)
    if b == 0:
        return out
    scratch = torch.empty(int(_lib.load().kp_image_metrics_masked_scratch_bytes(b, h, w)), dtype=torch.uint8, device=pred.device)
    call("kp_image_metrics_masked", ptr(pred), ptr(target), c_void_p(mask.data_ptr()), b, h, w, c_void_p(scratch.data_ptr()),
         ptr(out), stream_ptr())
    return out


def depth_metrics(pred: torch.Tensor, gt: torch.Tensor, directions_norm: Optional[torch.Tensor] = None,
                  mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Per-image depth error of rendered depth against ground truth on the device (kp_depth_metrics): pred, gt and
    ``directions_norm`` fp32 CUDA [B,H,W] or [B,H,W,1], mask bool or uint8 [B,H,W] (non-zero: the dynamic region) ->
    float64 [B,R,8], row = (n_valid, abs_rel, sq_rel, rmse, rmse_log, delta1, delta2, delta3); R = 1 (whole image)
    without a mask, 3 (whole, dynamic, static) with one.  With ``directions_norm`` the ground truth is z-depth and is
    compared as gt * directions_norm (``is_euclidean_depth=False``).  Equal to ``utils.image_metrics.depth_metrics``;
    NaN for a region without a valid pixel.  No host synchronisation, so it can be captured in a CUDA graph."""
    maps = {"pred": pred, "gt": gt, "directions_norm": directions_norm}
    for name, t in maps.items():
        if t is not None and t.dim() == 4 and t.shape[-1] == 1:
            maps[name] = t = t.squeeze(-1)
        if t is not None and t.dim() != 3:
            raise ValueError(f"depth_metrics: {name} must be [B,H,W] or [B,H,W,1] (got {tuple(t.shape)})")
    pred, gt, directions_norm = maps["pred"], maps["gt"], maps["directions_norm"]
    if gt.shape != pred.shape or (directions_norm is not None and directions_norm.shape != pred.shape):
        raise ValueError(f"depth_metrics: pred, gt and directions_norm must have one shape (got {tuple(pred.shape)}, "
                         f"{tuple(gt.shape)}, {None if directions_norm is None else tuple(directions_norm.shape)})")
    if mask is not None and mask.shape != pred.shape:
        raise ValueError(f"depth_metrics: mask must be [B,H,W] = {tuple(pred.shape)} (got {tuple(mask.shape)})")
    b, h, w = pred.shape
    if h * w == 0:
        raise ValueError(f"depth_metrics: {h}x{w} images have no pixel")
    if any(t is not None and t.dtype != torch.float32 for t in (pred, gt, directions_norm)):
        raise TypeError("depth_metrics: pred, gt and directions_norm must be float32")
    if mask is not None and mask.dtype not in (torch.bool, torch.uint8):
        raise TypeError(f"depth_metrics: mask must be bool or uint8 (got {mask.dtype})")
    if not pred.is_cuda or any(t is not None and t.device != pred.device for t in (gt, directions_norm, mask)):
        raise RuntimeError("depth_metrics: every tensor must be a CUDA tensor on one device (there is no CPU path)")
    pred, gt = pred.contiguous(), gt.contiguous()
    directions_norm = None if directions_norm is None else directions_norm.contiguous()
    if mask is not None:
        mask = mask.contiguous()
        if mask.dtype == torch.bool:
            mask = mask.view(torch.uint8)  # one byte, 0 or 1
    out = torch.empty((b, 1 if mask is None else 3, 8), dtype=torch.float64, device=pred.device)
    if b == 0:
        return out
    scratch = torch.empty(int(_lib.load().kp_depth_metrics_scratch_bytes(b, h * w, int(mask is not None))), dtype=torch.uint8,
                          device=pred.device)
    call("kp_depth_metrics", ptr(pred), ptr(gt), ptr(directions_norm), c_void_p(0 if mask is None else mask.data_ptr()), b,
         h * w, c_void_p(scratch.data_ptr()), ptr(out), stream_ptr())
    return out


def eval_maps(pred: torch.Tensor, gt: torch.Tensor, depth: Optional[torch.Tensor] = None, gt_depth: Optional[torch.Tensor] = None,
              directions_norm: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    """Per-pixel error maps of a batch on the device (kp_eval_maps): pred, gt fp32 CUDA [B,H,W,3] with H, W >= 11; depth,
    gt_depth and directions_norm fp32 [B,H,W] or [B,H,W,1] -> fp32 [B,H,W] maps in physical units:

    - ``error``: the channel mean of |pred - gt|;
    - ``ssim``: the channel mean of the SSIM window centred on each pixel (``image_metrics``' window, constants and data
      range: ``utils.image_metrics.ssim_map`` averaged over channels), NaN on the 5-pixel border;
    - ``depth_error`` (with ``depth`` and ``gt_depth``): |max(depth, 1e-6) - g| / g, g = gt_depth * directions_norm (fp32)
      or gt_depth, NaN where g is not finite or not > 0 (``depth_metrics``' rule).

    No host synchronisation, so it can be captured in a CUDA graph."""
    if pred.dim() != 4 or pred.shape[-1] != 3 or gt.shape != pred.shape:
        raise ValueError(f"eval_maps: pred and gt must both be [B,H,W,3] (got {tuple(pred.shape)}, {tuple(gt.shape)})")
    if (depth is None) != (gt_depth is None):
        raise ValueError("eval_maps: depth and gt_depth are given together")
    if directions_norm is not None and depth is None:
        raise ValueError("eval_maps: directions_norm needs depth and gt_depth")
    maps = {"depth": depth, "gt_depth": gt_depth, "directions_norm": directions_norm}
    for name, t in maps.items():
        if t is not None and t.dim() == 4 and t.shape[-1] == 1:
            maps[name] = t = t.squeeze(-1)
        if t is not None and t.shape != pred.shape[:3]:
            raise ValueError(f"eval_maps: {name} must be [B,H,W] or [B,H,W,1] = {tuple(pred.shape[:3])} (got {tuple(t.shape)})")
    depth, gt_depth, directions_norm = maps["depth"], maps["gt_depth"], maps["directions_norm"]
    b, h, w = pred.shape[:3]
    if h < 11 or w < 11:
        raise ValueError(f"eval_maps: {h}x{w} images are smaller than the 11x11 SSIM window")
    tensors = [t for t in (pred, gt, depth, gt_depth, directions_norm) if t is not None]
    if any(t.dtype != torch.float32 for t in tensors):
        raise TypeError("eval_maps: every input must be float32")
    if not pred.is_cuda or any(t.device != pred.device for t in tensors):
        raise RuntimeError("eval_maps: every tensor must be a CUDA tensor on one device (there is no CPU path)")
    pred, gt = pred.contiguous(), gt.contiguous()
    depth, gt_depth, directions_norm = (None if t is None else t.contiguous() for t in (depth, gt_depth, directions_norm))
    out = {"error": torch.empty((b, h, w), dtype=torch.float32, device=pred.device),
           "ssim": torch.empty((b, h, w), dtype=torch.float32, device=pred.device)}
    if depth is not None:
        out["depth_error"] = torch.empty((b, h, w), dtype=torch.float32, device=pred.device)
    if b == 0:
        return out
    scratch = torch.empty(int(_lib.load().kp_eval_maps_scratch_bytes(b, h, w)), dtype=torch.uint8, device=pred.device)
    call("kp_eval_maps", ptr(pred), ptr(gt), ptr(depth), ptr(gt_depth), ptr(directions_norm), b, h, w,
         c_void_p(scratch.data_ptr()), ptr(out["error"]), ptr(out["ssim"]), ptr(out.get("depth_error")), stream_ptr())
    return out


COMPOSE_MAX_PANELS = 8
_COLORMAP_TABLES: Dict = {}


SCALAR_PANELS = ("accumulation", "accumulation_static", "dynamic", "error", "ssim", "depth_error", "dynamic_mask")


def panel_kind(name: str) -> int:
    """How ``compose_frame`` maps a rendered output: 1 = a scalar in [0, 1] through viridis (``SCALAR_PANELS``: the
    accumulations, the dynamics score ``dynamic`` and the eval maps the Evaluator scales into [0, 1]), 2 = a depth (turbo,
    blended with its accumulation; ns-render's rule: any other name containing "depth"), 0 = a colour shown as it is."""
    if name in SCALAR_PANELS:
        return 1
    return 2 if "depth" in name else 0


def accumulation_of(name: str) -> str:
    """The accumulation a depth panel is blended with: the static render's for ``depth_static``, the ground truth's
    validity mask ``depth_gt_valid`` (white where it has no depth) for the eval ground truth ``depth_gt``, else the
    frame's."""
    if name == "depth_gt":
        return "depth_gt_valid"
    return "accumulation_static" if name.endswith("_static") else "accumulation"


def _colormap_tables(device) -> Tuple[torch.Tensor, torch.Tensor]:
    key = str(device)
    if key not in _COLORMAP_TABLES:  # copied once per device: no host-to-device copy per frame
        from .utils import colormaps

        _COLORMAP_TABLES[key] = tuple(colormaps._table(c).to(device).contiguous() for c in ("turbo", "viridis"))
    return _COLORMAP_TABLES[key]


def compose_frame(frames: Dict[str, torch.Tensor], names: Sequence[str]) -> torch.Tensor:
    """The outputs ``names`` of one rendered frame (fp32 CUDA [H,W,3] colours, [H,W,1] accumulation / depths) ->
    uint8 [H, W*len(names), 3], side by side in that order, colour-mapped as ``get_image_metrics_and_images`` maps them
    (utils/colormaps.py; see ``panel_kind``) and quantised as floor(clamp(x, 0, 1) * 255 + 0.5) (kp_compose_frame_accs).
    A depth panel also needs its accumulation (``accumulation_of``): ``frames["accumulation"]``, or
    ``frames["accumulation_static"]`` for ``depth_static``.  On the current stream, no host synchronisation."""
    names = list(names)
    if not 1 <= len(names) <= COMPOSE_MAX_PANELS:
        raise ValueError(f"compose_frame: 1..{COMPOSE_MAX_PANELS} outputs per frame (got {len(names)})")
    missing = [n for n in names if n not in frames]
    if missing:
        raise ValueError(f"compose_frame: {missing} not among the frame's outputs {sorted(frames)}")
    kinds = [panel_kind(n) for n in names]
    acc_names = [accumulation_of(n) if k == 2 else None for n, k in zip(names, kinds)]
    lacking = sorted({a for a in acc_names if a is not None and a not in frames})
    if lacking:
        raise ValueError(f"compose_frame: a depth panel is blended with its accumulation, which the frame lacks: {lacking}")
    first = frames[names[0]]
    h, w = first.shape[:2]
    panels = []
    for name, kind in zip(names, kinds):
        t = frames[name]
        if t.dim() != 3 or tuple(t.shape[:2]) != (h, w) or t.shape[2] != (3 if kind == 0 else 1):
            raise ValueError(f"compose_frame: {name} is {tuple(t.shape)}; expected [{h},{w},{3 if kind == 0 else 1}]")
        if t.dtype != torch.float32:
            raise TypeError(f"compose_frame: {name} must be float32")
        if not t.is_cuda or t.device != first.device:
            raise RuntimeError("compose_frame: the outputs must be CUDA tensors on one device (there is no CPU path)")
        panels.append(t.contiguous())
    accs: Dict[str, torch.Tensor] = {}
    for a in acc_names:
        if a is None or a in accs:
            continue
        acc = frames[a]
        if tuple(acc.shape) != (h, w, 1) or acc.dtype != torch.float32 or acc.device != first.device:
            raise ValueError(f"compose_frame: {a} must be fp32 [{h},{w},1] on {first.device}")
        accs[a] = acc.contiguous()
    turbo, viridis = _colormap_tables(first.device)
    p = len(panels)
    out = torch.empty((h, w * p, 3), dtype=torch.uint8, device=first.device)
    scratch = torch.empty(int(_lib.load().kp_compose_frame_scratch_bytes(h, w, p)), dtype=torch.uint8, device=first.device)
    kind_arr = (c_int32 * p)(*kinds)
    call("kp_compose_frame_accs", _lib.ptr_array(panels), kind_arr, _lib.ptr_array([accs.get(a) for a in acc_names]), p, h, w,
         ptr(turbo), ptr(viridis), c_void_p(scratch.data_ptr()), c_void_p(out.data_ptr()), stream_ptr())
    return out


_JPEG_HEADERS: Dict = {}
JPEG_HEADER_BYTES = 613  # KP_JPEG_HEADER_BYTES


def _jpeg_header(device, h: int, w: int, quality: int) -> torch.Tensor:
    key = (str(device), h, w, quality)
    if key not in _JPEG_HEADERS:  # built on the host and copied once per (device, size, quality): no copy per frame
        host = torch.empty(JPEG_HEADER_BYTES, dtype=torch.uint8)
        call("kp_jpeg_header", h, w, quality, c_void_p(host.data_ptr()))
        _JPEG_HEADERS[key] = host.to(device)
    return _JPEG_HEADERS[key]


def jpeg_capacity(h: int, w: int) -> int:
    """Bytes ``encode_jpeg`` reserves for an h x w image: the worst-case file size (kp_jpeg_encode_capacity)."""
    return int(_lib.load().kp_jpeg_encode_capacity(h, w))


def encode_jpeg(image: torch.Tensor, quality: int = 95) -> Tuple[torch.Tensor, torch.Tensor]:
    """A uint8 RGB CUDA image [H, W, 3] -> one baseline JPEG (JFIF, YCbCr 4:2:0, IJG ``quality`` 1..100) encoded on the
    device (kp_jpeg_encode): ``(bytes uint8 [jpeg_capacity(H, W)], length int64 [1])``, both on the image's device; the
    file is ``bytes[:length]``.  On the current stream, no host synchronisation (graph-capturable once the header for
    this size and quality has been built by an earlier call)."""
    if not isinstance(quality, int) or isinstance(quality, bool) or not 1 <= quality <= 100:
        raise ValueError(f"encode_jpeg: quality {quality!r} is not an integer in 1..100")
    if image.dim() != 3 or image.shape[2] != 3:
        raise ValueError(f"encode_jpeg: image is {tuple(image.shape)}; expected [H, W, 3]")
    h, w = int(image.shape[0]), int(image.shape[1])
    if not (1 <= h <= 65535 and 1 <= w <= 65535):
        raise ValueError(f"encode_jpeg: a {h}x{w} image; JPEG needs 1..65535 rows and columns")
    if image.dtype != torch.uint8:
        raise TypeError(f"encode_jpeg: image must be uint8 (got {image.dtype})")
    if not image.is_cuda:
        raise RuntimeError("encode_jpeg: image must be a CUDA tensor (there is no CPU path)")
    image = image.contiguous()
    dev = image.device
    header = _jpeg_header(dev, h, w, quality)
    out = torch.empty(jpeg_capacity(h, w), dtype=torch.uint8, device=dev)
    length = torch.empty(1, dtype=torch.int64, device=dev)
    scratch = torch.empty(int(_lib.load().kp_jpeg_encode_scratch_bytes(h, w)), dtype=torch.uint8, device=dev)
    call("kp_jpeg_encode", c_void_p(image.data_ptr()), h, w, c_void_p(header.data_ptr()), c_void_p(scratch.data_ptr()),
         c_void_p(out.data_ptr()), ptr(length), stream_ptr())
    return out, length


_HEAD_WS: Dict = {}


def _head_workspace(device) -> torch.Tensor:
    key = (device.type, device.index)
    if key not in _HEAD_WS:
        _HEAD_WS[key] = torch.zeros(4, dtype=torch.float64, device=device)
    return _HEAD_WS[key]


class _LossHead(torch.autograd.Function):
    """(vals3, total, psnr) from the per-ray / per-sample loss tensors; see csrc/loss_head.cu."""

    @staticmethod
    def forward(ctx, coefs, extra, pred, image, dist, *il):
        ctx.set_materialize_grads(False)
        pred_c, image_c = f32c(pred.detach()), f32c(image.detach())
        n = pred_c.shape[0]
        dist_c = None if dist is None else f32c(dist.detach()).view(-1)
        il_c = [f32c(t.detach()) for t in il]
        counts = (c_int64 * max(1, len(il_c)))(*[t.numel() for t in il_c])
        ptrs = (c_void_p * max(1, len(il_c)))(*[t.data_ptr() for t in il_c])
        dev = pred_c.device
        vals = torch.empty(3, dtype=torch.float32, device=dev)
        total, psnr = torch.empty((), dtype=torch.float32, device=dev), torch.empty((), dtype=torch.float32, device=dev)
        extra_c = None if extra is None else f32c(extra.detach()).view(-1)
        call("kp_loss_head_fwd", ptr(pred_c), ptr(image_c), n, ptr(dist_c), ptrs, counts, len(il_c), float(coefs[0]),
             float(coefs[1]), float(coefs[2]), ptr(extra_c), 0 if extra_c is None else extra_c.numel(),
             ptr(_head_workspace(dev)), ptr(vals), ptr(total), ptr(psnr), stream_ptr())
        ctx.save_for_backward(pred_c, image_c)
        ctx.meta = (coefs, n, dist is not None, [tuple(t.shape) for t in il], counts)
        ctx.mark_non_differentiable(psnr)
        return vals, total, psnr

    @staticmethod
    def backward(ctx, g_vals, g_total, _g_psnr):
        pred_c, image_c = ctx.saved_tensors
        coefs, n, has_dist, il_shapes, counts = ctx.meta
        dev = pred_c.device
        need = ctx.needs_input_grad
        g_pred = torch.empty_like(pred_c) if need[2] else None
        g_dist = torch.empty(n, dtype=torch.float32, device=dev) if (has_dist and need[4]) else None
        g_il = [torch.empty(sh, dtype=torch.float32, device=dev) if need[5 + i] else None for i, sh in enumerate(il_shapes)]
        gptrs = (c_void_p * max(1, len(g_il)))(*[0 if t is None else t.data_ptr() for t in g_il])
        call("kp_loss_head_bwd", ptr(pred_c), ptr(image_c), n, counts, len(il_shapes), float(coefs[0]), float(coefs[1]),
             float(coefs[2]), ptr(None if g_total is None else f32c(g_total)), ptr(None if g_vals is None else f32c(g_vals)),
             ptr(g_pred), ptr(g_dist), gptrs, stream_ptr())
        return (None, None, g_pred, None, g_dist, *g_il)


def loss_head(pred: torch.Tensor, image: torch.Tensor, dist_per_ray: Optional[torch.Tensor], interlevel: Sequence[torch.Tensor],
              coef_rgb: float, coef_dist: float, coef_il: float, extra: Optional[torch.Tensor] = None):
    """-> (vals [3] = scaled rgb / distortion / interlevel losses, total = their sum + sum(extra), psnr), one kernel.
    ``dist_per_ray`` [N] from lossfun_distortion, ``interlevel`` = per-level lossfun_outer outputs [N,S_l]."""
    pred2 = pred.reshape(-1, 3)
    dist = None if dist_per_ray is None else dist_per_ray.reshape(-1)
    return _LossHead.apply((coef_rgb, coef_dist, coef_il), extra, pred2, image.reshape(-1, 3), dist, *interlevel)


class _PlaneReg(torch.autograd.Function):
    """sums[p] = (sum dh^2, sum dw^2, sum (d2h)^2, sum |1-t|) for each plane p, masked by terms[p].
    The forward is one sums-only ``plane_reg_fused`` sweep; the backward one gradient-only sweep per target kind."""

    @staticmethod
    def forward(ctx, terms: Tuple[int, ...], *planes):
        ctx.sinks = [grad_sink(p) for p in planes]
        ctx.planes, ctx.terms = [as_channel_last(p.detach()) for p in planes], terms
        return plane_reg_fused(ctx.planes, terms, None, [None] * len(planes), accumulate=False).float()

    @staticmethod
    def backward(ctx, gsums):
        global PLANE_REG_BACKWARDS
        PLANE_REG_BACKWARDS += 1
        planes = ctx.planes
        need = [bool(t) and ctx.needs_input_grad[1 + i] for i, t in enumerate(ctx.terms)]
        idx = [i for i, n in enumerate(need) if n]
        if not idx:
            return (None,) * (1 + len(planes))
        g = f32c(gsums)
        grads = [None] * len(planes)
        for accumulate in (True, False):  # sunk planes: accumulate into the sink; others: write a fresh gradient tensor
            sub = [i for i in idx if (ctx.sinks[i] is not None) == accumulate]
            if not sub:
                continue
            if accumulate:
                tgt = [ctx.sinks[i] for i in sub]
            else:
                flat = torch.empty(sum(planes[i].numel() for i in sub), dtype=torch.float32, device=g.device)
                tgt, off = [], 0
                for i in sub:
                    _, c, h, w = planes[i].shape
                    grads[i] = flat[off: off + planes[i].numel()].view(1, h, w, c).permute(0, 3, 1, 2)
                    tgt.append(grads[i])
                    off += planes[i].numel()
            coef = g if len(sub) == len(planes) else g[sub].contiguous()
            plane_reg_fused([planes[i] for i in sub], [ctx.terms[i] for i in sub], coef, tgt, accumulate, want_sums=False)
        return (None, *grads)


def plane_reg_fused(planes: Sequence[torch.Tensor], terms: Sequence[int], coef_dev: Optional[torch.Tensor],
                    targets: Sequence[Optional[torch.Tensor]], accumulate: bool, want_sums: bool = True,
                    write_range: Optional[torch.Tensor] = None, sums_in_range: bool = False) -> Optional[torch.Tensor]:
    """One sweep per plane: -> sums [P,4] (float64) of the regulariser terms, and targets[p] (channel-last gradient
    buffers, entries may be None) = / += sum_i coef_dev[p,i] * d(sums[p,i])/d(plane).  ``coef_dev`` may be None when
    every target is None.  No autograd: the training step's gradient goes straight into the parameter's bucket (and,
    with accumulate=False, replaces the bucket's memset); ``plane_reg_sums`` wraps it for autograd."""
    planes = [as_channel_last(p.detach()) for p in planes]
    for p, t in zip(planes, targets):
        ptr_cl(p)
        if t is not None and (t.shape != p.shape or t.stride() != p.stride() or t.dtype != torch.float32):
            raise RuntimeError("plane_reg_fused: a gradient target must have the plane's channel-last layout")
    sums = torch.zeros((len(planes), 4), dtype=torch.float64, device=planes[0].device) if want_sums else None
    coef = None if coef_dev is None else f32c(coef_dev)
    hwc, tm = _reg_tables(planes, terms)
    if write_range is not None:  # int64 [P,2] on the device: float4 element range of each plane whose gradient is written
        if write_range.dtype != torch.int64 or tuple(write_range.shape) != (len(planes), 2):
            raise RuntimeError("plane_reg_fused: write_range must be int64 [P,2]")
        # sums_in_range: the shard form -- sums restricted to the range too, tiles outside it skipped
        call("kp_plane_reg_fused_shard" if sums_in_range else "kp_plane_reg_fused_range", _plane_ptrs(planes),
             _plane_ptrs(list(targets)), hwc, tm, len(planes), ptr(coef), int(accumulate), ptr(sums), ptr(write_range),
             stream_ptr())
        return sums
    call("kp_plane_reg_fused", _plane_ptrs(planes), _plane_ptrs(list(targets)), hwc, tm, len(planes), ptr(coef),
         int(accumulate), ptr(sums), stream_ptr())
    return sums


def repack(src: torch.Tensor, dst: torch.Tensor, to_channel_last: bool) -> None:
    """One plane [1,C,H,W]: NCHW-contiguous ``src`` -> channel-last ``dst`` (or the reverse), on the device."""
    _, c, h, w = src.shape
    if dst.shape != src.shape:
        raise RuntimeError("repack: shape mismatch")
    call("kp_repack_nchw_to_hwc" if to_channel_last else "kp_repack_hwc_to_nchw", c_void_p(src.data_ptr()),
         c_void_p(dst.data_ptr()), c, h, w, stream_ptr())


def ptr_cl(p: torch.Tensor) -> c_void_p:
    if not p.is_cuda:
        raise RuntimeError("soccernerfs_b200 kernels need CUDA tensors (there is no CPU path)")
    return c_void_p(p.data_ptr())


def plane_reg_sums(planes: Sequence[torch.Tensor], terms: Sequence[int]) -> torch.Tensor:
    """-> [P,4] raw sums; bit i of terms[p] selects sum i (see include/kplanes_b200.h)."""
    return _PlaneReg.apply(tuple(int(t) for t in terms), *planes)


# ------------------------------------------------------------------------------------------------
# (f1) Adam
# ------------------------------------------------------------------------------------------------
def plane_reg_adam_supported(c: int) -> bool:
    return bool(_lib.load().kp_plane_reg_adam_supported(int(c)))


def plane_reg_adam_scratch_bytes(planes: Sequence[torch.Tensor]) -> int:
    hwc, _ = _reg_tables(planes, [0] * len(planes))
    return int(_lib.load().kp_plane_reg_adam_scratch_bytes(hwc, len(planes)))


def plane_reg_adam_(planes, grads, exp_avgs, exp_avg_sqs, terms, coef_dev, lr, beta1, beta2, eps, weight_decay, step,
                    grad_scale, scratch: torch.Tensor, sums: Optional[torch.Tensor] = None, zero_grads: bool = True,
                    hyper_dev: Optional[torch.Tensor] = None) -> None:
    """(f1) regulariser stencil + Adam in one streaming pass per plane (kp_plane_reg_adam): planes / grads / moments are
    channel-last [1,C,H,W] tensors sharing one layout; ``coef_dev`` [P,4] weights the four regulariser sums' gradients,
    which are computed from the pre-update planes and added to ``grads * grad_scale``; ``sums`` [P,4] float64 (optional)
    accumulates the sums themselves (the loss values); ``zero_grads`` leaves the gradient buffers zeroed for the next
    step.  ``scratch``: uint8 CUDA tensor of >= plane_reg_adam_scratch_bytes(planes) bytes."""
    n = len(planes)
    if n == 0:
        return
    for p, g, m, v in zip(planes, grads, exp_avgs, exp_avg_sqs):
        if not is_channel_last(p) or not (g.stride() == p.stride() == m.stride() == v.stride()) or g.dtype != torch.float32:
            raise RuntimeError("plane_reg_adam_: plane / grad / moments must share one channel-last fp32 layout")
        ptr_cl(p)
    hwc, tm = _reg_tables(planes, terms)
    call("kp_plane_reg_adam", _plane_ptrs(planes), _plane_ptrs(grads), _plane_ptrs(exp_avgs), _plane_ptrs(exp_avg_sqs), hwc, tm, n,
         ptr(f32c(coef_dev)), float(lr), float(beta1), float(beta2), float(eps), float(weight_decay), int(step), float(grad_scale),
         ptr(hyper_dev), ptr(sums), c_void_p(scratch.data_ptr()), int(scratch.numel() * scratch.element_size()), int(zero_grads),
         stream_ptr())


def adam_multi_(params, grads, exp_avgs, exp_avg_sqs, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0,
                hyper_dev: Optional[torch.Tensor] = None) -> None:
    """One launch of torch.optim.Adam's update over a list of dense fp32 tensors (same layout per tuple)."""
    from ctypes import c_int64

    n = len(params)
    if n == 0:
        return
    sizes = (c_int64 * n)()
    for i, (p, g, m, v) in enumerate(zip(params, grads, exp_avgs, exp_avg_sqs)):
        if not (g.stride() == p.stride() == m.stride() == v.stride()) or g.dtype != torch.float32:
            raise RuntimeError("adam_multi_: param/grad/state must share one dense fp32 layout")
        sizes[i] = p.numel()
    call("kp_adam_multi", _plane_ptrs(params), _plane_ptrs(grads), _plane_ptrs(exp_avgs), _plane_ptrs(exp_avg_sqs), sizes, n,
         float(lr), float(beta1), float(beta2), float(eps), float(weight_decay), int(step), float(grad_scale),
         ptr(hyper_dev), stream_ptr())
