"""Losses of the K-Planes training step on the B200 kernels.

Same function names / arguments as NS/model_components/losses.py: ``outer``-based ``lossfun_outer`` :78-95 and
``interlevel_loss`` :106-121, ``lossfun_distortion`` :125-136 and ``distortion_loss`` :139-144, the K-Planes plane
regularisers ``compute_plane_tv`` :356-366, ``compute_plane_smoothness`` :369-380, ``space_tv_loss`` :383-406,
``time_smoothness_loss`` :409-428, ``sparse_transients_loss`` :431-452, and the DS-NeRF ``depth_loss`` :213-313.
The plane regularisers stream every plane once (forward) / once more (backward) with analytic gradients
instead of building an autograd graph of slices.
"""
from __future__ import annotations

from enum import Enum
from typing import List, Sequence

import torch
from torch import nn

from .. import ops
from ..cameras.rays import RaySamples

L1Loss = nn.L1Loss
MSELoss = nn.MSELoss
LOSSES = {"L1": L1Loss, "MSE": MSELoss}
EPS = 1.0e-7
URF_SIGMA_SCALE_FACTOR = 3.0

T_H, T_W, T_SMOOTH, T_L1 = 1, 2, 4, 8  # term bits of kp_plane_reg_*


class DepthLossType(Enum):
    DS_NERF = 1
    URF = 2


def lossfun_outer(t: torch.Tensor, w: torch.Tensor, t_env: torch.Tensor, w_env: torch.Tensor) -> torch.Tensor:
    """clip(w - w_outer, 0)^2 / (w + eps) with w_outer the envelope histogram (t_env, w_env) resampled onto t."""
    s, sp = w.shape[-1], w_env.shape[-1]
    out = ops.lossfun_outer(t.reshape(-1, s + 1), w.reshape(-1, s), t_env.reshape(-1, sp + 1), w_env.reshape(-1, sp))
    return out.view(w.shape)


def ray_samples_to_sdist(ray_samples: RaySamples) -> torch.Tensor:
    """[N,S+1] bin edges in the normalised spacing domain (losses.py:98-103)."""
    from .ray_samplers import spacing_edges

    return spacing_edges(ray_samples)


def interlevel_loss(weights_list: List[torch.Tensor], ray_samples_list: List[RaySamples]) -> torch.Tensor:
    """mip-NeRF 360 proposal loss; only the proposal weights receive gradient (losses.py:106-121)."""
    c = ray_samples_to_sdist(ray_samples_list[-1]).detach()
    w = weights_list[-1][..., 0].detach()
    loss_interlevel = 0.0
    for ray_samples, weights in zip(ray_samples_list[:-1], weights_list[:-1]):
        cp = ray_samples_to_sdist(ray_samples)
        wp = weights[..., 0]
        loss_interlevel = loss_interlevel + torch.mean(lossfun_outer(c, w, cp, wp))
    return loss_interlevel


def interlevel_terms(weights_list: List[torch.Tensor], ray_samples_list: List[RaySamples]) -> List[torch.Tensor]:
    """The per-level [N,S] tensors whose means ``interlevel_loss`` adds up (for the fused loss head)."""
    c = ray_samples_to_sdist(ray_samples_list[-1]).detach()
    w = weights_list[-1][..., 0].detach()
    return [lossfun_outer(c, w, ray_samples_to_sdist(rs), ws[..., 0]) for rs, ws in zip(ray_samples_list[:-1], weights_list[:-1])]


def lossfun_distortion(t: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """Per-ray distortion (inter + intra terms), t [..., S+1], w [..., S] -> [...]."""
    s = w.shape[-1]
    return ops.distortion_per_ray(t.reshape(-1, s + 1), w.reshape(-1, s)).view(w.shape[:-1])


def distortion_per_ray(weights_list, ray_samples_list) -> torch.Tensor:
    """[N] per-ray distortion of the last level; ``distortion_loss`` is its mean."""
    c = ray_samples_to_sdist(ray_samples_list[-1])
    w = weights_list[-1][..., 0]
    return lossfun_distortion(c, w)


def distortion_loss(weights_list, ray_samples_list) -> torch.Tensor:
    return torch.mean(distortion_per_ray(weights_list, ray_samples_list))


# ---- K-Planes plane regularisers ----------------------------------------------------------------------
def compute_plane_tv(t: torch.Tensor, only_w: bool = False) -> torch.Tensor:
    """mean squared first difference along H (unless only_w) and W of a [1,C,H,W] plane (losses.py:356-366)."""
    _, c, h, w = t.shape
    sums = ops.plane_reg_sums([t], [T_W if only_w else T_H | T_W])[0]
    w_tv = sums[1] / (c * h * (w - 1))
    return w_tv if only_w else sums[0] / (c * (h - 1) * w) + w_tv


def compute_plane_smoothness(t: torch.Tensor) -> torch.Tensor:
    """mean squared second difference along H (= time for space-time planes) (losses.py:369-380)."""
    _, c, h, w = t.shape
    return ops.plane_reg_sums([t], [T_SMOOTH])[0][2] / (c * (h - 2) * w)


_CONST_CACHE = {}


def _const(values, device) -> torch.Tensor:
    """Small constant tensors (normalisers) cached per device so a training step makes no H2D copy for them."""
    key = (repr(values), str(device))
    if key not in _CONST_CACHE:
        _CONST_CACHE[key] = torch.tensor(values, dtype=torch.float32, device=device)
    return _CONST_CACHE[key]


def _flatten_grids(multi_res_grids) -> List[Sequence[torch.Tensor]]:
    return [list(g) for g in multi_res_grids]


def space_tv_loss(multi_res_grids) -> torch.Tensor:
    """TV in space: 2-D on space planes, 1-D (along the spatial axis = W) on space-time planes (losses.py:383-406)."""
    planes, terms, norms = [], [], []
    for grids in _flatten_grids(multi_res_grids):
        spatial = [0, 1, 2] if len(grids) == 3 else [0, 1, 3]
        for gid, g in enumerate(grids):
            _, c, h, w = g.shape
            planes.append(g)
            if gid in spatial:
                terms.append(T_H | T_W)
                norms.append([1.0 / (c * (h - 1) * w), 1.0 / (c * h * (w - 1))])
            else:
                terms.append(T_W)
                norms.append([0.0, 1.0 / (c * h * (w - 1))])
    sums = ops.plane_reg_sums(planes, terms)
    return (sums[:, :2] * _const(norms, sums.device)).sum()


def time_smoothness_loss(multi_res_grids) -> torch.Tensor:
    """Second-derivative penalty along time on the space-time planes (losses.py:409-428)."""
    planes, norms = [], []
    for grids in _flatten_grids(multi_res_grids):
        for gid in [] if len(grids) == 3 else [2, 4, 5]:
            _, c, h, w = grids[gid].shape
            planes.append(grids[gid])
            norms.append(1.0 / (c * (h - 2) * w))
    if not planes:
        return torch.as_tensor(0.0)
    sums = ops.plane_reg_sums(planes, [T_SMOOTH] * len(planes))
    return (sums[:, 2] * _const(norms, sums.device)).sum()


def sparse_transients_loss(multi_res_grids) -> torch.Tensor:
    """L1 distance of the space-time planes from 1 (losses.py:431-452)."""
    planes, norms = [], []
    for grids in _flatten_grids(multi_res_grids):
        if len(grids) == 3:
            continue
        for gid in [2, 4, 5]:
            planes.append(grids[gid])
            norms.append(1.0 / grids[gid].numel())
    if not planes:
        return torch.as_tensor(0.0)
    sums = ops.plane_reg_sums(planes, [T_L1] * len(planes))
    return (sums[:, 3] * _const(norms, sums.device)).sum()


# ---- depth supervision (plain torch: [N,S] elementwise, only when depth images are in the batch) -----
def ds_nerf_depth_loss(weights, termination_depth, steps, lengths, sigma) -> torch.Tensor:
    """losses.py:213-235."""
    depth_mask = termination_depth > 0
    loss = -torch.log(weights + EPS) * torch.exp(-((steps - termination_depth[:, None]) ** 2) / (2 * sigma)) * lengths
    loss = loss.sum(-2) * depth_mask
    return torch.mean(loss)


def urban_radiance_field_depth_loss(weights, termination_depth, predicted_depth, steps, sigma) -> torch.Tensor:
    """losses.py:238-274."""
    depth_mask = termination_depth > 0
    expected_depth_loss = (termination_depth - predicted_depth) ** 2
    target_distribution = torch.distributions.normal.Normal(0.0, sigma / URF_SIGMA_SCALE_FACTOR)
    termination_depth = termination_depth[:, None]
    near_mask = torch.logical_and(steps <= termination_depth + sigma, steps >= termination_depth - sigma)
    near = (weights - torch.exp(target_distribution.log_prob(steps - termination_depth))) ** 2
    near = (near_mask * near).sum(-2)
    empty = ((steps < termination_depth - sigma) * weights**2).sum(-2)
    return torch.mean((expected_depth_loss + near + empty) * depth_mask)


def depth_loss(weights, ray_samples, termination_depth, predicted_depth, sigma, directions_norm, is_euclidean,
               depth_loss_type) -> torch.Tensor:
    """losses.py:277-313."""
    if not is_euclidean:
        termination_depth = termination_depth * directions_norm
    steps = (ray_samples.frustums.starts + ray_samples.frustums.ends) / 2
    if depth_loss_type == DepthLossType.DS_NERF:
        lengths = ray_samples.frustums.ends - ray_samples.frustums.starts
        return ds_nerf_depth_loss(weights, termination_depth, steps, lengths, sigma)
    if depth_loss_type == DepthLossType.URF:
        return urban_radiance_field_depth_loss(weights, termination_depth, predicted_depth, steps, sigma)
    raise NotImplementedError("Provided depth loss type not implemented.")


REG_NAMES = ["space_tv_loss", "time_smoothness_loss", "sparse_transients_loss",
             "space_tv_proposal_loss", "time_smoothness_proposal_loss", "sparse_transients_proposal_loss"]


def regularizer_plan(ms_grids_nerf, ms_grids_prop):
    """(planes, terms, norm rows [P][6][4]) of the six plane regularisers of NS/models/kplanes.py:430-446: which sums of
    which plane enter which loss, with the reference's mean normalisers (losses.py:356-452)."""
    planes, terms, rows = [], [], []
    for group, ms in enumerate((_flatten_grids(ms_grids_nerf), _flatten_grids(ms_grids_prop))):
        for grids in ms:
            dynamic = len(grids) == 6
            spatial = [0, 1, 3] if dynamic else [0, 1, 2]
            for gid, g in enumerate(grids):
                _, c, h, w = g.shape
                row = [[0.0] * 4 for _ in range(6)]
                if gid in spatial:
                    t = T_H | T_W
                    row[3 * group + 0][0] = 1.0 / (c * (h - 1) * w)
                    row[3 * group + 0][1] = 1.0 / (c * h * (w - 1))
                else:
                    t = T_W | T_SMOOTH | T_L1
                    row[3 * group + 0][1] = 1.0 / (c * h * (w - 1))
                    row[3 * group + 1][2] = 1.0 / (c * (h - 2) * w)
                    row[3 * group + 2][3] = 1.0 / g.numel()
                planes.append(g)
                terms.append(t)
                rows.append(row)
    return planes, terms, rows


def kplanes_regularizers_into_grads(ms_grids_nerf, ms_grids_prop, loss_coefficients, accumulate: bool = False,
                                    write_range=None, grad_scale=None, sums_in_range: bool = False, sum_scale=None):
    """The training step's form of ``kplanes_regularizers``: ONE sweep per plane that returns the six SCALED loss values
    (detached; keyed like the reference's loss dict) and writes (``accumulate=False``: the sweep replaces the gradient
    buffer's memset) or adds the scaled regularisers' gradient into every plane's gradient sink (``ops.grad_sink``).
    Planes without a sink (frozen / no bucket attached) only contribute their value.
    ``write_range`` (int64 [P,2] device tensor) / ``grad_scale`` ([P] device tensor): the data-parallel step with the sparse
    gradient exchange writes each plane's gradient only inside this rank's shard of the bucket, pre-multiplied by the world
    size (the reduction then divides the sum by it).  ``sums_in_range``: the loss VALUES are this rank's share as well (the
    sweep reads only its shard; the caller sums the returned values over the ranks); ``sum_scale`` ([P] device tensor) then
    weights each plane's share (1/world for a plane every rank sweeps in full)."""
    planes, terms, rows = regularizer_plan(ms_grids_nerf, ms_grids_prop)
    dev = planes[0].device
    scale = [float(loss_coefficients.get(n, 0.0)) for n in REG_NAMES]
    norm = _const(rows, dev)  # [P,6,4]
    coef = _const([[sum(scale[j] * r[j][i] for j in range(6)) for i in range(4)] for r in rows], dev)  # [P,4]
    if grad_scale is not None:  # [P] per-plane factor on the GRADIENT only (the values below stay unscaled)
        coef = coef * grad_scale[:, None]
    targets = [ops.grad_sink(p) for p in planes]
    sums = ops.plane_reg_fused(planes, terms, coef, targets, accumulate, write_range=write_range, sums_in_range=sums_in_range)
    if sum_scale is not None:
        sums = sums * sum_scale.to(sums.dtype)[:, None]
    vals = (sums.float()[:, None, :] * norm).sum(dim=(0, 2)) * _const(scale, dev)  # [6], already scaled
    return {name: vals[i] for i, name in enumerate(REG_NAMES) if name in loss_coefficients}, targets


def kplanes_regularizers(ms_grids_nerf, ms_grids_prop):
    """All six plane regularisers of ``KPlanesModel.get_loss_dict`` (NS/models/kplanes.py:430-446) from ONE pass over
    the planes: identical values to ``space_tv_loss`` / ``time_smoothness_loss`` / ``sparse_transients_loss`` called on
    the field grids and on the proposal grids, but each plane is streamed once forward and once backward and receives
    a single gradient contribution.  Returns a dict keyed like the reference's loss dict."""
    planes, terms, rows = regularizer_plan(ms_grids_nerf, ms_grids_prop)
    sums = ops.plane_reg_sums(planes, terms)  # [P,4]
    norm = _const(rows, sums.device)  # [P,6,4]
    vals = (sums[:, None, :] * norm).sum(dim=(0, 2))  # [6]
    return {name: vals[i] for i, name in enumerate(REG_NAMES)}
