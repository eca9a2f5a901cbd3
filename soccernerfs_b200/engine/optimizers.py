"""Optimizer / scheduler pieces the K-Planes training step needs (SURVEY.md 8f rank 1).

``FusedAdam`` has torch.optim.Adam's math (the reference uses ``AdamOptimizerConfig(lr=1e-2, eps=1e-12)``,
NS/configs/method_configs.py:546-557, NS/engine/optimizers.py:74-160) executed by ``kp_adam_multi``: one
vectorised pass over param / grad / exp_avg / exp_avg_sq of every parameter of a group that shares a step count.
``cosine_decay_factor`` is the reference's ``CosineDecayScheduler`` lambda (NS/engine/schedulers.py:126-142).
"""
from __future__ import annotations

from typing import Callable, Dict, Iterable, Optional

import numpy as np
import torch

from .. import ops


class FusedAdam(torch.optim.Optimizer):
    def __init__(self, params: Iterable, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))

    @torch.no_grad()
    def step(self, closure=None, grad_scale: float = 1.0, use_device_hyper: bool = True, plane_reg: "PlaneRegAdamPlan" = None):
        """``grad_scale`` multiplies every gradient before use (e.g. 1/GradScaler scale, or 1/world_size).
        ``use_device_hyper``: read lr / bias corrections from the group's ``hyper_dev`` device triple when it has one (the
        graph-replayed step keeps them there); False = the host-side values of this call.
        ``plane_reg``: the planes it lists are updated by the fused regulariser + Adam pass (their regulariser gradient is
        computed inside that pass, their gradient buffers are left zeroed); everything else by the plain Adam kernel."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        for group in self.param_groups:
            b1, b2 = group["betas"]
            launches = {}  # step count -> (params, grads, exp_avgs, exp_avg_sqs)
            rp = []  # planes of this group routed through the fused regulariser + Adam pass
            for p in group["params"]:
                if p.grad is None or p.numel() == 0:
                    continue
                g = p.grad
                if g.dtype != torch.float32 or g.stride() != p.stride():
                    g = torch.empty_like(p, memory_format=torch.preserve_format).copy_(g)
                st = self.state[p]
                if not st:
                    st["step"] = 0
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st["step"] += 1
                if plane_reg is not None and plane_reg.covers(p):
                    if g is not p.grad:  # (never with the gradient buckets: their views share the planes' layout)
                        raise RuntimeError("fused regulariser + Adam pass: a plane's gradient must share the plane's layout")
                    rp.append(p)
                    continue
                ps, gs, ms, vs = launches.setdefault(st["step"], ([], [], [], []))
                ps.append(p), gs.append(g), ms.append(st["exp_avg"]), vs.append(st["exp_avg_sq"])
            if rp:
                steps = {self.state[p]["step"] for p in rp}
                if len(steps) != 1:
                    raise RuntimeError("fused regulariser + Adam pass: the planes of a group must share one step count")
                plane_reg.step_group(rp, [p.grad for p in rp], [self.state[p]["exp_avg"] for p in rp],
                                     [self.state[p]["exp_avg_sq"] for p in rp], group["lr"], b1, b2, group["eps"],
                                     group["weight_decay"], steps.pop(), grad_scale,
                                     hyper_dev=group.get("hyper_dev") if use_device_hyper else None)
            # parameters that joined the optimizer at different times have different step counts: one launch per count,
            # with the host's scalars (the device triple holds the bias corrections of one step count)
            hyper_dev = group.get("hyper_dev") if use_device_hyper and len(launches) == 1 else None
            for step, (ps, gs, ms, vs) in launches.items():
                ops.adam_multi_(ps, gs, ms, vs, group["lr"], b1, b2, group["eps"], group["weight_decay"], step, grad_scale,
                                hyper_dev=hyper_dev)
        return loss


def cosine_decay_factor(step: int, warm_up_end: int, max_steps: int, learning_rate_alpha: float = 0.0) -> float:
    if step < warm_up_end:
        return step / warm_up_end
    progress = (step - warm_up_end) / (max_steps - warm_up_end)
    return float((np.cos(np.pi * progress) + 1.0) * 0.5 * (1 - learning_rate_alpha) + learning_rate_alpha)


class Optimizers:
    """One FusedAdam + cosine LambdaLR per parameter group, keyed like ``Model.get_param_groups()`` /
    ``TrainerConfig.optimizers`` ("proposal_networks", "fields")."""

    def __init__(self, param_groups: Dict[str, list], lr: float = 1e-2, eps: float = 1e-12, warm_up_end: int = 512,
                 max_steps: int = 30000, learning_rate_alpha: float = 0.0) -> None:
        self.optimizers, self.schedulers, self.parameters = {}, {}, param_groups
        for name, params in param_groups.items():
            opt = FusedAdam(params, lr=lr, eps=eps)
            self.optimizers[name] = opt
            self.schedulers[name] = torch.optim.lr_scheduler.LambdaLR(
                opt, lr_lambda=lambda s: cosine_decay_factor(s, warm_up_end, max_steps, learning_rate_alpha))

    def zero_grad_all(self) -> None:
        for opt in self.optimizers.values():
            opt.zero_grad(set_to_none=True)

    def optimizer_step_all(self, grad_scale: float = 1.0, use_device_hyper: bool = True, plane_reg: "PlaneRegAdamPlan" = None,
                           before: Optional[Dict[str, Callable[[], None]]] = None) -> None:
        """``before[name]()`` runs right before group ``name`` is stepped (e.g. a stream join only that group needs);
        groups with such a hook are stepped last."""
        if plane_reg is not None:
            plane_reg.begin_step()
        before = before or {}
        for name in sorted(self.optimizers, key=lambda n: n in before):  # (stable: the other groups keep their order)
            if name in before:
                before[name]()
            self.optimizers[name].step(grad_scale=grad_scale, use_device_hyper=use_device_hyper, plane_reg=plane_reg)

    def scheduler_step_all(self, step: int = 0) -> None:
        for sch in self.schedulers.values():
            sch.step()


class PlaneRegAdamPlan:
    """(f1, SURVEY.md 8f rank 1) Everything ``kp_plane_reg_adam`` needs to fold the six plane regularisers of
    NS/models/kplanes.py:430-446 into the optimizer pass: which sums of which plane enter which loss with which
    normaliser (``losses.regularizer_plan``), the per-plane gradient weights ``coef`` = sum_j loss_coefficient_j *
    normaliser, the halo scratch, and the [P,4] sums the pass accumulates (-> the six SCALED loss values of the step,
    available once the optimizer has run)."""

    def __init__(self, model) -> None:
        from ..model_components.losses import REG_NAMES, _const, regularizer_plan

        planes, terms, rows = regularizer_plan(model.field.grids, [p.grids for p in model.proposal_networks])
        coefs = model.config.loss_coefficients
        self.names = [n for n in REG_NAMES if n in coefs]
        self.planes, self.terms = planes, terms
        self.index = {id(p): i for i, p in enumerate(planes)}
        dev = planes[0].device
        scale = [float(coefs.get(n, 0.0)) for n in REG_NAMES]
        self.norm = _const(rows, dev)  # [P,6,4]
        self.scale = _const(scale, dev)  # [6]
        self.coef = _const([[sum(scale[j] * r[j][i] for j in range(6)) for i in range(4)] for r in rows], dev)  # [P,4]
        self.sums = torch.zeros((len(planes), 4), dtype=torch.float64, device=dev)
        self._groups: Dict[tuple, dict] = {}
        self.supported = bool(planes) and planes[0].is_cuda and all(
            ops.plane_reg_adam_supported(p.shape[1]) and p.requires_grad for p in planes)

    def covers(self, p) -> bool:
        return self.supported and id(p) in self.index

    def begin_step(self) -> None:
        self.sums.zero_()

    def step_group(self, planes, grads, exp_avgs, exp_avg_sqs, lr, b1, b2, eps, weight_decay, step, grad_scale, hyper_dev=None):
        key = tuple(self.index[id(p)] for p in planes)
        st = self._groups.get(key)
        if st is None:
            idx = torch.tensor(key, dtype=torch.int64, device=self.sums.device)
            st = {"idx": idx, "coef": self.coef[idx].contiguous(), "terms": [self.terms[i] for i in key],
                  "sums": torch.zeros((len(key), 4), dtype=torch.float64, device=self.sums.device),
                  "scratch": torch.empty(max(16, ops.plane_reg_adam_scratch_bytes(planes)), dtype=torch.uint8, device=self.sums.device)}
            self._groups[key] = st
        st["sums"].zero_()
        ops.plane_reg_adam_(planes, grads, exp_avgs, exp_avg_sqs, st["terms"], st["coef"], lr, b1, b2, eps, weight_decay, step,
                            grad_scale, st["scratch"], sums=st["sums"], zero_grads=True, hyper_dev=hyper_dev)
        self.sums.index_copy_(0, st["idx"], st["sums"])

    def values(self) -> Dict[str, torch.Tensor]:
        """The six SCALED regulariser terms of the step whose optimizer pass has just run (pre-update planes), keyed like
        the reference's loss dict."""
        from ..model_components.losses import REG_NAMES

        vals = (self.sums.float()[:, None, :] * self.norm).sum(dim=(0, 2)) * self.scale
        return {name: vals[i] for i, name in enumerate(REG_NAMES) if name in self.names}
