"""K-Planes model on the B200 hot path.

``KPlanesModelConfig`` has the reference's fields and defaults (NS/models/kplanes.py:67-177) and ``KPlanesModel``
its surface: ``populate_modules`` :188-309, ``get_param_groups`` :311-316, ``get_training_callbacks`` :318-347,
``get_outputs`` :349-388, ``get_metrics_dict`` :390-412, ``get_loss_dict`` :414-452,
``get_image_metrics_and_images`` :454-515 (PSNR / SSIM restated in torch, colour maps in ``utils/colormaps.py``; the
pretrained-network metrics LPIPS and DynMetric are used through the reference's objects when importable).
"""
from __future__ import annotations

import functools
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple, Type

import numpy as np
import torch
from torch.nn import Parameter

from .. import ops
from ..cameras.rays import RayBundle
from ..field_components.spatial_distortions import SceneContraction
from ..fields.base_field import FieldHeadNames
from ..fields.kplanes_field import KPlanesDensityField, KPlanesField
from ..model_components.losses import (
    REG_NAMES,
    DepthLossType,
    MSELoss,
    depth_loss,
    distortion_loss,
    distortion_per_ray,
    interlevel_loss,
    interlevel_terms,
    kplanes_regularizers,
    space_tv_loss,
    sparse_transients_loss,
    time_smoothness_loss,
)
from ..model_components.ray_samplers import ProposalNetworkSampler, UniformSampler
from ..model_components.renderers import AccumulationRenderer, DepthRenderer, MedianRGBRenderer, RGBRenderer
from ..model_components.scene_colliders import AABBBoxCollider, NearFarCollider
from .base_model import Model, ModelConfig, to_immutable_dict


class TrainingCallbackLocation:
    """NS/engine/callbacks.py:44-48."""

    BEFORE_TRAIN_ITERATION = 1
    AFTER_TRAIN_ITERATION = 2


@dataclass
class TrainingCallback:
    """Callback run by the trainer before/after each iteration (NS/engine/callbacks.py:51-103)."""

    where_to_run: List[int]
    func: callable
    update_every_num_iters: Optional[int] = None
    iters: Optional[Tuple[int, ...]] = None
    args: Optional[List] = None
    kwargs: Optional[Dict] = None

    def run_callback(self, step: int):
        args, kwargs = self.args or [], self.kwargs or {}
        if self.update_every_num_iters is not None:
            if step % self.update_every_num_iters == 0:
                self.func(*args, **kwargs, step=step)
        elif self.iters is not None:
            if step in self.iters:
                self.func(*args, **kwargs, step=step)

    def run_callback_at_location(self, step: int, location: int):
        if location in self.where_to_run:
            self.run_callback(step=step)


@dataclass
class KPlanesModelConfig(ModelConfig):
    """K-Planes model config: field names, types and defaults of NS/models/kplanes.py:67-177."""

    _target: Type = field(default_factory=lambda: KPlanesModel)
    near_plane: float = 0.05
    far_plane: float = 1000.0
    bounded: bool = True
    spacetime_resolution: Sequence[int] = (64, 64, 64, 50)
    feature_dim: int = 32
    multiscale_res: Sequence[int] = (1, 2, 4, 8)
    concat_features_across_scales: bool = True
    linear_decoder: bool = False
    linear_decoder_layers: Optional[int] = 1
    sigma_net_layers: int = 1
    sigma_net_hidden_dim: int = 64
    rgb_net_layers: int = 2
    rgb_net_hidden_dim: int = 64
    background_color_train: str = "random"
    background_color_eval: str = "last_sample"
    num_proposal_iterations: int = 2
    use_same_proposal_network: bool = False
    proposal_net_args_list: List[Dict] = field(
        default_factory=lambda: [
            {"feature_dim": 8, "resolution": [128, 128, 128, 150]},
            {"feature_dim": 8, "resolution": [256, 256, 256, 150]},
        ]
    )
    num_nerf_samples_per_ray: int = 48
    num_proposal_samples_per_ray: Tuple[int, ...] = (256, 128)
    use_single_jitter: bool = False
    proposal_warmup: int = 5000
    proposal_update_every: int = 5
    use_proposal_weight_anneal: bool = True
    proposal_weights_anneal_max_num_iters: int = 1000
    proposal_weights_anneal_slope: float = 10.0
    use_appearance_embedding: bool = False
    appearance_embedding_dim: int = 0
    disable_viewing_dependent: bool = False
    loss_coefficients: Dict[str, float] = to_immutable_dict(
        {
            "rgb_loss": 1.0,
            "interlevel_loss": 1.0,
            "distortion_loss": 0.001,
            "space_tv_loss": 0.0002,
            "time_smoothness_loss": 0.001,
            "sparse_transients_loss": 0.0001,
            "space_tv_proposal_loss": 0.0002,
            "time_smoothness_proposal_loss": 0.00001,
            "sparse_transients_proposal_loss": 0.0001,
            "depth_loss": 0.05,
        }
    )
    is_euclidean_depth: bool = True
    depth_sigma: float = 0.01
    should_decay_sigma: bool = False
    starting_depth_sigma: float = 0.2
    sigma_decay_rate: float = 0.99985
    depth_loss_type: DepthLossType = DepthLossType.DS_NERF
    freeze_time_planes: bool = False
    freeze_space_planes: bool = False


class LossDict(dict):
    """Loss dictionary (same keys / scaled scalar tensors as the reference's) that may also carry ``total``: the sum of
    its values when the fused loss head already produced it (saves the trainer's sum(loss_dict.values()) kernels)."""

    total: Optional[torch.Tensor] = None


def scale_dict(dictionary: Dict, coefficients: Dict[str, float]) -> Dict:
    """NS/utils/misc.py:116-129."""
    for key in dictionary:
        if key in coefficients:
            dictionary[key] *= coefficients[key]
    return dictionary


class _branch:
    """``with _branch(streams, i):`` runs the body on ``streams[i % len(streams)]`` (forked from the current stream);
    ``join_now()`` makes the current stream wait for it; branch 0 is joined by the owner of the streams (the training step
    does, before it returns).  ``streams`` None / empty: a no-op."""

    def __init__(self, streams, index: int) -> None:
        self.stream = streams[index % len(streams)] if streams else None

    def __enter__(self):
        if self.stream is not None:
            self.main = torch.cuda.current_stream()
            self.stream.wait_stream(self.main)
            self.ctx = torch.cuda.stream(self.stream)
            self.ctx.__enter__()
        return self

    def __exit__(self, *exc):
        if self.stream is not None:
            self.ctx.__exit__(*exc)
        return False

    def join_now(self) -> None:
        if self.stream is not None:
            torch.cuda.current_stream().wait_stream(self.stream)


class KPlanesModel(Model):
    config: KPlanesModelConfig
    _kp_branch_streams = None  # engine/trainer.py: CUDA streams for the independent small branches of a training step

    def populate_modules(self):
        super().populate_modules()
        cfg = self.config
        # unbounded scenes: L-infinity scene contraction (kplanes.py:203-206), evaluated inside the field kernels
        scene_contraction = None if cfg.bounded else SceneContraction(order=float("inf"))
        self.field = KPlanesField(
            self.scene_box.aabb,
            feat_dim=cfg.feature_dim,
            spacetime_resolution=cfg.spacetime_resolution,
            concat_features_across_scales=cfg.concat_features_across_scales,
            multiscale_res=cfg.multiscale_res,
            use_appearance_embedding=cfg.use_appearance_embedding,
            appearance_dim=cfg.appearance_embedding_dim,
            spatial_distortion=scene_contraction,
            linear_decoder=cfg.linear_decoder,
            linear_decoder_layers=cfg.linear_decoder_layers,
            num_images=self.num_train_data,
            disable_viewing_dependent=cfg.disable_viewing_dependent,
            sigma_net_layers=cfg.sigma_net_layers,
            sigma_net_hidden_dim=cfg.sigma_net_hidden_dim,
            rgb_net_layers=cfg.rgb_net_layers,
            rgb_net_hidden_dim=cfg.rgb_net_hidden_dim,
            freeze_time_planes=cfg.freeze_time_planes,
            freeze_space_planes=cfg.freeze_space_planes,
        )
        self.depth_sigma = torch.tensor([cfg.starting_depth_sigma if cfg.should_decay_sigma else cfg.depth_sigma])

        self.density_fns = []
        num_prop_nets = cfg.num_proposal_iterations
        self.proposal_networks = torch.nn.ModuleList()
        common = dict(spatial_distortion=scene_contraction, linear_decoder=cfg.linear_decoder, freeze_time_planes=cfg.freeze_time_planes,
                      freeze_space_planes=cfg.freeze_space_planes)
        if cfg.use_same_proposal_network:
            assert len(cfg.proposal_net_args_list) == 1, "Only one proposal network is allowed."
            network = KPlanesDensityField(self.scene_box.aabb, **common, **cfg.proposal_net_args_list[0])
            self.proposal_networks.append(network)
            self.density_fns.extend([network.density_fn for _ in range(num_prop_nets)])
        else:
            for i in range(num_prop_nets):
                args = cfg.proposal_net_args_list[min(i, len(cfg.proposal_net_args_list) - 1)]
                self.proposal_networks.append(KPlanesDensityField(self.scene_box.aabb, **common, **args))
            self.density_fns.extend([network.density_fn for network in self.proposal_networks])

        def update_schedule(step):
            return np.clip(np.interp(step, [0, cfg.proposal_warmup], [0, cfg.proposal_update_every]), 1,
                           cfg.proposal_update_every)

        # bounded => uniform; unbounded => None = ProposalNetworkSampler's piecewise default (kplanes.py:261-264)
        initial_sampler = UniformSampler(single_jitter=cfg.use_single_jitter) if cfg.bounded else None
        self.proposal_sampler = ProposalNetworkSampler(
            num_nerf_samples_per_ray=cfg.num_nerf_samples_per_ray,
            num_proposal_samples_per_ray=cfg.num_proposal_samples_per_ray,
            num_proposal_network_iterations=cfg.num_proposal_iterations,
            single_jitter=cfg.use_single_jitter,
            update_sched=update_schedule,
            initial_sampler=initial_sampler,
        )
        if cfg.bounded:  # kplanes.py:275-278
            self.collider = AABBBoxCollider(scene_box=self.scene_box)
        else:
            self.collider = NearFarCollider(near_plane=cfg.near_plane, far_plane=cfg.far_plane)
        self.renderer_rgb = RGBRenderer(background_color=cfg.background_color_train)
        self.renderer_accumulation = AccumulationRenderer()
        self.renderer_depth = DepthRenderer()
        self.medianrgb_renderer = MedianRGBRenderer()
        self.rgb_loss = MSELoss()
        self.temporal_distortion = len(cfg.spacetime_resolution) == 4  # viewer flag (kplanes.py:297)

    def get_param_groups(self) -> Dict[str, List[Parameter]]:
        return {
            "proposal_networks": list(self.proposal_networks.parameters()),
            "fields": list(self.field.parameters()),
        }

    def get_training_callbacks(self, training_callback_attributes=None) -> List[TrainingCallback]:
        callbacks = []
        if self.config.use_proposal_weight_anneal:
            n_iters = self.config.proposal_weights_anneal_max_num_iters

            def set_anneal(step):  # https://arxiv.org/pdf/2111.12077.pdf eq. 18 (kplanes.py:326-331)
                train_frac = np.clip(step / n_iters, 0, 1)
                b = self.config.proposal_weights_anneal_slope
                self.proposal_sampler.set_anneal((b * train_frac) / ((b - 1) * train_frac + 1))

            callbacks.append(TrainingCallback(where_to_run=[TrainingCallbackLocation.BEFORE_TRAIN_ITERATION],
                                              update_every_num_iters=1, func=set_anneal))
            callbacks.append(TrainingCallback(where_to_run=[TrainingCallbackLocation.AFTER_TRAIN_ITERATION],
                                              update_every_num_iters=1, func=self.proposal_sampler.step_cb))
        return callbacks

    def get_outputs(self, ray_bundle: RayBundle):
        density_fns = self.density_fns
        if ray_bundle.times is not None:
            density_fns = [functools.partial(f, times=ray_bundle.times) for f in density_fns]
        ray_samples, weights_list, ray_samples_list = self.proposal_sampler(ray_bundle, density_fns=density_fns)
        field_out = self.field(ray_samples)
        weights = ray_samples.get_weights(field_out[FieldHeadNames.DENSITY])
        weights_list.append(weights)
        ray_samples_list.append(ray_samples)

        self.renderer_rgb.background_color = (
            self.config.background_color_train if self.training else self.config.background_color_eval
        )
        rgb = self.renderer_rgb(rgb=field_out[FieldHeadNames.RGB], weights=weights)
        # outputs no loss term reads (accumulation, depths, median colour): on the trainer's auxiliary stream when it
        # gave us one, next to the loss kernels instead of in front of them
        with _branch(self._kp_branch_streams if (self.training and rgb.is_cuda) else None, 0):
            accumulation = self.renderer_accumulation(weights)
            depth = self.renderer_depth(weights, ray_samples)
            median_rgb = self.medianrgb_renderer(rgb=field_out[FieldHeadNames.RGB], weights=weights)
            outputs = {"rgb": rgb, "accumulation": accumulation, "depth": depth, "median_rgb": median_rgb}
            if "dynamic" in field_out:  # base_model.dynamics_output: composited like the accumulation, [N, 1]
                outputs["dynamic"] = torch.sum(weights * field_out["dynamic"], dim=-2)
            if self.training:
                outputs["weights_list"] = weights_list
                outputs["ray_samples_list"] = ray_samples_list
            for i in range(self.config.num_proposal_iterations):
                outputs[f"prop_depth_{i}"] = self.renderer_depth(weights=weights_list[i], ray_samples=ray_samples_list[i])
        if ray_bundle.metadata is not None and "directions_norm" in ray_bundle.metadata:
            outputs["directions_norm"] = ray_bundle.metadata["directions_norm"]
        return outputs

    def get_metrics_dict(self, outputs, batch):
        metrics_dict = {}
        image = batch["image"].to(self.device)
        head = self._loss_head(outputs, image)
        if head is not None:
            metrics_dict["psnr"] = head[2]
        else:
            with torch.no_grad():  # PSNR with data_range 1.0 (torchmetrics.PeakSignalNoiseRatio in the reference)
                metrics_dict["psnr"] = -10.0 * torch.log10(torch.mean((outputs["rgb"] - image) ** 2))
        if self.training and "depth_image" in batch and self.config.loss_coefficients["depth_loss"] > 0:
            metrics_dict["depth_loss"] = self._mean_depth_loss(outputs, batch["depth_image"].to(self.device))
        return metrics_dict

    def _loss_head(self, outputs, image):
        """Training on CUDA: rgb / distortion / interlevel losses (scaled), their total and the PSNR from ONE kernel
        (ops.loss_head), computed once per forward and cached in ``outputs``.  None when not applicable."""
        if "_loss_head" in outputs:
            return outputs["_loss_head"]
        head = None
        coef = self.config.loss_coefficients
        rgb = outputs["rgb"]
        if (self.training and rgb.is_cuda and "weights_list" in outputs and "rgb_loss" in coef
                and len(outputs["weights_list"]) - 1 <= 4 and image.shape == rgb.shape):
            wl, rl = outputs["weights_list"], outputs["ray_samples_list"]
            # the distortion term and the interlevel terms are independent warp-per-ray kernels of a few microseconds
            # each: as parallel branches (trainer-provided streams) they and their backward kernels overlap; autograd
            # replays every backward on its forward's stream
            br, forks = self._kp_branch_streams, []
            with _branch(br, 1) as b:
                dist = distortion_per_ray(wl, rl) if "distortion_loss" in coef else None
            forks.append(b)
            il = []
            if "interlevel_loss" in coef:
                for lvl in range(len(wl) - 1):
                    with _branch(br, 2 + lvl) as b:
                        il += interlevel_terms([wl[lvl], wl[-1]], [rl[lvl], rl[-1]])
                    forks.append(b)
            for b in forks:  # (joined only after every branch was forked: a join in between would serialise them)
                b.join_now()
            extra = outputs.get("_scaled_regularizers_vec")
            head = ops.loss_head(rgb, image, dist, il, coef["rgb_loss"], coef.get("distortion_loss", 0.0),
                                 coef.get("interlevel_loss", 0.0), extra) + (extra is not None,)
        outputs["_loss_head"] = head
        return head

    def regularizer_losses(self) -> Dict[str, torch.Tensor]:
        """The plane regularisers of the loss dict (kplanes.py:430-446), UNSCALED.  They depend on the planes only,
        not on the batch, which lets a training step evaluate them off the critical path."""
        loss_coef = self.config.loss_coefficients
        out: Dict[str, torch.Tensor] = {}
        ms_grids_nerf = self.field.grids
        ms_grids_prop = [p.grids for p in self.proposal_networks]
        if self._all_six_regularizers():
            # the six regularisers of kplanes.py:430-446 from one pass over the planes (same values)
            out.update(kplanes_regularizers(ms_grids_nerf, ms_grids_prop))
            return out
        dynamic = self._dynamic()
        if "space_tv_loss" in loss_coef:
            out["space_tv_loss"] = space_tv_loss(ms_grids_nerf)
        if "space_tv_proposal_loss" in loss_coef:
            out["space_tv_proposal_loss"] = space_tv_loss(ms_grids_prop)
        if dynamic:
            if "sparse_transients_loss" in loss_coef:
                out["sparse_transients_loss"] = sparse_transients_loss(ms_grids_nerf)
            if "sparse_transients_proposal_loss" in loss_coef:
                out["sparse_transients_proposal_loss"] = sparse_transients_loss(ms_grids_prop)
            if "time_smoothness_loss" in loss_coef:
                out["time_smoothness_loss"] = time_smoothness_loss(ms_grids_nerf)
            if "time_smoothness_proposal_loss" in loss_coef:
                out["time_smoothness_proposal_loss"] = time_smoothness_loss(ms_grids_prop)
        return out

    def _dynamic(self) -> bool:
        return len(self.config.spacetime_resolution) > 3 and not self.config.freeze_time_planes

    def _all_six_regularizers(self) -> bool:
        """Dynamic scene with all six regulariser keys: they are evaluated together, in one pass over the planes."""
        return self._dynamic() and all(k in self.config.loss_coefficients for k in REG_NAMES)

    def fused_regularizers_applicable(self) -> bool:
        """Whether ``regularizers_into_grads`` covers this configuration (dynamic scene, all six regulariser keys)."""
        return self._all_six_regularizers() and not self.config.freeze_space_planes

    def regularized_planes(self) -> List[Parameter]:
        return [p for g in self.field.grids for p in g] + [p for net in self.proposal_networks for p in net.grids]

    def regularizers_into_grads(self, accumulate: bool = False, write_range=None, grad_scale=None, sums_in_range: bool = False,
                                sum_scale=None) -> Dict[str, torch.Tensor]:
        """Training-step form of ``regularizer_losses`` (kplanes.py:430-446): the six SCALED, detached loss values from
        ONE sweep per plane that also writes (or adds) the scaled regularisers' gradient into every plane's gradient
        sink -- no autograd graph, no separate backward sweep, and no memset of the planes' part of the bucket."""
        from ..model_components.losses import kplanes_regularizers_into_grads

        vals, _ = kplanes_regularizers_into_grads(self.field.grids, [p.grids for p in self.proposal_networks],
                                                  self.config.loss_coefficients, accumulate=accumulate,
                                                  write_range=write_range, grad_scale=grad_scale,
                                                  sums_in_range=sums_in_range, sum_scale=sum_scale)
        ops.PLANE_REG_BACKWARDS += 1
        return vals

    def get_loss_dict(self, outputs, batch, metrics_dict=None, regularizers=None) -> Dict[str, torch.Tensor]:
        """kplanes.py:410-452.  ``regularizers`` (extension): already SCALED regulariser terms computed (and possibly
        already back-propagated) by the caller; they are merged instead of being evaluated here."""
        device = outputs["rgb"].device
        image = batch["image"].to(device)
        loss_coef = self.config.loss_coefficients
        head = self._loss_head(outputs, image)
        if head is not None:
            vals, total, _psnr, has_extra = head
            loss_dict = LossDict(rgb_loss=vals[0])
            if "distortion_loss" in loss_coef:
                loss_dict["distortion_loss"] = vals[1]
            if "interlevel_loss" in loss_coef:
                loss_dict["interlevel_loss"] = vals[2]
            rest: Dict[str, torch.Tensor] = {}
            if regularizers is None:
                rest.update(self.regularizer_losses())
            if "depth_image" in batch.keys() and loss_coef["depth_loss"] > 0:
                rest["depth_loss"] = metrics_dict["depth_loss"]
            rest = scale_dict(rest, loss_coef)
            if regularizers is not None and not has_extra:
                rest.update(regularizers)
            for v in rest.values():
                total = total + v
            loss_dict.update(rest)
            if regularizers is not None and has_extra:
                loss_dict.update(regularizers)
            loss_dict.total = total
            return loss_dict
        loss_dict = {"rgb_loss": self.rgb_loss(image, outputs["rgb"])}
        if self.training:
            if "distortion_loss" in loss_coef:
                loss_dict["distortion_loss"] = distortion_loss(outputs["weights_list"], outputs["ray_samples_list"])
            if "interlevel_loss" in loss_coef:
                loss_dict["interlevel_loss"] = interlevel_loss(outputs["weights_list"], outputs["ray_samples_list"])
            if regularizers is None:
                loss_dict.update(self.regularizer_losses())
            if "depth_image" in batch.keys() and loss_coef["depth_loss"] > 0:
                loss_dict["depth_loss"] = metrics_dict["depth_loss"]
        loss_dict = scale_dict(loss_dict, loss_coef)
        if self.training and regularizers is not None:
            loss_dict.update(regularizers)
        return loss_dict

    def get_image_metrics_and_images(self, outputs: Dict[str, torch.Tensor], batch: Dict[str, torch.Tensor]
                                     ) -> Tuple[Dict[str, float], Dict[str, torch.Tensor]]:
        """Eval-image metrics and visualisations (kplanes.py:454-515; called by the pipeline every ``steps_per_eval_image``).
        ``psnr`` / ``ssim`` always; ``lpips`` and the dynamic-region ``dpsnr/dssim/dlpips`` + ``bbox`` image when the
        reference's pretrained-network metrics are importable (their keys are absent otherwise, never an exception)."""
        from ..utils import colormaps, image_metrics

        image = batch["image"].to(outputs["rgb"].device)
        rgb = outputs["rgb"]
        acc = colormaps.apply_colormap(outputs["accumulation"])
        depth = colormaps.apply_depth_colormap(outputs["depth"], accumulation=outputs["accumulation"])
        combined_rgb = torch.cat([image, rgb], dim=1)
        # [H, W, C] -> [1, C, H, W] for the metrics
        image_m = torch.moveaxis(image, -1, 0)[None, ...]
        rgb_m = torch.moveaxis(rgb, -1, 0)[None, ...]
        metrics_dict = {"psnr": float(image_metrics.psnr(image_m, rgb_m)), "ssim": float(image_metrics.ssim(image_m, rgb_m))}
        images_dict = {"img": combined_rgb, "accumulation": acc, "depth": depth}
        if not hasattr(self, "_lpips"):
            self._lpips = image_metrics.optional_lpips(rgb.device)
            self._dynmetric = image_metrics.optional_dynmetric(rgb.device)
        if self._lpips is not None:
            metrics_dict["lpips"] = float(self._lpips(image_m, rgb_m))
        if self._dynmetric is not None:
            bbox_img, dpsnr, dssim, dlpips = self._dynmetric(image_m, rgb_m)
            metrics_dict.update({"dpsnr": float(dpsnr), "dssim": float(dssim), "dlpips": float(dlpips)})
            images_dict["bbox"] = bbox_img
        for i in range(self.config.num_proposal_iterations):
            key = f"prop_depth_{i}"
            images_dict[key] = colormaps.apply_depth_colormap(outputs[key], accumulation=outputs["accumulation"])
        if "depth_image" in batch.keys():  # ground-truth depth beside the prediction (kplanes.py:503-510)
            ground_truth_depth = batch["depth_image"].to(rgb.device)
            if not self.config.is_euclidean_depth:
                ground_truth_depth = ground_truth_depth * outputs["directions_norm"]
            images_dict["depth"] = torch.cat([colormaps.apply_depth_colormap(ground_truth_depth), depth], dim=1)
        images_dict["median_rgb"] = outputs["median_rgb"]
        return metrics_dict, images_dict

    def _mean_depth_loss(self, outputs, termination_depth: torch.Tensor) -> torch.Tensor:
        """Depth supervision averaged over every sampling level, proposal levels included (kplanes.py:395-410): each
        level's weights are compared with the sensor depth along its own samples."""
        levels = list(zip(outputs["weights_list"], outputs["ray_samples_list"]))
        sigma = self._get_sigma().to(self.device)
        per_level = [depth_loss(weights=w, ray_samples=rs, termination_depth=termination_depth, predicted_depth=outputs["depth"],
                                sigma=sigma, directions_norm=outputs["directions_norm"],
                                is_euclidean=self.config.is_euclidean_depth, depth_loss_type=self.config.depth_loss_type)
                     for w, rs in levels]
        return sum(per_level) / len(per_level)

    def _get_sigma(self):
        if not self.config.should_decay_sigma:
            return self.depth_sigma
        self.depth_sigma = torch.maximum(self.config.sigma_decay_rate * self.depth_sigma,
                                         torch.tensor([self.config.depth_sigma]))
        return self.depth_sigma
