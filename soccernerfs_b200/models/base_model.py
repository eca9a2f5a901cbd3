"""Model base class and config plumbing.  Mirror of NS/models/base_model.py:38-217 and of the two config classes
K-Planes needs from NS/configs/base_config.py:33-58 (``PrintableConfig`` / ``InstantiateConfig``)."""
from __future__ import annotations

import contextlib

from abc import abstractmethod
from collections import defaultdict
from dataclasses import dataclass, field
from typing import Any, Dict, List, Optional, Tuple, Type

import torch
from torch import nn
from torch.nn import Parameter

from ..cameras.rays import RayBundle
from ..data.scene_box import SceneBox
from ..model_components.scene_colliders import NearFarCollider


class PrintableConfig:
    def __str__(self):
        lines = [self.__class__.__name__ + ":"]
        for key, val in vars(self).items():
            if isinstance(val, tuple):
                val = "[" + "\n".join(str(v) for v in val) + "]"
            lines += f"{key}: {str(val)}".split("\n")
        return "\n    ".join(lines)


@dataclass
class InstantiateConfig(PrintableConfig):
    """``_target(self, **kwargs)`` instantiation contract (base_config.py:50-58)."""

    _target: Type

    def setup(self, **kwargs) -> Any:
        return self._target(self, **kwargs)


def to_immutable_dict(d: Dict[str, Any]):
    return field(default_factory=lambda: dict(d))


@dataclass
class ModelConfig(InstantiateConfig):
    _target: Type = field(default_factory=lambda: Model)
    enable_collider: bool = True
    collider_params: Optional[Dict[str, float]] = to_immutable_dict({"near_plane": 2.0, "far_plane": 6.0})
    loss_coefficients: Dict[str, float] = to_immutable_dict({"rgb_loss_coarse": 1.0, "rgb_loss_fine": 1.0})
    eval_num_rays_per_chunk: int = 4096


@contextlib.contextmanager
def coherent_rays(model, tile: int = 4):
    """Tell the model's field that consecutive rays of the bundles it is about to see are neighbouring pixels of one frame:
    its gather then lets a warp take one sample index of ``tile`` neighbouring rays (``KpPoints.ray_tile``), whose texel
    reads coalesce.  Inference only (the field ignores it while gradients are enabled); no effect on results."""
    field = getattr(model, "field", None)
    old = getattr(field, "coherent_ray_tile", 0) if field is not None else 0
    if field is not None:
        field.coherent_ray_tile = tile
    try:
        yield
    finally:
        if field is not None:
            field.coherent_ray_tile = old


@contextlib.contextmanager
def static_scene(model):
    """Render the static part of a dynamic scene: inside, the model's field and every proposal network leave their time
    planes (XT, YT, ZT) out of each feature product -- the space planes alone, which is the scene with its time planes
    set to the identity 1 -- so the proposals place samples on the static scene too.  Time is not read: cameras need no
    times, and their times do not change the result.  Inference only: raises while gradients are enabled.  Outside the
    context nothing changes; a static model renders as it always does."""
    if torch.is_grad_enabled():
        raise RuntimeError("static_scene is an inference mode: use it under torch.no_grad()")
    field = getattr(model, "field", None)
    modules = ([field] if field is not None else []) + list(getattr(model, "proposal_networks", []))
    old = [m.static_scene for m in modules]
    for m in modules:
        m.static_scene = True
    try:
        yield
    finally:
        for m, o in zip(modules, old):
            m.static_scene = o


@contextlib.contextmanager
def dynamics_output(model, enabled: bool = True):
    """Ask the model for its per-ray dynamics output ``dynamic`` [N, 1]: the final level's weights composite the
    samples' dynamics scores, sum_i w_i delta_i, delta = mean over scales and channels of |1 - product of the time planes'
    interpolants| (ops.hexplane_features_dyn); 0 where the time planes are the identity.  Inference only (the field
    ignores it while gradients are enabled); no effect on the other outputs."""
    field = getattr(model, "field", None)
    old = getattr(field, "dynamic_output", False)
    if field is not None:
        field.dynamic_output = enabled
    try:
        yield
    finally:
        if field is not None:
            field.dynamic_output = old


class Model(nn.Module):
    config: ModelConfig

    def __init__(self, config: ModelConfig, scene_box: SceneBox, num_train_data: int, **kwargs) -> None:
        super().__init__()
        self.config = config
        self.scene_box = scene_box
        self.render_aabb = None
        self.num_train_data = num_train_data
        self.kwargs = kwargs
        self.collider = None
        self.populate_modules()
        self.callbacks = None
        self.device_indicator_param = nn.Parameter(torch.empty(0))

    @property
    def device(self):
        return self.device_indicator_param.device

    def get_training_callbacks(self, training_callback_attributes) -> List:
        return []

    def populate_modules(self):
        if self.config.enable_collider:
            self.collider = NearFarCollider(near_plane=self.config.collider_params["near_plane"],
                                            far_plane=self.config.collider_params["far_plane"])

    @abstractmethod
    def get_param_groups(self) -> Dict[str, List[Parameter]]:
        """parameter groups for the optimizers."""

    @abstractmethod
    def get_outputs(self, ray_bundle: RayBundle) -> Dict[str, torch.Tensor]:
        """ray bundle -> outputs."""

    def forward(self, ray_bundle: RayBundle) -> Dict[str, torch.Tensor]:
        """Collider (near / far planes) first, then the model's ``get_outputs`` (base_model.py:131-143)."""
        bundle = ray_bundle if self.collider is None else self.collider(ray_bundle)
        return self.get_outputs(bundle)

    def get_metrics_dict(self, outputs, batch) -> Dict[str, torch.Tensor]:
        return {}

    @abstractmethod
    def get_loss_dict(self, outputs, batch, metrics_dict=None) -> Dict[str, torch.Tensor]:
        """losses."""

    @torch.no_grad()
    def get_outputs_for_camera_ray_bundle(self, camera_ray_bundle: RayBundle) -> Dict[str, torch.Tensor]:
        """Full-image inference: the [H,W] bundle is rendered in row-major chunks of ``eval_num_rays_per_chunk`` rays
        and every tensor output is stitched back to [H,W,C] (base_model.py:162-186).  ``engine.frame_renderer`` is the
        pipelined variant that also generates the rays on the device."""
        chunk = self.config.eval_num_rays_per_chunk
        height, width = camera_ray_bundle.origins.shape[:2]
        pieces: Dict[str, List[torch.Tensor]] = defaultdict(list)
        with coherent_rays(self):  # row-major chunks: neighbouring rays are neighbouring pixels
            for begin in range(0, len(camera_ray_bundle), chunk):
                part = self.forward(ray_bundle=camera_ray_bundle.get_row_major_sliced_ray_bundle(begin, begin + chunk))
                for name, value in part.items():
                    if torch.is_tensor(value):
                        pieces[name].append(value)
        return {name: torch.cat(values).view(height, width, -1) for name, values in pieces.items()}

    def get_image_metrics_and_images(self, outputs, batch) -> Tuple[Dict[str, float], Dict[str, torch.Tensor]]:
        raise NotImplementedError

    def load_model(self, loaded_state: Dict[str, Any]) -> None:
        """Load ``loaded_state["model"]``, tolerating a DDP ``module.`` prefix (base_model.py:201-208)."""
        self.load_state_dict({k.replace("module.", ""): v for k, v in loaded_state["model"].items()})
