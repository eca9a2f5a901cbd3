"""IST / ISG datamanager options (the surface `ns-train k-planes --pipeline.datamanager.*` exposes).

Field names, types and defaults of ``DynamicDataManagerConfig`` (NS/data/datamanagers/dynamic_datamanager.py:34-59;
preset overrides at NS/configs/method_configs.py:491-511).  The reference's own ``DynamicDataManager`` (image cache,
dataparsers, ray generator) is a caller of the hot path and is used unchanged when this package is plugged into
nerfstudio (INTEGRATION.md); ``importance_weights`` / ``make_pixel_sampler`` below give the same behaviour to users of
this package alone (synthetic data, tests).

``DeviceImageCache`` + ``DynamicDataManager`` are the B200 form of the caller side: the reference keeps the collated image
batch on the host (``CacheDataloader``, NS/data/utils/dataloaders.py:43-232), samples pixels there and ships rays to the GPU
every step; a broadcast-style training set (19 cameras x 25 frames at 960x540: 2.9 GB fp32, plus 0.5 GB of weight maps) is
1.6 % of one B200's HBM, so here the whole cache, its weight maps, the pixel sampler, the pixel gather and the ray generator
live on the device and ``next_train`` (NS/data/datamanagers/base_datamanager.py:486-494) moves nothing over PCIe.
"""
from __future__ import annotations

import random
from dataclasses import dataclass, replace
from typing import Any, Dict, Iterator, Literal, Optional, Tuple

import torch

from ..dynamic_dataset import compute_isg, compute_ist
from ..pixel_samplers import DynamicBasedPixelSampler, EquirectangularPixelSampler, PatchPixelSampler, PixelSampler


@dataclass
class DynamicDataManagerConfig:
    """The dynamic-scene options of the reference; everything else of VanillaDataManagerConfig is out of scope."""

    train_num_rays_per_batch: int = 1024
    eval_num_rays_per_batch: int = 1024
    use_importance_sampling: bool = True
    """Whether to use importance sampling for the dynamic dataset."""
    is_pixel_ratio: float = 0.1
    """The ratio of pixels to sample using importance sampling per iteration."""
    ist_range: float = 0.25
    """The range of time differences to use for importance sampling."""
    isg: bool = False
    """Use ISG (true) or IST (False)."""
    isg_gamma: float = 5e-2
    """ISG gamma."""
    iters_to_start_is: int = 5000
    """Iterations before starting IST sampling."""
    pick_mode: Literal["normal", "randsteps", "lowfps"] = "normal"
    """Method for picking images in random loading."""
    patch_size: int = 1
    """Size of patch to sample from. If >1, patch-based sampling will be used (VanillaDataManagerConfig)."""


class ImportanceState:
    """What ``DynamicBasedPixelSampler`` reads from the dataset object (dynamic_dataset.py:60-68)."""

    def __init__(self, config: DynamicDataManagerConfig) -> None:
        self.use_importance_sampling = config.use_importance_sampling
        self.is_pixel_ratio = config.is_pixel_ratio
        self.ist_range = config.ist_range
        self.isg = config.isg
        self.isg_gamma = config.isg_gamma
        self.iters_to_start_ist = config.iters_to_start_is
        self.pick_mode = config.pick_mode


def importance_weights(config: DynamicDataManagerConfig, images: torch.Tensor, cam_ids: torch.Tensor,
                       cam_times: torch.Tensor, device="cpu") -> Optional[torch.Tensor]:
    """fp16 [B,H,W] weight maps for a cached image batch: ISG if ``config.isg`` else IST (dynamic_dataset.py:97-110)."""
    if not config.use_importance_sampling:
        return None
    if config.isg:
        return compute_isg(images, cam_ids, config.isg_gamma, device=device)
    return compute_ist(images, cam_ids, cam_times, config.ist_range, device=device)


def make_pixel_sampler(config: DynamicDataManagerConfig, num_rays_per_batch: int, cameras=None, **kwargs: Any) -> PixelSampler:
    """DynamicDataManager._get_pixel_sampler (dynamic_datamanager.py:97-113): patches if ``patch_size > 1``, sphere-uniform
    sampling if every camera is equirectangular, else the importance sampler (if enabled) or the uniform one."""
    if config.patch_size > 1:
        return PatchPixelSampler(num_rays_per_batch, patch_size=config.patch_size, **kwargs)
    if cameras is not None and bool((cameras.camera_type == 3).all()):  # CameraType.EQUIRECTANGULAR
        return EquirectangularPixelSampler(num_rays_per_batch, **kwargs)
    if config.use_importance_sampling:
        return DynamicBasedPixelSampler(num_rays_per_batch, dataset=ImportanceState(config), **kwargs)
    return PixelSampler(num_rays_per_batch, **kwargs)


class DeviceImageCache:
    """``CacheDataloader`` in its cache-all-images mode (dataloaders.py:66-92, 208-232) with the collated batch on the
    device: ``image`` [B,H,W,3] fp32, ``image_idx`` [B], the IST / ISG maps computed once by ``kp_ist_map`` /
    ``kp_isg_map`` when importance sampling is on (``ist_weights`` fp16 [B,H,W]), optional ``depth_image`` / ``mask``;
    iterating yields that batch with ``iter_steps`` counted up like the reference's loader (:230-231)."""

    def __init__(self, images: torch.Tensor, config: DynamicDataManagerConfig, cam_ids: Optional[torch.Tensor] = None,
                 cam_times: Optional[torch.Tensor] = None, device="cuda", image_idx: Optional[torch.Tensor] = None,
                 extras: Optional[Dict[str, torch.Tensor]] = None) -> None:
        if images.dim() != 4 or images.shape[-1] != 3:
            raise ValueError("DeviceImageCache: images must be [B,H,W,3]")
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("DeviceImageCache keeps the image batch on a CUDA device (there is no CPU path)")
        b = images.shape[0]
        self.batch: Dict[str, Any] = {
            "image": images.to(dev, dtype=torch.float32).contiguous(),
            "image_idx": (torch.arange(b) if image_idx is None else image_idx).to(dev),
        }
        for k, v in (extras or {}).items():
            self.batch[k] = v.to(dev)
        if config.use_importance_sampling:
            if cam_ids is None or (cam_times is None and not config.isg):
                raise ValueError("importance sampling needs the cameras' ids (and times for IST)")
            self.batch["ist_weights"] = importance_weights(config, self.batch["image"], cam_ids, cam_times, device=dev)
        self.iter_step = 0

    def __iter__(self) -> Iterator[Dict[str, Any]]:
        while True:
            self.iter_step += 1
            self.batch["iter_steps"] = self.iter_step
            yield self.batch


class DynamicDataManager:
    """``DynamicDataManager`` / ``VanillaDataManager`` (dynamic_datamanager.py:60-113, base_datamanager.py:486-494) on
    device-resident image caches: pixel sampler -> pixel gather -> ray generator, every tensor a CUDA tensor.  ``cameras``:
    one camera per cached image (nerfstudio's convention: ``image_idx`` indexes them), carrying ``times`` and ``ids``.
    ``next_train`` serves the train split; ``next_eval`` / ``next_eval_image`` the optional eval split."""

    def __init__(self, config: DynamicDataManagerConfig, cameras, images: torch.Tensor, device="cuda",
                 extras: Optional[Dict[str, torch.Tensor]] = None, prefetch: bool = False, eval_cameras=None,
                 eval_images: Optional[torch.Tensor] = None, eval_extras: Optional[Dict[str, torch.Tensor]] = None,
                 **sampler_kwargs: Any) -> None:
        """``prefetch``: the batch ``next_train`` returns was produced on a side stream while the previous step ran, and
        the next one is enqueued there before returning -- the ~0.5 ms of sampler / gather / ray-generation kernels and
        their launch latencies leave the training stream (same batches in the same order as without it).
        ``eval_cameras`` / ``eval_images`` [B,H,W,3]: the eval split, cached on the device beside the train images (without
        importance maps: eval batches are drawn uniformly).  ``eval_extras``: per-pixel maps of the eval images, cached
        with them as ``extras`` is with the train images; ``depth_image`` [B_eval,H,W,1] (ground-truth depth in the units
        of the train ``depth_image``) travels with the ``next_eval`` pixels and ``next_eval_image``, and turns on the
        ``Evaluator``'s depth metrics."""
        from ...model_components.ray_generators import RayGenerator

        if eval_extras is not None and eval_images is None:
            raise ValueError("eval_extras needs the eval split (eval_cameras and eval_images)")
        depth = (eval_extras or {}).get("depth_image")
        if depth is not None and tuple(depth.shape) != (*eval_images.shape[:3], 1):
            raise ValueError(f"eval_extras['depth_image'] must be [B_eval,H,W,1] = {(*eval_images.shape[:3], 1)} "
                             f"(got {tuple(depth.shape)})")
        self.config = config
        self.device = torch.device(device)
        self.cameras = cameras.to(self.device)
        if len(self.cameras) != images.shape[0]:
            raise ValueError(f"{images.shape[0]} images for {len(self.cameras)} cameras")
        ids = getattr(cameras, "ids", None)
        self.image_cache = DeviceImageCache(images, config, cam_ids=ids, cam_times=cameras.times, device=self.device,
                                            extras=extras)
        self.iter_train_image_dataloader = iter(self.image_cache)
        self.train_pixel_sampler = make_pixel_sampler(config, config.train_num_rays_per_batch, cameras=self.cameras,
                                                      **sampler_kwargs)
        self.train_ray_generator = RayGenerator(self.cameras)
        self.train_count = 0
        self._side = torch.cuda.Stream(device=self.device) if prefetch else None
        self._ready = None  # (ray_bundle, batch, event) produced ahead on the side stream
        self.eval_cameras = self.eval_image_cache = None
        if (eval_cameras is None) != (eval_images is None):
            raise ValueError("eval_cameras and eval_images come together")
        if eval_cameras is not None:
            self.eval_cameras = eval_cameras.to(self.device)
            if len(self.eval_cameras) != eval_images.shape[0]:
                raise ValueError(f"{eval_images.shape[0]} eval images for {len(self.eval_cameras)} eval cameras")
            self.eval_image_cache = DeviceImageCache(eval_images, replace(config, use_importance_sampling=False), device=self.device,
                                                     extras=eval_extras)
            self.iter_eval_image_dataloader = iter(self.eval_image_cache)
            self.eval_pixel_sampler = PixelSampler(config.eval_num_rays_per_batch)
            self.eval_ray_generator = RayGenerator(self.eval_cameras)
        self.eval_count = 0

    def _produce(self) -> Tuple[Any, Dict[str, Any]]:
        image_batch = next(self.iter_train_image_dataloader)
        batch = self.train_pixel_sampler.sample(image_batch)
        ray_bundle = self.train_ray_generator(batch["indices"])
        return ray_bundle, batch

    def _produce_ahead(self, main: torch.cuda.Stream) -> None:
        if self._ready is None:
            self._side.wait_stream(main)  # the cache and its weight maps were built on the calling stream
        # later batches read only those constants and allocate their own outputs: no dependency on the training stream,
        # so the producer is NOT made to wait for the step in flight (that would serialise it behind the step again)
        with torch.cuda.stream(self._side):
            ray_bundle, batch = self._produce()
            done = torch.cuda.Event()
            done.record(self._side)
        self._ready = (ray_bundle, batch, done)

    @staticmethod
    def _tensors(ray_bundle, batch):
        for t in (ray_bundle.origins, ray_bundle.directions, ray_bundle.pixel_area, ray_bundle.camera_indices,
                  ray_bundle.nears, ray_bundle.fars, ray_bundle.times, *(ray_bundle.metadata or {}).values(), *batch.values()):
            if torch.is_tensor(t) and t.is_cuda:
                yield t

    def next_train(self, step: int) -> Tuple[Any, Dict[str, Any]]:
        """-> (RayBundle, batch): base_datamanager.py:486-494."""
        self.train_count += 1
        if self._side is None:
            return self._produce()
        main = torch.cuda.current_stream(self.device)
        if self._ready is None:
            self._produce_ahead(main)
        ray_bundle, batch, done = self._ready
        main.wait_event(done)
        for t in self._tensors(ray_bundle, batch):
            t.record_stream(main)  # allocated on the side stream, consumed on the training stream
        self._produce_ahead(main)
        return ray_bundle, batch

    def _need_eval(self) -> None:
        if self.eval_image_cache is None:
            raise RuntimeError("this datamanager has no eval split: pass eval_cameras and eval_images")

    def next_eval(self, step: int) -> Tuple[Any, Dict[str, Any]]:
        """-> (RayBundle, batch) of ``eval_num_rays_per_batch`` pixels drawn uniformly from the eval images
        (``VanillaDataManager.next_eval``)."""
        self._need_eval()
        self.eval_count += 1
        batch = self.eval_pixel_sampler.sample(next(self.iter_eval_image_dataloader))
        return self.eval_ray_generator(batch["indices"]), batch

    def next_eval_image(self, step: int) -> Tuple[int, Dict[str, torch.Tensor]]:
        """-> (camera index, {"image": [H,W,3] device tensor, and "depth_image": [H,W,1] when the eval split has one}) of a
        random eval image (``VanillaDataManager.next_eval_image``: a random draw of the eval dataloader); render the camera
        with ``engine.frame_renderer.FrameRenderer``."""
        self._need_eval()
        i = random.randrange(len(self.eval_cameras))
        batch = self.eval_image_cache.batch
        return i, {k: batch[k][i] for k in ("image", "depth_image") if k in batch}
