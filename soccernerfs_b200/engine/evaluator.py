"""Evaluation of a trained model over its eval split: the eval side of ``VanillaPipeline``
(``get_eval_loss_dict``, ``get_eval_image_metrics_and_images``, ``get_average_eval_image_metrics``,
NS/pipelines/base_pipeline.py:343-352) and the JSON that ``ns-eval`` writes (REF/nerfstudio/scripts/eval.py:20-44).

``get_average_eval_image_metrics`` keeps the frames on the device: each image is rendered by ``FrameRenderer`` into device
tensors, and the PSNR / SSIM of all of a rank's images come from one ``ops.image_metrics`` call (three kernel launches)
instead of the torch restatement and its host synchronisations per image.  With ``world > 1`` rank r renders the images
``i % world == r``; one ``all_gather`` brings every image's row to every rank, and each key is averaged in image order,
so the result does not depend on the world size.

With ``regions`` the same images are also measured per region: ``ops.image_metrics_masked`` gives the PSNR / SSIM of a
dynamic-region mask and of its complement (``psnr_dynamic`` ... ``ssim_static``).  The masks are the caller's, or
``median_dynamic_masks`` of the eval images: the pixels that differ from their camera's per-pixel temporal median, which
for a broadcast clip with moving players is the empty pitch.  These are not the reference's ``DynMetric`` (detector
boxes), hence keys of their own rather than its ``dpsnr`` / ``dssim``.

When the eval split carries ground-truth depth (``DynamicDataManager(eval_extras={"depth_image": ...})``), the rendered
``depth`` frames of the same images go through one ``ops.depth_metrics`` call per rank (``depth_abs_rel`` ...
``depth_delta3``, per region too with ``regions``): the geometry the preset's depth supervision trains, which colour
metrics cannot tell apart from a flat billboard that looks right from near the training cameras.
"""
from __future__ import annotations

import math
from typing import Any, Callable, Dict, List, Optional, Sequence, Tuple, Union

import torch

from .. import ops
from ..configs.method_configs import KPLANES_DATAMANAGER, KPLANES_TRAINER
from ..utils import image_metrics
from .frame_renderer import FrameRenderer


def images_of_rank(n_images: int, rank: int, world: int) -> List[int]:
    """Eval images rank ``rank`` of ``world`` renders: i % world == rank."""
    return list(range(rank, n_images, world))


def average_metrics(rows: Dict[int, Dict[str, float]], keys: Sequence[str]) -> Dict[str, float]:
    """Mean of every key over the images, in image order, as the reference averages its per-image dicts
    (``float(torch.mean(torch.tensor([...])))``)."""
    order = sorted(rows)
    return {k: float(torch.mean(torch.tensor([rows[i][k] for i in order]))) for k in keys}


REGION_KEYS = ("psnr_dynamic", "ssim_dynamic", "psnr_static", "ssim_static")


def average_region_metrics(rows: Dict[int, Dict[str, float]], keys: Sequence[str]) -> Dict[str, float]:
    """``average_metrics``, except that each of ``REGION_KEYS`` is averaged over the images where it is defined (not
    NaN), still in image order; then ``num_images_dynamic`` / ``num_images_static``: the images whose region has a pixel
    (an image whose region only touches the 5-pixel border has a PSNR but no SSIM)."""
    order = sorted(rows)
    out = {}
    for k in keys:
        vals = [rows[i][k] for i in order]
        if k in REGION_KEYS:
            vals = [v for v in vals if not math.isnan(v)]
        out[k] = float(torch.mean(torch.tensor(vals)))
    out["num_images_dynamic"] = sum(not math.isnan(rows[i]["psnr_dynamic"]) for i in order)
    out["num_images_static"] = sum(not math.isnan(rows[i]["psnr_static"]) for i in order)
    return out


DEPTH_KEYS = ("depth_abs_rel", "depth_sq_rel", "depth_rmse", "depth_rmse_log", "depth_delta1", "depth_delta2", "depth_delta3")
REGION_SUFFIXES = ("_dynamic", "_static")


def depth_row_keys(regions: bool) -> List[str]:
    """Per-image depth keys: ``DEPTH_KEYS`` (columns 1-7 of ``ops.depth_metrics``' whole-image row), then with regions
    the same with ``_dynamic`` and with ``_static``."""
    return list(DEPTH_KEYS) + ([k + s for s in REGION_SUFFIXES for k in DEPTH_KEYS] if regions else [])


def average_depth_metrics(rows: Dict[int, Dict[str, float]], regions: bool) -> Dict[str, float]:
    """Each of ``depth_row_keys(regions)`` averaged in image order over the images where it is defined (not NaN), with
    ``num_images_depth`` (the images with a valid ground-truth pixel) after ``DEPTH_KEYS``; with regions
    ``num_images_depth_dynamic`` / ``num_images_depth_static`` come last."""
    order = sorted(rows)
    out: Dict[str, float] = {}
    for s in ("",) + (REGION_SUFFIXES if regions else ()):
        for k in DEPTH_KEYS:
            out[k + s] = float(torch.mean(torch.tensor([v for v in (rows[i][k + s] for i in order) if not math.isnan(v)])))
        if not s:
            out["num_images_depth"] = sum(not math.isnan(rows[i]["depth_abs_rel"]) for i in order)
    for s in REGION_SUFFIXES if regions else ():
        out["num_images_depth" + s] = sum(not math.isnan(rows[i]["depth_abs_rel" + s]) for i in order)
    return out


def median_dynamic_masks(images: torch.Tensor, cam_ids: Optional[torch.Tensor], gamma: float = KPLANES_DATAMANAGER.isg_gamma,
                         threshold: float = 0.5) -> torch.Tensor:
    """Dynamic-region masks of a clip, bool [B,H,W]: ``ops.isg_map(images, cam_ids, gamma) >= threshold``.

    That map is the reference's ISG residual (``compute_isg``): per pixel the channel mean of the Geman-McClure distance
    d^2 / (d^2 + gamma^2) of the frame from its camera's per-pixel temporal median.  Where the players move, the median
    is the background, so the mask marks what differs from the background in this frame (the IST map would also mark
    where the players were in neighbouring frames).  The policy: ``threshold`` 0.5 is the residual's midpoint, about
    |d| >= gamma; ``gamma`` defaults to the preset's ``isg_gamma``.  images: fp32 CUDA [B,H,W,3]; cam_ids [B]: every
    camera needs at least 3 images, since the median of 1 or 2 frames is not a background."""
    if cam_ids is None:
        raise ValueError("median_dynamic_masks: the cameras have no ids; the median is taken per camera")
    ids = cam_ids.reshape(-1).cpu()
    if ids.numel() != images.shape[0]:
        raise ValueError(f"median_dynamic_masks: {ids.numel()} camera ids for {images.shape[0]} images")
    for cam, n in zip(*(t.tolist() for t in torch.unique(ids, return_counts=True))):
        if n < 3:
            raise ValueError(f"median_dynamic_masks: camera {cam} has {n} image(s); its median needs at least 3")
    return ops.isg_map(images, ids, gamma) >= threshold


def pack_rows(rows: Dict[int, Dict[str, float]], keys: Sequence[str], n_rows: int) -> torch.Tensor:
    """float64 [n_rows, 1 + len(keys)] = (image index, values...) for ``all_gather``; unused rows have index -1."""
    out = torch.full((n_rows, 1 + len(keys)), -1.0, dtype=torch.float64)
    for r, i in enumerate(sorted(rows)):
        out[r, 0] = i
        out[r, 1:] = torch.tensor([rows[i][k] for k in keys], dtype=torch.float64)
    return out


def unpack_rows(packed: Sequence[torch.Tensor], keys: Sequence[str]) -> Dict[int, Dict[str, float]]:
    rows: Dict[int, Dict[str, float]] = {}
    for t in packed:
        for row in t.cpu().tolist():
            if row[0] >= 0:
                rows[int(row[0])] = dict(zip(keys, row[1:]))
    return rows


def eval_report(results: Dict[str, float], experiment_name: str, checkpoint: str,
                method_name: str = KPLANES_TRAINER["method_name"]) -> Dict[str, Any]:
    """The JSON ``ns-eval`` writes: {experiment_name, method_name, checkpoint, results}."""
    return {"experiment_name": experiment_name, "method_name": method_name, "checkpoint": str(checkpoint),
            "results": dict(results)}


class Evaluator:
    """Eval metrics of ``model`` on the eval split of ``datamanager`` (a ``DynamicDataManager`` built with
    ``eval_cameras`` / ``eval_images``).  ``rank`` / ``world``: this process' share of ``get_average_eval_image_metrics``
    (``torch.distributed`` must be initialised when ``world > 1``).  ``regions``: None, ``"median"`` (the
    ``median_dynamic_masks`` of the eval images and ``eval_cameras.ids``, computed here once) or a mask [B_eval,H,W]
    (non-zero: dynamic), e.g. rasterised player boxes; with it the averages also carry the per-region metrics.  When the
    eval image cache holds a ``depth_image``, the averages also carry the depth metrics (``average_depth_metrics``)."""

    regions: Optional[torch.Tensor] = None  # bool [B_eval,H,W] on the device
    depth: bool = False  # the eval split has ground-truth depth

    def __init__(self, model, datamanager, rank: int = 0, world: int = 1,
                 regions: Union[None, str, torch.Tensor] = None) -> None:
        if datamanager.eval_cameras is None:
            raise ValueError("Evaluator: the datamanager has no eval split (eval_cameras / eval_images)")
        self.model, self.datamanager = model, datamanager
        self.rank, self.world = rank, world
        if regions is not None:
            images = datamanager.eval_image_cache.batch["image"]
            if isinstance(regions, str):
                if regions != "median":
                    raise ValueError(f'Evaluator: regions must be None, "median" or a mask tensor (got {regions!r})')
                self.regions = median_dynamic_masks(images, datamanager.eval_cameras.ids)
            elif regions.shape != images.shape[:3]:
                raise ValueError(f"Evaluator: regions must be [B_eval,H,W] = {tuple(images.shape[:3])} (got {tuple(regions.shape)})")
            else:
                self.regions = regions.to(images.device) != 0
        self.depth = "depth_image" in datamanager.eval_image_cache.batch
        outputs = ["rgb", "depth", "accumulation", "median_rgb"]
        outputs += [f"prop_depth_{i}" for i in range(getattr(model.config, "num_proposal_iterations", 0))]
        if self.depth and not getattr(model.config, "is_euclidean_depth", True):
            outputs.append("directions_norm")  # the ground truth is z-depth: compared along the unit ray
        # whole frames per rank: the renderer itself is not sharded
        self.renderer = FrameRenderer(model, datamanager.eval_cameras, outputs=outputs)
        self._warm: set = set()
        self._lpips = None
        self._lpips_checked = False

    def _size(self, i: int) -> Tuple[int, int]:
        cams = self.datamanager.eval_cameras
        return cams._height_host[i], cams._width_host[i]

    def get_eval_loss_dict(self, step: int) -> Tuple[Dict[str, torch.Tensor], Dict[str, torch.Tensor], Dict[str, torch.Tensor]]:
        """-> (outputs, loss_dict, metrics_dict) of the model in eval mode on a ``next_eval`` batch."""
        was_training = self.model.training
        self.model.eval()
        try:
            with torch.no_grad():
                ray_bundle, batch = self.datamanager.next_eval(step)
                outputs = self.model(ray_bundle)
                metrics_dict = self.model.get_metrics_dict(outputs, batch)
                loss_dict = self.model.get_loss_dict(outputs, batch, metrics_dict)
        finally:
            self.model.train(was_training)
        return outputs, loss_dict, metrics_dict

    def get_eval_image_metrics_and_images(self, step: int) -> Tuple[Dict[str, float], Dict[str, torch.Tensor]]:
        """One random eval image, rendered whole and passed to the model's ``get_image_metrics_and_images``."""
        i, batch = self.datamanager.next_eval_image(step)
        outputs = self.renderer.render(i, device_frames=True)
        metrics_dict, images_dict = self.model.get_image_metrics_and_images(outputs, batch)
        h, w = self._size(i)
        metrics_dict["image_idx"] = i
        metrics_dict["num_rays"] = h * w
        return metrics_dict, images_dict

    def _render_timed(self, i: int, depth: bool = False) -> Tuple[Union[torch.Tensor, Callable[[], float], None], ...]:
        """-> (rgb [H,W,3] on the device, seconds of the render: call once the stream has passed the render); with
        ``depth`` then also the frame's depth [H,W,1] and its directions_norm [H,W,1] (None when not rendered)."""
        if self._size(i) not in self._warm:  # the first frame of a size captures the tile graphs: not part of the time
            self.renderer.render(i, device_frames=True)
            self._warm.add(self._size(i))
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        out = self.renderer.render(i, device_frames=True)
        end.record()
        timed = (out["rgb"], lambda: start.elapsed_time(end) / 1e3)
        return timed + (out["depth"], out.get("directions_norm")) if depth else timed

    def _lpips_metric(self, device):
        if not self._lpips_checked:  # the model's rule: LPIPS only when its pretrained network is available
            self._lpips = image_metrics.optional_lpips(device)
            self._lpips_checked = True
        return self._lpips

    def _rank_rows(self, mine: Sequence[int]) -> Dict[int, Dict[str, float]]:
        """Per-image rows {psnr, ssim, [lpips], num_rays_per_sec, fps, [REGION_KEYS, dynamic_fraction],
        [depth_row_keys]} of this rank's images."""
        if not mine:
            return {}
        renders = [self._render_timed(i, depth=True) if self.depth else self._render_timed(i) for i in mine]
        pred = torch.stack([r[0] for r in renders])
        idx = torch.tensor(mine, device=pred.device)
        target = self.datamanager.eval_image_cache.batch["image"][idx]
        values = ops.image_metrics(pred, target)
        mask = None
        if self.regions is not None:
            mask = self.regions.to(pred.device)[idx]
            fraction = mask.flatten(1).sum(1, dtype=torch.float64) / mask[0].numel()
            values = torch.cat([values.double(), ops.image_metrics_masked(pred, target, mask).double(), fraction[:, None]], 1)
        if self.depth:
            norms = [r[3] for r in renders]
            depth = ops.depth_metrics(torch.stack([r[2] for r in renders]), self.datamanager.eval_image_cache.batch["depth_image"][idx],
                                      None if norms[0] is None else torch.stack(norms), mask)
            values = torch.cat([values.double(), depth[:, :, 1:].flatten(1)], 1)  # (n_valid dropped: NaN marks "undefined")
        values = values.tolist()  # the one host synchronisation: the events have completed too
        n_colour = 2 if self.regions is None else 7
        lpips = self._lpips_metric(pred.device)
        rows = {}
        for k, i in enumerate(mine):
            h, w = self._size(i)
            row = {"psnr": values[k][0], "ssim": values[k][1]}
            if lpips is not None:
                row["lpips"] = float(lpips(torch.moveaxis(target[k], -1, 0)[None], torch.moveaxis(pred[k], -1, 0)[None]))
            row["num_rays_per_sec"] = h * w / renders[k][1]()
            row["fps"] = row["num_rays_per_sec"] / (h * w)
            if self.regions is not None:
                row.update(zip(REGION_KEYS + ("dynamic_fraction",), values[k][2:n_colour]))
            if self.depth:
                row.update(zip(depth_row_keys(self.regions is not None), values[k][n_colour:]))
            rows[i] = row
        return rows

    def _keys(self, device) -> List[str]:
        keys = ["psnr", "ssim"] + (["lpips"] if self._lpips_metric(device) is not None else []) + ["num_rays_per_sec", "fps"]
        keys = keys if self.regions is None else keys + list(REGION_KEYS) + ["dynamic_fraction"]
        return keys + depth_row_keys(self.regions is not None) if self.depth else keys

    def _all_gather(self, rows: Dict[int, Dict[str, float]], keys: Sequence[str], n_images: int) -> Dict[int, Dict[str, float]]:
        import torch.distributed as dist

        dev = torch.device("cuda", torch.cuda.current_device())
        packed = pack_rows(rows, keys, -(-n_images // self.world)).to(dev)
        gathered = [torch.empty_like(packed) for _ in range(self.world)]
        dist.all_gather(gathered, packed)
        return unpack_rows(gathered, keys)

    def get_average_eval_image_metrics(self, step: int = 0) -> Dict[str, float]:
        """Every eval image: ``psnr``, ``ssim`` (and ``lpips`` when available), ``num_rays_per_sec`` and ``fps`` averaged
        over the images (``VanillaPipeline.get_average_eval_image_metrics``).  With ``regions``, then ``REGION_KEYS``,
        ``dynamic_fraction`` (the mean share of dynamic pixels), ``num_images_dynamic`` and ``num_images_static``
        (``average_region_metrics``).  With eval depth, then the depth keys (``average_depth_metrics``)."""
        n = len(self.datamanager.eval_cameras)
        rows = self._rank_rows(images_of_rank(n, self.rank, self.world))
        keys = self._keys(self.datamanager.device)
        if self.world > 1:
            rows = self._all_gather(rows, keys, n)
        colour = keys[:len(keys) - len(depth_row_keys(self.regions is not None))] if self.depth else keys
        out = average_metrics(rows, colour) if self.regions is None else average_region_metrics(rows, colour)
        if self.depth:
            out.update(average_depth_metrics(rows, self.regions is not None))
        return out
