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

``write_eval_images`` / ``write_eval_videos`` show where those numbers come from: each eval image is rendered once, its
per-pixel error, SSIM and depth-error maps come from ``ops.eval_maps``, and the panels (``eval_panels``) are composed
and, for JPEG and video, encoded on the device through the render side's frame loop (``path_renderer._frame_loop``).
The per-image rows written beside the images come from ``_measure``, the same kernels ``get_average_eval_image_metrics``
averages with, one image at a time.
"""
from __future__ import annotations

import json
import math
import os
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


MAP_PANELS = ("error", "ssim", "depth_error")  # the panels of ops.eval_maps


def eval_panels(model, depth: bool, regions: bool) -> List[str]:
    """The panels ``Evaluator.write_eval_images`` can show: the eval image ``gt``, the renderer's outputs, the error maps;
    with eval depth the ground-truth depth ``depth_gt`` and ``depth_error``; with regions the ``dynamic_mask``."""
    names = ["gt", "rgb", "median_rgb", "error", "ssim", "depth", "accumulation"]
    names += [f"prop_depth_{i}" for i in range(getattr(model.config, "num_proposal_iterations", 0))]
    names += ["depth_gt", "depth_error"] if depth else []
    return names + (["dynamic_mask"] if regions else [])


def check_eval_panels(available: Sequence[str], panels: Sequence[str], error_range: float, depth_error_range: float) -> List[str]:
    """The ValueErrors of ``write_eval_images`` / ``write_eval_videos``, raised before anything is rendered."""
    names = list(panels)
    if not names:
        raise ValueError(f"no panels; available panels: {list(available)}")
    missing = [n for n in names if n not in available]
    if missing:
        raise ValueError(f"panel(s) {missing} not available (depth_gt and depth_error need eval depth, dynamic_mask needs "
                         f"regions); available panels: {list(available)}")
    if len(names) > ops.COMPOSE_MAX_PANELS:
        raise ValueError(f"at most {ops.COMPOSE_MAX_PANELS} panels per image (got {len(names)})")
    for name, r in (("error_range", error_range), ("depth_error_range", depth_error_range)):
        if isinstance(r, bool) or not isinstance(r, (int, float)) or not (r > 0 and math.isfinite(r)):
            raise ValueError(f"{name} must be positive and finite (got {r!r})")
    return names


def eval_video_sequences(ids: Optional[torch.Tensor], times: Optional[torch.Tensor], n_images: int) -> Dict[str, List[int]]:
    """{video file name: eval image indices in play order}: ``camera_{id:03d}.avi`` per camera id with that camera's
    images ordered by time (equal times in image order); without ids one ``eval.avi`` in image order."""
    if ids is None:
        return {"eval.avi": list(range(n_images))}
    cam = [int(v) for v in ids.reshape(-1).tolist()]
    t = [0.0] * n_images if times is None else [float(v) for v in times.reshape(-1).tolist()]
    if len(cam) != n_images or len(t) != n_images:
        raise ValueError(f"{len(cam)} camera ids and {len(t)} times for {n_images} eval images")
    return {f"camera_{c:03d}.avi": sorted((i for i in range(n_images) if cam[i] == c), key=lambda i: (t[i], i))
            for c in sorted(set(cam))}


def metrics_file_name(rank: int, world: int, gathered: bool) -> Optional[str]:
    """The file rank ``rank`` writes the per-image rows to: ``metrics.json`` with one rank, or on rank 0 when the rows
    were gathered over a process group (None on the other ranks); else ``metrics.rank{r}.json`` with its own rows."""
    if world == 1 or gathered:
        return "metrics.json" if rank == 0 else None
    return f"metrics.rank{rank}.json"


def metrics_document(rows: Dict[int, Dict[str, float]], extension: str) -> Dict[str, Any]:
    """The content of ``metrics.json``: {"images": [{"image": i, "file": "{i:05d}.{extension}", <row>}, ...]} in image
    order."""
    return {"images": [dict({"image": i, "file": f"{i:05d}.{extension}"}, **rows[i]) for i in sorted(rows)]}


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

    def _value_keys(self) -> List[str]:
        """The columns of ``_measure``: psnr, ssim, [REGION_KEYS, dynamic_fraction], [depth_row_keys]."""
        keys = ["psnr", "ssim"] + (list(REGION_KEYS) + ["dynamic_fraction"] if self.regions is not None else [])
        return keys + depth_row_keys(self.regions is not None) if self.depth else keys

    def _measure(self, sel: Union[torch.Tensor, slice], pred: torch.Tensor, depth: Optional[torch.Tensor] = None,
                 norms: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The ``_value_keys`` columns [B, K] on the device of the renders ``pred`` [B,H,W,3] (``depth``, ``norms``
        [B,H,W,1] with eval depth) of the eval images ``sel`` (an index tensor or a slice).  No host synchronisation.
        A row depends only on its own image, so one image at a time gives the bits of the whole batch."""
        batch = self.datamanager.eval_image_cache.batch
        target = batch["image"][sel]
        values = ops.image_metrics(pred, target)
        mask = None
        if self.regions is not None:
            mask = self.regions.to(pred.device)[sel]
            fraction = mask.flatten(1).sum(1, dtype=torch.float64) / mask[0].numel()
            values = torch.cat([values.double(), ops.image_metrics_masked(pred, target, mask).double(), fraction[:, None]], 1)
        if self.depth:
            depth = ops.depth_metrics(depth, batch["depth_image"][sel], norms, mask)
            values = torch.cat([values.double(), depth[:, :, 1:].flatten(1)], 1)  # (n_valid dropped: NaN marks "undefined")
        return values

    def _rank_rows(self, mine: Sequence[int]) -> Dict[int, Dict[str, float]]:
        """Per-image rows {psnr, ssim, [lpips], num_rays_per_sec, fps, [REGION_KEYS, dynamic_fraction],
        [depth_row_keys]} of this rank's images."""
        if not mine:
            return {}
        renders = [self._render_timed(i, depth=True) if self.depth else self._render_timed(i) for i in mine]
        pred = torch.stack([r[0] for r in renders])
        idx = torch.tensor(mine, device=pred.device)
        depth = norms = None
        if self.depth:
            depth = torch.stack([r[2] for r in renders])
            norms = None if renders[0][3] is None else torch.stack([r[3] for r in renders])
        values = self._measure(idx, pred, depth, norms).tolist()  # the one host synchronisation: the events have completed too
        keys = self._value_keys()
        target = self.datamanager.eval_image_cache.batch["image"][idx]
        lpips = self._lpips_metric(pred.device)
        rows = {}
        for k, i in enumerate(mine):
            h, w = self._size(i)
            row = {"psnr": values[k][0], "ssim": values[k][1]}
            if lpips is not None:
                row["lpips"] = float(lpips(torch.moveaxis(target[k], -1, 0)[None], torch.moveaxis(pred[k], -1, 0)[None]))
            row["num_rays_per_sec"] = h * w / renders[k][1]()
            row["fps"] = row["num_rays_per_sec"] / (h * w)
            row.update(zip(keys[2:], values[k][2:]))
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

    # ---- the eval images as files ----
    def _eval_frame(self, i: int, names: Sequence[str], error_range: float, depth_error_range: float,
                    values: Optional[Dict[int, torch.Tensor]] = None) -> torch.Tensor:
        """Render eval image i once and compose ``names`` on the device (uint8 [H, W*P, 3]); with ``values``, also put
        its ``_measure`` row (on the device) in ``values[i]``."""
        out = self.renderer.render(i, device_frames=True)
        batch = self.datamanager.eval_image_cache.batch
        pred, target = out["rgb"], batch["image"][i]
        norms = out.get("directions_norm")
        depth = gt_depth = None
        if self.depth:
            depth, gt_depth = out["depth"], batch["depth_image"][i]
        if values is not None:
            values[i] = self._measure(slice(i, i + 1), pred[None], None if depth is None else depth[None],
                                      None if norms is None else norms[None])
        frames = dict(out, gt=target)
        if any(n in MAP_PANELS for n in names):
            maps = ops.eval_maps(pred[None], target[None], None if depth is None else depth[None],
                                 None if gt_depth is None else gt_depth[None], None if norms is None else norms[None])
            frames["error"] = (maps["error"][0] / error_range)[..., None]
            frames["ssim"] = (1 - maps["ssim"][0])[..., None]  # bright = bad, as for the error; the NaN border shows as 0
            if depth is not None:
                frames["depth_error"] = (maps["depth_error"][0] / depth_error_range)[..., None]  # NaN (invalid) shows as 0
        if "depth_gt" in names:
            g = gt_depth if norms is None else gt_depth * norms  # z-depth -> distance along the ray, as the metrics compare
            valid = torch.isfinite(g) & (g > 0)
            # invalid pixels: white (accumulation 0) and the valid minimum, so they set neither near nor far
            frames["depth_gt"] = torch.where(valid, g, torch.where(valid, g, math.inf).amin())
            frames["depth_gt_valid"] = valid.float()
        if "dynamic_mask" in names:
            frames["dynamic_mask"] = self.regions[i].float()[..., None]
        return ops.compose_frame(frames, names)

    def _check_write(self, panels, error_range: float, depth_error_range: float) -> List[str]:
        return check_eval_panels(eval_panels(self.model, self.depth, self.regions is not None), panels, error_range,
                                 depth_error_range)

    def write_eval_images(self, output_dir: Union[str, os.PathLike], panels: Sequence[str] = ("gt", "rgb", "error", "ssim"),
                          image_format: str = "png", jpeg_quality: int = 95, error_range: float = 0.25,
                          depth_error_range: float = 0.25) -> List[int]:
        """Write this rank's eval images (``i % world == rank``) as ``output_dir/{i:05d}.png`` (PIL on the host) or
        ``.jpg`` (``image_format="jpeg"``, encoded on the device): the ``panels`` side by side (``eval_panels``).
        ``error``: viridis of the per-pixel error / ``error_range``; ``ssim``: viridis of 1 - the per-pixel SSIM (the
        5-pixel border, where no window lies inside, shows as 0); ``depth_gt``: the ground-truth depth through turbo over
        its own near / far, white where it is invalid; ``depth_error``: viridis of the relative depth error /
        ``depth_error_range`` (0 where the ground truth is invalid); ``dynamic_mask``: the ``regions`` mask.  Values
        beyond a range show as its top colour.

        Each image is rendered once; maps, composition and JPEG run on the device while the previous image is written.
        Also writes the per-image rows (psnr, ssim, the region and depth keys; bit for bit the rows
        ``get_average_eval_image_metrics`` averages) to ``metrics.json`` (``metrics_document``): with a process group
        rank 0 writes every rank's rows, without one each rank of several writes ``metrics.rank{r}.json``.  Returns the
        image indices this rank wrote."""
        from .path_renderer import IMAGE_FORMATS, _frame_loop, check_jpeg_quality, file_writer

        names = self._check_write(panels, error_range, depth_error_range)
        if image_format not in IMAGE_FORMATS:
            raise ValueError(f"image_format {image_format!r} is not one of {IMAGE_FORMATS}")
        check_jpeg_quality(jpeg_quality)
        out = os.fspath(output_dir)
        os.makedirs(out, exist_ok=True)
        n = len(self.datamanager.eval_cameras)
        mine = images_of_rank(n, self.rank, self.world)
        h, w = self.datamanager.eval_image_cache.batch["image"].shape[1:3]
        values: Dict[int, torch.Tensor] = {}
        _frame_loop(lambda i: self._eval_frame(i, names, error_range, depth_error_range, values), mine, (h, w * len(names)),
                    self.datamanager.device, None if image_format == "png" else jpeg_quality, file_writer(out, image_format))
        keys = self._value_keys()
        table = torch.cat([values[i] for i in mine]).tolist() if mine else []
        rows = {i: dict(zip(keys, table[k])) for k, i in enumerate(mine)}
        gathered = self.world > 1 and torch.distributed.is_available() and torch.distributed.is_initialized()
        if gathered:
            rows = self._all_gather(rows, keys, n)
        name = metrics_file_name(self.rank, self.world, gathered)
        if name is not None:
            with open(os.path.join(out, name), "w", encoding="utf-8") as f:
                json.dump(metrics_document(rows, "png" if image_format == "png" else "jpg"), f, indent=1)
        return mine

    def write_eval_videos(self, output_dir: Union[str, os.PathLike], fps: float,
                          panels: Sequence[str] = ("gt", "rgb", "error", "ssim"), jpeg_quality: int = 95,
                          error_range: float = 0.25, depth_error_range: float = 0.25) -> Dict[str, List[int]]:
        """Write the eval split as Motion-JPEG AVIs at ``fps`` frames per second: ``camera_{id:03d}.avi`` per eval camera
        id with its images in time order, or one ``eval.avi`` in image order without ids (``eval_video_sequences``);
        each frame is ``panels`` side by side, as ``write_eval_images`` composes them.  The k-th frame of a video goes to
        rank ``k % world``, which encodes it into its part file.  With one rank the videos are written at once; with a
        process group the ranks meet at a barrier and rank 0 assembles them; without one the caller runs
        ``assemble_video(path, world, fps)`` for each returned path once every rank is done.  ``fps`` is required:
        eval frames are usually subsampled from the clip, so only the caller knows their rate.  Returns {video path:
        the image indices this rank encoded into it}."""
        from .path_renderer import assemble_video, check_jpeg_quality, write_part

        names = self._check_write(panels, error_range, depth_error_range)
        check_jpeg_quality(jpeg_quality)
        if isinstance(fps, bool) or not isinstance(fps, (int, float)) or not (fps > 0 and math.isfinite(fps)):
            raise ValueError(f"fps must be positive and finite (got {fps!r})")
        out = os.fspath(output_dir)
        os.makedirs(out, exist_ok=True)
        cams = self.datamanager.eval_cameras
        h, w = self.datamanager.eval_image_cache.batch["image"].shape[1:3]
        written = {}
        for name, seq in eval_video_sequences(cams.ids, cams.times, len(cams)).items():
            path = os.path.join(out, name)
            written[path] = write_part(path, self.rank, lambda i: self._eval_frame(i, names, error_range, depth_error_range),
                                       seq[self.rank::self.world], (h, w * len(names)), self.datamanager.device, jpeg_quality)
        if self.world == 1:
            for path in written:
                assemble_video(path, 1, fps)
        elif torch.distributed.is_available() and torch.distributed.is_initialized():
            torch.distributed.barrier()
            if self.rank == 0:
                for path in written:
                    assemble_video(path, self.world, fps)
        return written
