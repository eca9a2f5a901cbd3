"""Rendering a camera path to image files: what ``ns-render --camera-path-filename`` does for a trained model
(REF/nerfstudio/scripts/render.py ``_render_trajectory_video``), writing PNG frames.

Per frame: ``FrameRenderer.render(i, device_frames=True)`` renders the requested outputs into device tensors (one
CUDA-graph replay per tile), ``ops.compose_frame`` colour-maps them and lays them side by side as one uint8 image on the
same stream, a copy stream moves the image into one of a small ring of pinned host buffers, and a thread pool encodes
the PNG ``output_dir/{i:05d}.png`` with PIL.  The GPU renders frame k+1 while frame k is encoded; the render loop waits
only when the ring is full.

With ``world > 1`` rank r renders the whole frames ``i % world == r``.  A file's name depends only on its frame index,
so the ranks write disjoint files, need no collective, and together write the same set of files as one rank does.
For a dynamic model the path must carry a render time per camera: that is what makes the players move.
"""
from __future__ import annotations

import contextlib
import json
import os
from concurrent.futures import Future, ThreadPoolExecutor
from typing import Dict, List, Optional, Sequence, Tuple, Union

import torch

from .. import ops
from ..cameras.camera_paths import CropData, get_crop_from_json, get_path_from_json
from ..cameras.cameras import Cameras
from ..model_components.renderers import background_color_override_context
from .evaluator import images_of_rank
from .frame_renderer import FrameRenderer

RING_SLOTS = 3  # pinned host images in flight: one being filled by the copy, the others being encoded


def load_camera_path(path_or_dict: Union[str, os.PathLike, Dict]) -> Tuple[Cameras, Optional[CropData]]:
    """A camera-path JSON file (or its already-parsed dict) -> (cameras on the host, crop or None)."""
    if isinstance(path_or_dict, dict):
        camera_path = path_or_dict
    else:
        with open(path_or_dict, "r", encoding="utf-8") as f:
            camera_path = json.load(f)
    return get_path_from_json(camera_path), get_crop_from_json(camera_path)


def available_outputs(model) -> List[str]:
    """The per-pixel outputs of the model that can be written as images."""
    names = ["rgb", "depth", "accumulation", "median_rgb"]
    return names + [f"prop_depth_{i}" for i in range(getattr(model.config, "num_proposal_iterations", 0))]


def check_render_inputs(model, cameras: Cameras, rendered_output_names: Sequence[str]) -> None:
    """The ValueErrors of ``render_camera_path``, raised before anything is rendered."""
    available = available_outputs(model)
    names = list(rendered_output_names)
    if not names:
        raise ValueError(f"no rendered_output_names; available outputs: {available}")
    unknown = [n for n in names if n not in available]
    if unknown:
        raise ValueError(f"unknown rendered output(s) {unknown}; available outputs: {available}")
    if len(names) > ops.COMPOSE_MAX_PANELS:
        raise ValueError(f"at most {ops.COMPOSE_MAX_PANELS} rendered outputs per frame (got {len(names)})")
    if getattr(model.field, "has_time_planes", False) and cameras.times is None:
        raise ValueError("the model is dynamic (its field has time planes) but the cameras have no times: every camera of "
                         "the path needs a render_time")
    sizes = sorted(set(zip(cameras._height_host, cameras._width_host)))
    if len(sizes) > 1:
        raise ValueError(f"the cameras' frames differ in size (H, W): {sizes}; one image size per path")


def _write_png(done: torch.cuda.Event, image: torch.Tensor, path: str) -> None:
    from PIL import Image

    done.synchronize()  # the copy into this pinned buffer has landed
    Image.fromarray(image.numpy()).save(path)


def render_camera_path(model, cameras: Cameras, output_dir: Union[str, os.PathLike],
                       rendered_output_names: Sequence[str] = ("rgb",), rank: int = 0, world: int = 1,
                       crop: Optional[CropData] = None) -> List[int]:
    """Render this rank's frames of ``cameras`` (``i % world == rank``) and write each as ``output_dir/{i:05d}.png``:
    the ``rendered_output_names`` side by side, colour-mapped like the model's eval images.  ``crop``: rays start and
    end at the crop box and the crop's background colour shows outside it (ns-render's crop).  Returns the frame
    indices this rank wrote."""
    check_render_inputs(model, cameras, rendered_output_names)
    names = list(rendered_output_names)
    dev = model.device
    if cameras.device != dev:
        cameras = cameras.to(dev)
    outputs = names + (["accumulation"] if "accumulation" not in names and any(ops.panel_kind(n) == 2 for n in names) else [])
    os.makedirs(output_dir, exist_ok=True)
    mine = images_of_rank(len(cameras), rank, world)
    aabb_box = None
    bg = None
    if crop is not None:
        aabb_box = crop.scene_box
        bg = crop.background_color.to(dev, torch.float32)  # on the device: the tile graphs read it, no copy in the capture
    renderer = FrameRenderer(model, cameras, outputs=outputs, aabb_box=aabb_box)  # whole frames per rank
    h, w = cameras._height_host[0], cameras._width_host[0]
    ring = [torch.empty((h, w * len(names), 3), dtype=torch.uint8).pin_memory() for _ in range(min(RING_SLOTS, len(mine)))]
    pending: List[Optional[Future]] = [None] * len(ring)
    copy_stream = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream(dev)
    with ThreadPoolExecutor(max_workers=max(1, len(ring))) as pool, \
            (background_color_override_context(bg) if bg is not None else contextlib.nullcontext()):
        for k, i in enumerate(mine):
            slot = k % len(ring)
            if pending[slot] is not None:
                pending[slot].result()  # ring full: this buffer's PNG is still being encoded
            frames = renderer.render(i, device_frames=True)
            image = ops.compose_frame(frames, names)
            copy_stream.wait_stream(main)
            with torch.cuda.stream(copy_stream):
                ring[slot].copy_(image, non_blocking=True)
                image.record_stream(copy_stream)
                done = torch.cuda.Event()
                done.record(copy_stream)
            pending[slot] = pool.submit(_write_png, done, ring[slot], os.path.join(os.fspath(output_dir), f"{i:05d}.png"))
        for fut in pending:
            if fut is not None:
                fut.result()
    return mine

