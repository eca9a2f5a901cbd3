"""Camera paths: the camera-path JSON the viewer exports and ``ns-render --camera-path-filename`` reads, as
``get_path_from_json`` (NS/cameras/camera_paths.py) and ``get_crop_from_json`` (scripts/render.py) read it.

The format, as this module reads it (tests/test_render_path_host.py pins each rule):
  * ``render_height`` / ``render_width``: H and W of every camera; cx = W/2, cy = H/2.
  * ``camera_type``: absent (perspective), "perspective", "fisheye" or "equirectangular"; anything else is a ValueError
    (the reference falls back to perspective silently).
  * ``camera_path``: one entry per camera.  ``camera_to_world`` is a row-major 4x4 matrix of 16 floats; its top three
    rows are the camera-to-world pose.  Perspective and fisheye: ``fov`` is the vertical field of view in degrees
    (three.js), fx = fy = 0.5*H / tan(0.5*fov*pi/180).  Equirectangular: fx = W/2, fy = H.  ``aspect`` is not read:
    W and H are given.
  * ``render_time`` in [0, 1] (the training cameras' time range): the cameras carry times only when every entry has
    one, else ``times`` is None.
  * an optional top-level ``crop``: ``{crop_bg_color: {r, g, b} in 0-255, crop_center: [3], crop_scale: [3]}`` ->
    ``CropData``: background colour rgb/255 and the box center +- scale/2.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Any, Dict, Optional

import torch

from ..data.scene_box import SceneBox
from .cameras import Cameras, CameraType

_CAMERA_TYPES = {"perspective": CameraType.PERSPECTIVE, "fisheye": CameraType.FISHEYE,
                 "equirectangular": CameraType.EQUIRECTANGULAR}


def three_js_perspective_camera_focal_length(fov: float, image_height: int) -> float:
    """Focal length in pixels of a three.js camera with vertical field of view ``fov`` degrees."""
    return 0.5 * image_height / math.tan(0.5 * fov * math.pi / 180.0)


def get_path_from_json(camera_path: Dict[str, Any]) -> Cameras:
    """A camera-path dict -> ``Cameras`` on the host (one camera per ``camera_path`` entry)."""
    h, w = int(camera_path["render_height"]), int(camera_path["render_width"])
    name = camera_path.get("camera_type", "perspective")
    if name not in _CAMERA_TYPES:
        raise ValueError(f"camera path: camera_type {name!r} is not one of {sorted(_CAMERA_TYPES)}")
    camera_type = _CAMERA_TYPES[name]
    entries = camera_path["camera_path"]
    if not entries:
        raise ValueError("camera path: camera_path holds no cameras")
    c2ws, fxs, fys = [], [], []
    for cam in entries:
        c2ws.append(torch.tensor(cam["camera_to_world"], dtype=torch.float32).view(4, 4)[:3])
        if camera_type == CameraType.EQUIRECTANGULAR:
            fxs.append(w / 2)
            fys.append(float(h))
        else:
            f = three_js_perspective_camera_focal_length(cam["fov"], h)
            fxs.append(f)
            fys.append(f)
    times = None
    if all("render_time" in cam for cam in entries):
        times = torch.tensor([float(cam["render_time"]) for cam in entries], dtype=torch.float32)
    return Cameras(torch.stack(c2ws), torch.tensor(fxs), torch.tensor(fys), w / 2, h / 2, width=w, height=h,
                   camera_type=camera_type, times=times)


def get_seconds_from_json(camera_path: Dict[str, Any]) -> float:
    """The path's ``seconds``: how long its video plays (``len(camera_path) / seconds`` frames per second)."""
    if "seconds" not in camera_path:
        raise ValueError("camera path: no 'seconds' entry; a video needs the path's length in seconds")
    seconds = float(camera_path["seconds"])
    if not seconds > 0 or not math.isfinite(seconds):
        raise ValueError(f"camera path: seconds must be positive and finite (got {camera_path['seconds']!r})")
    return seconds


@dataclass
class CropData:
    """A crop of the render (scripts/render.py ``CropData``): outside the box the background colour shows."""

    background_color: torch.Tensor  # [3] in [0, 1]
    center: torch.Tensor  # [3]
    scale: torch.Tensor  # [3]

    @property
    def scene_box(self) -> SceneBox:
        return SceneBox(aabb=torch.stack([self.center - self.scale / 2.0, self.center + self.scale / 2.0]))


def get_crop_from_json(camera_path: Dict[str, Any]) -> Optional[CropData]:
    """The path's ``crop`` entry -> ``CropData``, or None when the path has none."""
    crop = camera_path.get("crop")
    if crop is None:
        return None
    bg = crop["crop_bg_color"]
    return CropData(background_color=torch.tensor([bg["r"] / 255.0, bg["g"] / 255.0, bg["b"] / 255.0], dtype=torch.float32),
                    center=torch.tensor(crop["crop_center"], dtype=torch.float32),
                    scale=torch.tensor(crop["crop_scale"], dtype=torch.float32))
