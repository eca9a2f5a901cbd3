"""Cameras: the subset of NS/cameras/cameras.py the K-Planes path's callers use -- a flat batch of perspective,
fisheye or equirectangular cameras (mixed types allowed) with optional OpenCV lens distortion, as the reference's
dataparsers build them (broadcaststyle_dataparser.py:465-509) -- with ray generation on the device
(``kp_generate_rays``).

Same constructor argument names, attribute names (``camera_to_worlds, fx, fy, cx, cy, width, height, times``) and
``generate_rays`` call forms as the reference (cameras.py:38-120, 327-502):
  * ``generate_rays(camera_indices=c[:, None], coords=coords)`` -- RayGenerator.forward, ray_generators.py:43-59
  * ``generate_rays(camera_indices=i, keep_shape=True)``          -- a whole frame (scripts/render.py, eval)
plus ``generate_tile(camera_index, start, end)`` (a row-major pixel range of a frame without materialising coords).
All-zero distortion parameters are dropped at construction: the reference's Newton iteration leaves such points
unchanged bit for bit (residual 0, step 0), so those cameras take the plain perspective kernel.  Camera-optimizer
deltas (``camera_opt_to_camera``, ``distortion_params_delta``) and multi-dimensional camera batches are not built: they
raise NotImplementedError instead of taking another route.
"""
from __future__ import annotations

from enum import Enum, auto
from typing import List, Optional, Union

import torch

from .. import ops
from ..data.scene_box import SceneBox
from .rays import RayBundle


class CameraType(Enum):
    """cameras.py:28-33."""

    PERSPECTIVE = auto()
    FISHEYE = auto()
    EQUIRECTANGULAR = auto()


def _col(v, n: int, device, dtype=torch.float32) -> torch.Tensor:
    if not torch.is_tensor(v):
        v = torch.tensor([float(v)], dtype=dtype)
    v = v.to(device=device, dtype=dtype).reshape(-1, 1)
    return v.expand(n, 1).contiguous() if v.shape[0] == 1 else v.contiguous()


class Cameras:
    def __init__(self, camera_to_worlds: torch.Tensor, fx, fy, cx, cy, width=None, height=None,
                 distortion_params: Optional[torch.Tensor] = None, camera_type=CameraType.PERSPECTIVE,
                 times: Optional[torch.Tensor] = None, ids: Optional[torch.Tensor] = None) -> None:
        c2w = camera_to_worlds
        if c2w.dim() == 2:
            c2w = c2w[None]
        if c2w.dim() != 3 or c2w.shape[-2:] != (3, 4):
            raise NotImplementedError("Cameras: a flat batch [num_cameras, 3, 4] of camera-to-world matrices is supported")
        dev = c2w.device
        n = c2w.shape[0]
        self.camera_type = self._parse_camera_type(camera_type, n, dev)
        self.distortion_params = self._parse_distortion(distortion_params, n, dev)
        self.camera_to_worlds = c2w.float().contiguous()
        self.fx, self.fy, self.cx, self.cy = (_col(v, n, dev) for v in (fx, fy, cx, cy))
        h = height if height is not None else (self.cy * 2).to(torch.int64)
        w = width if width is not None else (self.cx * 2).to(torch.int64)
        self.height, self.width = _col(h, n, dev, torch.int64), _col(w, n, dev, torch.int64)
        # host copies: reading a size back from the device would synchronise every tile of a frame
        self._height_host, self._width_host = self.height.view(-1).tolist(), self.width.view(-1).tolist()
        self.times = None if times is None else times.to(dev).float().reshape(n, 1).contiguous()
        self.ids = ids
        self._intrinsics = None
        # what the kernel takes: NULL for "all perspective" / "no distortion" (the plain kernel), else per-camera tables
        plain = bool((self.camera_type == CameraType.PERSPECTIVE.value).all())
        self._cam_types = None if plain else self.camera_type.view(-1).to(torch.int32).contiguous()
        self._distortion = self.distortion_params

    @classmethod
    def from_reference(cls, cameras, device=None) -> "Cameras":
        """A flat batch of the reference's ``Cameras`` (NS/cameras/cameras.py:56-146; same field names, read by duck
        typing) -> this class, on ``device`` (default: where the reference object lives)."""
        dev = cameras.camera_to_worlds.device if device is None else device
        to = lambda t: None if t is None else t.to(dev)  # noqa: E731
        return cls(to(cameras.camera_to_worlds), to(cameras.fx), to(cameras.fy), to(cameras.cx), to(cameras.cy),
                   width=to(cameras.width), height=to(cameras.height), distortion_params=getattr(cameras, "distortion_params", None),
                   camera_type=cameras.camera_type, times=getattr(cameras, "times", None), ids=getattr(cameras, "ids", None))

    @staticmethod
    def _parse_camera_type(camera_type, n: int, dev) -> torch.Tensor:
        """cameras.py:178-218: CameraType | List[CameraType] | int | integer tensor -> int64 [n,1]; values outside the
        enum raise like the reference does at ray generation (cameras.py:699-701)."""
        if isinstance(camera_type, CameraType):
            t = torch.tensor([camera_type.value])
        elif isinstance(camera_type, (list, tuple)) and len(camera_type) and isinstance(camera_type[0], CameraType):
            t = torch.tensor([c.value for c in camera_type])
        elif isinstance(camera_type, int):
            t = torch.tensor([camera_type])
        elif torch.is_tensor(camera_type):
            if torch.is_floating_point(camera_type):
                raise AssertionError(f"camera_type tensor must be of type int, not: {camera_type.dtype}")
            t = camera_type
        else:
            raise ValueError('Invalid camera_type. Must be CameraType, List[CameraType], int, or torch.Tensor["num_cameras"]. '
                             "Received: " + str(type(camera_type)))
        t = t.reshape(-1, 1).to(device=dev, dtype=torch.int64)
        if t.shape[0] not in (1, n):
            raise ValueError(f"camera_type has {t.shape[0]} entries for {n} cameras")
        t = t.expand(n, 1).contiguous()
        valid = [c.value for c in CameraType]
        for v in torch.unique(t.cpu()).tolist():
            if v not in valid:
                raise ValueError(f"Camera type {v} not supported.")
        return t

    @staticmethod
    def _parse_distortion(distortion_params, n: int, dev) -> Optional[torch.Tensor]:
        """[6] or [n,6] OpenCV (k1,k2,k3,k4,p1,p2), camera_utils.get_distortion_params order -> fp32 [n,6] | None."""
        if distortion_params is None:
            return None
        d = torch.as_tensor(distortion_params, dtype=torch.float32)
        if d.shape[-1] != 6 or d.dim() > 2:
            raise ValueError("distortion_params must be [6] or [num_cameras, 6] (k1, k2, k3, k4, p1, p2)")
        d = d.reshape(-1, 6)
        if d.shape[0] not in (1, n):
            raise ValueError(f"distortion_params has {d.shape[0]} rows for {n} cameras")
        if not bool((d != 0).any()):
            return None
        return d.expand(n, 6).to(dev).contiguous()

    # -- bookkeeping -----------------------------------------------------------------------------------
    @property
    def device(self):
        return self.camera_to_worlds.device

    @property
    def image_height(self) -> torch.Tensor:
        return self.height

    @property
    def image_width(self) -> torch.Tensor:
        return self.width

    @property
    def shape(self):
        return self.camera_to_worlds.shape[:-2]

    @property
    def size(self) -> int:
        return self.camera_to_worlds.shape[0]

    def __len__(self) -> int:
        return self.size

    def to(self, device) -> "Cameras":
        out = Cameras(self.camera_to_worlds.to(device), self.fx.to(device), self.fy.to(device), self.cx.to(device),
                      self.cy.to(device), self.width.to(device), self.height.to(device),
                      distortion_params=self.distortion_params, camera_type=self.camera_type, times=self.times, ids=self.ids)
        return out

    def rescale_output_resolution(self, scaling_factor: Union[float, int, torch.Tensor]) -> None:
        """Scale the output resolution in place (cameras.py ``rescale_output_resolution``, ns-render's
        ``--downscale-factor``): fx, fy, cx, cy times the factor, height / width = (size * factor) cast to int64.
        ``scaling_factor``: a number or a tensor [num_cameras] / [num_cameras, 1]."""
        if isinstance(scaling_factor, (float, int)):
            scaling_factor = torch.tensor([scaling_factor]).to(self.device).broadcast_to(self.cx.shape)
        elif torch.is_tensor(scaling_factor) and tuple(scaling_factor.shape) in ((self.size,), (self.size, 1)):
            scaling_factor = scaling_factor.to(self.device, torch.float32).reshape(self.size, 1)  # fp32 intrinsics
        else:
            raise ValueError(f"scaling_factor must be a number or a tensor of shape [{self.size}] or [{self.size}, 1]")
        self.fx, self.fy = self.fx * scaling_factor, self.fy * scaling_factor
        self.cx, self.cy = self.cx * scaling_factor, self.cy * scaling_factor
        self.height = (self.height * scaling_factor).to(torch.int64)
        self.width = (self.width * scaling_factor).to(torch.int64)
        self._height_host, self._width_host = self.height.view(-1).tolist(), self.width.view(-1).tolist()
        self._intrinsics = None  # packed again from the new fx, fy, cx, cy on the next ray generation

    def get_image_coords(self, pixel_offset: float = 0.5, index=None) -> torch.Tensor:
        """[H,W,2] (y, x) pixel-centre coordinates (cameras.py:299-326)."""
        if index is None:
            h, w = int(self.height.max()), int(self.width.max())
        else:
            h, w = int(self.height[index]), int(self.width[index])
        yy, xx = torch.meshgrid(torch.arange(h), torch.arange(w), indexing="ij")
        return torch.stack([yy, xx], dim=-1) + pixel_offset

    def _lens(self, disable_distortion: bool) -> Optional[torch.Tensor]:
        """cameras.py:636: ``disable_distortion`` skips the undistortion, not the camera-type direction model."""
        return None if disable_distortion else self._distortion

    def _packed_intrinsics(self) -> torch.Tensor:
        if self._intrinsics is None:
            self._intrinsics = torch.cat([self.fx, self.fy, self.cx, self.cy], dim=-1).contiguous()
        return self._intrinsics

    def _bundle(self, out, camera_indices: torch.Tensor, shape, aabb_box: Optional[SceneBox]) -> RayBundle:
        origins, directions, pixel_area, norm, times = out
        rb = RayBundle(origins=origins.view(*shape, 3), directions=directions.view(*shape, 3),
                       pixel_area=pixel_area.view(*shape, 1), camera_indices=camera_indices,
                       times=None if times is None else times.view(*shape, 1),
                       metadata={"directions_norm": norm.view(*shape, 1)})
        if aabb_box is not None:
            # cameras.py:478-497: nears / fars from utils.math.intersect_aabb (a crop-box render, scripts/render.py:101-106);
            # a bundle that carries them passes the model's collider unchanged (scene_colliders.py:41-45)
            t_min, t_max = ops.intersect_aabb(origins, directions, self.box6(aabb_box))
            rb.nears, rb.fars = t_min.view(*shape, 1), t_max.view(*shape, 1)
        return rb

    @staticmethod
    def box6(aabb_box) -> tuple:
        """A SceneBox (or six floats already on the host) -> (x, y, z min, x, y, z max) host floats.  Reading a device
        box synchronises: callers inside a CUDA-graph capture convert once beforehand and pass the tuple."""
        if isinstance(aabb_box, (tuple, list)):
            if len(aabb_box) != 6:
                raise ValueError("aabb_box as a sequence must hold six floats (min then max)")
            return tuple(float(v) for v in aabb_box)
        return tuple(float(v) for v in aabb_box.aabb.detach().flatten().tolist())

    # -- ray generation -------------------------------------------------------------------------------
    def generate_rays(self, camera_indices: Union[torch.Tensor, int], coords: Optional[torch.Tensor] = None,
                      camera_opt_to_camera: Optional[torch.Tensor] = None, distortion_params_delta: Optional[torch.Tensor] = None,
                      keep_shape: Optional[bool] = None, disable_distortion: bool = False,
                      aabb_box: Optional[SceneBox] = None) -> RayBundle:
        if camera_opt_to_camera is not None or distortion_params_delta is not None:
            raise NotImplementedError("camera-optimizer deltas are not built")
        if isinstance(camera_indices, int):
            cam = camera_indices
            if coords is None:  # the whole frame of one camera, [H,W] rays (cameras.py:405-440 case 1)
                h, w = self._height_host[cam], self._width_host[cam]
                rb = self.generate_tile(cam, 0, h * w, aabb_box=aabb_box, disable_distortion=disable_distortion)
                return rb.reshape((h, w)) if keep_shape in (None, True) else rb
            camera_indices = torch.full((*coords.shape[:-1], 1), cam, dtype=torch.int64, device=coords.device)
        if coords is None:
            raise NotImplementedError("tensor camera_indices without coords (stacked full frames) is not built")
        shape = camera_indices.shape[:-1]
        if camera_indices.shape[-1] != 1 or coords.shape[:-1] != shape:
            raise ValueError("camera_indices must be [..., 1] and coords [..., 2] with the same batch shape")
        dev = self.device
        # coords are (y, x) image coordinates = integer index + one sub-pixel offset: 0.5 for pixel centres
        # (image_coords[y, x], what RayGenerator and the eval loaders pass), 0 for integer coordinates (the reference's own
        # tests/cameras/test_cameras.py:119-122).  The kernel adds the offset itself -- (float)index + offset is exactly the
        # coordinate again -- so hand it the integer part.  Coordinates with differing fractional parts are not built.
        flat = coords.to(dev).to(torch.float32).reshape(-1, 2)
        whole = torch.floor(flat)
        frac = flat - whole
        offset = float(frac[0, 0]) if flat.numel() else 0.5
        if not bool((frac == offset).all()):
            raise NotImplementedError("generate_rays: coords must share one sub-pixel offset (pixel centres: integer + 0.5)")
        tri = torch.cat([camera_indices.to(dev).reshape(-1, 1).to(torch.int64), whole.to(torch.int64)], dim=-1).contiguous()
        out = ops.generate_rays(self.camera_to_worlds, self._packed_intrinsics(), self.times, ray_indices=tri,
                                pixel_offset=offset, distortion=self._lens(disable_distortion), cam_types=self._cam_types)
        return self._bundle(out, camera_indices.to(dev), shape, aabb_box)

    def generate_rays_from_indices(self, ray_indices: torch.Tensor, aabb_box=None) -> RayBundle:
        """(camera,row,col) triplets -> rays, what RayGenerator.forward computes, without building coords.
        Indices that arrive on the host (the pixel samplers produce them there) are range-checked like the reference's
        tensor indexing would; device-resident indices are trusted (checking them would cost a synchronisation) and the
        kernel clamps the camera index."""
        if not ray_indices.is_cuda and ray_indices.numel():
            cam, row, col = ray_indices[:, 0], ray_indices[:, 1], ray_indices[:, 2]
            if int(cam.min()) < 0 or int(cam.max()) >= self.size:
                raise IndexError(f"camera index out of range [0, {self.size})")
            h, w = self.height.cpu()[cam.long(), 0], self.width.cpu()[cam.long(), 0]
            if bool((row < 0).any() or (col < 0).any() or (row >= h).any() or (col >= w).any()):
                raise IndexError("pixel index outside its camera's image")
        tri = ray_indices.to(self.device).to(torch.int64).contiguous()
        out = ops.generate_rays(self.camera_to_worlds, self._packed_intrinsics(), self.times, ray_indices=tri,
                                distortion=self._distortion, cam_types=self._cam_types)
        return self._bundle(out, tri[:, 0:1], (tri.shape[0],), aabb_box)

    def generate_tile(self, camera_index: int, start: int, end: int, aabb_box: Optional[SceneBox] = None,
                      disable_distortion: bool = False) -> RayBundle:
        """Rays of the row-major pixels [start, end) of one camera's frame (flat)."""
        w = self._width_host[camera_index]
        out = ops.generate_rays(self.camera_to_worlds, self._packed_intrinsics(), self.times, cam=int(camera_index), width=w,
                                first_pixel=int(start), n=int(end - start), distortion=self._lens(disable_distortion),
                                cam_types=self._cam_types)
        ci = torch.full((end - start, 1), int(camera_index), dtype=torch.int64, device=self.device)
        return self._bundle(out, ci, (end - start,), aabb_box)
