"""Rendering a camera path to image files: what ``ns-render --camera-path-filename`` does for a trained model
(REF/nerfstudio/scripts/render.py ``_render_trajectory_video``), writing PNG or JPEG frames, or a Motion-JPEG video.

Per frame: ``FrameRenderer.render(i, device_frames=True)`` renders the requested outputs into device tensors (one
CUDA-graph replay per tile), ``ops.compose_frame`` colour-maps them and lays them side by side as one uint8 image on the
same stream, a copy stream moves the image into one of a small ring of pinned host buffers, and a thread pool encodes
the PNG ``output_dir/{i:05d}.png`` with PIL.  For JPEG frames and video, ``ops.encode_jpeg`` encodes the image on the
same stream and only the file's bytes are copied.  The GPU renders frame k+1 while frame k is written; the render loop
waits only when the ring is full.

With ``world > 1`` rank r renders the whole frames ``i % world == r``.  A file's name depends only on its frame index,
so the ranks write disjoint files, need no collective, and together write the same set of files as one rank does.  A
video is written per rank as a part file and interleaved into the AVI afterwards (``assemble_video``).
For a dynamic model the path must carry a render time per camera: that is what makes the players move.
"""
from __future__ import annotations

import contextlib
import json
import math
import os
import struct
from concurrent.futures import Future, ThreadPoolExecutor
from fractions import Fraction
from typing import Callable, Dict, List, Optional, Sequence, Tuple, Union

import torch

from .. import ops
from ..cameras.camera_paths import CropData, get_crop_from_json, get_path_from_json
from ..cameras.cameras import Cameras
from ..model_components.renderers import background_color_override_context
from .evaluator import images_of_rank
from .frame_renderer import STATIC_OUTPUTS, FrameRenderer

RING_SLOTS = 3  # pinned host images in flight: one being filled by the copy, the others being encoded
IMAGE_FORMATS = ("png", "jpeg")


def load_camera_path(path_or_dict: Union[str, os.PathLike, Dict]) -> Tuple[Cameras, Optional[CropData]]:
    """A camera-path JSON file (or its already-parsed dict) -> (cameras on the host, crop or None)."""
    if isinstance(path_or_dict, dict):
        camera_path = path_or_dict
    else:
        with open(path_or_dict, "r", encoding="utf-8") as f:
            camera_path = json.load(f)
    return get_path_from_json(camera_path), get_crop_from_json(camera_path)


def available_outputs(model) -> List[str]:
    """The per-pixel outputs of the model that can be written as images.  A dynamic model (its field has time planes) also
    has its space-time decomposition: the static scene (``rgb_static``, ``depth_static``, ``accumulation_static``: the
    render with the time planes left out, models.base_model.static_scene) and ``dynamic``, how far the time planes move
    the scene from it (models.base_model.dynamics_output)."""
    names = ["rgb", "depth", "accumulation", "median_rgb"]
    names += [f"prop_depth_{i}" for i in range(getattr(model.config, "num_proposal_iterations", 0))]
    if getattr(model.field, "has_time_planes", False):
        names += list(STATIC_OUTPUTS) + ["dynamic"]
    return names


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
    timed = [n for n in names if n not in STATIC_OUTPUTS]  # the static render reads no time
    if getattr(model.field, "has_time_planes", False) and cameras.times is None and timed:
        raise ValueError(f"the model is dynamic (its field has time planes) but the cameras have no times: every camera of "
                         f"the path needs a render_time for the outputs {timed}")
    sizes = sorted(set(zip(cameras._height_host, cameras._width_host)))
    if len(sizes) > 1:
        raise ValueError(f"the cameras' frames differ in size (H, W): {sizes}; one image size per path")


def check_jpeg_quality(jpeg_quality) -> None:
    if isinstance(jpeg_quality, bool) or not isinstance(jpeg_quality, int) or not 1 <= jpeg_quality <= 100:
        raise ValueError(f"jpeg_quality {jpeg_quality!r} is not an integer in 1..100")


def _land_image(done: torch.cuda.Event, image: torch.Tensor, i: int, write: Callable):
    done.synchronize()  # the copy into this pinned buffer has landed
    return write(i, image)


def _land_jpeg(done: torch.cuda.Event, data: torch.Tensor, ring: List[torch.Tensor], lengths: torch.Tensor, slot: int,
               stream: torch.cuda.Stream, i: int, write: Callable):
    done.synchronize()  # the encoded length has landed (so the encoding is finished)
    n = int(lengths[slot])
    if ring[slot].numel() < n:
        ring[slot] = torch.empty(n, dtype=torch.uint8).pin_memory()
    host = ring[slot][:n]
    with torch.cuda.stream(stream):
        host.copy_(data[:n], non_blocking=True)
        landed = torch.cuda.Event()
        landed.record(stream)
    landed.synchronize()  # ``data`` stays referenced until here, so its device memory is not reused under the copy
    return write(i, host)


def _path_frames(model, cameras: Cameras, names: List[str], crop: Optional[CropData]):
    """-> (produce, context, (H, W*P)): ``produce(i)`` renders frame i of the path and composes ``names`` on the device
    (uint8 [H, W*P, 3]); it runs inside ``context`` (the crop's background colour)."""
    dev = model.device
    if cameras.device != dev:
        cameras = cameras.to(dev)
    outputs = list(names)
    for n in names:  # each depth panel is blended with its own accumulation
        if ops.panel_kind(n) == 2 and ops.accumulation_of(n) not in outputs:
            outputs.append(ops.accumulation_of(n))
    aabb_box = None
    bg = None
    if crop is not None:
        aabb_box = crop.scene_box
        bg = crop.background_color.to(dev, torch.float32)  # on the device: the tile graphs read it, no copy in the capture
    renderer = FrameRenderer(model, cameras, outputs=outputs, aabb_box=aabb_box)  # whole frames per rank
    context = background_color_override_context(bg) if bg is not None else contextlib.nullcontext()
    return (lambda i: ops.compose_frame(renderer.render(i, device_frames=True), names)), context, \
        (cameras._height_host[0], cameras._width_host[0] * len(names))


def _frame_loop(produce: Callable[[int], torch.Tensor], mine: Sequence[int], size: Tuple[int, int], dev,
                jpeg_quality: Optional[int], write: Callable, collect: Optional[Callable] = None) -> List[int]:
    """The write loop of every output format.  For each frame i of ``mine`` in order, ``produce(i)`` gives the composed
    uint8 image [H, W', 3] (``size`` = (H, W')) on the current stream, which is encoded on the device with a
    ``jpeg_quality``; a copy stream moves it into a ring of pinned host buffers and ``write(i, data)`` runs on a pool
    thread once it has landed: ``data`` is the composed image, or the JPEG file's bytes (uint8 [n]; the length is copied
    first, then exactly n bytes).  ``collect(i, result)`` gets the results of ``write`` on this thread in frame order.
    The loop itself never synchronises with the device; it waits only for the pool when every ring buffer is still in
    use, so the device produces frame k+1 while frame k is written.  Returns ``mine``."""
    mine = list(mine)
    h, w = size
    slots = min(RING_SLOTS, len(mine))
    # JPEG: sized like the raw image, grown by the pool thread in the rare case a file is larger
    shape = (h, w, 3) if jpeg_quality is None else (h * w * 3,)
    ring = [torch.empty(shape, dtype=torch.uint8).pin_memory() for _ in range(slots)]
    lengths = torch.empty(max(slots, 1), dtype=torch.int64).pin_memory() if jpeg_quality is not None else None
    pending: List[Optional[Future]] = [None] * slots
    copy_stream = torch.cuda.Stream(device=dev)
    bytes_stream = torch.cuda.Stream(device=dev)  # the pool's byte copies: never queued behind the next frame's wait
    main = torch.cuda.current_stream(dev)

    def finish(k: int) -> None:
        result = pending[k % slots].result()
        if collect is not None:
            collect(mine[k], result)

    with ThreadPoolExecutor(max_workers=max(1, slots)) as pool:
        for k, i in enumerate(mine):
            slot = k % slots
            if k >= slots:
                finish(k - slots)  # ring full: this buffer's frame is still being written
            image = produce(i)
            if jpeg_quality is None:
                copy_stream.wait_stream(main)
                with torch.cuda.stream(copy_stream):
                    ring[slot].copy_(image, non_blocking=True)
                    image.record_stream(copy_stream)
                    done = torch.cuda.Event()
                    done.record(copy_stream)
                pending[slot] = pool.submit(_land_image, done, ring[slot], i, write)
            else:
                data, length = ops.encode_jpeg(image, jpeg_quality)
                copy_stream.wait_stream(main)
                with torch.cuda.stream(copy_stream):
                    lengths[slot:slot + 1].copy_(length, non_blocking=True)
                    length.record_stream(copy_stream)
                    done = torch.cuda.Event()
                    done.record(copy_stream)
                pending[slot] = pool.submit(_land_jpeg, done, data, ring, lengths, slot, bytes_stream, i, write)
        for k in range(max(0, len(mine) - slots), len(mine)):
            finish(k)
    return mine


def render_camera_path(model, cameras: Cameras, output_dir: Union[str, os.PathLike],
                       rendered_output_names: Sequence[str] = ("rgb",), rank: int = 0, world: int = 1,
                       crop: Optional[CropData] = None, image_format: str = "png", jpeg_quality: int = 95) -> List[int]:
    """Render this rank's frames of ``cameras`` (``i % world == rank``) and write each as ``output_dir/{i:05d}.png``
    (``image_format="png"``, encoded by PIL on the host) or ``{i:05d}.jpg`` (``"jpeg"``, baseline 4:2:0 at
    ``jpeg_quality``, encoded on the device by ``ops.encode_jpeg``): the ``rendered_output_names`` side by side,
    colour-mapped like the model's eval images.  ``crop``: rays start and end at the crop box and the crop's background
    colour shows outside it (ns-render's crop).  Returns the frame indices this rank wrote."""
    check_render_inputs(model, cameras, rendered_output_names)
    if image_format not in IMAGE_FORMATS:
        raise ValueError(f"image_format {image_format!r} is not one of {IMAGE_FORMATS}")
    check_jpeg_quality(jpeg_quality)
    out = os.fspath(output_dir)
    os.makedirs(out, exist_ok=True)
    produce, context, size = _path_frames(model, cameras, list(rendered_output_names), crop)
    with context:
        return _frame_loop(produce, images_of_rank(len(cameras), rank, world), size, model.device,
                           None if image_format == "png" else jpeg_quality, file_writer(out, image_format))


def file_writer(out: str, image_format: str) -> Callable:
    """The ``write`` of ``_frame_loop`` for image files: a composed image to ``out/{i:05d}.png`` through PIL, or the JPEG
    bytes to ``out/{i:05d}.jpg``."""
    def write_png(i: int, image: torch.Tensor) -> None:
        from PIL import Image

        Image.fromarray(image.numpy()).save(os.path.join(out, f"{i:05d}.png"))

    def write_jpeg(i: int, data: torch.Tensor) -> None:
        with open(os.path.join(out, f"{i:05d}.jpg"), "wb") as f:
            f.write(data.numpy().tobytes())

    return write_png if image_format == "png" else write_jpeg


# ---- Motion-JPEG AVI (RIFF AVI 1.0): every frame a baseline JPEG in a '00dc' chunk of 'movi', all keyframes ----
AVI_MAX_MOVI_BYTES = 1 << 30  # AVI 1.0 addresses 1 GiB of 'movi' data (OpenDML, which goes past it, is not written)
_AVIF_HASINDEX = 0x10
_AVIIF_KEYFRAME = 0x10


def part_path(output_path: Union[str, os.PathLike], rank: int) -> str:
    """The file rank ``rank`` writes its encoded frames to before ``assemble_video`` interleaves them."""
    return f"{os.fspath(output_path)}.part{rank}"


def write_part(output_path: Union[str, os.PathLike], rank: int, produce: Callable[[int], torch.Tensor], frames: Sequence[int],
               size: Tuple[int, int], dev, jpeg_quality: int) -> List[int]:
    """Encode ``produce(i)`` of each of ``frames`` in order on the device and append the JPEGs to rank ``rank``'s part file
    of ``output_path`` (records of uint32 little-endian n, n bytes).  Returns ``frames``."""
    with open(part_path(output_path, rank), "wb") as part:

        def append(i: int, data: bytes) -> None:
            part.write(struct.pack("<I", len(data)) + data)

        return _frame_loop(produce, frames, size, dev, jpeg_quality, lambda i, data: data.numpy().tobytes(), append)


def _read_part(path: str) -> List[Tuple[int, int]]:
    """A part file is a sequence of records (uint32 little-endian n, n JPEG bytes): -> [(offset of the bytes, n)]."""
    records, size = [], os.path.getsize(path)
    with open(path, "rb") as f:
        pos = 0
        while pos < size:
            (n,) = struct.unpack("<I", f.read(4))
            records.append((pos + 4, n))
            pos += 4 + n
            f.seek(pos)
    return records


def _jpeg_size(data: bytes) -> Tuple[int, int]:
    """(width, height) from a JPEG's SOF0."""
    sof = data.index(b"\xff\xc0")
    h, w = struct.unpack(">HH", data[sof + 5:sof + 9])
    return w, h


def assemble_video(output_path: Union[str, os.PathLike], world: int, fps: float) -> None:
    """Interleave the part files of ranks 0..world-1 (frame i is record i // world of part i % world) into the
    Motion-JPEG AVI ``output_path`` at ``fps`` frames per second (stored as dwRate / dwScale), then delete the parts.
    Raises ValueError when the frames would pass AVI 1.0's 1 GiB of 'movi' data, saying how many frames fit."""
    if not fps > 0 or not math.isfinite(fps):
        raise ValueError(f"fps must be positive and finite (got {fps})")
    parts = [part_path(output_path, r) for r in range(world)]
    records = [_read_part(p) for p in parts]
    n = sum(len(r) for r in records)
    if n == 0:
        raise ValueError("the part files hold no frames")
    if [len(r) for r in records] != [len(range(r, n, world)) for r in range(world)]:
        raise ValueError(f"part files of {[len(r) for r in records]} frames do not interleave into {n} frames")
    order = [(i % world, records[i % world][i // world]) for i in range(n)]
    movi = 4
    for k, (_, (_, size)) in enumerate(order):
        step = 8 + size + (size & 1)
        if movi + step > AVI_MAX_MOVI_BYTES:
            raise ValueError(f"{n} frames need more than the 1 GiB of 'movi' data an AVI 1.0 file holds: {k} frames fit "
                             f"at this size and quality")
        movi += step
    files = [open(p, "rb") for p in parts]
    try:
        r0, (off0, n0) = order[0]
        files[r0].seek(off0)
        width, height = _jpeg_size(files[r0].read(n0))
        rate = Fraction(fps).limit_denominator(1 << 16)
        biggest = max(size for _, (_, size) in order)
        chunk = lambda fourcc, body: fourcc + struct.pack("<I", len(body)) + body  # noqa: E731
        u32 = lambda v: min(int(v), 0xFFFFFFFF)  # noqa: E731
        avih = struct.pack("<14I", u32(round(1e6 / fps)), u32(biggest * fps + 1), 0, _AVIF_HASINDEX, n, 0, 1, biggest + 8,
                           width, height, 0, 0, 0, 0)
        strh = b"vidsMJPG" + struct.pack("<IHHIIIIIIiI4H", 0, 0, 0, 0, u32(rate.denominator), u32(rate.numerator), 0,
                                          n, biggest + 8, -1, 0, 0, 0, width, height)
        strf = struct.pack("<IiiHH4sIiiII", 40, width, height, 1, 24, b"MJPG", u32(width * height * 3), 0, 0, 0, 0)
        hdrl = b"hdrl" + chunk(b"avih", avih) + chunk(b"LIST", b"strl" + chunk(b"strh", strh) + chunk(b"strf", strf))
        idx1_size = 16 * n
        riff_size = 4 + (8 + len(hdrl)) + (8 + movi) + (8 + idx1_size)
        index = bytearray()
        with open(output_path, "wb") as out:
            out.write(b"RIFF" + struct.pack("<I", riff_size) + b"AVI " + chunk(b"LIST", hdrl))
            out.write(b"LIST" + struct.pack("<I", movi) + b"movi")
            pos = 4  # idx1 offsets count from the 'movi' fourcc
            for r, (off, size) in order:
                files[r].seek(off)
                out.write(b"00dc" + struct.pack("<I", size) + files[r].read(size) + b"\x00" * (size & 1))
                index += b"00dc" + struct.pack("<III", _AVIIF_KEYFRAME, pos, size)
                pos += 8 + size + (size & 1)
            out.write(b"idx1" + struct.pack("<I", idx1_size) + bytes(index))
    finally:
        for f in files:
            f.close()
    for p in parts:
        os.remove(p)


def render_camera_path_video(model, cameras: Cameras, output_path: Union[str, os.PathLike], seconds: float,
                             rendered_output_names: Sequence[str] = ("rgb",), rank: int = 0, world: int = 1,
                             crop: Optional[CropData] = None, jpeg_quality: int = 95) -> List[int]:
    """Render the path as a Motion-JPEG AVI ``output_path`` at ``len(cameras) / seconds`` frames per second (what
    ns-render's default video output plays at), the frames encoded on the device as ``render_camera_path(...,
    image_format="jpeg")`` encodes them.  Rank r encodes the frames ``i % world == r`` into its part file.  With one
    rank the video is written at once; with a ``torch.distributed`` group the ranks meet at a barrier and rank 0
    assembles the parts; without one the caller runs ``assemble_video(output_path, world, fps)`` once every rank is
    done.  Returns the frame indices this rank rendered."""
    check_render_inputs(model, cameras, rendered_output_names)
    check_jpeg_quality(jpeg_quality)
    if not seconds > 0 or not math.isfinite(seconds):
        raise ValueError(f"seconds must be positive and finite (got {seconds})")
    fps = len(cameras) / seconds
    out_dir = os.path.dirname(os.path.abspath(output_path))
    os.makedirs(out_dir, exist_ok=True)
    produce, context, size = _path_frames(model, cameras, list(rendered_output_names), crop)
    with context:
        mine = write_part(output_path, rank, produce, images_of_rank(len(cameras), rank, world), size, model.device, jpeg_quality)
    if world == 1:
        assemble_video(output_path, 1, fps)
    elif torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.barrier()
        if rank == 0:
            assemble_video(output_path, world, fps)
    return mine


