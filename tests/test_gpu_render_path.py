"""Camera-path rendering on the device: kp_compose_frame against the torch restatement of the model's eval images
(utils/colormaps.py + the uint8 quantisation), byte for byte on the same device, and render_camera_path on the tiny model:
the PNG files against direct renders, the frame sharding over ranks, render times, the crop and the rescale."""
import json
import math

import numpy as np
import pytest
import torch

from tests.conftest import load_golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ALL = ["rgb", "depth", "accumulation", "median_rgb", "prop_depth_0", "prop_depth_1"]


def _quantise(img):
    return torch.floor(torch.nan_to_num(img).clamp(0, 1) * 255 + 0.5).to(torch.uint8)


def _cmap_clamped(x, cmap):
    """colormaps.apply_colormap with an out-of-range index clamped to the table (apply_colormap asserts instead)."""
    from soccernerfs_b200.utils import colormaps

    idx = (torch.nan_to_num(x, 0) * 255).long().clamp(0, 255)
    return colormaps._table(cmap).to(x.device)[idx[..., 0]]


def _depth_clamped(depth, acc):
    """colormaps.apply_depth_colormap over _cmap_clamped, same operations in the same order."""
    near, far = float(torch.min(depth)), float(torch.max(depth))
    d = torch.clip((depth - near) / (far - near + 1e-10), 0, 1)
    return _cmap_clamped(d, "turbo") * acc + (1 - acc)


def _restate(frames, names, clamp=False):
    """The torch restatement: the model's eval visualisations (get_image_metrics_and_images) of each output, side by
    side, quantised.  ``clamp``: the clamped colour-map index of the kernel instead of apply_colormap's assertion."""
    from soccernerfs_b200 import ops
    from soccernerfs_b200.utils import colormaps

    acc = frames.get("accumulation")
    panels = []
    for name in names:
        x, kind = frames[name], ops.panel_kind(name)
        if kind == 0:
            panels.append(x)
        elif kind == 1:
            panels.append(_cmap_clamped(x, "viridis") if clamp else colormaps.apply_colormap(x))
        else:
            panels.append(_depth_clamped(x, acc) if clamp else colormaps.apply_depth_colormap(x, accumulation=acc))
    return _quantise(torch.cat(panels, dim=1))


def _check(frames, names, clamp=False):
    from soccernerfs_b200 import ops

    got = ops.compose_frame(frames, names)
    h, w = frames[names[0]].shape[:2]
    assert got.dtype == torch.uint8 and got.shape == (h, w * len(names), 3) and got.is_cuda
    want = _restate(frames, names, clamp)
    if not clamp:  # the clamped restatement is the library's own where no index leaves the table
        assert torch.equal(_restate(frames, names, clamp=True), want)
    assert torch.equal(got, want), (names, int((got.int() - want.int()).abs().max()), int((got != want).sum()))
    return got


def _random_frames(h, w, seed, acc_lo=0.0, acc_hi=1.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    r = lambda c: torch.rand((h, w, c), generator=g, device=DEV)  # noqa: E731
    return {"rgb": r(3) * 1.2 - 0.1, "median_rgb": r(3), "accumulation": acc_lo + (acc_hi - acc_lo) * r(1),
            "depth": 0.5 + 20.0 * r(1) ** 2, "prop_depth_0": 3.0 + r(1), "prop_depth_1": r(1) * 1e-3}


def test_compose_random_frames_every_panel_count_and_order():
    from soccernerfs_b200 import ops

    frames = _random_frames(270, 480, 0)
    for name in ALL:  # P = 1 of every kind
        _check(frames, [name])
    _check(frames, ["depth", "rgb", "accumulation", "prop_depth_1", "median_rgb"])  # P = 5, mixed order
    _check(frames, ALL + ["rgb", "depth"])  # P = 8
    _check(_random_frames(1080, 1920, 1), ["rgb", "depth", "accumulation"])  # the 1080p frame of the benchmark
    _check(_random_frames(5, 7, 2), ["accumulation", "depth", "rgb"])  # fewer pixels than one 4-pixel group per row
    # panels whose storage is not 16-byte aligned (the scalar load path) give the same bytes
    shifted = {}
    for k, v in frames.items():
        buf = torch.empty(v.numel() + 1, device=DEV)
        buf[1:].copy_(v.flatten())
        shifted[k] = buf[1:].view(v.shape)
    names = ["prop_depth_0", "accumulation", "rgb"]
    assert torch.equal(ops.compose_frame(shifted, names), _check(frames, names))
    assert torch.equal(ops.compose_frame(frames, names), ops.compose_frame(frames, names))


def test_compose_constant_depth_and_accumulation_outside_the_table():
    frames = _random_frames(64, 96, 3)
    frames["depth"] = torch.full((64, 96, 1), 2.5, device=DEV)  # far == near: d' = 0 everywhere
    _check(frames, ["depth", "accumulation", "rgb"])
    frames["prop_depth_0"] = torch.zeros((64, 96, 1), device=DEV)
    _check(frames, ["prop_depth_0"])
    # an accumulation just above 1 (index 256, apply_colormap would assert) and slightly below 0: clamped to the table
    acc = frames["accumulation"].clone()
    acc[0, :8, 0] = 1.0 + 2.0 / 255
    acc[1, :8, 0] = 1.0000001
    acc[2, :8, 0] = -0.01
    frames["accumulation"] = acc
    got = _check(frames, ["accumulation", "depth", "prop_depth_1"], clamp=True)
    from soccernerfs_b200.utils import colormaps

    top = _quantise(colormaps._table("viridis")[255].to(DEV))
    assert torch.equal(got[0, :8], top.expand(8, 3)) and torch.equal(got[2, :8], _quantise(colormaps._table("viridis")[0].to(DEV)).expand(8, 3))


def test_compose_rejects_bad_inputs():
    from soccernerfs_b200 import ops

    frames = _random_frames(16, 16, 4)
    with pytest.raises(ValueError, match="not among"):
        ops.compose_frame(frames, ["normals"])
    with pytest.raises(ValueError, match="accumulation"):
        ops.compose_frame({"depth": frames["depth"]}, ["depth"])
    with pytest.raises(ValueError):
        ops.compose_frame(frames, [])
    with pytest.raises(ValueError):
        ops.compose_frame(frames, ["rgb"] * 9)
    with pytest.raises(ValueError):
        ops.compose_frame({"rgb": frames["depth"]}, ["rgb"])  # a colour panel must have 3 channels
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.compose_frame({"rgb": frames["rgb"].cpu()}, ["rgb"])


def _tiny_model():
    from tests.helpers import build_model
    from tests.test_oracle_golden import load_tiny_model

    gm = load_golden("model_tiny")
    model = build_model("tiny", load_tiny_model(gm), gm["aabb"], DEV)
    model.eval()
    model.config.eval_num_rays_per_chunk = 256
    return model


def _c2w(k, n):
    return [1.0, 0.0, 0.0, 0.1 + 0.2 * (k / max(n - 1, 1) - 0.5),
            0.0, 1.0, 0.0, -0.2,
            0.0, 0.0, 1.0, 2.5,
            0.0, 0.0, 0.0, 1.0]


def _camera_path(n=3, h=37, w=53, fov=60.0, times=None, same_pose=False, crop=None):
    times = [0.2 + 0.6 * k / max(n - 1, 1) for k in range(n)] if times is None else times
    cams = [{"camera_to_world": _c2w(0 if same_pose else k, n), "fov": fov, "aspect": w / h, "render_time": t}
            for k, t in zip(range(n), times)]
    out = {"render_height": h, "render_width": w, "camera_path": cams}
    if crop is not None:
        out["crop"] = crop
    return out


def _direct(model, cams, i, names, aabb_box=None):
    """FrameRenderer.render(i, device_frames=True) of the same cameras, composed by the torch restatement."""
    from soccernerfs_b200 import ops
    from soccernerfs_b200.engine.frame_renderer import FrameRenderer

    outputs = list(names) + (["accumulation"] if any(ops.panel_kind(n) == 2 for n in names) and "accumulation" not in names else [])
    frames = FrameRenderer(model, cams.to(DEV), outputs=outputs, aabb_box=aabb_box).render(i, device_frames=True)
    return _restate(frames, names).cpu().numpy()


def _png(path):
    from PIL import Image

    with Image.open(path) as im:
        assert im.mode == "RGB"
        return np.asarray(im).copy()


def test_rendered_frames_compose_like_the_restatement():
    from soccernerfs_b200.engine.frame_renderer import FrameRenderer

    model = _tiny_model()
    from soccernerfs_b200.cameras.camera_paths import get_path_from_json

    cams = get_path_from_json(_camera_path(n=3)).to(DEV)
    frames = FrameRenderer(model, cams, outputs=ALL).render(1, device_frames=True)  # 37 x 53
    _check(frames, ALL)
    _check(frames, ["prop_depth_1", "rgb", "accumulation", "depth", "median_rgb"])
    _check(frames, ["depth"])


def test_render_camera_path_end_to_end_and_over_ranks(tmp_path):
    from soccernerfs_b200.engine.path_renderer import load_camera_path, render_camera_path

    model = _tiny_model()
    path_file = tmp_path / "camera_path.json"
    path_file.write_text(json.dumps(_camera_path(n=3)))
    cams, crop = load_camera_path(path_file)
    assert crop is None and cams.times is not None
    names = ("rgb", "depth", "accumulation")
    one = tmp_path / "world1"
    assert render_camera_path(model, cams, one, rendered_output_names=names) == [0, 1, 2]
    assert sorted(p.name for p in one.iterdir()) == ["00000.png", "00001.png", "00002.png"]
    for i in range(3):
        img = _png(one / f"{i:05d}.png")
        assert img.shape == (37, 53 * 3, 3)
        assert np.array_equal(img, _direct(model, cams, i, names)), i
    # two ranks in one process (there is no collective): rank 0 writes 0 and 2, rank 1 writes 1, the same files
    two = tmp_path / "world2"
    assert render_camera_path(model, cams, two, rendered_output_names=names, rank=0, world=2) == [0, 2]
    assert render_camera_path(model, cams, two, rendered_output_names=names, rank=1, world=2) == [1]
    assert sorted(p.name for p in two.iterdir()) == sorted(p.name for p in one.iterdir())
    for i in range(3):
        assert np.array_equal(_png(two / f"{i:05d}.png"), _png(one / f"{i:05d}.png")), i
    # a default call writes the rgb alone
    rgb_only = tmp_path / "rgb"
    render_camera_path(model, cams, rgb_only)
    assert np.array_equal(_png(rgb_only / "00001.png"), _png(one / "00001.png")[:, :53])


def test_render_time_moves_the_scene(tmp_path):
    from soccernerfs_b200.cameras.cameras import Cameras
    from soccernerfs_b200.engine.path_renderer import load_camera_path, render_camera_path

    model = _tiny_model()
    assert model.field.has_time_planes
    cams, _ = load_camera_path(_camera_path(n=2, times=[0.0, 1.0], same_pose=True))
    render_camera_path(model, cams, tmp_path, rendered_output_names=("rgb", "depth"))
    a, b = _png(tmp_path / "00000.png"), _png(tmp_path / "00001.png")
    assert not np.array_equal(a, b)
    # each frame equals a render of a hand-built camera with that time
    f = 0.5 * 37 / math.tan(0.5 * 60.0 * math.pi / 180.0)  # the three.js focal length of camera_paths.py
    c2w = torch.tensor(_c2w(0, 2)).view(4, 4)[:3]
    for t, got in ((0.0, a), (1.0, b)):
        own = Cameras(c2w[None], float(f), float(f), 53 / 2, 37 / 2, 53, 37, times=torch.tensor([[t]]))
        assert np.array_equal(got, _direct(model, own, 0, ("rgb", "depth"))), t


def test_crop_box_and_background(tmp_path):
    from soccernerfs_b200.engine.frame_renderer import FrameRenderer
    from soccernerfs_b200.engine.path_renderer import load_camera_path, render_camera_path
    from soccernerfs_b200.model_components.renderers import background_color_override_context

    model = _tiny_model()
    crop = {"crop_bg_color": {"r": 255, "g": 51, "b": 0}, "crop_center": [0.0, 0.0, 0.0], "crop_scale": [0.6, 0.6, 0.6]}
    cams, cd = load_camera_path(_camera_path(n=2, crop=crop))
    names = ("rgb", "accumulation")
    render_camera_path(model, cams, tmp_path, rendered_output_names=names, crop=cd)
    for i in range(2):
        with background_color_override_context(cd.background_color.to(DEV)):
            frames = FrameRenderer(model, cams.to(DEV), outputs=list(names), aabb_box=cd.scene_box).render(i, device_frames=True)
        want = _restate(frames, names).cpu().numpy()
        got = _png(tmp_path / f"{i:05d}.png")
        assert np.array_equal(got, want), i
        outside = (got[:, :53] == np.array([255, 51, 0], dtype=np.uint8)).all(-1)
        assert 0 < outside.sum() < 37 * 53, int(outside.sum())  # the background shows where rays miss the box
    uncropped = tmp_path / "full"
    render_camera_path(model, cams, uncropped, rendered_output_names=names)
    assert not np.array_equal(_png(uncropped / "00000.png"), _png(tmp_path / "00000.png"))


def test_rescaled_path(tmp_path):
    from soccernerfs_b200.cameras.cameras import Cameras
    from soccernerfs_b200.engine.path_renderer import load_camera_path, render_camera_path

    model = _tiny_model()
    cams, _ = load_camera_path(_camera_path(n=2, h=48, w=80, fov=50.0))
    fx = float(cams.fx[0])
    cams.rescale_output_resolution(0.5)
    render_camera_path(model, cams, tmp_path, rendered_output_names=("rgb", "depth"))
    times = [0.2, 0.8]
    for i in range(2):
        got = _png(tmp_path / f"{i:05d}.png")
        assert got.shape == (24, 40 * 2, 3)
        c2w = torch.tensor(_c2w(i, 2)).view(4, 4)[:3]
        half = Cameras(c2w[None], fx / 2, fx / 2, 20.0, 12.0, 40, 24, times=torch.tensor([[times[i]]]))
        assert np.array_equal(got, _direct(model, half, 0, ("rgb", "depth"))), i
