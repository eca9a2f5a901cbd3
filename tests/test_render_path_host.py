"""Host side of camera-path rendering without a GPU: the camera-path JSON (cameras/camera_paths.py), the in-place
resolution rescale of Cameras, which frames a rank renders, and the input checks of render_camera_path."""
import json
import math
import types

import pytest
import torch

from soccernerfs_b200.cameras.camera_paths import get_crop_from_json, get_path_from_json
from soccernerfs_b200.cameras.cameras import Cameras, CameraType
from soccernerfs_b200.engine import path_renderer as pr
from soccernerfs_b200.engine.evaluator import images_of_rank

POSE = [1.0, 0.0, 0.0, 0.5,
        0.0, 0.0, -1.0, -2.0,
        0.0, 1.0, 0.0, 3.0,
        0.0, 0.0, 0.0, 1.0]


def _path(n=3, h=1080, w=1920, fov=90.0, times=True, **extra):
    cams = []
    for k in range(n):
        c = {"camera_to_world": list(POSE), "fov": fov, "aspect": 1.0}
        if times is True or (times == "some" and k != 1):
            c["render_time"] = k / max(n - 1, 1)
        cams.append(c)
    return {"render_height": h, "render_width": w, "seconds": 1.0, "camera_path": cams, **extra}


def test_perspective_intrinsics_and_row_major_pose():
    cams = get_path_from_json(_path(fov=90.0))
    assert len(cams) == 3
    assert cams._height_host == [1080] * 3 and cams._width_host == [1920] * 3
    assert torch.equal(cams.height, torch.full((3, 1), 1080)) and torch.equal(cams.width, torch.full((3, 1), 1920))
    assert torch.allclose(cams.fx, torch.full((3, 1), 540.0)) and torch.allclose(cams.fy, torch.full((3, 1), 540.0))
    assert float(cams.fx[0]) == pytest.approx(540.0, abs=1e-4)
    assert torch.equal(cams.cx, torch.full((3, 1), 960.0)) and torch.equal(cams.cy, torch.full((3, 1), 540.0))
    want = torch.tensor([[1.0, 0.0, 0.0, 0.5], [0.0, 0.0, -1.0, -2.0], [0.0, 1.0, 0.0, 3.0]])
    assert torch.equal(cams.camera_to_worlds[1], want)  # row-major: the translation is the last column
    assert bool((cams.camera_type == CameraType.PERSPECTIVE.value).all())
    # fov 60 at H 37 (odd): 18.5 / tan(30 deg)
    odd = get_path_from_json(_path(h=37, w=53, fov=60.0))
    assert float(odd.fx[0]) == pytest.approx(18.5 / math.tan(math.pi / 6), rel=1e-6)
    assert float(odd.cx[0]) == 26.5 and float(odd.cy[0]) == 18.5 and odd._height_host[0] == 37 and odd._width_host[0] == 53


def test_camera_types_and_equirectangular_intrinsics():
    eq = get_path_from_json(_path(h=512, w=1024, camera_type="equirectangular"))
    assert torch.equal(eq.fx, torch.full((3, 1), 512.0)) and torch.equal(eq.fy, torch.full((3, 1), 512.0))
    assert bool((eq.camera_type == CameraType.EQUIRECTANGULAR.value).all())
    eq2 = get_path_from_json(_path(h=300, w=1000, camera_type="equirectangular"))
    assert float(eq2.fx[0]) == 500.0 and float(eq2.fy[0]) == 300.0
    fish = get_path_from_json(_path(camera_type="fisheye"))
    assert bool((fish.camera_type == CameraType.FISHEYE.value).all()) and float(fish.fx[0]) == pytest.approx(540.0, abs=1e-4)
    persp = get_path_from_json(_path(camera_type="perspective"))
    assert bool((persp.camera_type == CameraType.PERSPECTIVE.value).all())
    with pytest.raises(ValueError, match="orthographic"):
        get_path_from_json(_path(camera_type="orthographic"))


def test_render_times_on_all_some_and_no_cameras():
    cams = get_path_from_json(_path(n=3, times=True))
    assert cams.times is not None and torch.equal(cams.times, torch.tensor([[0.0], [0.5], [1.0]]))
    assert get_path_from_json(_path(n=3, times="some")).times is None
    assert get_path_from_json(_path(n=3, times=False)).times is None


def test_crop_box_and_background():
    assert get_crop_from_json(_path()) is None
    assert get_crop_from_json(_path(crop=None)) is None
    crop = get_crop_from_json(_path(crop={"crop_bg_color": {"r": 255, "g": 51, "b": 0},
                                          "crop_center": [0.5, -1.0, 2.0], "crop_scale": [1.0, 4.0, 0.5]}))
    assert torch.equal(crop.background_color, torch.tensor([1.0, 0.2, 0.0]))
    assert torch.equal(crop.scene_box.aabb, torch.tensor([[0.0, -3.0, 1.75], [1.0, 1.0, 2.25]]))


def test_load_camera_path_from_a_file_or_a_dict(tmp_path):
    d = _path(n=2, h=40, w=60, crop={"crop_bg_color": {"r": 0, "g": 0, "b": 255}, "crop_center": [0, 0, 0],
                                      "crop_scale": [2, 2, 2]})
    f = tmp_path / "path.json"
    f.write_text(json.dumps(d))
    for src in (d, f, str(f)):
        cams, crop = pr.load_camera_path(src)
        assert len(cams) == 2 and cams._height_host == [40, 40] and torch.equal(crop.background_color, torch.tensor([0.0, 0.0, 1.0]))


def test_rescale_output_resolution_in_place():
    cams = get_path_from_json(_path(n=2, h=1080, w=1920, fov=90.0))
    packed = cams._packed_intrinsics()
    assert torch.equal(packed[0], torch.tensor([540.0, 540.0, 960.0, 540.0]))
    cams.rescale_output_resolution(0.5)
    assert torch.allclose(cams.fx, torch.full((2, 1), 270.0)) and torch.allclose(cams.fy, torch.full((2, 1), 270.0))
    assert torch.equal(cams.cx, torch.full((2, 1), 480.0)) and torch.equal(cams.cy, torch.full((2, 1), 270.0))
    assert cams.height.dtype == torch.int64 and torch.equal(cams.height, torch.full((2, 1), 540))
    assert torch.equal(cams.width, torch.full((2, 1), 960))
    assert cams._height_host == [540, 540] and cams._width_host == [960, 960]
    assert torch.allclose(cams._packed_intrinsics()[1], torch.tensor([270.0, 270.0, 480.0, 270.0]))
    assert cams.fx.dtype == torch.float32 and cams.fx.shape == (2, 1)
    # an odd size truncates, like the cast to int64: 37 * 0.5 = 18.5 -> 18
    odd = get_path_from_json(_path(n=1, h=37, w=53))
    odd.rescale_output_resolution(0.5)
    assert odd._height_host == [18] and odd._width_host == [26] and float(odd.cy[0]) == 9.25
    per_camera = get_path_from_json(_path(n=2, h=100, w=200))
    per_camera.rescale_output_resolution(torch.tensor([0.5, 2.0], dtype=torch.float64))
    assert per_camera._height_host == [50, 200] and per_camera._width_host == [100, 400]
    assert per_camera.fx.dtype == torch.float32
    with pytest.raises(ValueError):
        per_camera.rescale_output_resolution(torch.tensor([0.5, 2.0, 1.0]))


def test_frame_assignment_per_rank():
    for n in (0, 1, 3, 7, 16):
        for world in (1, 2, 3, 4, 8):
            parts = [images_of_rank(n, r, world) for r in range(world)]
            assert sorted(i for p in parts for i in p) == list(range(n)), (n, world)
            assert all(i % world == r for r, p in enumerate(parts) for i in p)
            names = sorted(f"{i:05d}.png" for p in parts for i in p)
            assert names == [f"{i:05d}.png" for i in range(n)]  # the same files for every world size
    assert images_of_rank(7, 1, 3) == [1, 4]


def _stub_model(dynamic=True, proposals=2):
    return types.SimpleNamespace(config=types.SimpleNamespace(num_proposal_iterations=proposals),
                                 field=types.SimpleNamespace(has_time_planes=dynamic))


def test_render_camera_path_input_errors(tmp_path):
    cams = get_path_from_json(_path(n=2, h=24, w=40))
    with pytest.raises(ValueError, match="available outputs.*prop_depth_1"):
        pr.render_camera_path(_stub_model(), cams, tmp_path, rendered_output_names=("rgb", "normals"))
    with pytest.raises(ValueError, match="available"):
        pr.render_camera_path(_stub_model(), cams, tmp_path, rendered_output_names=())
    no_times = get_path_from_json(_path(n=2, h=24, w=40, times="some"))
    with pytest.raises(ValueError, match="render_time"):
        pr.render_camera_path(_stub_model(dynamic=True), no_times, tmp_path)
    mixed = Cameras(torch.eye(4)[:3].repeat(2, 1, 1), 30.0, 30.0, torch.tensor([20.0, 30.0]), 12.0,
                    width=torch.tensor([40, 60]), height=24, times=torch.tensor([0.0, 1.0]))
    with pytest.raises(ValueError, match="size"):
        pr.render_camera_path(_stub_model(), mixed, tmp_path)
    with pytest.raises(ValueError, match="at most 8"):
        pr.render_camera_path(_stub_model(), cams, tmp_path, rendered_output_names=["rgb"] * 9)
    assert list(tmp_path.iterdir()) == []  # nothing was written
    # a static model renders a path without times; the names the model can render pass the checks
    pr.check_render_inputs(_stub_model(dynamic=False), no_times, ["rgb", "depth", "accumulation", "median_rgb", "prop_depth_0"])


def test_panel_kinds():
    from soccernerfs_b200 import ops

    assert [ops.panel_kind(n) for n in ("rgb", "median_rgb", "accumulation", "depth", "prop_depth_0", "prop_depth_1")] == \
        [0, 0, 1, 2, 2, 2]
