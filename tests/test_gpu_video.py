"""The device JPEG encoder (kp_jpeg_encode / ops.encode_jpeg) against the numpy reference (tests/jpeg_reference.py), and
the JPEG frames and Motion-JPEG video of render_camera_path / render_camera_path_video on the tiny model.

For every encoded file: PIL decodes it (up to libjpeg's 65500 columns); its quantised coefficients equal the reference's
fp64 forward transform except where coef / Q lies within 1e-3 of a .5 rounding boundary (the fp32 DCT may round either
way there, and then by one); the reference entropy coder fed those coefficients reproduces the file byte for byte;
nothing is written past the returned length; on smooth content the PSNR is at most 0.1 dB below PIL's own 4:2:0
encoder at the same quality."""
import io
import json
from ctypes import c_void_p

import numpy as np
import pytest
import torch

from tests import jpeg_reference as jr
from tests.test_video_host import _image, _parse_avi

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CANARY = 0xA5
TIE = 1e-3
SMALL = ((1, 1), (7, 9), (16, 16), (17, 33))
KINDS = ("noise", "constant", "gradient", "saturated", "checker")
QUALITIES = (1, 50, 95, 100)
# the large sizes: smooth and flat content at every quality, noise where the reference coder stays quick in Python
LARGE = [((1080, 1920), k, q) for k in ("gradient", "constant") for q in QUALITIES] + \
        [((1080, 5760), "gradient", q) for q in (50, 95)] + [((1080, 5760), "saturated", 1)] + \
        [((8, 65535), k, q) for k, q in (("gradient", 95), ("noise", 1), ("checker", 50))] + [((8, 65500), "gradient", 95)] + \
        [((1080, 1920), "noise", 1)]
TIES = {"coefs": 0, "near_tie": 0, "differ": 0}
PIL_MAX_DIMENSION = 65500  # libjpeg's JPEG_MAX_DIMENSION: PIL decodes nothing wider, the reference decoder does


def _encode_with_canary(img: torch.Tensor, quality: int):
    """kp_jpeg_encode into a buffer 256 bytes longer than the capacity, pre-filled with CANARY: -> (file bytes, the
    untouched tail's check)."""
    from soccernerfs_b200 import _lib, ops

    h, w = img.shape[:2]
    cap = ops.jpeg_capacity(h, w)
    out = torch.full((cap + 256,), CANARY, dtype=torch.uint8, device=DEV)
    length = torch.zeros(1, dtype=torch.int64, device=DEV)
    scratch = torch.empty(int(_lib.load().kp_jpeg_encode_scratch_bytes(h, w)), dtype=torch.uint8, device=DEV)
    _lib.call("kp_jpeg_encode", c_void_p(img.data_ptr()), h, w, c_void_p(ops._jpeg_header(img.device, h, w, quality).data_ptr()),
              c_void_p(scratch.data_ptr()), c_void_p(out.data_ptr()), _lib.ptr(length), _lib.stream_ptr())
    n = int(length)
    assert 0 < n <= cap
    host = out.cpu().numpy()
    assert (host[n:] == CANARY).all(), f"bytes written past the length {n}"
    return host[:n].tobytes()


def _psnr(a: np.ndarray, b: np.ndarray) -> float:
    mse = float(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2))
    return float("inf") if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)


def _check_file(img_np: np.ndarray, data: bytes, quality: int, smooth: bool):
    from PIL import Image

    h, w = img_np.shape[:2]
    if max(h, w) <= PIL_MAX_DIMENSION:
        with Image.open(io.BytesIO(data)) as im:
            im.load()
            assert im.size == (w, h) and im.mode == "RGB"
            decoded = np.asarray(im).copy()
    dec = jr.decode(data)
    want, ratio = jr.forward(img_np, quality)
    got = dec["coefs"]
    diff = got != want
    near = np.abs(np.abs(ratio) - np.floor(np.abs(ratio)) - 0.5) < TIE
    assert not (diff & ~near).any(), f"{int((diff & ~near).sum())} coefficients differ away from a rounding tie"
    assert (np.abs(got - want) <= 1).all()
    TIES["coefs"] += got.size
    TIES["near_tie"] += int(near.sum())
    TIES["differ"] += int(diff.sum())
    assert jr.encode(got, h, w, quality) == data, "the reference coder does not reproduce the file"
    if smooth and min(h, w) >= 16 and max(h, w) <= PIL_MAX_DIMENSION:
        buf = io.BytesIO()
        Image.fromarray(img_np).save(buf, "JPEG", quality=quality, subsampling=2)
        with Image.open(buf) as pil:
            theirs = np.asarray(pil.convert("RGB"))
        ours_db, pil_db = _psnr(decoded, img_np), _psnr(theirs, img_np)
        assert ours_db >= pil_db - 0.1, (h, w, quality, ours_db, pil_db)


def _run(size, kind, quality):
    from soccernerfs_b200 import ops

    h, w = size
    img_np = _image(kind, h, w, seed=h * 7 + w)
    img = torch.from_numpy(img_np).to(DEV)
    data = _encode_with_canary(img, quality)
    out, length = ops.encode_jpeg(img, quality)
    assert out.dtype == torch.uint8 and length.dtype == torch.int64 and out.numel() == ops.jpeg_capacity(h, w)
    assert out[:int(length)].cpu().numpy().tobytes() == data
    _check_file(img_np, data, quality, smooth=kind in ("gradient", "constant"))


@pytest.mark.parametrize("kind", KINDS)
def test_encoder_small_sizes(kind):
    for size in SMALL:
        for q in QUALITIES:
            _run(size, kind, q)


@pytest.mark.parametrize("size,kind,quality", LARGE)
def test_encoder_large_sizes(size, kind, quality):
    _run(size, kind, quality)


def test_encoder_tie_share():
    """Runs after the encoder tests: the share of coefficients near a .5 boundary, and of those that differ."""
    if TIES["coefs"] == 0:  # run on its own
        _run((1080, 1920), "noise", 1)
    near, differ = TIES["near_tie"] / TIES["coefs"], TIES["differ"] / TIES["coefs"]
    print(f"jpeg: {TIES['coefs']} coefficients, {near:.2e} within {TIE} of a .5 boundary, {differ:.2e} differ by one")
    assert near < 5e-3 and differ <= near


def test_encoder_in_a_cuda_graph():
    from soccernerfs_b200 import ops

    img = torch.from_numpy(_image("noise", 96, 200, seed=3)).to(DEV)
    want, n = ops.encode_jpeg(img, 90)  # builds the header (a host copy) before the capture
    want = want[:int(n)].clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.encode_jpeg(img, 90)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out, length = ops.encode_jpeg(img, 90)
    for _ in range(3):
        out.fill_(0)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out[:int(length)], want)
    img.copy_(torch.from_numpy(_image("gradient", 96, 200)).to(DEV))  # new pixels, same graph
    graph.replay()
    _check_file(_image("gradient", 96, 200), out[:int(length)].cpu().numpy().tobytes(), 90, smooth=True)


# ---- the render path ----
def _tiny_model():
    from tests.test_gpu_render_path import _tiny_model as tiny

    return tiny()


def _composed(model, cams, i, names, crop=None):
    """compose_frame of a direct FrameRenderer render of camera i (the crop's box and background as the path uses)."""
    import contextlib

    from soccernerfs_b200 import ops
    from soccernerfs_b200.engine.frame_renderer import FrameRenderer
    from soccernerfs_b200.model_components.renderers import background_color_override_context

    outputs = list(names) + (["accumulation"] if any(ops.panel_kind(n) == 2 for n in names) and "accumulation" not in names else [])
    ctx = background_color_override_context(crop.background_color.to(DEV)) if crop is not None else contextlib.nullcontext()
    with ctx:
        frames = FrameRenderer(model, cams.to(DEV), outputs=outputs,
                               aabb_box=crop.scene_box if crop is not None else None).render(i, device_frames=True)
    return ops.compose_frame(frames, list(names))


def _jpeg_of(image, quality):
    from soccernerfs_b200 import ops

    out, n = ops.encode_jpeg(image, quality)
    return out[:int(n)].cpu().numpy().tobytes()


def test_render_camera_path_jpeg_frames(tmp_path):
    from soccernerfs_b200.engine.path_renderer import load_camera_path, render_camera_path
    from tests.test_gpu_render_path import _camera_path

    model = _tiny_model()
    cams, _ = load_camera_path(_camera_path(n=3))
    names = ("rgb", "depth", "accumulation")
    assert render_camera_path(model, cams, tmp_path, rendered_output_names=names, image_format="jpeg", jpeg_quality=90) == [0, 1, 2]
    assert sorted(p.name for p in tmp_path.iterdir()) == ["00000.jpg", "00001.jpg", "00002.jpg"]
    for i in range(3):
        image = _composed(model, cams, i, names)
        data = (tmp_path / f"{i:05d}.jpg").read_bytes()
        assert data == _jpeg_of(image, 90), i
        _check_file(image.cpu().numpy(), data, 90, smooth=False)


def test_render_camera_path_video(tmp_path):
    from soccernerfs_b200.cameras.camera_paths import get_seconds_from_json
    from soccernerfs_b200.engine.path_renderer import assemble_video, load_camera_path, render_camera_path_video
    from tests.test_gpu_render_path import _camera_path

    model = _tiny_model()
    path = dict(_camera_path(n=5), seconds=2.0)  # 2.5 fps, render times 0.2 .. 0.8
    path_file = tmp_path / "camera_path.json"
    path_file.write_text(json.dumps(path))
    cams, _ = load_camera_path(path_file)
    seconds = get_seconds_from_json(json.loads(path_file.read_text()))
    names = ("rgb", "depth")
    one = tmp_path / "one.avi"
    assert render_camera_path_video(model, cams, one, seconds, rendered_output_names=names, jpeg_quality=85) == list(range(5))
    avi = _parse_avi(one)
    assert avi["fps"] == pytest.approx(2.5) and (avi["width"], avi["height"]) == (53 * 2, 37)
    assert len(avi["frames"]) == 5
    for i, data in enumerate(avi["frames"]):
        assert data == _jpeg_of(_composed(model, cams, i, names), 85), i
    # two ranks in one process (no process group): each writes its part, the caller assembles
    two = tmp_path / "two.avi"
    assert render_camera_path_video(model, cams, two, seconds, rendered_output_names=names, rank=0, world=2, jpeg_quality=85) == [0, 2, 4]
    assert render_camera_path_video(model, cams, two, seconds, rendered_output_names=names, rank=1, world=2, jpeg_quality=85) == [1, 3]
    assert not two.exists()
    assemble_video(two, 2, len(cams) / seconds)
    assert two.read_bytes() == one.read_bytes()
    assert sorted(p.name for p in tmp_path.iterdir()) == ["camera_path.json", "one.avi", "two.avi"]


def test_crop_path_video_and_jpeg(tmp_path):
    from soccernerfs_b200.engine.path_renderer import load_camera_path, render_camera_path, render_camera_path_video
    from tests.test_gpu_render_path import _camera_path

    model = _tiny_model()
    crop = {"crop_bg_color": {"r": 255, "g": 51, "b": 0}, "crop_center": [0.0, 0.0, 0.0], "crop_scale": [0.6, 0.6, 0.6]}
    cams, cd = load_camera_path(_camera_path(n=2, crop=crop))
    names = ("rgb", "accumulation")
    render_camera_path_video(model, cams, tmp_path / "crop.avi", 1.0, rendered_output_names=names, crop=cd)
    render_camera_path(model, cams, tmp_path / "jpg", rendered_output_names=names, crop=cd, image_format="jpeg")
    frames = _parse_avi(tmp_path / "crop.avi")["frames"]
    for i in range(2):
        want = _jpeg_of(_composed(model, cams, i, names, crop=cd), 95)
        assert frames[i] == want == (tmp_path / "jpg" / f"{i:05d}.jpg").read_bytes(), i
