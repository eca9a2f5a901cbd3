"""Eval images on the device: kp_eval_maps (ops.eval_maps) against a float64 restatement, the eval panels against the
torch restatement of their colour maps and quantisation, and Evaluator.write_eval_images / write_eval_videos on the tiny
model: PNG, JPEG and AVI bytes, the (camera, time) order, two ranks against one, and metrics.json against the
Evaluator's own per-image rows."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.test_gpu_render_path import _cmap_clamped, _png, _quantise

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
# per pixel, absolute: fp32 moments cancel in E[x^2] - mu^2 where a window is flat against a narrow data range (small
# C2); the largest deviation these inputs met on a B200 was 5.9e-5 (test_observed_maxima prints it)
SSIM_TOL = 1e-4
MAXIMA = {"err": 0.0, "ssim": 0.0, "depth_err": 0.0}


def _ref_maps(pred, gt, depth=None, gt_depth=None, norms=None):
    """float64 restatement -> (err, ssim, depth_err) [B,H,W]: ssim from utils.image_metrics.ssim_map per image (its own
    data range), the channel mean, NaN on the 5-pixel border; depth_err from kp_depth_metrics' rule with the fp32 product."""
    from soccernerfs_b200.utils import image_metrics

    b, h, w = pred.shape[:3]
    err = (pred.double() - gt.double()).abs().mean(-1)
    ssim = torch.full((b, h, w), math.nan, dtype=torch.float64, device=pred.device)
    for k in range(b):
        p4, t4 = (torch.moveaxis(x[k].double(), -1, 0)[None] for x in (pred, gt))
        ssim[k, 5:h - 5, 5:w - 5] = image_metrics.ssim_map(t4, p4)[0].mean(0)
    derr = None
    if depth is not None:
        depth, gt_depth, norms = (None if t is None else t.reshape(b, h, w) for t in (depth, gt_depth, norms))
        g = gt_depth if norms is None else gt_depth * norms
        valid = torch.isfinite(g) & (g > 0)
        p, gd = depth.double().clamp_min(1e-6), g.double()
        derr = torch.where(valid, (p - gd).abs() / gd, math.nan)
    return err, ssim, derr


def _check_maps(pred, gt, depth=None, gt_depth=None, norms=None):
    from soccernerfs_b200 import ops
    from soccernerfs_b200.utils import image_metrics

    got = ops.eval_maps(pred, gt, depth, gt_depth, norms)
    b, h, w = pred.shape[:3]
    assert set(got) == ({"error", "ssim"} | ({"depth_error"} if depth is not None else set()))
    assert all(t.shape == (b, h, w) and t.dtype == torch.float32 and t.is_cuda for t in got.values())
    err, ssim, derr = _ref_maps(pred, gt, depth, gt_depth, norms)
    e = float((got["error"].double() - err).abs().max())
    MAXIMA["err"] = max(MAXIMA["err"], e)
    assert e <= 1e-6, e
    border = torch.ones((h, w), dtype=torch.bool, device=DEV)
    border[5:h - 5, 5:w - 5] = False
    assert bool(got["ssim"][:, border].isnan().all()) and not bool(got["ssim"][:, ~border].isnan().any())
    s = float((got["ssim"][:, ~border].double() - ssim[:, ~border]).abs().max())
    MAXIMA["ssim"] = max(MAXIMA["ssim"], s)
    assert s <= SSIM_TOL, s
    metrics = ops.image_metrics(pred, gt).cpu()
    for k in range(b):  # the interior mean is the image's SSIM
        want = float(image_metrics.ssim(*(torch.moveaxis(x[k].double(), -1, 0)[None] for x in (gt, pred))))
        mean = float(got["ssim"][k, 5:h - 5, 5:w - 5].double().mean())
        assert abs(mean - want) <= 1e-5 and abs(mean - float(metrics[k, 1])) <= 1e-5, (k, mean, want)
    if depth is not None:
        nan = derr.isnan()
        assert torch.equal(got["depth_error"].isnan(), nan)
        rel = float(((got["depth_error"].double() - derr).abs() / derr.abs().clamp_min(1e-30))[~nan].max()) if bool((~nan).any()) else 0.0
        MAXIMA["depth_err"] = max(MAXIMA["depth_err"], rel)
        assert rel <= 1e-6, rel
        rows = ops.depth_metrics(depth, gt_depth, norms).cpu()
        for k in range(b):
            valid = ~nan[k]
            if bool(valid.any()):
                mean = float(got["depth_error"][k][valid].double().mean())
                assert abs(mean - float(rows[k, 0, 1])) <= 1e-6 * float(rows[k, 0, 1]), (k, mean, float(rows[k, 0, 1]))
            else:
                assert math.isnan(float(rows[k, 0, 1]))
    return got


def _images(b, h, w, seed):
    """b pairs with a different data range per image: full-range noise, a narrow band around 0.4, a ramp, a flat grey."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    r = lambda: torch.rand((h, w, 3), generator=g, device=DEV)  # noqa: E731
    ramp = torch.linspace(0, 1, w, device=DEV)[None, :, None].expand(h, w, 3)
    kinds = [r(), 0.4 + 0.1 * r(), ramp * 0.8 + 0.05 * r(), torch.full((h, w, 3), 0.5, device=DEV) + 1e-3 * r()]
    pred = torch.stack([kinds[k % 4] for k in range(b)])
    gt = (pred + 0.05 * torch.randn(pred.shape, generator=g, device=DEV)).clamp(0, 1)
    return pred.contiguous(), gt


def _depths(b, h, w, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    gt = 1.0 + 30.0 * torch.rand((b, h, w), generator=g, device=DEV)
    pred = gt * torch.exp(0.3 * torch.randn((b, h, w), generator=g, device=DEV))
    pred[0, 0, :7] = 0.0  # clamped to 1e-6
    gt[0, 1, :5] = 0.0  # sky
    gt[0, 2, :3] = math.inf
    gt[0, 3, :2] = -1.0
    gt[-1, :, :] = 0.0  # an image without a valid pixel
    norms = 1.0 + 0.2 * torch.rand((b, h, w), generator=g, device=DEV)
    return pred, gt, norms


@pytest.mark.parametrize("h,w,b", [(11, 11, 2), (37, 53, 4), (1080, 1920, 2)])
def test_eval_maps_against_float64(h, w, b):
    pred, gt = _images(b, h, w, seed=h + w)
    _check_maps(pred, gt)
    d, gd, norms = _depths(b, h, w, seed=h * w)
    _check_maps(pred, gt, d, gd)
    _check_maps(pred, gt, d[..., None], gd[..., None], norms[..., None])  # [B,H,W,1] like the renderer's frames


def test_eval_maps_bitwise_repeatable_and_graph_replay():
    from soccernerfs_b200 import ops

    pred, gt = _images(3, 270, 480, seed=5)
    d, gd, norms = _depths(3, 270, 480, seed=6)
    a, b = ops.eval_maps(pred, gt, d, gd, norms), ops.eval_maps(pred, gt, d, gd, norms)
    assert all(torch.equal(a[k].nan_to_num(7.0), b[k].nan_to_num(7.0)) and torch.equal(a[k].isnan(), b[k].isnan()) for k in a)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.eval_maps(pred, gt, d, gd, norms)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = ops.eval_maps(pred, gt, d, gd, norms)
    graph.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(captured[k].nan_to_num(7.0), a[k].nan_to_num(7.0)) for k in a)
    pred.copy_(gt)  # new inputs, same buffers: the replay follows them
    graph.replay()
    torch.cuda.synchronize()
    assert float(captured["error"].abs().max()) == 0.0 and float((captured["ssim"][:, 5:-5, 5:-5] - 1).abs().max()) < 1e-5


def test_eval_maps_input_errors():
    from ctypes import c_void_p

    from soccernerfs_b200 import _lib, ops

    x = torch.rand((2, 16, 16, 3), device=DEV)
    d = torch.rand((2, 16, 16), device=DEV)
    with pytest.raises(ValueError, match="11x11"):
        ops.eval_maps(torch.rand((1, 10, 40, 3), device=DEV), torch.rand((1, 10, 40, 3), device=DEV))
    with pytest.raises(ValueError, match="11x11"):
        ops.eval_maps(torch.rand((1, 40, 10, 3), device=DEV), torch.rand((1, 40, 10, 3), device=DEV))
    with pytest.raises(ValueError):
        ops.eval_maps(x, x[:1])
    with pytest.raises(ValueError):
        ops.eval_maps(torch.rand((2, 16, 16, 4), device=DEV), torch.rand((2, 16, 16, 4), device=DEV))
    with pytest.raises(ValueError, match="together"):
        ops.eval_maps(x, x, depth=d)
    with pytest.raises(ValueError, match="directions_norm"):
        ops.eval_maps(x, x, directions_norm=d)
    with pytest.raises(ValueError, match="gt_depth"):
        ops.eval_maps(x, x, d, d[:, :8])
    with pytest.raises(TypeError):
        ops.eval_maps(x.double(), x.double())
    with pytest.raises(TypeError):
        ops.eval_maps(x, x, d.double(), d)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.eval_maps(x.cpu(), x.cpu())
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.eval_maps(x, x, d, d.cpu())
    small = torch.rand((1, 10, 40, 3), device=DEV)
    out = torch.empty((1, 10, 40), device=DEV)
    scratch = torch.empty(1 << 16, dtype=torch.uint8, device=DEV)
    with pytest.raises(RuntimeError, match="smaller than"):  # the library checks it too
        _lib.call("kp_eval_maps", _lib.ptr(small), _lib.ptr(small), None, None, None, 1, 10, 40, c_void_p(scratch.data_ptr()),
                  _lib.ptr(out), _lib.ptr(out), None, _lib.stream_ptr())
    empty = ops.eval_maps(torch.empty((0, 16, 16, 3), device=DEV), torch.empty((0, 16, 16, 3), device=DEV))
    assert empty["error"].shape == (0, 16, 16)


# ---- the tiny model ----
def _tiny_model():
    from tests.test_gpu_eval import _tiny_model as tiny

    model = tiny()
    model.config.is_euclidean_depth = False  # the preset's convention: z-depth ground truth
    return model


def _setup(model, depth=True):
    """6 eval images of 2 cameras (ids 0, 1, alternating), times out of image order within each camera, noisy ground
    truth; with ``depth`` a z-depth ground truth with invalid pixels and an image without any."""
    from soccernerfs_b200.cameras.cameras import Cameras
    from soccernerfs_b200.data.datamanagers.dynamic_datamanager import DynamicDataManager, DynamicDataManagerConfig
    from soccernerfs_b200.engine.frame_renderer import FrameRenderer

    n, h, w = 6, 24, 40
    c2w = torch.tensor([[1.0, 0, 0, 0.1], [0, 1.0, 0, -0.2], [0, 0, 1.0, 2.5]]).repeat(n, 1, 1)
    c2w[:, 0, 3] += torch.tensor([-0.1, 0.1] * 3)
    times = torch.tensor([0.8, 0.5, 0.2, 0.9, 0.5, 0.1])[:, None]
    cams = Cameras(c2w.to(DEV), 40.0, 40.0, w / 2, h / 2, w, h, times=times.to(DEV), ids=torch.tensor([0, 1] * 3).to(DEV))
    out = [FrameRenderer(model, cams, outputs=("rgb", "depth", "directions_norm")).render(i, device_frames=True) for i in range(n)]
    g = torch.Generator(device=DEV).manual_seed(11)
    images = torch.stack([(o["rgb"] + 0.05 * torch.randn(o["rgb"].shape, generator=g, device=DEV)).clamp(0, 1) for o in out])
    cfg = DynamicDataManagerConfig(train_num_rays_per_batch=128, eval_num_rays_per_batch=256, use_importance_sampling=False)
    extras = None
    if depth:
        gt = torch.stack([o["depth"] / o["directions_norm"] for o in out])
        gt = gt * torch.exp(0.1 * torch.randn(gt.shape, generator=g, device=DEV))
        gt[0, :4] = 0.0
        gt[1, 5:9, :6] = math.inf
        gt[3] = 0.0  # no valid pixel
        extras = {"depth_image": gt}
    return DynamicDataManager(cfg, cams, torch.full_like(images, 2.0), device=DEV, eval_cameras=cams, eval_images=images,
                              eval_extras=extras)


def _regions(dm):
    g = torch.Generator(device=DEV).manual_seed(12)
    mask = torch.rand(dm.eval_image_cache.batch["image"].shape[:3], generator=g, device=DEV) < 0.3
    mask[2] = False
    return mask


def _restated_panels(model, dm, regions, i, names, error_range=0.25, depth_error_range=0.25):
    """Image i of the eval split composed by the torch restatement: a direct FrameRenderer render, ops.eval_maps, then
    each panel through utils/colormaps (the kernel's clamped index) and the uint8 quantisation."""
    from soccernerfs_b200 import ops
    from soccernerfs_b200.engine.frame_renderer import FrameRenderer
    from soccernerfs_b200.utils import colormaps

    frames = FrameRenderer(model, dm.eval_cameras, outputs=("rgb", "depth", "accumulation", "median_rgb", "prop_depth_0",
                                                            "prop_depth_1", "directions_norm")).render(i, device_frames=True)
    batch = dm.eval_image_cache.batch
    target = batch["image"][i]
    depth = "depth_image" in batch
    maps = ops.eval_maps(frames["rgb"][None], target[None], frames["depth"][None] if depth else None,
                         batch["depth_image"][i][None] if depth else None, frames["directions_norm"][None] if depth else None)
    acc = frames["accumulation"]
    panels = []
    for name in names:
        if name in ("gt", "rgb", "median_rgb"):
            panels.append(target if name == "gt" else frames[name])
        elif name in ("depth", "prop_depth_0", "prop_depth_1"):
            x = frames[name]
            near, far = float(x.min()), float(x.max())
            panels.append(_cmap_clamped(torch.clip((x - near) / (far - near + 1e-10), 0, 1), "turbo") * acc + (1 - acc))
        elif name == "depth_gt":
            g = batch["depth_image"][i] * frames["directions_norm"]
            valid = torch.isfinite(g) & (g > 0)
            if bool(valid.any()):
                near, far = float(g[valid].min()), float(g[valid].max())
                col = _cmap_clamped(torch.clip((g - near) / (far - near + 1e-10), 0, 1).nan_to_num(0.0), "turbo")
            else:
                col = torch.zeros((*g.shape[:2], 3), device=DEV)
            panels.append(torch.where(valid, col, 1.0))  # white where the ground truth is invalid
        else:
            x = {"accumulation": acc, "error": maps["error"][0, ..., None] / error_range,
                 "ssim": 1 - maps["ssim"][0, ..., None], "dynamic_mask": None if regions is None else regions[i, ..., None].float(),
                 "depth_error": maps["depth_error"][0, ..., None] / depth_error_range if depth else None}[name]
            panels.append(_cmap_clamped(x, "viridis"))
    assert colormaps._table("viridis").shape == (256, 3)
    return _quantise(torch.cat(panels, dim=1))


ALL_PANELS = ("gt", "rgb", "error", "ssim", "depth_gt", "depth_error", "depth", "dynamic_mask")


def test_every_panel_kind_against_the_restatement():
    from soccernerfs_b200.engine.evaluator import Evaluator

    model = _tiny_model()
    dm = _setup(model)
    regions = _regions(dm)
    ev = Evaluator(model, dm, regions=regions)
    for i in (0, 1, 3):  # invalid ground-truth rows, an inf patch, no valid pixel at all
        got = ev._eval_frame(i, ALL_PANELS, 0.25, 0.25)
        want = _restated_panels(model, dm, regions, i, ALL_PANELS)
        assert torch.equal(got, want), (i, int((got.int() - want.int()).abs().max()), int((got != want).any(-1).sum()))
        if i == 0:
            white = got[:4, 4 * 40:5 * 40]  # depth_gt of the invalid rows
            assert bool((white == 255).all())
            assert bool((got[:5, 3 * 40:4 * 40] ==_quantise(_cmap_clamped(torch.zeros(1, 1, 1, device=DEV), "viridis"))[0, 0]).all())
    other = ("median_rgb", "accumulation", "prop_depth_1", "error")
    for rng in (0.05, 1.0):
        assert torch.equal(ev._eval_frame(2, other, rng, rng), _restated_panels(model, dm, regions, 2, other, rng, rng))
    depth_err = ("depth_error",)
    assert torch.equal(ev._eval_frame(2, depth_err, 0.25, 0.05), _restated_panels(model, dm, regions, 2, depth_err, 0.25, 0.05))


def _jpeg(image, quality):
    from soccernerfs_b200 import ops

    out, n = ops.encode_jpeg(image, quality)
    return out[:int(n)].cpu().numpy().tobytes()


def _same(a, b):
    return a == b or (isinstance(a, float) and math.isnan(a) and math.isnan(b))


def test_write_eval_images_png_jpeg_and_metrics(tmp_path):
    from soccernerfs_b200.engine.evaluator import Evaluator

    model = _tiny_model()
    for depth, with_regions in ((False, False), (True, True)):
        dm = _setup(model, depth=depth)
        regions = _regions(dm) if with_regions else None
        ev = Evaluator(model, dm, regions=regions)
        before = ev.get_average_eval_image_metrics(0)
        names = ("gt", "rgb", "error", "ssim") + (("depth_gt", "depth_error", "dynamic_mask") if depth else ())
        png = tmp_path / f"png_{depth}"
        assert ev.write_eval_images(png, panels=names) == list(range(6))
        assert sorted(p.name for p in png.iterdir()) == [f"{i:05d}.png" for i in range(6)] + ["metrics.json"]
        for i in range(6):
            img = _png(png / f"{i:05d}.png")
            assert img.shape == (24, 40 * len(names), 3)
            assert np.array_equal(img, _restated_panels(model, dm, regions, i, names).cpu().numpy()), (depth, i)
        jpg = tmp_path / f"jpg_{depth}"
        ev.write_eval_images(jpg, panels=names, image_format="jpeg", jpeg_quality=80)
        for i in range(6):
            want = _jpeg(torch.from_numpy(_png(png / f"{i:05d}.png")).to(DEV), 80)
            assert (jpg / f"{i:05d}.jpg").read_bytes() == want, (depth, i)
        # metrics.json: the Evaluator's own per-image rows, bit for bit (NaN where NaN)
        rows = ev._rank_rows(list(range(6)))
        keys = ev._value_keys()
        for path, ext in ((png, "png"), (jpg, "jpg")):
            doc = json.loads((path / "metrics.json").read_text())["images"]
            assert [e["image"] for e in doc] == list(range(6)) and [e["file"] for e in doc] == [f"{i:05d}.{ext}" for i in range(6)]
            for e in doc:
                assert list(e)[2:] == keys
                assert all(_same(e[k], rows[e["image"]][k]) for k in keys), (e, rows[e["image"]])
        if depth:
            assert math.isnan(doc[3]["depth_abs_rel"]) and math.isnan(doc[2]["psnr_dynamic"])
        after = ev.get_average_eval_image_metrics(1)
        assert list(after) == list(before)
        assert all(_same(after[k], before[k]) for k in before if k not in ("num_rays_per_sec", "fps")), (before, after)


def test_write_eval_videos_in_camera_time_order(tmp_path):
    from soccernerfs_b200.engine.evaluator import Evaluator
    from soccernerfs_b200.engine.path_renderer import assemble_video
    from tests.test_video_host import _parse_avi

    model = _tiny_model()
    dm = _setup(model)
    ev = Evaluator(model, dm)
    names = ("gt", "rgb", "error", "depth_error")
    one = tmp_path / "one"
    written = ev.write_eval_videos(one, 12.5, panels=names, jpeg_quality=85)
    assert written == {str(one / "camera_000.avi"): [2, 4, 0], str(one / "camera_001.avi"): [5, 1, 3]}  # by time
    assert sorted(p.name for p in one.iterdir()) == ["camera_000.avi", "camera_001.avi"]
    for name, seq in (("camera_000.avi", [2, 4, 0]), ("camera_001.avi", [5, 1, 3])):
        avi = _parse_avi(one / name)
        assert avi["fps"] == pytest.approx(12.5) and (avi["width"], avi["height"]) == (40 * len(names), 24)
        assert avi["frames"] == [_jpeg(ev._eval_frame(i, names, 0.25, 0.25), 85) for i in seq], name
    # two ranks in one process (no process group): each writes its parts, the caller assembles them
    two = tmp_path / "two"
    parts = [Evaluator(model, dm, rank=r, world=2).write_eval_videos(two, 12.5, panels=names, jpeg_quality=85) for r in range(2)]
    assert parts[0] == {str(two / "camera_000.avi"): [2, 0], str(two / "camera_001.avi"): [5, 3]}
    assert parts[1] == {str(two / "camera_000.avi"): [4], str(two / "camera_001.avi"): [1]}
    for path in parts[0]:
        assert not os.path.exists(path)
        assemble_video(path, 2, 12.5)
    for name in ("camera_000.avi", "camera_001.avi"):
        assert (two / name).read_bytes() == (one / name).read_bytes(), name
    # without camera ids: one video in image order
    dm.eval_cameras.ids = None
    ev.write_eval_videos(tmp_path / "noid", 5.0, panels=("rgb",))
    assert len(_parse_avi(tmp_path / "noid" / "eval.avi")["frames"]) == 6


def test_two_ranks_write_the_files_of_one_rank(tmp_path):
    from soccernerfs_b200.engine.evaluator import Evaluator

    model = _tiny_model()
    dm = _setup(model)
    regions = _regions(dm)
    names = ("gt", "rgb", "error", "ssim", "depth_gt", "dynamic_mask")
    one, two = tmp_path / "one", tmp_path / "two"
    Evaluator(model, dm, regions=regions).write_eval_images(one, panels=names, image_format="jpeg")
    mine = [Evaluator(model, dm, rank=r, world=2, regions=regions).write_eval_images(two, panels=names, image_format="jpeg")
            for r in range(2)]
    assert mine == [[0, 2, 4], [1, 3, 5]]
    assert sorted(p.name for p in two.iterdir()) == [f"{i:05d}.jpg" for i in range(6)] + ["metrics.rank0.json", "metrics.rank1.json"]
    for i in range(6):
        assert (two / f"{i:05d}.jpg").read_bytes() == (one / f"{i:05d}.jpg").read_bytes(), i
    single = json.loads((one / "metrics.json").read_text())["images"]
    merged = sorted(sum((json.loads((two / f"metrics.rank{r}.json").read_text())["images"] for r in range(2)), []),
                    key=lambda e: e["image"])
    assert [list(e) for e in merged] == [list(e) for e in single]
    assert all(_same(a[k], b[k]) for a, b in zip(merged, single) for k in a)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_eval_images_two_processes_equal_one():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29583", os.path.join(root, "tests", "_eval_images_worker.py")]
    res = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "EVAL_IMAGES_MULTI_OK" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]


def test_observed_maxima():
    """Runs after the map tests: the largest deviations from float64 they met (the ground for SSIM_TOL)."""
    if MAXIMA["ssim"] == 0.0:  # run on its own
        test_eval_maps_against_float64(1080, 1920, 2)
    print(f"eval_maps: max |err - ref| {MAXIMA['err']:.3e}, max |ssim - ref| {MAXIMA['ssim']:.3e}, "
          f"max depth_err relative {MAXIMA['depth_err']:.3e}")
