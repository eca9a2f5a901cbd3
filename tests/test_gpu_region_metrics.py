"""Per-region eval metrics on the device: kp_image_metrics_masked against the float64 utils/image_metrics.region_psnr_ssim,
its agreement with kp_image_metrics for all-true / all-false masks, repeatability and graph replay, median_dynamic_masks on
a synthetic eval camera, and Evaluator(regions=...) on the tiny model (one GPU and, with >= 2 GPUs, two ranks)."""
import math
import os
import subprocess
import sys

import pytest
import torch

from tests.test_gpu_eval import _eval_setup, _tiny_model

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _check(pred, target, mask):
    """ops.image_metrics_masked == region_psnr_ssim in float64: PSNR to 1e-5 relative, SSIM to 1e-5, NaN where it is NaN."""
    from soccernerfs_b200 import ops
    from soccernerfs_b200.utils import image_metrics

    got = ops.image_metrics_masked(pred, target, mask).cpu()
    assert got.shape == (pred.shape[0], 4) and got.dtype == torch.float32
    ref = image_metrics.region_psnr_ssim(pred.double(), target.double(), mask).cpu()
    assert torch.equal(got.isnan(), ref.isnan()), (got, ref)
    ok = ~ref.isnan()
    tol = torch.where(torch.arange(4)[None] % 2 == 0, 1e-5 * ref.abs(), torch.full_like(ref, 1e-5))
    assert bool(((got.double() - ref).abs() <= tol)[ok].all()), (got, ref)
    return got


def _masks(b, h, w, g):
    """random, blob, single pixel, border only, all true, all false: one kind per image, cycling."""
    out = []
    for k in range(b):
        kind = k % 6
        m = torch.zeros((h, w), dtype=torch.bool, device=DEV)
        if kind == 0:
            m = torch.rand((h, w), generator=g, device=DEV) < 0.3
        elif kind == 1:
            yy, xx = torch.meshgrid(torch.arange(h, device=DEV), torch.arange(w, device=DEV), indexing="ij")
            m = (yy - h * 0.4) ** 2 + (xx - w * 0.6) ** 2 < (min(h, w) * 0.3) ** 2
        elif kind == 2:
            m[h // 2, w // 2] = True
        elif kind == 3:
            m[:5, :] = True
            m[:, -5:] = True
        elif kind == 4:
            m[:] = True
        out.append(m)
    return torch.stack(out)


@pytest.mark.parametrize("h,w,b", [(11, 11, 6), (37, 53, 6), (23, 300, 6), (1080, 1920, 2)])
def test_masked_metrics_against_float64(h, w, b):
    g = torch.Generator(device=DEV).manual_seed(h * 7 + w)
    pred = torch.rand((b, h, w, 3), generator=g, device=DEV)
    target = (pred + 0.1 * torch.randn(pred.shape, generator=g, device=DEV)).clamp(0, 1)
    target[-1] = torch.rand(target[-1].shape, generator=g, device=DEV)  # an unrelated pair
    masks = _masks(b, h, w, g)
    if b == 2:
        masks[1] = _masks(3, h, w, g)[2] | _masks(4, h, w, g)[3]  # single pixel + border at 1080p
    _check(pred, target, masks)
    _check(pred, target, masks.to(torch.uint8) * 200)  # any non-zero byte is dynamic


def test_mixed_batch_rows_equal_single_images():
    from soccernerfs_b200 import ops

    g = torch.Generator(device=DEV).manual_seed(5)
    ramp = torch.linspace(0, 1, 53, device=DEV)[None, :, None].expand(37, 53, 3)
    pred = torch.stack([ramp, torch.full((37, 53, 3), 0.5, device=DEV) + 1e-3 * torch.randn((37, 53, 3), generator=g, device=DEV),
                        0.2 + 0.2 * torch.rand((37, 53, 3), generator=g, device=DEV),
                        (torch.rand((37, 53, 3), generator=g, device=DEV) > 0.5).float(), torch.rand((37, 53, 3), generator=g, device=DEV),
                        torch.rand((37, 53, 3), generator=g, device=DEV)])
    target = (pred + 0.03 * torch.randn(pred.shape, generator=g, device=DEV)).clamp(0, 1)
    masks = _masks(6, 37, 53, g)
    batch = _check(pred, target, masks)
    for k in range(6):
        one = ops.image_metrics_masked(pred[k:k + 1], target[k:k + 1], masks[k:k + 1]).cpu()
        assert torch.equal(one.isnan(), batch[k:k + 1].isnan()) and torch.equal(one.nan_to_num(), batch[k:k + 1].nan_to_num()), k


@pytest.mark.parametrize("h,w", [(11, 11), (37, 53), (540, 960)])
def test_all_true_and_all_false_masks_equal_image_metrics_bit_for_bit(h, w):
    from soccernerfs_b200 import ops

    g = torch.Generator(device=DEV).manual_seed(h)
    pred = torch.rand((3, h, w, 3), generator=g, device=DEV)
    target = (pred + 0.05 * torch.randn(pred.shape, generator=g, device=DEV)).clamp(0, 1)
    whole = ops.image_metrics(pred, target)
    ones = torch.ones((3, h, w), dtype=torch.bool, device=DEV)
    dyn, static = ops.image_metrics_masked(pred, target, ones), ops.image_metrics_masked(pred, target, ~ones)
    assert torch.equal(dyn[:, :2], whole) and torch.equal(static[:, 2:], whole)
    assert bool(dyn[:, 2:].isnan().all()) and bool(static[:, :2].isnan().all())


def test_bitwise_repeatable_and_graph_replay():
    from soccernerfs_b200 import ops

    g = torch.Generator(device=DEV).manual_seed(2)
    pred = torch.rand((3, 270, 480, 3), generator=g, device=DEV)
    target = (pred + 0.05 * torch.randn(pred.shape, generator=g, device=DEV)).clamp(0, 1)
    mask = _masks(3, 270, 480, g)
    a, b = ops.image_metrics_masked(pred, target, mask), ops.image_metrics_masked(pred, target, mask)
    assert torch.equal(a, b)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.image_metrics_masked(pred, target, mask)  # warm-up on the capturing stream
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = ops.image_metrics_masked(pred, target, mask)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, a)
    mask.copy_(~mask)  # new mask, same buffer: the replay follows it
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, ops.image_metrics_masked(pred, target, mask))
    assert torch.equal(captured[:, :2], a[:, 2:]) and torch.equal(captured[:, 2:], a[:, :2])


def test_input_errors():
    from ctypes import c_void_p

    from soccernerfs_b200 import _lib, ops

    small = torch.rand((1, 10, 40, 3), device=DEV)
    with pytest.raises(ValueError, match="11x11"):
        ops.image_metrics_masked(small, small, torch.ones((1, 10, 40), dtype=torch.bool, device=DEV))
    out = torch.empty((1, 4), device=DEV)
    scratch = torch.empty(1 << 20, dtype=torch.uint8, device=DEV)
    mask = torch.ones((1, 10, 40), dtype=torch.uint8, device=DEV)
    with pytest.raises(RuntimeError, match="smaller than"):  # the library checks it too
        _lib.call("kp_image_metrics_masked", _lib.ptr(small), _lib.ptr(small), c_void_p(mask.data_ptr()), 1, 10, 40,
                  c_void_p(scratch.data_ptr()), _lib.ptr(out), _lib.stream_ptr())
    img = torch.rand((2, 16, 16, 3), device=DEV)
    with pytest.raises(ValueError, match="mask must be"):
        ops.image_metrics_masked(img, img, torch.ones((1, 16, 16), dtype=torch.bool, device=DEV))
    with pytest.raises(ValueError):
        ops.image_metrics_masked(torch.rand((2, 16, 16, 4), device=DEV), torch.rand((2, 16, 16, 4), device=DEV),
                                 torch.ones((2, 16, 16), dtype=torch.bool, device=DEV))
    with pytest.raises(TypeError):
        ops.image_metrics_masked(img.double(), img.double(), torch.ones((2, 16, 16), dtype=torch.bool, device=DEV))
    with pytest.raises(TypeError):
        ops.image_metrics_masked(img, img, torch.ones((2, 16, 16), dtype=torch.int32, device=DEV))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.image_metrics_masked(img, img, torch.ones((2, 16, 16), dtype=torch.bool))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.image_metrics_masked(img.cpu(), img.cpu(), torch.ones((2, 16, 16), dtype=torch.bool))


def _moving_square_clip():
    """Two cameras over a constant background: camera 7 has 4 frames, camera 2 has 3, and in every frame a square
    sits at a position it occupies in no other frame of its camera."""
    h, w, s = 40, 64, 8
    spots = {7: [(2, 3), (20, 10), (5, 40), (28, 50)], 2: [(10, 5), (10, 20), (10, 35)]}
    images, ids, squares = [], [], []
    for cam, places in spots.items():
        for y, x in places:
            img = torch.full((h, w, 3), 0.3, device=DEV)
            img[..., 1] = 0.45
            sq = torch.zeros((h, w), dtype=torch.bool, device=DEV)
            sq[y:y + s, x:x + s] = True
            img[sq] = torch.tensor([0.9, 0.1, 0.8], device=DEV)
            images.append(img)
            ids.append(cam)
            squares.append(sq)
    return torch.stack(images), torch.tensor(ids), torch.stack(squares)


def test_median_dynamic_masks_mark_the_square_of_each_frame():
    from soccernerfs_b200.engine.evaluator import median_dynamic_masks

    images, ids, squares = _moving_square_clip()
    masks = median_dynamic_masks(images, ids)
    assert masks.dtype == torch.bool and masks.shape == squares.shape
    assert torch.equal(masks, squares)
    with pytest.raises(ValueError, match="camera 2 has 2 image"):
        median_dynamic_masks(images[:6], ids[:6])


def _region_reference(frames, images, masks):
    from soccernerfs_b200.utils import image_metrics

    rows = image_metrics.region_psnr_ssim(torch.stack(frames).double(), images.double(), masks).tolist()
    out = {}
    for c, k in enumerate(("psnr_dynamic", "ssim_dynamic", "psnr_static", "ssim_static")):
        vals = [r[c] for r in rows if not math.isnan(r[c])]
        out[k] = sum(vals) / len(vals) if vals else float("nan")
    out["dynamic_fraction"] = float(masks.flatten(1).double().mean(1).mean())
    out["num_images_dynamic"] = sum(not math.isnan(r[0]) for r in rows)
    out["num_images_static"] = sum(not math.isnan(r[2]) for r in rows)
    return out


def _compare(avg, ref):
    for k in ("psnr_dynamic", "psnr_static"):
        assert abs(avg[k] - ref[k]) <= 1e-5 * abs(ref[k]), (k, avg, ref)
    for k in ("ssim_dynamic", "ssim_static", "dynamic_fraction"):
        assert abs(avg[k] - ref[k]) <= 1e-5, (k, avg, ref)
    assert avg["num_images_dynamic"] == ref["num_images_dynamic"] and avg["num_images_static"] == ref["num_images_static"]


def test_evaluator_regions_on_the_tiny_model():
    from soccernerfs_b200.engine.evaluator import Evaluator, median_dynamic_masks

    model = _tiny_model()
    dm, frames, images = _eval_setup(model, n=4)
    plain = Evaluator(model, dm).get_average_eval_image_metrics(0)

    g = torch.Generator(device=DEV).manual_seed(9)
    caller = torch.rand(images.shape[:3], generator=g, device=DEV) < 0.25
    caller[1] = False  # an image without a dynamic pixel
    caller[2, :, :] = False
    caller[2, :3, :] = True  # dynamic pixels on the border only
    avg = Evaluator(model, dm, regions=caller.to(torch.uint8)).get_average_eval_image_metrics(0)
    assert list(avg)[:len(plain)] == list(plain)
    assert list(avg)[len(plain):] == ["psnr_dynamic", "ssim_dynamic", "psnr_static", "ssim_static", "dynamic_fraction",
                                      "num_images_dynamic", "num_images_static"]
    assert all(avg[k] == plain[k] for k in ("psnr", "ssim"))
    ref = _region_reference(frames, images, caller)
    assert ref["num_images_dynamic"] == 3
    _compare(avg, ref)

    dm.eval_cameras.ids = torch.zeros(4, dtype=torch.int64)
    ev = Evaluator(model, dm, regions="median")
    masks = median_dynamic_masks(images, dm.eval_cameras.ids)
    assert torch.equal(ev.regions, masks)
    _compare(ev.get_average_eval_image_metrics(0), _region_reference(frames, images, masks))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_evaluator_regions_two_ranks_equal_one_rank():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29579", os.path.join(root, "tests", "_region_eval_worker.py")]
    res = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "REGION_EVAL_MULTI_OK" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]
