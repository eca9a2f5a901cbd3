"""Eval depth metrics on the device: kp_depth_metrics against the float64 utils/image_metrics.depth_metrics, masks that
reproduce the unmasked row, repeatability and graph replay, input errors, and the Evaluator with eval depth on the tiny
model (one GPU and, with >= 2 GPUs, two ranks)."""
import math
import os
import subprocess
import sys
from ctypes import c_void_p

import pytest
import torch

from tests.test_gpu_eval import _eval_cameras, _tiny_model

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _same(a, b):
    return torch.equal(a.isnan(), b.isnan()) and torch.equal(a.nan_to_num(), b.nan_to_num())


def _inputs(b, h, w, g):
    """Rendered-like depth, a noisy ground truth with every kind of invalid pixel, and ray-direction norms."""
    pred = 0.5 + 10 * torch.rand((b, h, w), generator=g, device=DEV)
    pred[torch.rand(pred.shape, generator=g, device=DEV) < 0.02] = 0.0  # clamped to 1e-6
    norm = 1 + 0.4 * torch.rand((b, h, w), generator=g, device=DEV)
    gt = pred / norm * torch.exp(0.3 * torch.randn(pred.shape, generator=g, device=DEV))
    u = torch.rand(pred.shape, generator=g, device=DEV)
    gt[u < 0.1] = 0.0
    gt[(u >= 0.1) & (u < 0.13)] = math.inf
    gt[(u >= 0.13) & (u < 0.15)] = math.nan
    gt[(u >= 0.15) & (u < 0.17)] = -1.0
    pred[0, 0, 0], gt[0, 0, 0] = 4.0, 5.0  # a ratio exactly on a threshold (without directions_norm)
    return pred, gt, norm


def _check(pred, gt, norm=None, mask=None):
    """ops.depth_metrics == the float64 restatement: n_valid and the deltas exactly, the four error sums to 1e-12
    relative, NaN where it is NaN."""
    from soccernerfs_b200 import ops
    from soccernerfs_b200.utils import image_metrics

    got = ops.depth_metrics(pred, gt, norm, mask)
    assert got.dtype == torch.float64 and got.shape == (pred.shape[0], 1 if mask is None else 3, 8)
    ref = image_metrics.depth_metrics(pred, gt, norm, mask)
    assert torch.equal(got.isnan(), ref.isnan()), (got, ref)
    exact = [0, 5, 6, 7]
    assert _same(got[..., exact], ref[..., exact]), (got, ref)
    ok = ~ref[..., 1:5].isnan()
    err = (got[..., 1:5] - ref[..., 1:5]).abs()
    assert bool((err <= 1e-12 * ref[..., 1:5].abs())[ok].all()), (got, ref)
    return got


def _masks(b, h, w, g):
    """random, single pixel, all true, all false: one kind per image, cycling."""
    out = []
    for k in range(b):
        m = torch.zeros((h, w), dtype=torch.bool, device=DEV)
        if k % 4 == 0:
            m = torch.rand((h, w), generator=g, device=DEV) < 0.3
        elif k % 4 == 1:
            m[h // 2, w // 2] = True
        elif k % 4 == 2:
            m[:] = True
        out.append(m)
    return torch.stack(out)


@pytest.mark.parametrize("h,w,b", [(1, 1, 4), (37, 53, 5), (23, 300, 4), (1080, 1920, 2)])
def test_depth_metrics_against_float64(h, w, b):
    g = torch.Generator(device=DEV).manual_seed(h * 7 + w)
    pred, gt, norm = _inputs(b, h, w, g)
    gt[-1] = 0.0  # an image without a valid pixel
    masks = _masks(b, h, w, g)
    if b == 2:
        masks[1] = _masks(2, h, w, g)[1]  # single pixel at 1080p
    whole = _check(pred, gt)
    assert whole[0, 0, 0] > 0 and whole[-1, 0, 0] == 0 and bool(whole[-1, 0, 1:].isnan().all())
    _check(pred, gt, norm)
    _check(pred[..., None], gt[..., None], norm[..., None])  # [B,H,W,1]
    _check(pred, gt, norm, masks)
    _check(pred, gt, None, masks.to(torch.uint8) * 200)  # any non-zero byte is dynamic


def test_directions_norm_is_an_fp32_product():
    from soccernerfs_b200 import ops

    g = torch.Generator(device=DEV).manual_seed(3)
    pred, gt, norm = _inputs(3, 45, 61, g)
    assert torch.equal(ops.depth_metrics(pred, gt, norm).nan_to_num(), ops.depth_metrics(pred, gt * norm).nan_to_num())


@pytest.mark.parametrize("h,w", [(1, 1), (37, 53), (540, 960)])
def test_all_true_and_all_false_masks_reproduce_the_whole_row_bit_for_bit(h, w):
    from soccernerfs_b200 import ops

    g = torch.Generator(device=DEV).manual_seed(h)
    pred, gt, norm = _inputs(3, h, w, g)
    whole = ops.depth_metrics(pred, gt, norm)
    ones = torch.ones((3, h, w), dtype=torch.bool, device=DEV)
    dyn, static = ops.depth_metrics(pred, gt, norm, ones), ops.depth_metrics(pred, gt, norm, ~ones)
    for out, r in ((dyn, 1), (static, 2)):
        assert _same(out[:, 0], whole[:, 0]) and _same(out[:, r], whole[:, 0])
        assert bool((out[:, 3 - r, 0] == 0).all()) and bool(out[:, 3 - r, 1:].isnan().all())


def test_bitwise_repeatable_and_graph_replay():
    from soccernerfs_b200 import ops

    g = torch.Generator(device=DEV).manual_seed(2)
    pred, gt, norm = _inputs(3, 270, 480, g)
    mask = _masks(3, 270, 480, g)
    a, b = ops.depth_metrics(pred, gt, norm, mask), ops.depth_metrics(pred, gt, norm, mask)
    assert _same(a, b)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.depth_metrics(pred, gt, norm, mask)  # warm-up on the capturing stream
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = ops.depth_metrics(pred, gt, norm, mask)
    graph.replay()
    torch.cuda.synchronize()
    assert _same(captured, a)
    mask.copy_(~mask)  # new mask, same buffer: the replay follows it
    graph.replay()
    torch.cuda.synchronize()
    assert _same(captured, ops.depth_metrics(pred, gt, norm, mask))
    assert _same(captured[:, 1], a[:, 2]) and _same(captured[:, 2], a[:, 1]) and _same(captured[:, 0], a[:, 0])


def test_input_errors():
    from soccernerfs_b200 import _lib, ops

    d = torch.rand((2, 16, 16), device=DEV)
    out = torch.empty((2, 3, 8), dtype=torch.float64, device=DEV)
    scratch = torch.empty(1 << 20, dtype=torch.uint8, device=DEV)
    args = (_lib.ptr(d), _lib.ptr(d), c_void_p(0), c_void_p(0))
    with pytest.raises(RuntimeError, match="B=-1"):
        _lib.call("kp_depth_metrics", *args, -1, 256, c_void_p(scratch.data_ptr()), _lib.ptr(out), _lib.stream_ptr())
    with pytest.raises(RuntimeError, match="HW=0"):
        _lib.call("kp_depth_metrics", *args, 2, 0, c_void_p(scratch.data_ptr()), _lib.ptr(out), _lib.stream_ptr())
    with pytest.raises(RuntimeError, match="NULL"):
        _lib.call("kp_depth_metrics", *args, 2, 256, c_void_p(0), _lib.ptr(out), _lib.stream_ptr())
    with pytest.raises(RuntimeError, match="NULL"):
        _lib.call("kp_depth_metrics", c_void_p(0), *args[1:], 2, 256, c_void_p(scratch.data_ptr()), _lib.ptr(out),
                  _lib.stream_ptr())
    assert ops.depth_metrics(d[:0], d[:0]).shape == (0, 1, 8)
    assert ops.depth_metrics(d[:0], d[:0], mask=torch.ones((0, 16, 16), dtype=torch.bool, device=DEV)).shape == (0, 3, 8)
    with pytest.raises(ValueError, match="one shape"):
        ops.depth_metrics(d, d[:, :8])
    with pytest.raises(ValueError, match="mask must be"):
        ops.depth_metrics(d, d, mask=torch.ones((2, 16, 15), dtype=torch.bool, device=DEV))
    with pytest.raises(TypeError):
        ops.depth_metrics(d, d.half())
    with pytest.raises(TypeError):
        ops.depth_metrics(d, d, mask=d)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.depth_metrics(d, d.cpu())
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.depth_metrics(d, d, mask=torch.ones((2, 16, 16), dtype=torch.bool))


def _depth_setup(model, n=4, h=24, w=40, scale=1.0):
    """The eval setup of test_gpu_eval with ground-truth depth: the model's own rendered depth as z-depth
    (depth / directions_norm, the preset's convention), times ``scale``.  -> (dm, frames, images, depth, norms, gt)."""
    from soccernerfs_b200.data.datamanagers.dynamic_datamanager import DynamicDataManager, DynamicDataManagerConfig
    from soccernerfs_b200.engine.frame_renderer import FrameRenderer

    cams = _eval_cameras(h, w, n)
    renderer = FrameRenderer(model, cams, outputs=("rgb", "depth", "directions_norm"))
    out = [renderer.render(i, device_frames=True) for i in range(n)]
    frames = [o["rgb"] for o in out]
    depth, norms = torch.stack([o["depth"] for o in out]), torch.stack([o["directions_norm"] for o in out])
    g = torch.Generator(device=DEV).manual_seed(3)
    images = torch.stack([(f + 0.05 * torch.randn(f.shape, generator=g, device=DEV)).clamp(0, 1) for f in frames])
    gt = depth / norms * scale
    cfg = DynamicDataManagerConfig(train_num_rays_per_batch=128, eval_num_rays_per_batch=256, use_importance_sampling=False)
    dm = DynamicDataManager(cfg, cams, torch.full_like(images, 2.0), device=DEV, eval_cameras=cams, eval_images=images,
                            eval_extras={"depth_image": gt})
    return dm, frames, images, depth, norms, gt


def _region_reference(depth, gt, norms, mask):
    """The Evaluator's depth keys from the float64 restatement, averaged over the images where each is defined."""
    from soccernerfs_b200.engine.evaluator import DEPTH_KEYS
    from soccernerfs_b200.utils import image_metrics

    rows = image_metrics.depth_metrics(depth, gt, norms, mask).cpu()
    out = {}
    for r, s in enumerate(("", "_dynamic", "_static")[:rows.shape[1]]):
        for c, k in enumerate(DEPTH_KEYS):
            vals = [v for v in rows[:, r, c + 1].tolist() if not math.isnan(v)]
            out[k + s] = sum(vals) / len(vals) if vals else math.nan
        out["num_images_depth" + s] = int((rows[:, r, 0] > 0).sum())
    return out


def test_evaluator_with_eval_depth_on_the_tiny_model():
    import random

    from soccernerfs_b200.engine.evaluator import DEPTH_KEYS, REGION_KEYS, Evaluator, depth_row_keys

    model = _tiny_model()
    model.config.is_euclidean_depth = False  # the preset's convention: z-depth ground truth
    dm, frames, images, depth, norms, gt = _depth_setup(model)
    ev = Evaluator(model, dm)
    assert ev.depth and "directions_norm" in ev.renderer.outputs
    avg = ev.get_average_eval_image_metrics(0)
    colour = [k for k in avg if k not in DEPTH_KEYS and k != "num_images_depth"]
    assert colour in (["psnr", "ssim", "num_rays_per_sec", "fps"], ["psnr", "ssim", "lpips", "num_rays_per_sec", "fps"])
    assert list(avg) == colour + list(DEPTH_KEYS) + ["num_images_depth"]
    # the ground truth is the rendered depth, up to the two fp32 roundings of / and * directions_norm
    assert avg["num_images_depth"] == 4
    assert avg["depth_abs_rel"] < 1e-6 and avg["depth_sq_rel"] < 1e-12 * float(depth.max()) and avg["depth_rmse_log"] < 1e-6
    assert avg["depth_rmse"] < 1e-6 * float(depth.max())
    assert avg["depth_delta1"] == avg["depth_delta2"] == avg["depth_delta3"] == 1.0

    # the same Evaluator without eval depth: the parent's keys, and colour values that depth did not change
    plain_dm = _depth_setup(model)[0]
    plain_dm.eval_image_cache.batch.pop("depth_image")
    plain = Evaluator(model, plain_dm)
    assert not plain.depth and "directions_norm" not in plain.renderer.outputs
    plain_avg = plain.get_average_eval_image_metrics(0)
    assert list(plain_avg) == colour and all(plain_avg[k] == avg[k] for k in ("psnr", "ssim"))

    # eval batches and eval images carry the ground truth; the reference's depth panel shows it beside the prediction
    random.seed(0)
    torch.manual_seed(0)
    rb, batch = dm.next_eval(1)
    idx = batch["indices"]
    assert torch.equal(batch["depth_image"], gt[idx[:, 0], idx[:, 1], idx[:, 2]])
    i, image_batch = dm.next_eval_image(2)
    assert set(image_batch) == {"image", "depth_image"} and torch.equal(image_batch["depth_image"], gt[i])
    metrics, images_dict = ev.get_eval_image_metrics_and_images(3)
    assert images_dict["depth"].shape == (24, 80, 3) and images_dict["img"].shape == (24, 80, 3)
    assert "psnr" in metrics and not any(k.startswith("depth") for k in metrics)

    # twice the z-depth: abs_rel 0.5, rmse_log log 2, no pixel within 1.25^3
    twice = Evaluator(model, _depth_setup(model, scale=2.0)[0]).get_average_eval_image_metrics(0)
    assert abs(twice["depth_abs_rel"] - 0.5) < 1e-6 and abs(twice["depth_rmse_log"] - math.log(2)) < 1e-6
    assert twice["depth_delta1"] == twice["depth_delta2"] == twice["depth_delta3"] == 0.0

    # regions: each region key equals the restatement over that region; a noisy ground truth with invalid pixels
    g = torch.Generator(device=DEV).manual_seed(9)
    noisy = gt * torch.exp(0.2 * torch.randn(gt.shape, generator=g, device=DEV))
    noisy[0, :5] = 0.0  # sky
    noisy[2] = math.inf  # no valid pixel
    dm.eval_image_cache.batch["depth_image"] = noisy
    caller = torch.rand(images.shape[:3], generator=g, device=DEV) < 0.3
    caller[1] = False  # no dynamic pixel
    regioned = Evaluator(model, dm, regions=caller).get_average_eval_image_metrics(0)
    n_region = len(colour) + len(REGION_KEYS) + 3
    assert list(regioned)[n_region:] == (list(DEPTH_KEYS) + ["num_images_depth"] + depth_row_keys(True)[7:]
                                         + ["num_images_depth_dynamic", "num_images_depth_static"])
    ref = _region_reference(depth, noisy, norms, caller)
    assert (ref["num_images_depth"], ref["num_images_depth_dynamic"], ref["num_images_depth_static"]) == (3, 2, 3)
    for k, v in ref.items():
        assert abs(regioned[k] - v) <= 1e-6 * abs(v), (k, regioned[k], v)


def test_euclidean_ground_truth_needs_no_directions_norm():
    from soccernerfs_b200.engine.evaluator import Evaluator

    model = _tiny_model()
    model.config.is_euclidean_depth = True
    dm, _, _, depth, norms, gt = _depth_setup(model, n=3)
    dm.eval_image_cache.batch["depth_image"] = depth.clone()  # distance along the unit ray, compared as is
    ev = Evaluator(model, dm)
    assert "directions_norm" not in ev.renderer.outputs
    avg = ev.get_average_eval_image_metrics(0)
    assert avg["depth_abs_rel"] < 1e-6 and avg["depth_delta1"] == 1.0


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_evaluator_depth_two_ranks_equal_one_rank():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29581", os.path.join(root, "tests", "_depth_eval_worker.py")]
    res = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "DEPTH_EVAL_MULTI_OK" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]
