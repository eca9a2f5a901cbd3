"""Eval side on the device: kp_image_metrics against utils/image_metrics.py, FrameRenderer(device_frames=True), the eval
split of DynamicDataManager and the Evaluator on the tiny model (one GPU and, with >= 2 GPUs, two ranks)."""
import os
import subprocess
import sys

import pytest
import torch

from tests.conftest import load_golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _reference(pred, target):
    """image_metrics.psnr / ssim of one [H,W,3] pair in the model's argument order, in float64 (so the reference itself
    carries no fp32 / TF32 convolution rounding)."""
    from soccernerfs_b200.utils import image_metrics

    p = torch.moveaxis(pred.double(), -1, 0)[None]
    t = torch.moveaxis(target.double(), -1, 0)[None]
    return float(image_metrics.psnr(t, p)), float(image_metrics.ssim(t, p))


def _check(pred, target):
    from soccernerfs_b200 import ops

    got = ops.image_metrics(pred, target).cpu()
    assert got.shape == (pred.shape[0], 2) and got.dtype == torch.float32
    for k in range(pred.shape[0]):
        psnr, ssim = _reference(pred[k], target[k])
        assert abs(float(got[k, 0]) - psnr) <= 1e-5 * abs(psnr), (k, float(got[k, 0]), psnr)
        assert abs(float(got[k, 1]) - ssim) <= 1e-5, (k, float(got[k, 1]), ssim)
    return got


def _tiny_model():
    from tests.helpers import build_model
    from tests.test_oracle_golden import load_tiny_model

    gm = load_golden("model_tiny")
    model = build_model("tiny", load_tiny_model(gm), gm["aabb"], DEV)
    model.eval()
    model.config.eval_num_rays_per_chunk = 256
    return model


def _eval_cameras(h=24, w=40, n=3):
    from soccernerfs_b200.cameras.cameras import Cameras

    c2w = torch.tensor([[1.0, 0, 0, 0.1], [0, 1.0, 0, -0.2], [0, 0, 1.0, 2.5]]).repeat(n, 1, 1)
    c2w[:, 0, 3] += torch.linspace(-0.1, 0.1, n)
    return Cameras(c2w.to(DEV), 40.0, 40.0, w / 2, h / 2, w, h, times=torch.linspace(0.2, 0.8, n)[:, None].to(DEV))


def _renders(model, cams):
    return [model.get_outputs_for_camera_ray_bundle(cams.generate_rays(camera_indices=i, keep_shape=True))["rgb"]
            for i in range(len(cams))]


def test_image_metrics_random_pairs():
    g = torch.Generator(device=DEV).manual_seed(0)
    pred = torch.rand((2, 540, 960, 3), generator=g, device=DEV)
    target = (pred + 0.1 * torch.randn(pred.shape, generator=g, device=DEV)).clamp(0, 1)
    target[1] = torch.rand(target[1].shape, generator=g, device=DEV)  # an unrelated pair: SSIM near 0
    _check(pred, target)


def test_image_metrics_rendered_frames_odd_and_minimum_sizes_and_a_mixed_batch():
    model = _tiny_model()
    frames = _renders(model, _eval_cameras(37, 53))
    g = torch.Generator(device=DEV).manual_seed(1)
    noisy = [(f + 0.05 * torch.randn(f.shape, generator=g, device=DEV)).clamp(0, 1) for f in frames]
    _check(torch.stack(frames), torch.stack(noisy))  # rendered frames with seeded noise, 37x53
    _check(torch.rand((1, 11, 11, 3), generator=g, device=DEV), torch.rand((1, 11, 11, 3), generator=g, device=DEV))
    # a batch of 5 different kinds of image: each row equals the image on its own
    ramp = torch.linspace(0, 1, 53, device=DEV)[None, :, None].expand(37, 53, 3)
    pred = torch.stack([frames[0], ramp, torch.full((37, 53, 3), 0.5, device=DEV) + 1e-3 * torch.randn((37, 53, 3), generator=g, device=DEV),
                        0.2 + 0.2 * torch.rand((37, 53, 3), generator=g, device=DEV), (torch.rand((37, 53, 3), generator=g, device=DEV) > 0.5).float()])
    target = (pred + 0.03 * torch.randn(pred.shape, generator=g, device=DEV)).clamp(0, 1)
    batch = _check(pred, target)
    from soccernerfs_b200 import ops

    for k in range(5):
        assert torch.equal(ops.image_metrics(pred[k:k + 1], target[k:k + 1]).cpu(), batch[k:k + 1])


def test_image_metrics_rejects_small_images_and_bad_inputs():
    from ctypes import c_void_p

    from soccernerfs_b200 import _lib, ops

    small = torch.rand((1, 10, 40, 3), device=DEV)
    with pytest.raises(ValueError, match="11x11"):
        ops.image_metrics(small, small)
    with pytest.raises(ValueError):
        ops.image_metrics(torch.rand((1, 40, 10, 3), device=DEV), torch.rand((1, 40, 10, 3), device=DEV))
    out = torch.empty((1, 2), device=DEV)
    scratch = torch.empty(1 << 20, dtype=torch.uint8, device=DEV)
    with pytest.raises(RuntimeError, match="smaller than"):  # the library checks it too
        _lib.call("kp_image_metrics", _lib.ptr(small), _lib.ptr(small), 1, 10, 40, c_void_p(scratch.data_ptr()), _lib.ptr(out),
                  _lib.stream_ptr())
    with pytest.raises(TypeError):
        ops.image_metrics(small.double(), small.double())
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.image_metrics(torch.rand((1, 16, 16, 3)), torch.rand((1, 16, 16, 3)))
    with pytest.raises(ValueError):
        ops.image_metrics(torch.rand((1, 16, 16, 4), device=DEV), torch.rand((1, 16, 16, 4), device=DEV))


def test_image_metrics_bitwise_repeatable_and_graph_capturable():
    from soccernerfs_b200 import ops

    g = torch.Generator(device=DEV).manual_seed(2)
    pred = torch.rand((3, 270, 480, 3), generator=g, device=DEV)
    target = (pred + 0.05 * torch.randn(pred.shape, generator=g, device=DEV)).clamp(0, 1)
    a, b = ops.image_metrics(pred, target), ops.image_metrics(pred, target)
    assert torch.equal(a, b)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.image_metrics(pred, target)  # warm-up on the capturing stream
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = ops.image_metrics(pred, target)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, a)
    pred.copy_(target)  # new inputs, same buffers: the replay follows them
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, ops.image_metrics(pred, target)) and float((captured[:, 1] - 1).abs().max()) < 1e-5


def test_frame_renderer_device_frames_equal_host_frames():
    from soccernerfs_b200.engine.frame_renderer import FrameRenderer

    model = _tiny_model()
    cams = _eval_cameras()
    host = FrameRenderer(model, cams, chunk=200).render(1)
    for graph in (True, False):
        dev = FrameRenderer(model, cams, chunk=200, use_cuda_graph=graph).render(1, device_frames=True)
        for k in ("rgb", "depth", "accumulation"):
            assert dev[k].is_cuda and dev[k].shape == host[k].shape
            assert torch.equal(dev[k].cpu(), host[k]), (k, graph)


def _eval_setup(model, n=3, h=24, w=40):
    from soccernerfs_b200.data.datamanagers.dynamic_datamanager import DynamicDataManager, DynamicDataManagerConfig

    cams = _eval_cameras(h, w, n)
    g = torch.Generator(device=DEV).manual_seed(3)
    with torch.no_grad():
        frames = _renders(model, cams)
    images = torch.stack([(f + 0.05 * torch.randn(f.shape, generator=g, device=DEV)).clamp(0, 1) for f in frames])
    cfg = DynamicDataManagerConfig(train_num_rays_per_batch=128, eval_num_rays_per_batch=256, use_importance_sampling=False)
    dm = DynamicDataManager(cfg, cams, torch.full_like(images, 2.0), device=DEV, eval_cameras=cams, eval_images=images)
    return dm, frames, images


def test_evaluator_on_the_tiny_model():
    import random

    from soccernerfs_b200.engine.evaluator import Evaluator

    model = _tiny_model()
    dm, frames, images = _eval_setup(model)
    ev = Evaluator(model, dm)
    avg = ev.get_average_eval_image_metrics(0)
    assert list(avg) == ["psnr", "ssim", "num_rays_per_sec", "fps"] or list(avg) == ["psnr", "ssim", "lpips", "num_rays_per_sec", "fps"]
    ref = [_reference(f, t) for f, t in zip(frames, images)]
    assert abs(avg["psnr"] - sum(r[0] for r in ref) / 3) <= 1e-5 * abs(avg["psnr"]), (avg, ref)
    assert abs(avg["ssim"] - sum(r[1] for r in ref) / 3) <= 1e-5, (avg, ref)
    assert avg["num_rays_per_sec"] > 0 and avg["fps"] > 0
    again = ev.get_average_eval_image_metrics(1)
    assert again["psnr"] == avg["psnr"] and again["ssim"] == avg["ssim"]

    # next_eval draws eval pixels only (the train cache holds 2.0 everywhere), with the eval cameras' rays
    random.seed(0)
    torch.manual_seed(0)
    for step in range(3):
        rb, batch = dm.next_eval(step)
        idx = batch["indices"]
        assert idx.shape == (256, 3) and bool((idx[:, 0] < 3).all())
        assert torch.equal(batch["image"], images[idx[:, 0], idx[:, 1], idx[:, 2]])
        assert torch.equal(rb.times, dm.eval_cameras.times[idx[:, 0]])
    assert dm.eval_count == 3 and dm.train_count == 0

    outputs, loss_dict, metrics_dict = ev.get_eval_loss_dict(4)
    rb, batch = dm.next_eval(5)
    with torch.no_grad():
        own_out = model(rb)
        own_loss = model.get_loss_dict(own_out, batch, model.get_metrics_dict(own_out, batch))
    assert set(loss_dict) == set(own_loss) and "rgb_loss" in loss_dict and "psnr" in metrics_dict
    assert outputs["rgb"].shape == (256, 3)

    metrics, images_dict = ev.get_eval_image_metrics_and_images(6)
    i = metrics["image_idx"]
    assert 0 <= i < 3 and metrics["num_rays"] == 24 * 40
    assert abs(metrics["psnr"] - ref[i][0]) <= 1e-4 * abs(ref[i][0]) and abs(metrics["ssim"] - ref[i][1]) <= 1e-4
    assert images_dict["img"].shape == (24, 80, 3)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_evaluator_two_ranks_equal_one_rank():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29578", os.path.join(root, "tests", "_eval_worker.py")]
    res = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "EVAL_MULTI_OK" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]
