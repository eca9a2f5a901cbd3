"""Per-region eval metrics without a GPU: utils/image_metrics.region_psnr_ssim (the statement the kernel is tested
against), the averaging of region keys with undefined (NaN) rows, the Evaluator's key order and its independence of the
world size with the kernels replaced by CPU stand-ins, and the input errors."""
import math
import types

import pytest
import torch

from soccernerfs_b200 import ops
from soccernerfs_b200.engine import evaluator as ev
from soccernerfs_b200.utils import image_metrics

N_IMAGES, H, W = 7, 16, 20


def _pair(seed, b=2, h=H, w=W):
    g = torch.Generator().manual_seed(seed)
    pred = torch.rand((b, h, w, 3), generator=g, dtype=torch.float64)
    return pred, (pred + 0.1 * torch.randn(pred.shape, generator=g, dtype=torch.float64)).clamp(0, 1)


def _whole(pred, target):
    """psnr / ssim of each image in the model's argument order."""
    out = []
    for p, t in zip(pred, target):
        p4, t4 = torch.moveaxis(p, -1, 0)[None], torch.moveaxis(t, -1, 0)[None]
        out.append([float(image_metrics.psnr(t4, p4)), float(image_metrics.ssim(t4, p4))])
    return torch.tensor(out, dtype=torch.float64)


def test_all_true_and_all_false_masks_give_the_whole_image_metrics():
    pred, target = _pair(0)
    whole = _whole(pred, target)
    ones = torch.ones(pred.shape[:3], dtype=torch.bool)
    dyn = image_metrics.region_psnr_ssim(pred, target, ones)
    static = image_metrics.region_psnr_ssim(pred, target, torch.zeros_like(ones))
    assert dyn.dtype == torch.float64 and dyn.shape == (2, 4)
    torch.testing.assert_close(dyn[:, :2], whole, rtol=1e-13, atol=1e-13)
    torch.testing.assert_close(static[:, 2:], whole, rtol=1e-13, atol=1e-13)
    assert dyn[:, 2:].isnan().all() and static[:, :2].isnan().all()


def test_psnr_by_hand_on_12x12():
    pred = torch.zeros((1, 12, 12, 3), dtype=torch.float64)
    target = torch.full_like(pred, 0.2)
    mask = torch.zeros((1, 12, 12), dtype=torch.uint8)
    mask[0, 3:7, 2:5] = 7  # any non-zero byte is dynamic
    target[0, 3:7, 2:5] = 0.1
    out = image_metrics.region_psnr_ssim(pred, target, mask)
    assert abs(float(out[0, 0]) - 20.0) < 1e-12  # mse 0.01 over the 12 dynamic pixels
    assert abs(float(out[0, 2]) - 10 * math.log10(1 / 0.04)) < 1e-12  # mse 0.04 over the other 132


def test_empty_regions_and_border_only_masks_are_nan():
    pred, target = _pair(1, b=1, h=13, w=15)
    border = torch.zeros((1, 13, 15), dtype=torch.bool)
    border[0, :5, :] = True  # rows 0-4: no window centre (the centres are rows 5-7, columns 5-9)
    border[0, :, 10:] = True  # columns 10-14
    out = image_metrics.region_psnr_ssim(pred, target, border)
    assert not math.isnan(float(out[0, 0])) and math.isnan(float(out[0, 1]))
    assert not out[0, 2:].isnan().any()  # the static region holds every window centre
    centre = torch.zeros_like(border)
    centre[0, 6, 7] = True  # one pixel, one window centre
    out = image_metrics.region_psnr_ssim(pred, target, centre)
    full = image_metrics.ssim_map(torch.moveaxis(target[0], -1, 0)[None], torch.moveaxis(pred[0], -1, 0)[None])[0]
    assert float(out[0, 1]) == float(full[:, 1, 2].mean())
    assert float(out[0, 0]) == float(10 * torch.log10(1 / ((pred[0, 6, 7] - target[0, 6, 7]) ** 2).mean()))


def test_average_skips_undefined_regions_and_counts_images():
    nan = float("nan")
    keys = ["psnr", "ssim", "num_rays_per_sec", "fps", *ev.REGION_KEYS, "dynamic_fraction"]
    vals = {0: [30.0, 0.9, 1e6, 2.0, 25.0, 0.8, 31.0, 0.91, 0.1],
            1: [29.0, 0.8, 2e6, 4.0, nan, nan, 29.0, 0.8, 0.0],  # no dynamic pixel
            2: [28.0, 0.7, 3e6, 6.0, 24.0, nan, 28.5, 0.75, 0.01],  # dynamic pixels on the border only
            3: [27.0, 0.6, 4e6, 8.0, 21.0, 0.5, nan, nan, 1.0]}  # no static pixel
    rows = {i: dict(zip(keys, v)) for i, v in vals.items()}
    out = ev.average_region_metrics(rows, keys)
    assert list(out) == keys + ["num_images_dynamic", "num_images_static"]
    mean = lambda xs: float(torch.mean(torch.tensor(xs)))  # noqa: E731  (the reference's averaging)
    assert out["psnr"] == mean([30.0, 29.0, 28.0, 27.0]) == ev.average_metrics(rows, ["psnr"])["psnr"]
    assert out["psnr_dynamic"] == mean([25.0, 24.0, 21.0]) and out["ssim_dynamic"] == mean([0.8, 0.5])
    assert out["psnr_static"] == mean([31.0, 29.0, 28.5]) and out["ssim_static"] == mean([0.91, 0.8, 0.75])
    assert out["dynamic_fraction"] == mean([0.1, 0.0, 0.01, 1.0])
    assert out["num_images_dynamic"] == 3 and out["num_images_static"] == 3
    # NaNs travel through the all_gather rows unchanged
    packed = ev.pack_rows(rows, keys, 5)
    back = ev.unpack_rows([packed], keys)
    assert all(math.isnan(back[i][k]) == math.isnan(rows[i][k]) for i in rows for k in keys)
    assert ev.average_region_metrics(back, keys) == pytest.approx(out, nan_ok=True)
    only_static = {i: dict(rows[i], psnr_dynamic=nan, ssim_dynamic=nan) for i in rows}
    out = ev.average_region_metrics(only_static, keys)
    assert math.isnan(out["psnr_dynamic"]) and out["num_images_dynamic"] == 0


class _Cams:
    def __init__(self, n, h, w):
        self._height_host, self._width_host = [h] * n, [w] * n

    def __len__(self):
        return len(self._height_host)


def _cpu_image_metrics(pred, target):
    return _whole(pred.double(), target.double()).float()


def _cpu_image_metrics_masked(pred, target, mask):
    return image_metrics.region_psnr_ssim(pred, target, mask)


def _masks():
    m = torch.zeros((N_IMAGES, H, W), dtype=torch.bool)
    for i in range(N_IMAGES):
        m[i, 2 + i % 5:8 + i % 5, 3:3 + 2 * i] = True  # image 0: empty region
    m[3, :, :] = True  # no static pixel
    m[5] = False
    m[5, :4, :] = True  # border only
    return m


def _evaluator(rank, world, monkeypatch):
    g = torch.Generator().manual_seed(1)
    targets, renders = torch.rand((N_IMAGES, H, W, 3), generator=g), torch.rand((N_IMAGES, H, W, 3), generator=g)
    dm = types.SimpleNamespace(eval_cameras=_Cams(N_IMAGES, H, W), device=torch.device("cpu"),
                               eval_image_cache=types.SimpleNamespace(batch={"image": targets}))
    e = ev.Evaluator.__new__(ev.Evaluator)
    e.model, e.datamanager, e.rank, e.world = None, dm, rank, world
    e._lpips, e._lpips_checked = None, True
    e.regions = _masks()
    e._render_timed = lambda i: (renders[i], lambda: 0.01 * (i + 1))
    monkeypatch.setattr(ev.ops, "image_metrics", _cpu_image_metrics)
    monkeypatch.setattr(ev.ops, "image_metrics_masked", _cpu_image_metrics_masked)
    return e, renders, targets


def test_region_keys_and_independence_of_the_world_size(monkeypatch):
    one, renders, targets = _evaluator(0, 1, monkeypatch)
    ref = one.get_average_eval_image_metrics()
    assert list(ref) == ["psnr", "ssim", "num_rays_per_sec", "fps", "psnr_dynamic", "ssim_dynamic", "psnr_static",
                         "ssim_static", "dynamic_fraction", "num_images_dynamic", "num_images_static"]
    regions = image_metrics.region_psnr_ssim(renders, targets, _masks()).tolist()
    mean = lambda xs: float(torch.mean(torch.tensor([x for x in xs if not math.isnan(x)])))  # noqa: E731
    for c, k in enumerate(ev.REGION_KEYS):
        assert ref[k] == mean([r[c] for r in regions]), k
    assert ref["dynamic_fraction"] == mean((_masks().flatten(1).double().mean(1)).tolist())
    assert ref["num_images_dynamic"] == N_IMAGES - 1 and ref["num_images_static"] == N_IMAGES - 1

    for world in (2, 3):
        ranks = [_evaluator(r, world, monkeypatch)[0] for r in range(world)]
        keys = ranks[0]._keys(torch.device("cpu"))
        per_rank = [e._rank_rows(ev.images_of_rank(N_IMAGES, e.rank, world)) for e in ranks]
        packed = [ev.pack_rows(rows, keys, -(-N_IMAGES // world)) for rows in per_rank]
        for e in ranks:
            e._rank_rows = lambda mine, e=e: per_rank[e.rank]
            e._all_gather = lambda rows, keys, n: ev.unpack_rows(packed, keys)
            got = e.get_average_eval_image_metrics()
            assert list(got) == list(ref), world
            assert all(got[k] == ref[k] or (math.isnan(got[k]) and math.isnan(ref[k])) for k in ref), (world, got, ref)


def test_without_regions_the_keys_are_unchanged(monkeypatch):
    e, _, _ = _evaluator(0, 1, monkeypatch)
    e.regions = None
    assert list(e.get_average_eval_image_metrics()) == ["psnr", "ssim", "num_rays_per_sec", "fps"]


def test_input_errors():
    images = torch.rand((4, 12, 12, 3))
    with pytest.raises(ValueError, match="no ids"):
        ev.median_dynamic_masks(images, None)
    with pytest.raises(ValueError, match="camera 1 has 1 image"):
        ev.median_dynamic_masks(images, torch.tensor([0, 0, 0, 1]))
    with pytest.raises(ValueError, match="3 camera ids for 4 images"):
        ev.median_dynamic_masks(images, torch.tensor([0, 0, 0]))

    dm = types.SimpleNamespace(eval_cameras=types.SimpleNamespace(ids=None), eval_image_cache=types.SimpleNamespace(
        batch={"image": images}))
    with pytest.raises(ValueError, match="regions must be None"):
        ev.Evaluator(None, dm, regions="boxes")
    with pytest.raises(ValueError, match=r"\[B_eval,H,W\]"):
        ev.Evaluator(None, dm, regions=torch.ones((4, 12, 11), dtype=torch.bool))
    with pytest.raises(ValueError, match="no ids"):
        ev.Evaluator(None, dm, regions="median")

    pred = torch.rand((2, 12, 12, 3))
    with pytest.raises(ValueError):
        image_metrics.region_psnr_ssim(pred, pred, torch.ones((2, 12, 13)))
    with pytest.raises(ValueError, match="11x11"):
        image_metrics.region_psnr_ssim(pred[:, :10], pred[:, :10], torch.ones((2, 10, 12)))
    with pytest.raises(ValueError, match="mask must be"):
        ops.image_metrics_masked(pred, pred, torch.ones((2, 12, 11), dtype=torch.bool))
    with pytest.raises(ValueError, match="both be"):
        ops.image_metrics_masked(pred, pred[:1], torch.ones((2, 12, 12), dtype=torch.bool))
    with pytest.raises(TypeError):
        ops.image_metrics_masked(pred, pred, torch.ones((2, 12, 12)))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.image_metrics_masked(pred, pred, torch.ones((2, 12, 12), dtype=torch.bool))
