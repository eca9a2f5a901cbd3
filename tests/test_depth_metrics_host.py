"""Eval depth metrics without a GPU: utils/image_metrics.depth_metrics (the statement the kernel is tested against) on
hand-computed cases, the averaging of depth keys with undefined (NaN) rows, the Evaluator's key order and its
independence of the world size with the kernels replaced by CPU stand-ins, and the input errors."""
import math
import types

import pytest
import torch

from soccernerfs_b200 import ops
from soccernerfs_b200.engine import evaluator as ev
from soccernerfs_b200.utils import image_metrics

N_IMAGES, H, W = 7, 16, 20
NAN = float("nan")


def test_thresholds_are_exact_and_strict():
    # g = 1 and p = 1.25^k (or g = 1.25^k and p = 1): the ratio is exactly on the threshold, which is not "below" it
    pred = torch.tensor([[[1.25, 1.0, 1.5625, 1.953125, 1.0, 2.0]]], dtype=torch.float32)
    gt = torch.tensor([[[1.0, 1.25, 1.0, 1.0, 1.953125, 1.0]]], dtype=torch.float32)
    row = image_metrics.depth_metrics(pred, gt)[0, 0]
    assert row.dtype == torch.float64 and row[0] == 6
    # ratios 1.25, 1.25, 1.5625, 1.953125, 1.953125, 2: < 1.25 none, < 1.5625 two, < 1.953125 three
    assert row[5:].tolist() == [0.0, 2 / 6, 3 / 6]
    p, g = pred.double()[0, 0], gt.double()[0, 0]
    e = p - g
    assert row[1] == (e.abs() / g).mean() and row[2] == (e * e / g).mean()
    assert row[3] == (e * e).mean().sqrt() and row[4] == ((p.log() - g.log()) ** 2).mean().sqrt()


def test_by_hand_with_directions_norm_and_the_clamp():
    gt = torch.tensor([[[2.0, 4.0, 1.0]]], dtype=torch.float32)
    norm = torch.tensor([[[1.5, 0.5, 3.0]]], dtype=torch.float32)
    pred = torch.tensor([[[3.0, 2.5, -1.0]]], dtype=torch.float32)  # g = 3, 2, 3; the last prediction clamps to 1e-6
    row = image_metrics.depth_metrics(pred, gt, norm[..., None])[0, 0].tolist()  # [B,H,W,1] is accepted too
    p, g = [3.0, 2.5, 1e-6], [3.0, 2.0, 3.0]
    e = [a - b for a, b in zip(p, g)]
    assert row[0] == 3
    assert row[1] == pytest.approx(sum(abs(x) / y for x, y in zip(e, g)) / 3, rel=1e-14)
    assert row[2] == pytest.approx(sum(x * x / y for x, y in zip(e, g)) / 3, rel=1e-14)
    assert row[3] == pytest.approx(math.sqrt(sum(x * x for x in e) / 3), rel=1e-14)
    assert row[4] == pytest.approx(math.sqrt(sum((math.log(a) - math.log(b)) ** 2 for a, b in zip(p, g)) / 3), rel=1e-14)
    assert row[5:] == [1 / 3, 2 / 3, 2 / 3]  # ratios 1, 1.25 (not below 1.25) and 3e6
    # the ground truth is gt * directions_norm in fp32, before any double arithmetic
    assert torch.equal(image_metrics.depth_metrics(pred, gt, norm), image_metrics.depth_metrics(pred, gt * norm))


def test_invalid_ground_truth_pixels_are_left_out():
    gt = torch.tensor([[[2.0, 0.0, -1.0, math.inf, NAN, -math.inf, 4.0]]])
    pred = torch.tensor([[[2.2, 1.0, 1.0, 1.0, 1.0, 1.0, 3.0]]])
    row = image_metrics.depth_metrics(pred, gt)[0, 0]
    assert torch.equal(row, image_metrics.depth_metrics(pred[..., [0, 6]], gt[..., [0, 6]])[0, 0])
    assert row[0] == 2
    norm = torch.tensor([[[1.0, 1.0, 1.0, 1.0, 1.0, 1.0, math.inf]]])  # the product becomes inf: invalid too
    assert image_metrics.depth_metrics(pred, gt, norm)[0, 0, 0] == 1


def test_regions_and_empty_regions():
    g = torch.Generator().manual_seed(0)
    pred = 1 + 4 * torch.rand((3, 6, 7), generator=g)
    gt = pred * (1 + 0.3 * torch.randn(pred.shape, generator=g)).clamp_min(0.05)
    gt[1] = 0  # no valid pixel anywhere
    mask = torch.rand(pred.shape, generator=g) < 0.4
    mask[2] = True  # no static pixel
    out = image_metrics.depth_metrics(pred, gt, mask=mask.to(torch.uint8) * 9)
    assert out.shape == (3, 3, 8)
    torch.testing.assert_close(out[:, :1], image_metrics.depth_metrics(pred, gt), rtol=0, atol=0, equal_nan=True)
    assert out[1, :, 0].tolist() == [0, 0, 0] and out[1, :, 1:].isnan().all()
    assert out[2, 2, 0] == 0 and out[2, 2, 1:].isnan().all() and torch.equal(out[2, 1], out[2, 0])
    sel = mask[0]
    assert torch.equal(out[0, 1], image_metrics.depth_metrics(pred[0][sel][None, None], gt[0][sel][None, None])[0, 0])
    assert torch.equal(out[0, 2], image_metrics.depth_metrics(pred[0][~sel][None, None], gt[0][~sel][None, None])[0, 0])
    assert out[0, 1, 0] + out[0, 2, 0] == out[0, 0, 0]


def test_average_skips_undefined_images_and_counts_them():
    keys = ev.depth_row_keys(True)
    assert keys[:7] == list(ev.DEPTH_KEYS) and keys[7] == "depth_abs_rel_dynamic" and keys[-1] == "depth_delta3_static"
    rows = {}
    for i in range(4):
        vals = [0.1 * (i + 1) + 0.01 * c for c in range(21)]
        if i == 1:
            vals[7:14] = [NAN] * 7  # no valid dynamic pixel
        if i == 3:
            vals = [NAN] * 21  # no valid pixel at all
        rows[i] = dict(zip(keys, vals))
    out = ev.average_depth_metrics(rows, True)
    assert list(out) == (list(ev.DEPTH_KEYS) + ["num_images_depth"] + keys[7:]
                         + ["num_images_depth_dynamic", "num_images_depth_static"])
    mean = lambda xs: float(torch.mean(torch.tensor(xs)))  # noqa: E731  (the reference's averaging)
    assert out["depth_abs_rel"] == mean([rows[i]["depth_abs_rel"] for i in (0, 1, 2)])
    assert out["depth_rmse_dynamic"] == mean([rows[i]["depth_rmse_dynamic"] for i in (0, 2)])
    assert out["depth_delta3_static"] == mean([rows[i]["depth_delta3_static"] for i in (0, 1, 2)])
    assert (out["num_images_depth"], out["num_images_depth_dynamic"], out["num_images_depth_static"]) == (3, 2, 3)
    plain = ev.average_depth_metrics({i: {k: rows[i][k] for k in ev.DEPTH_KEYS} for i in rows}, False)
    assert list(plain) == list(ev.DEPTH_KEYS) + ["num_images_depth"]
    assert all(plain[k] == out[k] for k in plain)
    none = ev.average_depth_metrics({0: rows[3]}, False)
    assert math.isnan(none["depth_abs_rel"]) and none["num_images_depth"] == 0


class _Cams:
    def __init__(self, n, h, w):
        self._height_host, self._width_host = [h] * n, [w] * n

    def __len__(self):
        return len(self._height_host)


def _cpu_image_metrics(pred, target):
    return torch.stack([torch.stack([image_metrics.psnr(t, p), image_metrics.ssim(t, p)]) for p, t in
                        zip(torch.moveaxis(pred.double(), -1, 1)[:, None], torch.moveaxis(target.double(), -1, 1)[:, None])])


def _masks():
    m = torch.zeros((N_IMAGES, H, W), dtype=torch.bool)
    for i in range(N_IMAGES):
        m[i, 2 + i % 5:8 + i % 5, 3:3 + 2 * i] = True  # image 0: empty region
    m[3, :, :] = True  # no static pixel
    return m


def _evaluator(rank, world, monkeypatch, regions, euclidean=False):
    g = torch.Generator().manual_seed(1)
    targets, renders = torch.rand((N_IMAGES, H, W, 3), generator=g), torch.rand((N_IMAGES, H, W, 3), generator=g)
    frames = 1 + 3 * torch.rand((N_IMAGES, H, W, 1), generator=g)
    norms = 1 + 0.2 * torch.rand((N_IMAGES, H, W, 1), generator=g)
    gt = frames / norms * (1 + 0.2 * torch.randn(frames.shape, generator=g))
    gt[2] = 0  # no valid pixel
    gt[4, :6] = math.inf  # sky
    dm = types.SimpleNamespace(eval_cameras=_Cams(N_IMAGES, H, W), device=torch.device("cpu"),
                               eval_image_cache=types.SimpleNamespace(batch={"image": targets, "depth_image": gt}))
    e = ev.Evaluator.__new__(ev.Evaluator)
    e.model, e.datamanager, e.rank, e.world = None, dm, rank, world
    e._lpips, e._lpips_checked = None, True
    e.regions = _masks() if regions else None
    e.depth = True
    e._render_timed = lambda i, depth=False: ((renders[i], lambda: 0.01 * (i + 1))
                                              + ((frames[i], None if euclidean else norms[i]) if depth else ()))
    monkeypatch.setattr(ev.ops, "image_metrics", _cpu_image_metrics)
    monkeypatch.setattr(ev.ops, "image_metrics_masked", image_metrics.region_psnr_ssim)
    monkeypatch.setattr(ev.ops, "depth_metrics", image_metrics.depth_metrics)
    return e, (frames, gt, norms)


@pytest.mark.parametrize("regions", [False, True])
def test_depth_keys_and_independence_of_the_world_size(monkeypatch, regions):
    one, (depth, gt, norms) = _evaluator(0, 1, monkeypatch, regions)
    ref = one.get_average_eval_image_metrics()
    colour = ["psnr", "ssim", "num_rays_per_sec", "fps"]
    if regions:
        colour += list(ev.REGION_KEYS) + ["dynamic_fraction", "num_images_dynamic", "num_images_static"]
    depth_keys = list(ev.DEPTH_KEYS) + ["num_images_depth"]
    if regions:
        depth_keys += ev.depth_row_keys(True)[7:] + ["num_images_depth_dynamic", "num_images_depth_static"]
    assert list(ref) == colour + depth_keys

    rows = image_metrics.depth_metrics(depth, gt, norms, _masks() if regions else None)
    mean = lambda xs: float(torch.mean(torch.tensor([x for x in xs if not math.isnan(x)])))  # noqa: E731
    for r, s in enumerate(("", "_dynamic", "_static")[:3 if regions else 1]):
        for c, k in enumerate(ev.DEPTH_KEYS):
            assert ref[k + s] == mean(rows[:, r, c + 1].tolist()), k + s
        assert ref["num_images_depth" + s] == int((rows[:, r, 0] > 0).sum())
    assert ref["num_images_depth"] == N_IMAGES - 1
    if regions:
        assert ref["num_images_depth_dynamic"] == N_IMAGES - 2 and ref["num_images_depth_static"] == N_IMAGES - 2

    for world in (2, 3):
        ranks = [_evaluator(r, world, monkeypatch, regions)[0] for r in range(world)]
        keys = ranks[0]._keys(torch.device("cpu"))
        per_rank = [e._rank_rows(ev.images_of_rank(N_IMAGES, e.rank, world)) for e in ranks]
        packed = [ev.pack_rows(rows, keys, -(-N_IMAGES // world)) for rows in per_rank]
        for e in ranks:
            e._rank_rows = lambda mine, e=e: per_rank[e.rank]
            e._all_gather = lambda rows, keys, n: ev.unpack_rows(packed, keys)
            got = e.get_average_eval_image_metrics()
            assert list(got) == list(ref), world
            assert all(got[k] == ref[k] or (math.isnan(got[k]) and math.isnan(ref[k])) for k in ref), (world, got, ref)


def test_euclidean_ground_truth_is_compared_as_is(monkeypatch):
    e, (depth, gt, _) = _evaluator(0, 1, monkeypatch, False, euclidean=True)
    got = e.get_average_eval_image_metrics()
    rows = image_metrics.depth_metrics(depth, gt)
    assert got["depth_rmse"] == float(torch.mean(torch.tensor([x for x in rows[:, 0, 3].tolist() if not math.isnan(x)])))


def test_without_eval_depth_the_keys_are_unchanged(monkeypatch):
    e, _ = _evaluator(0, 1, monkeypatch, True)
    e.depth = False
    assert list(e.get_average_eval_image_metrics()) == ["psnr", "ssim", "num_rays_per_sec", "fps", *ev.REGION_KEYS,
                                                        "dynamic_fraction", "num_images_dynamic", "num_images_static"]


def test_input_errors():
    from soccernerfs_b200.data.datamanagers.dynamic_datamanager import DynamicDataManager, DynamicDataManagerConfig

    cfg = DynamicDataManagerConfig(use_importance_sampling=False)
    images = torch.rand((3, 8, 10, 3))
    for bad in (torch.ones((3, 8, 10)), torch.ones((3, 8, 10, 3)), torch.ones((2, 8, 10, 1)), torch.ones((3, 10, 8, 1))):
        with pytest.raises(ValueError, match=r"depth_image'\] must be \[B_eval,H,W,1\]"):
            DynamicDataManager(cfg, None, images, device="cpu", eval_cameras=object(), eval_images=images,
                               eval_extras={"depth_image": bad})
    with pytest.raises(ValueError, match="eval_extras needs the eval split"):
        DynamicDataManager(cfg, None, images, device="cpu", eval_extras={"depth_image": torch.ones((3, 8, 10, 1))})

    d = torch.rand((2, 5, 6))
    with pytest.raises(ValueError):
        image_metrics.depth_metrics(d, d[:, :4])
    with pytest.raises(ValueError):
        image_metrics.depth_metrics(d, d, mask=torch.ones((2, 5, 5), dtype=torch.bool))
    with pytest.raises(ValueError, match="gt must be"):
        ops.depth_metrics(d, d[..., None].expand(2, 5, 6, 2))
    with pytest.raises(ValueError, match="one shape"):
        ops.depth_metrics(d, d, d[:1])
    with pytest.raises(ValueError, match="mask must be"):
        ops.depth_metrics(d, d, mask=torch.ones((2, 5, 5), dtype=torch.bool))
    with pytest.raises(ValueError, match="no pixel"):
        ops.depth_metrics(d[:, :0], d[:, :0])
    with pytest.raises(TypeError):
        ops.depth_metrics(d.double(), d.double())
    with pytest.raises(TypeError):
        ops.depth_metrics(d, d, mask=torch.ones((2, 5, 6), dtype=torch.int32))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.depth_metrics(d, d, d[..., None], torch.ones((2, 5, 6), dtype=torch.bool))
