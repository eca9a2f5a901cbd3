"""Host logic of engine/evaluator.py without a GPU: which images a rank renders, how per-image rows travel through the
all_gather and are averaged (in image order, independent of the world size), and the ns-eval report shape.  The render
and the metric kernel are replaced by CPU stand-ins."""
import json
import types

import torch

from soccernerfs_b200.engine import evaluator as ev
from soccernerfs_b200.utils import image_metrics

N_IMAGES, H, W = 7, 16, 20


class _Cams:
    def __init__(self, n, h, w):
        self._height_host, self._width_host = [h] * n, [w] * n

    def __len__(self):
        return len(self._height_host)


def _images(seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand((N_IMAGES, H, W, 3), generator=g)


def _cpu_image_metrics(pred, target):
    """ops.image_metrics on the CPU: the torch restatement image by image."""
    out = []
    for p, t in zip(pred, target):
        p4, t4 = torch.moveaxis(p, -1, 0)[None], torch.moveaxis(t, -1, 0)[None]
        out.append([float(image_metrics.psnr(t4, p4)), float(image_metrics.ssim(t4, p4))])
    return torch.tensor(out)


def _evaluator(rank, world, monkeypatch):
    """An Evaluator over a stub datamanager whose renders are fixed 'rendered' frames with per-image render times."""
    targets, renders = _images(1), _images(2)
    dm = types.SimpleNamespace(eval_cameras=_Cams(N_IMAGES, H, W), device=torch.device("cpu"),
                               eval_image_cache=types.SimpleNamespace(batch={"image": targets}))
    e = ev.Evaluator.__new__(ev.Evaluator)
    e.model, e.datamanager, e.rank, e.world = None, dm, rank, world
    e._lpips, e._lpips_checked = None, True
    e.rendered = []
    e._render_timed = lambda i: (e.rendered.append(i) or renders[i], lambda: 0.01 * (i + 1))
    monkeypatch.setattr(ev.ops, "image_metrics", _cpu_image_metrics)
    return e


def test_images_of_rank_cover_every_image_once():
    for n in (0, 1, 5, 8, 9):
        for world in (1, 2, 3, 8):
            parts = [ev.images_of_rank(n, r, world) for r in range(world)]
            assert sorted(i for p in parts for i in p) == list(range(n))
            assert all(i % world == r for r, p in enumerate(parts) for i in p)


def test_average_is_independent_of_world_size(monkeypatch):
    one = _evaluator(0, 1, monkeypatch)
    ref = one.get_average_eval_image_metrics()
    assert one.rendered == list(range(N_IMAGES))
    assert list(ref) == ["psnr", "ssim", "num_rays_per_sec", "fps"]
    # the reference's averaging of its per-image dicts, in image order
    rows = [_cpu_image_metrics(_images(2)[i:i + 1], _images(1)[i:i + 1])[0].tolist() for i in range(N_IMAGES)]
    assert ref["psnr"] == float(torch.mean(torch.tensor([r[0] for r in rows])))
    assert ref["ssim"] == float(torch.mean(torch.tensor([r[1] for r in rows])))
    rays = [H * W / (0.01 * (i + 1)) for i in range(N_IMAGES)]
    assert ref["num_rays_per_sec"] == float(torch.mean(torch.tensor(rays)))
    assert ref["fps"] == float(torch.mean(torch.tensor([r / (H * W) for r in rays])))

    for world in (2, 3, 8):
        ranks = [_evaluator(r, world, monkeypatch) for r in range(world)]
        keys = ranks[0]._keys(torch.device("cpu"))
        per_rank = [e._rank_rows(ev.images_of_rank(N_IMAGES, e.rank, world)) for e in ranks]
        n_rows = -(-N_IMAGES // world)
        packed = [ev.pack_rows(rows, keys, n_rows) for rows in per_rank]
        assert all(p.shape == (n_rows, 1 + len(keys)) for p in packed)
        for e in ranks:
            e._rank_rows = lambda mine, e=e: per_rank[e.rank]
            e._all_gather = lambda rows, keys, n: ev.unpack_rows(packed, keys)
            assert e.get_average_eval_image_metrics() == ref, world  # bit for bit, on every rank


def test_eval_report_shape():
    res = {"psnr": 30.5, "ssim": 0.91, "num_rays_per_sec": 1.0e7, "fps": 4.8}
    rep = ev.eval_report(res, "soccer", "outputs/soccer/step-030000.ckpt")
    assert set(rep) == {"experiment_name", "method_name", "checkpoint", "results"}
    assert rep["method_name"] == "k-planes" and rep["results"] == res
    assert json.loads(json.dumps(rep)) == rep

