"""The host side of writing the eval split as images and videos: panel availability and every input error (raised before
anything is rendered), the image-to-rank assignment, the per-camera video order over ranks, and the metrics.json files
at world 1, 2 and 3."""
import json
import math
import struct
import types

import pytest
import torch

from soccernerfs_b200.engine import path_renderer as pr
from soccernerfs_b200.engine.evaluator import (Evaluator, check_eval_panels, eval_panels, eval_video_sequences, images_of_rank,
                                               metrics_document, metrics_file_name)
from tests.test_video_host import _frames, _parse_avi


def _stub_model(proposals=2):
    return types.SimpleNamespace(config=types.SimpleNamespace(num_proposal_iterations=proposals))


def test_panel_availability():
    base = ["gt", "rgb", "median_rgb", "error", "ssim", "depth", "accumulation", "prop_depth_0", "prop_depth_1"]
    assert eval_panels(_stub_model(), depth=False, regions=False) == base
    assert eval_panels(_stub_model(), depth=True, regions=False) == base + ["depth_gt", "depth_error"]
    assert eval_panels(_stub_model(), depth=True, regions=True) == base + ["depth_gt", "depth_error", "dynamic_mask"]
    assert eval_panels(_stub_model(0), depth=False, regions=True) == base[:7] + ["dynamic_mask"]


def test_panel_kinds_of_the_eval_panels():
    from soccernerfs_b200 import ops

    kinds = {n: ops.panel_kind(n) for n in eval_panels(_stub_model(), depth=True, regions=True)}
    assert kinds == {"gt": 0, "rgb": 0, "median_rgb": 0, "error": 1, "ssim": 1, "depth": 2, "accumulation": 1, "prop_depth_0": 2,
                     "prop_depth_1": 2, "depth_gt": 2, "depth_error": 1, "dynamic_mask": 1}
    assert ops.accumulation_of("depth_gt") == "depth_gt_valid" and ops.accumulation_of("depth") == "accumulation"


def test_panel_errors():
    avail = eval_panels(_stub_model(), depth=False, regions=False)
    assert check_eval_panels(avail, ("gt", "rgb", "error", "ssim"), 0.25, 0.25) == ["gt", "rgb", "error", "ssim"]
    with pytest.raises(ValueError, match="available panels.*prop_depth_1"):
        check_eval_panels(avail, ["rgb", "normals"], 0.25, 0.25)
    with pytest.raises(ValueError, match="need eval depth"):
        check_eval_panels(avail, ["depth_gt"], 0.25, 0.25)
    with pytest.raises(ValueError, match="not available"):
        check_eval_panels(avail, ["depth_error"], 0.25, 0.25)
    with pytest.raises(ValueError, match="needs regions"):
        check_eval_panels(avail, ["dynamic_mask"], 0.25, 0.25)
    with pytest.raises(ValueError, match="no panels"):
        check_eval_panels(avail, [], 0.25, 0.25)
    with pytest.raises(ValueError, match="at most 8"):
        check_eval_panels(avail, ["rgb"] * 9, 0.25, 0.25)
    for bad in (0.0, -1.0, math.inf, math.nan, True, "0.25"):
        with pytest.raises(ValueError, match="error_range"):
            check_eval_panels(avail, ["error"], bad, 0.25)
        with pytest.raises(ValueError, match="depth_error_range"):
            check_eval_panels(avail, ["error"], 0.25, bad)


def _stub_evaluator(depth=False, regions=False):
    """An Evaluator with the attributes the writers read before they render: no renderer, so any render would fail."""
    ev = Evaluator.__new__(Evaluator)
    ev.model = _stub_model()
    ev.rank, ev.world = 0, 1
    ev.depth = depth
    ev.regions = torch.zeros((3, 24, 40), dtype=torch.bool) if regions else None
    ev.renderer = None
    return ev


def test_writers_raise_before_rendering(tmp_path):
    ev = _stub_evaluator()
    out = tmp_path / "out"
    with pytest.raises(ValueError, match="available panels"):
        ev.write_eval_images(out, panels=("gt", "depth_gt"))
    with pytest.raises(ValueError, match="image_format"):
        ev.write_eval_images(out, image_format="bmp")
    with pytest.raises(ValueError, match="jpeg_quality"):
        ev.write_eval_images(out, image_format="jpeg", jpeg_quality=0)
    with pytest.raises(ValueError, match="error_range"):
        ev.write_eval_images(out, error_range=0.0)
    with pytest.raises(ValueError, match="dynamic_mask"):
        ev.write_eval_videos(out, 10.0, panels=("dynamic_mask",))
    for fps in (0.0, -5.0, math.inf, math.nan, None):
        with pytest.raises(ValueError, match="fps"):
            ev.write_eval_videos(out, fps)
    with pytest.raises(ValueError, match="jpeg_quality"):
        ev.write_eval_videos(out, 10.0, jpeg_quality=101)
    assert not out.exists()  # nothing was written
    assert check_eval_panels(eval_panels(ev.model, True, True), ["depth_gt", "depth_error", "dynamic_mask"], 1.0, 1.0)
    _stub_evaluator(depth=True, regions=True)._check_write(["depth_gt", "depth_error", "dynamic_mask"], 1.0, 1.0)


def test_image_assignment_over_ranks():
    for n in (1, 4, 7):
        for world in (1, 2, 3):
            parts = [images_of_rank(n, r, world) for r in range(world)]
            assert sorted(i for p in parts for i in p) == list(range(n))
            assert all(i % world == r for r, p in enumerate(parts) for i in p)


def test_video_sequences_per_camera_in_time_order():
    ids = torch.tensor([2, 0, 2, 0, 2, 7])
    times = torch.tensor([[0.5], [0.9], [0.1], [0.2], [0.5], [0.0]])
    seqs = eval_video_sequences(ids, times, 6)
    assert seqs == {"camera_000.avi": [3, 1], "camera_002.avi": [2, 0, 4], "camera_007.avi": [5]}  # equal times: image order
    assert eval_video_sequences(ids, None, 6) == {"camera_000.avi": [1, 3], "camera_002.avi": [0, 2, 4], "camera_007.avi": [5]}
    assert eval_video_sequences(None, times, 4) == {"eval.avi": [0, 1, 2, 3]}
    with pytest.raises(ValueError, match="camera ids"):
        eval_video_sequences(ids[:5], times, 6)
    # frame k of a video goes to rank k % world; every frame of a camera once
    for world in (1, 2, 3):
        for seq in seqs.values():
            parts = [seq[r::world] for r in range(world)]
            assert sorted(i for p in parts for i in p) == sorted(seq)
            assert all(seq.index(i) % world == r for r, p in enumerate(parts) for i in p)


def test_part_files_interleave_into_each_cameras_time_order(tmp_path):
    ids = torch.tensor([1, 1, 0, 1, 0, 1, 0])
    times = torch.tensor([0.6, 0.2, 0.3, 0.4, 0.1, 0.0, 0.9])
    seqs = eval_video_sequences(ids, times, 7)
    frames = _frames(7)  # frame i stands for eval image i
    for world in (1, 2, 3):
        for name, seq in seqs.items():
            path = tmp_path / f"w{world}_{name}"
            for r in range(world):  # what write_part writes on rank r: its share of the sequence, in order
                with open(pr.part_path(path, r), "wb") as f:
                    for i in seq[r::world]:
                        f.write(struct.pack("<I", len(frames[i])) + frames[i])
            pr.assemble_video(path, world, 10.0)
            assert _parse_avi(path)["frames"] == [frames[i] for i in seq], (world, name)


def _rows(n):
    return {i: {"psnr": 20.0 + i / 3, "ssim": 0.5 + i / 7, "psnr_dynamic": math.nan if i == 1 else 18.0 + i} for i in range(n)}


def test_metrics_files_at_world_1_2_3(tmp_path):
    assert metrics_file_name(0, 1, False) == metrics_file_name(0, 1, True) == "metrics.json"
    assert [metrics_file_name(r, 2, True) for r in range(2)] == ["metrics.json", None]
    assert [metrics_file_name(r, 3, False) for r in range(3)] == ["metrics.rank0.json", "metrics.rank1.json", "metrics.rank2.json"]
    rows = _rows(7)
    doc = metrics_document(rows, "png")
    assert [e["image"] for e in doc["images"]] == list(range(7))
    assert doc["images"][3] == {"image": 3, "file": "00003.png", "psnr": rows[3]["psnr"], "ssim": rows[3]["ssim"],
                                "psnr_dynamic": 21.0}
    assert metrics_document(rows, "jpg")["images"][6]["file"] == "00006.jpg"
    # the files round-trip every value exactly, NaN included; the ranks' files together hold the one-rank rows
    (tmp_path / "metrics.json").write_text(json.dumps(doc))
    one = json.loads((tmp_path / "metrics.json").read_text())["images"]
    for world in (2, 3):
        merged = []
        for r in range(world):
            mine = {i: rows[i] for i in images_of_rank(7, r, world)}
            path = tmp_path / metrics_file_name(r, world, False)
            path.write_text(json.dumps(metrics_document(mine, "png")))
            merged += json.loads(path.read_text())["images"]
        merged.sort(key=lambda e: e["image"])
        assert len(merged) == 7
        for a, b in zip(merged, one):
            assert a.keys() == b.keys()
            assert all(a[k] == b[k] or (math.isnan(a[k]) and math.isnan(b[k])) for k in a if k != "file")
            assert a["file"] == b["file"]
    assert math.isnan(one[1]["psnr_dynamic"]) and one[0]["psnr"] == rows[0]["psnr"]
