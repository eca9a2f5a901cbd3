#!/usr/bin/env python
"""bench_eval.py -- evaluation of a trained scene on B200s: Evaluator.get_average_eval_image_metrics over 8 eval images at
1920x1080 rendered from the 32x field (bench.py's cfg3 model, the BASELINE config-5 workload), and kp_image_metrics against
the torch restatement of PSNR + SSIM (utils/image_metrics.py) on the same frames and the same device.

    python scripts/bench_eval.py                                                       # 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 scripts/bench_eval.py   # 8 GPUs (images i % 8 == rank)
    python scripts/bench_eval.py --regions        # also the per-region metrics, the median masks, Evaluator(regions="median")
    python scripts/bench_eval.py --depth          # also the depth metrics (kp_depth_metrics) and the Evaluator with eval depth
    python scripts/bench_eval.py --write-images   # also the error maps (kp_eval_maps) and the eval image / video writers

Prints one JSON line (rank 0).  The eval targets are the model's own frames plus seeded noise: the metric values are
not a quality statement, the times are the point.  Kernel timing: CUDA events around each pass, after warm-up, with a
512 MB buffer written between passes so neither pass reads its frames from L2 (126 MB).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def card_info(index: int) -> dict:
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (p.strip() for p in out.split(","))
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as exc:  # the device name from torch is still recorded
        return {"name": torch.cuda.get_device_name(index), "power_limit": f"unknown ({exc})"}


def eval_cameras(n: int, h: int, w: int, dev):
    """bench.py's eval_leg camera path: a short arc of the broadcast ring, looking at the origin."""
    from soccernerfs_b200.cameras.cameras import Cameras

    ang = torch.linspace(0.0, 1.0, n) * 0.6
    pos = torch.stack([torch.cos(ang), torch.sin(ang), torch.full_like(ang, 0.35)], dim=-1)
    fwd = -pos / pos.norm(dim=-1, keepdim=True)
    right = torch.cross(fwd, torch.tensor([0.0, 0.0, 1.0]).expand_as(fwd), dim=-1)
    right = right / right.norm(dim=-1, keepdim=True)
    up = torch.cross(right, fwd, dim=-1)
    c2w = torch.cat([torch.stack([right, up, -fwd], dim=-1), pos[..., None]], dim=-1)
    return Cameras(c2w.to(dev), 1600.0, 1600.0, w / 2, h / 2, w, h, times=torch.linspace(0, 1, n)[:, None].to(dev))


def kernel_vs_torch(pred, target, reps: int) -> dict:
    """Median ms of ops.image_metrics on the batch vs image_metrics.psnr + ssim image by image (as
    get_image_metrics_and_images calls them), with L2 overwritten before every pass."""
    from soccernerfs_b200 import ops
    from soccernerfs_b200.utils import image_metrics

    flush = torch.empty(512 * 2**20 // 4, dtype=torch.float32, device=pred.device)
    p4 = [torch.moveaxis(p, -1, 0)[None] for p in pred]
    t4 = [torch.moveaxis(t, -1, 0)[None] for t in target]

    def torch_pass():
        return [(image_metrics.psnr(t, p), image_metrics.ssim(t, p)) for p, t in zip(p4, t4)]

    def timed(fn):
        times = []
        for _ in range(reps):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        return sorted(times)[len(times) // 2], times

    for _ in range(3):
        ops.image_metrics(pred, target)
        torch_pass()
    torch.cuda.synchronize()
    ours = ops.image_metrics(pred, target).cpu()
    ref = torch.tensor([[float(a), float(b)] for a, b in torch_pass()])
    k_ms, k_all = timed(lambda: ops.image_metrics(pred, target))
    t_ms, t_all = timed(torch_pass)
    b, h, w = pred.shape[:3]
    bytes_read = 2 * b * h * w * 3 * 4 * 2  # both images, read by the stats pass and by the SSIM pass
    return {"images": b, "hw": [h, w], "kp_image_metrics_ms": k_ms, "torch_psnr_ssim_ms": t_ms, "speedup": t_ms / k_ms,
            "kp_ms_all": k_all, "torch_ms_all": t_all, "kp_bytes_read_min": bytes_read,
            "kp_effective_gbs": bytes_read / (k_ms * 1e-3) / 1e9,
            "torch_tf32_conv": bool(torch.backends.cudnn.allow_tf32),
            "max_abs_diff_psnr": float((ours[:, 0] - ref[:, 0]).abs().max()),
            "max_abs_diff_ssim": float((ours[:, 1] - ref[:, 1]).abs().max()), "l2_flush": "512 MB written before every pass"}


def regions_timing(pred, target, cam_ids, reps: int) -> dict:
    """--regions: median ms of ops.image_metrics_masked on the batch against ops.image_metrics and the torch
    restatement (region_psnr_ssim, fp32), with L2 overwritten before every pass; and of median_dynamic_masks."""
    from soccernerfs_b200 import ops
    from soccernerfs_b200.engine.evaluator import median_dynamic_masks
    from soccernerfs_b200.utils import image_metrics

    flush = torch.empty(512 * 2**20 // 4, dtype=torch.float32, device=pred.device)

    def timed(fn):
        for _ in range(3):
            fn()
        times = []
        for _ in range(reps):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        return sorted(times)[len(times) // 2], times

    mask = median_dynamic_masks(target, cam_ids)
    ours = ops.image_metrics_masked(pred, target, mask).cpu()
    ref = image_metrics.region_psnr_ssim(pred, target, mask).cpu()
    whole = ops.image_metrics(pred, target).cpu()
    m_ms, m_all = timed(lambda: ops.image_metrics_masked(pred, target, mask))
    k_ms, k_all = timed(lambda: ops.image_metrics(pred, target))
    t_ms, _ = timed(lambda: image_metrics.region_psnr_ssim(pred, target, mask))
    d_ms, d_all = timed(lambda: median_dynamic_masks(target, cam_ids))
    ok = ~ref.isnan()
    return {"kp_image_metrics_masked_ms": m_ms, "kp_image_metrics_ms": k_ms, "masked_over_unmasked": m_ms / k_ms,
            "torch_region_psnr_ssim_ms": t_ms, "median_dynamic_masks_ms": d_ms, "masked_ms_all": m_all,
            "unmasked_ms_all": k_all, "median_masks_ms_all": d_all,
            "dynamic_fraction": float(mask.float().mean()), "max_abs_diff_vs_torch": float((ours - ref).abs()[ok].max()),
            "nan_pattern_equal": bool(torch.equal(ours.isnan(), ref.isnan())),
            "whole": whole.tolist(), "regions": ours.tolist(), "l2_flush": "512 MB written before every pass"}


def depth_timing(depth, gt, norms, mask, reps: int) -> dict:
    """--depth: median ms of ops.depth_metrics on the batch against the torch restatement (utils.image_metrics
    .depth_metrics, float64 terms) and of the masked call against the unmasked one, with L2 overwritten before every
    pass."""
    from soccernerfs_b200 import ops
    from soccernerfs_b200.utils import image_metrics

    flush = torch.empty(512 * 2**20 // 4, dtype=torch.float32, device=depth.device)

    def timed(fn):
        for _ in range(3):
            fn()
        times = []
        for _ in range(reps):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        return sorted(times)[len(times) // 2], times

    ours, ref = ops.depth_metrics(depth, gt, norms, mask).cpu(), image_metrics.depth_metrics(depth, gt, norms, mask).cpu()
    k_ms, k_all = timed(lambda: ops.depth_metrics(depth, gt, norms))
    m_ms, m_all = timed(lambda: ops.depth_metrics(depth, gt, norms, mask))
    t_ms, _ = timed(lambda: image_metrics.depth_metrics(depth, gt, norms))
    ok = ~ref.isnan()
    rel = ((ours - ref).abs() / ref.abs())[..., 1:5][ok[..., 1:5]]
    bytes_read = depth.numel() * 4 * 3  # pred, ground truth, directions_norm
    return {"kp_depth_metrics_ms": k_ms, "kp_depth_metrics_masked_ms": m_ms, "masked_over_unmasked": m_ms / k_ms,
            "torch_depth_metrics_ms": t_ms, "kp_ms_all": k_all, "masked_ms_all": m_all, "kp_bytes_read_min": bytes_read,
            "kp_effective_gbs": bytes_read / (k_ms * 1e-3) / 1e9, "dynamic_fraction": float(mask.float().mean()),
            "valid_fraction": float(ours[:, 0, 0].sum() / depth[0].numel() / depth.shape[0]),
            "counts_and_deltas_equal_torch": bool(torch.equal(ours[..., [0, 5, 6, 7]].nan_to_num(), ref[..., [0, 5, 6, 7]].nan_to_num())),
            "max_rel_diff_sums_vs_torch": float(rel.max()), "rows": ours.tolist(), "l2_flush": "512 MB written before every pass"}


def maps_timing(pred, target, reps: int) -> dict:
    """--write-images: median ms of ops.eval_maps on the batch against its torch restatement (fp32: the channel-mean
    error and utils.image_metrics.ssim_map image by image), with L2 overwritten before every pass."""
    from soccernerfs_b200 import ops
    from soccernerfs_b200.utils import image_metrics

    flush = torch.empty(512 * 2**20 // 4, dtype=torch.float32, device=pred.device)
    p4 = [torch.moveaxis(p, -1, 0)[None] for p in pred]
    t4 = [torch.moveaxis(t, -1, 0)[None] for t in target]

    def torch_pass():
        return (pred - target).abs().mean(-1), [image_metrics.ssim_map(t, p)[0].mean(0) for p, t in zip(p4, t4)]

    def timed(fn):
        for _ in range(3):
            fn()
        times = []
        for _ in range(reps):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        return sorted(times)[len(times) // 2], times

    ours = ops.eval_maps(pred, target)
    err, ssim = torch_pass()
    k_ms, k_all = timed(lambda: ops.eval_maps(pred, target))
    t_ms, _ = timed(torch_pass)
    b, h, w = pred.shape[:3]
    bytes_moved = 2 * b * h * w * 3 * 4 * 2 + 2 * b * h * w * 4  # both images read twice (min/max, map), two maps written
    return {"kp_eval_maps_ms": k_ms, "torch_maps_ms": t_ms, "speedup": t_ms / k_ms, "kp_ms_all": k_all,
            "kp_bytes_moved_min": bytes_moved, "kp_effective_gbs": bytes_moved / (k_ms * 1e-3) / 1e9,
            "max_abs_diff_error_vs_torch": float((ours["error"] - err).abs().max()),
            "max_abs_diff_ssim_vs_torch_fp32": float(max((ours["ssim"][k, 5:h - 5, 5:w - 5] - s).abs().max() for k, s in enumerate(ssim))),
            "l2_flush": "512 MB written before every pass"}


def write_timing(evaluator, n_images: int, repeats: int) -> dict:
    """--write-images: seconds per image of write_eval_images (PNG and JPEG) and write_eval_videos, each alternated with
    get_average_eval_image_metrics in the same run, into a temporary directory."""
    import shutil
    import tempfile

    out = tempfile.mkdtemp(prefix="bench_eval_images_")
    jobs = {"metrics": lambda r: evaluator.get_average_eval_image_metrics(r),
            "images_png": lambda r: evaluator.write_eval_images(os.path.join(out, "png")),
            "images_jpeg": lambda r: evaluator.write_eval_images(os.path.join(out, "jpeg"), image_format="jpeg"),
            "videos": lambda r: evaluator.write_eval_videos(os.path.join(out, "video"), 25.0)}
    try:
        for fn in jobs.values():  # warm-up
            fn(0)
        times = {k: [] for k in jobs}
        for r in range(repeats):
            for k, fn in jobs.items():
                if evaluator.world > 1:
                    torch.distributed.barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(r + 1)  # every writer ends once its files are written
                torch.cuda.synchronize()
                times[k].append((time.perf_counter() - t0) / n_images)
        sizes = {k: sum(os.path.getsize(os.path.join(out, k, f)) for f in os.listdir(os.path.join(out, k))) for k in ("png", "jpeg", "video")}
    finally:
        shutil.rmtree(out)
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    return {"seconds_per_image": med, "seconds_per_image_all": times, "bytes_written": sizes,
            "panels": ["gt", "rgb", "error", "ssim"], "overhead_over_metrics": {k: med[k] / med["metrics"] for k in med}}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=8)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--repeats", type=int, default=3, help="timed calls of get_average_eval_image_metrics")
    ap.add_argument("--kernel-reps", type=int, default=20)
    ap.add_argument("--out", help="also write the JSON result to this file")
    ap.add_argument("--regions", action="store_true",
                    help="also time the per-region metrics (kp_image_metrics_masked, median_dynamic_masks) and the "
                         'Evaluator with regions="median"')
    ap.add_argument("--depth", action="store_true",
                    help="also time the depth metrics (kp_depth_metrics against torch, masked against unmasked) and the "
                         "Evaluator with eval depth against the one without")
    ap.add_argument("--write-images", action="store_true",
                    help="also time the eval error maps (kp_eval_maps against torch) and writing the eval split as PNG, "
                         "JPEG and video (write_eval_images / write_eval_videos) against get_average_eval_image_metrics")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval.py measures on a CUDA device; none is visible")

    import bench
    from soccernerfs_b200.data.datamanagers.dynamic_datamanager import DynamicDataManager, DynamicDataManagerConfig
    from soccernerfs_b200.engine.evaluator import Evaluator

    rank, world, local = bench._dist_setup()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    model = bench.build_model("cfg3", dev)
    model.eval()
    cams = eval_cameras(args.images, args.height, args.width, dev)
    gen = torch.Generator(device=dev).manual_seed(7)
    renders, frames, geometry = [], [], []
    with torch.no_grad():
        from soccernerfs_b200.engine.frame_renderer import FrameRenderer

        renderer = FrameRenderer(model, cams, outputs=("rgb", "depth", "accumulation", "directions_norm") if args.depth
                                 else ("rgb", "depth", "accumulation"))
        for i in range(args.images):  # every rank builds the same targets (same model, same seed)
            out = renderer.render(i, device_frames=True)
            f = out["rgb"]
            renders.append(f)
            frames.append((f + 0.03 * torch.randn(f.shape, generator=gen, device=dev)).clamp(0, 1))
            if args.depth:
                geometry.append((out["depth"], out["accumulation"], out["directions_norm"]))
        del renderer
    targets = torch.stack(frames)
    cfg = DynamicDataManagerConfig(use_importance_sampling=False)
    dm = DynamicDataManager(cfg, cams, targets, device=dev, eval_cameras=cams, eval_images=targets)
    evaluator = Evaluator(model, dm, rank=rank, world=world)
    evaluator.get_average_eval_image_metrics(0)  # warm-up: tile graphs captured, kernels loaded
    calls = []
    for r in range(args.repeats):
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = evaluator.get_average_eval_image_metrics(r + 1)  # ends with the metrics on the host of every rank
        calls.append(time.perf_counter() - t0)
        torch.cuda.synchronize()
    result = {"metric": "eval over the eval split (Evaluator.get_average_eval_image_metrics)",
              "workload": f"kplanes-32x(cfg3 field), {args.images} eval images at {args.width}x{args.height}, chunk "
                          f"{model.config.eval_num_rays_per_chunk}, whole images per rank (i % world == rank)",
              "gpus": world, "card": card_info(local), "seconds_per_call": sorted(calls)[len(calls) // 2],
              "seconds_per_image": sorted(calls)[len(calls) // 2] / args.images, "seconds_per_call_all": calls,
              "results": res}
    if args.regions:  # the eval images form one camera's clip: its median is the background the masks leave out
        cams.ids = torch.zeros(args.images, dtype=torch.int64)
        dm.eval_cameras.ids = cams.ids
        t0 = time.perf_counter()
        region_evaluator = Evaluator(model, dm, rank=rank, world=world, regions="median")
        torch.cuda.synchronize()
        construct = time.perf_counter() - t0
        region_evaluator.get_average_eval_image_metrics(0)
        region_calls = []
        for r in range(args.repeats):
            if world > 1:
                torch.distributed.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            region_res = region_evaluator.get_average_eval_image_metrics(r + 1)
            region_calls.append(time.perf_counter() - t0)
            torch.cuda.synchronize()
        result["regions"] = {"evaluator_construct_s": construct, "seconds_per_call": sorted(region_calls)[len(region_calls) // 2],
                             "seconds_per_call_all": region_calls, "results": region_res}
    if args.depth:  # ground-truth z-depth (the preset's convention): the rendered depth with 5 % noise, 0 where the
        # frame accumulates less than half (background); the same evaluator with and without it, calls alternating
        depth, acc, norms = (torch.stack(t)[..., 0] for t in zip(*geometry))
        gt = depth / norms * torch.exp(0.05 * torch.randn(depth.shape, generator=gen, device=dev))
        gt[acc < 0.5] = 0.0
        model.config.is_euclidean_depth = False
        depth_dm = DynamicDataManager(cfg, cams, targets, device=dev, eval_cameras=cams, eval_images=targets,
                                      eval_extras={"depth_image": gt[..., None]})
        depth_evaluator = Evaluator(model, depth_dm, rank=rank, world=world)
        depth_evaluator.get_average_eval_image_metrics(0)
        plain_calls, depth_calls = [], []
        for r in range(args.repeats):
            for ev_, calls_ in ((evaluator, plain_calls), (depth_evaluator, depth_calls)):
                if world > 1:
                    torch.distributed.barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                res_ = ev_.get_average_eval_image_metrics(r + 1)
                calls_.append(time.perf_counter() - t0)
                torch.cuda.synchronize()
            depth_res = res_
        result["depth"] = {"seconds_per_call": sorted(depth_calls)[len(depth_calls) // 2],
                           "seconds_per_call_without_depth": sorted(plain_calls)[len(plain_calls) // 2],
                           "seconds_per_call_all": depth_calls, "seconds_per_call_without_depth_all": plain_calls,
                           "results": depth_res}
    if args.write_images:
        result["write_images"] = write_timing(evaluator, args.images, args.repeats)
    if rank == 0:
        if args.write_images:
            result["write_images"]["kernel"] = maps_timing(torch.stack(renders), targets, args.kernel_reps)
        result["kernel"] = kernel_vs_torch(torch.stack(renders), targets, args.kernel_reps)
        if args.depth:  # masks: the median masks of the 8 frames as one camera's clip, as --regions takes them
            from soccernerfs_b200.engine.evaluator import median_dynamic_masks

            mask = median_dynamic_masks(targets, torch.zeros(args.images, dtype=torch.int64))
            result["depth"]["kernel"] = depth_timing(depth, gt, norms, mask, args.kernel_reps)
        if args.regions:
            result["regions"]["kernel"] = regions_timing(torch.stack(renders), targets, cams.ids, args.kernel_reps)
        line = json.dumps(result)
        print(line)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
