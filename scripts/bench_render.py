#!/usr/bin/env python
"""bench_render.py -- rendering a camera path of a dynamic scene on B200s, to PNG files, to JPEG files and to a
Motion-JPEG video: render_camera_path / render_camera_path_video over a 1080p arc whose render times sweep [0, 1]
(bench_eval.py's eval cameras), from the 32x field (bench.py's cfg3 model), with the outputs rgb, depth and accumulation
side by side (a 5760x1080 frame); kp_compose_frame against the torch restatement of the same composition
(utils/colormaps.py + quantisation) on the same frames and device; and kp_jpeg_encode on the composed frame against PIL's
PNG and JPEG encoders on the host.

    python scripts/bench_render.py                                                       # 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 scripts/bench_render.py   # 8 GPUs (frames i % 8 == rank)

Prints one JSON line (rank 0).  The files go to a temporary directory that is removed afterwards.  Kernel timing: CUDA
events around each pass, after warm-up, with a 512 MB buffer written before every pass so no pass reads its frame from
L2 (126 MB).  End to end: the host wall time of one render_camera_path (or render_camera_path_video) call per rank
(tile-graph capture, renders, composition, encoding, copies, files written), the maximum over the ranks.
"""
from __future__ import annotations

import argparse
import io
import json
import os
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

NAMES = ("rgb", "depth", "accumulation")


def restated_compose(frames, names):
    """The torch restatement of ops.compose_frame: the model's eval visualisations, side by side, quantised."""
    from soccernerfs_b200 import ops
    from soccernerfs_b200.utils import colormaps

    panels = []
    for name in names:
        kind = ops.panel_kind(name)
        x = frames[name]
        if kind == 1:
            x = colormaps.apply_colormap(x)
        elif kind == 2:
            x = colormaps.apply_depth_colormap(x, accumulation=frames["accumulation"])
        panels.append(x)
    return torch.floor(torch.nan_to_num(torch.cat(panels, dim=1)).clamp(0, 1) * 255 + 0.5).to(torch.uint8)


def timed_ms(fn, reps: int, flush: torch.Tensor):
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


def compose_vs_torch(frames, reps: int) -> dict:
    from soccernerfs_b200 import ops

    flush = torch.empty(512 * 2**20 // 4, dtype=torch.float32, device=frames["rgb"].device)
    for _ in range(3):
        ops.compose_frame(frames, NAMES)
        restated_compose(frames, NAMES)
    torch.cuda.synchronize()
    equal = bool(torch.equal(ops.compose_frame(frames, NAMES), restated_compose(frames, NAMES)))
    k_ms, k_all = timed_ms(lambda: ops.compose_frame(frames, NAMES), reps, flush)
    t_ms, t_all = timed_ms(lambda: restated_compose(frames, NAMES), reps, flush)
    h, w = frames["rgb"].shape[:2]
    n_depth = sum(ops.panel_kind(n) == 2 for n in NAMES)
    # reads: every panel once, the depth panels twice (min / max pass), the accumulation once more per depth panel
    read = h * w * 4 * (sum(frames[n].shape[-1] for n in NAMES) + 2 * n_depth)
    written = h * w * len(NAMES) * 3
    return {"kp_compose_frame_ms": k_ms, "torch_restatement_ms": t_ms, "speedup": t_ms / k_ms, "identical_bytes": equal,
            "kp_ms_all": k_all, "torch_ms_all": t_all, "bytes_read_min": read, "bytes_written": written,
            "kp_effective_gbs": (read + written) / (k_ms * 1e-3) / 1e9, "l2_flush": "512 MB written before every pass"}


def png_encode_ms(image: torch.Tensor, reps: int = 5) -> float:
    from PIL import Image

    arr = image.cpu().numpy()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        Image.fromarray(arr).save(io.BytesIO(), format="PNG")
        times.append((time.perf_counter() - t0) * 1e3)
    return sorted(times)[len(times) // 2]


def jpeg_encode(image: torch.Tensor, reps: int, quality: int) -> dict:
    """kp_jpeg_encode on the composed frame (device events, L2 overwritten before each pass) and PIL's JPEG at the same
    quality and 4:2:0 on the host, with the encoded sizes."""
    from PIL import Image

    from soccernerfs_b200 import ops

    flush = torch.empty(512 * 2**20 // 4, dtype=torch.float32, device=image.device)
    for _ in range(3):
        ops.encode_jpeg(image, quality)
    torch.cuda.synchronize()
    k_ms, k_all = timed_ms(lambda: ops.encode_jpeg(image, quality), reps, flush)
    _, length = ops.encode_jpeg(image, quality)
    arr = image.cpu().numpy()
    times = []
    for _ in range(5):
        buf = io.BytesIO()
        t0 = time.perf_counter()
        Image.fromarray(arr).save(buf, format="JPEG", quality=quality, subsampling=2)
        times.append((time.perf_counter() - t0) * 1e3)
    h, w = arr.shape[:2]
    return {"kp_jpeg_encode_ms": k_ms, "kp_ms_all": k_all, "quality": quality, "frame": f"{w}x{h}",
            "encoded_bytes_per_frame": int(length), "pil_jpeg_ms_per_frame": sorted(times)[len(times) // 2],
            "pil_jpeg_bytes_per_frame": len(buf.getvalue()), "l2_flush": "512 MB written before every pass"}


def end_to_end(fn, world: int, dev) -> float:
    """Host seconds of fn() on every rank, ended by a device synchronise; the maximum over the ranks."""
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([wall], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        torch.distributed.barrier()
        wall = float(t)
    return wall


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--kernel-reps", type=int, default=20)
    ap.add_argument("--jpeg-quality", type=int, default=95)
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_render.py measures on a CUDA device; none is visible")

    import bench
    from bench_eval import card_info, eval_cameras
    from soccernerfs_b200.engine.frame_renderer import FrameRenderer
    from soccernerfs_b200.engine.path_renderer import render_camera_path, render_camera_path_video

    rank, world, local = bench._dist_setup()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    model = bench.build_model("cfg3", dev)
    model.eval()
    cams = eval_cameras(args.frames, args.height, args.width, dev)
    out_dir = tempfile.mkdtemp(prefix="bench_render_")
    try:
        # render seconds per frame: device events around FrameRenderer.render(device_frames=True), graphs warm
        renderer = FrameRenderer(model, cams, outputs=NAMES)
        with torch.no_grad():
            renderer.render(0, device_frames=True)
            events = []
            for i in range(min(4, args.frames)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                frames = renderer.render(i, device_frames=True)
                e1.record()
                events.append((e0, e1))
            torch.cuda.synchronize()
        render_s = sorted(a.elapsed_time(b) / 1e3 for a, b in events)[len(events) // 2]
        del renderer
        # end to end: one call per rank and output format, the files on disk
        mine = []
        wall = end_to_end(lambda: mine.extend(render_camera_path(model, cams, out_dir, rendered_output_names=NAMES,
                                                                 rank=rank, world=world)), world, dev)
        jpg_dir = os.path.join(out_dir, "jpeg")
        wall_jpeg = end_to_end(lambda: render_camera_path(model, cams, jpg_dir, rendered_output_names=NAMES, rank=rank,
                                                          world=world, image_format="jpeg",
                                                          jpeg_quality=args.jpeg_quality), world, dev)
        video = os.path.join(out_dir, "path.avi")
        wall_video = end_to_end(lambda: render_camera_path_video(model, cams, video, args.frames / 24.0,
                                                                 rendered_output_names=NAMES, rank=rank, world=world,
                                                                 jpeg_quality=args.jpeg_quality), world, dev)
        written = len([f for f in os.listdir(out_dir) if f.endswith(".png")])
        h, w = args.height, args.width
        result = {"metric": "camera-path render to PNG files, JPEG files and an MJPEG video (render_camera_path, "
                            "render_camera_path_video)",
                  "workload": f"kplanes-32x(cfg3 field), {args.frames} cameras at {w}x{h}, render times 0..1, outputs "
                              f"{list(NAMES)}, chunk {model.config.eval_num_rays_per_chunk}, whole frames per rank "
                              f"(i % world == rank)",
                  "gpus": world, "card": card_info(local), "render_seconds_per_frame": render_s,
                  "d2h_bytes_per_frame": h * w * len(NAMES) * 3,
                  "end_to_end_seconds": wall, "end_to_end_frames_per_second": args.frames / wall,
                  "end_to_end_frames_per_second_png": args.frames / wall,
                  "end_to_end_frames_per_second_jpeg": args.frames / wall_jpeg,
                  "end_to_end_frames_per_second_video": args.frames / wall_video,
                  "frames_this_rank": len(mine), "png_files_rank0_dir": written}
        if rank == 0:
            from soccernerfs_b200 import ops

            result["compose"] = compose_vs_torch(frames, args.kernel_reps)
            image = ops.compose_frame(frames, NAMES)
            result["png_encode_ms_per_frame"] = png_encode_ms(image)
            result["png_bytes_per_frame"] = os.path.getsize(os.path.join(out_dir, f"{mine[0]:05d}.png"))
            result["jpeg"] = jpeg_encode(image, args.kernel_reps, args.jpeg_quality)
            result["jpeg"]["share_of_render_time"] = result["jpeg"]["kp_jpeg_encode_ms"] / (render_s * 1e3)
            result["video_bytes"] = os.path.getsize(video)
            result["host_cpus"] = os.cpu_count()
            line = json.dumps(result)
            print(line)
            if args.out:
                os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
                with open(args.out, "w") as f:
                    f.write(line + "\n")
    finally:
        shutil.rmtree(out_dir, ignore_errors=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
