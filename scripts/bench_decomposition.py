#!/usr/bin/env python
"""bench_decomposition.py -- the space-time decomposition outputs on one B200, on the 32x field (bench.py's cfg3 model, time
planes perturbed) at 1920x1080 (bench_eval.py's eval cameras):

  * kp_hexplane_fwd_dyn against kp_hexplane_fwd on the samples of one tile of a frame (eval_num_rays_per_chunk rays of
    neighbouring pixels, coherent-ray gather as the renderer runs it), CUDA events per pass, a 512 MB buffer written
    before every pass so no pass reads the field from L2 (126 MB), the two kernels alternated;
  * seconds per frame of FrameRenderer.render(device_frames=True) for ("rgb",), ("rgb", "dynamic") and
    ("rgb", "rgb_static", "dynamic"): CUDA events around each render, tile graphs warm, the median of the frames.

    python scripts/bench_decomposition.py [--frames 4] [--reps 20] [--out result.json]

Prints one JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

OUTPUT_SETS = (("rgb",), ("rgb", "dynamic"), ("rgb", "rgb_static", "dynamic"))


def gather_legs(model, cams, reps: int) -> dict:
    from soccernerfs_b200 import ops
    from soccernerfs_b200.models.base_model import coherent_rays

    field = model.field
    n = model.config.eval_num_rays_per_chunk
    h, w = cams._height_host[0], cams._width_host[0]
    start = (h // 2) * w  # a tile from the middle of the frame
    with torch.no_grad():
        with coherent_rays(model):
            model.forward(ray_bundle=cams.generate_tile(0, start, start + n))
        points, ms = field._last_points, field._planes()
        concat, mask = field.concat_features_across_scales, 0x3F
        plain = lambda: ops.hexplane_features(ms, points, concat, mask)  # noqa: E731
        dyn = lambda: ops.hexplane_features_dyn(ms, points, concat, mask)  # noqa: E731
        flush = torch.empty(512 * 2**20 // 4, dtype=torch.float32, device=points.starts.device)
        for _ in range(3):
            plain(), dyn()
        same = bool(torch.equal(plain(), dyn()[0]))
        times = {"kp_hexplane_fwd": [], "kp_hexplane_fwd_dyn": []}
        for _ in range(reps):
            for name, fn in (("kp_hexplane_fwd", plain), ("kp_hexplane_fwd_dyn", dyn)):
                flush.fill_(1.0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                times[name].append(e0.elapsed_time(e1))
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    return {"samples": points.M, "rays": n, "samples_per_ray": points.S, "features_identical": same,
            "kp_hexplane_fwd_ms": med["kp_hexplane_fwd"], "kp_hexplane_fwd_dyn_ms": med["kp_hexplane_fwd_dyn"],
            "dyn_over_plain": med["kp_hexplane_fwd_dyn"] / med["kp_hexplane_fwd"], "ms_all": times,
            "l2_flush": "512 MB written before every pass"}


def frame_legs(model, cams, frames: int) -> dict:
    from soccernerfs_b200.engine.frame_renderer import FrameRenderer

    out = {}
    for names in OUTPUT_SETS:
        renderer = FrameRenderer(model, cams, outputs=names)
        with torch.no_grad():
            renderer.render(0, device_frames=True)  # capture the tile graphs
            events = []
            for i in range(frames):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                renderer.render(i, device_frames=True)
                e1.record()
                events.append((e0, e1))
            torch.cuda.synchronize()
        secs = sorted(a.elapsed_time(b) / 1e3 for a, b in events)
        out["+".join(names)] = {"seconds_per_frame": secs[len(secs) // 2], "all": secs}
        del renderer
        torch.cuda.empty_cache()
    base = out["rgb"]["seconds_per_frame"]
    for v in out.values():
        v["over_rgb"] = v["seconds_per_frame"] / base
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_decomposition.py measures on a CUDA device; none is visible")

    import bench
    from bench_eval import card_info, eval_cameras

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    model = bench.build_model("cfg3", dev)
    model.eval()
    cams = eval_cameras(args.frames, args.height, args.width, dev)
    result = {"metric": "space-time decomposition: kp_hexplane_fwd_dyn vs kp_hexplane_fwd, frame time with the new outputs",
              "workload": f"kplanes-32x (cfg3 field, time planes perturbed), {args.frames} cameras at {args.width}x{args.height}, "
                          f"chunk {model.config.eval_num_rays_per_chunk}",
              "card": card_info(0), "gather": gather_legs(model, cams, args.reps), "frames": frame_legs(model, cams, args.frames)}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
