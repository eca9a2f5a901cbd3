"""Worker for tests/test_gpu_eval_images.py::test_eval_images_two_processes_equal_one (torch.distributed.run, one process
per GPU): through the all_gather and the barrier, two ranks write the image files, metrics.json and per-camera videos
that one rank writes."""
import json
import math
import os
import shutil
import sys
import tempfile

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _same(a, b):
    return a == b or (isinstance(a, float) and math.isnan(a) and math.isnan(b))


def main() -> None:
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    import tests.test_gpu_eval as te
    import tests.test_gpu_eval_images as t
    from soccernerfs_b200.engine.evaluator import Evaluator

    t.DEV = te.DEV = f"cuda:{torch.cuda.current_device()}"
    model = t._tiny_model()
    dm = t._setup(model)
    regions = t._regions(dm)
    names = ("gt", "rgb", "error", "depth_error", "dynamic_mask")
    root = tempfile.mkdtemp(prefix=f"eval_images_rank{rank}_")  # each process' own single-rank reference
    shared = [None]
    if rank == 0:
        shared = [tempfile.mkdtemp(prefix="eval_images_shared_")]
    dist.broadcast_object_list(shared, src=0)
    one, two = os.path.join(root, "one"), shared[0]
    Evaluator(model, dm, regions=regions).write_eval_images(one, panels=names)
    Evaluator(model, dm, regions=regions).write_eval_videos(one, 10.0, panels=names)
    ev = Evaluator(model, dm, rank=rank, world=world, regions=regions)
    assert ev.write_eval_images(two, panels=names) == list(range(rank, 6, world))
    ev.write_eval_videos(two, 10.0, panels=names)  # barrier, then rank 0 assembles
    dist.barrier()
    if rank == 0:
        files = sorted(os.listdir(two))
        assert files == sorted(os.listdir(one)), (files, sorted(os.listdir(one)))
        for name in files:
            a, b = open(os.path.join(one, name), "rb").read(), open(os.path.join(two, name), "rb").read()
            if name == "metrics.json":
                ra, rb = json.loads(a)["images"], json.loads(b)["images"]
                assert [list(e) for e in ra] == [list(e) for e in rb]
                assert all(_same(x[k], y[k]) for x, y in zip(ra, rb) for k in x), name
            else:
                assert a == b, name
        print("EVAL_IMAGES_MULTI_OK")
    sys.stdout.flush()
    dist.barrier()
    shutil.rmtree(root)
    if rank == 0:
        shutil.rmtree(two)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
