"""Worker for tests/test_gpu_region_metrics.py::test_evaluator_regions_two_ranks_equal_one_rank (torch.distributed.run,
one process per GPU): with a caller mask and with "median" masks, the 2-rank averages equal the 1-rank ones bit for bit
(NaN where NaN), on every rank."""
import math
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _same(a, b):
    return a == b or (math.isnan(a) and math.isnan(b))


def main() -> None:
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    import tests.test_gpu_eval as t
    from soccernerfs_b200.engine.evaluator import Evaluator

    t.DEV = f"cuda:{torch.cuda.current_device()}"
    model = t._tiny_model()
    dm, _, images = t._eval_setup(model, n=5)  # 5 images over 2 ranks: 3 + 2
    dm.eval_cameras.ids = torch.zeros(5, dtype=torch.int64)
    caller = torch.zeros(images.shape[:3], dtype=torch.bool, device=images.device)
    caller[0, 4:12, 6:20] = True
    caller[3, :, :] = True  # image 1, 2, 4: no dynamic pixel; image 3: no static pixel
    for regions in (caller, "median"):
        single = Evaluator(model, dm, regions=regions).get_average_eval_image_metrics(0)
        shared = Evaluator(model, dm, rank=rank, world=world, regions=regions).get_average_eval_image_metrics(0)
        keys = [k for k in single if k not in ("num_rays_per_sec", "fps")]
        assert list(shared) == list(single) and all(_same(shared[k], single[k]) for k in keys), (rank, single, shared)
        mine = torch.tensor([shared[k] for k in keys], dtype=torch.float64, device="cuda")
        other = mine.clone()
        dist.broadcast(other, src=0)
        assert torch.equal(mine.isnan(), other.isnan()) and torch.equal(mine.nan_to_num(), other.nan_to_num()), "ranks disagree"
        if rank == 0:
            print("regions", "median" if isinstance(regions, str) else "caller", single)
    dist.barrier()
    if rank == 0:
        print("REGION_EVAL_MULTI_OK")
    sys.stdout.flush()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
