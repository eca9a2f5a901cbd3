"""Worker for tests/test_gpu_depth_metrics.py::test_evaluator_depth_two_ranks_equal_one_rank (torch.distributed.run, one
process per GPU): with eval depth, without and with regions, the 2-rank averages equal the 1-rank ones bit for bit (NaN
where NaN), on every rank."""
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
    import tests.test_gpu_depth_metrics as t
    import tests.test_gpu_eval as te
    from soccernerfs_b200.engine.evaluator import Evaluator

    t.DEV = te.DEV = f"cuda:{torch.cuda.current_device()}"
    model = te._tiny_model()
    model.config.is_euclidean_depth = False
    dm, _, images, _, _, gt = t._depth_setup(model, n=5)  # 5 images over 2 ranks: 3 + 2
    g = torch.Generator(device=t.DEV).manual_seed(4)
    noisy = gt * torch.exp(0.2 * torch.randn(gt.shape, generator=g, device=t.DEV))
    noisy[3] = 0.0  # image 3: no valid pixel
    dm.eval_image_cache.batch["depth_image"] = noisy
    caller = torch.zeros(images.shape[:3], dtype=torch.bool, device=images.device)
    caller[0, 4:12, 6:20] = True
    caller[4, :, :] = True  # image 1, 2, 3: no dynamic pixel; image 4: no static pixel
    for regions in (None, caller):
        single = Evaluator(model, dm, regions=regions).get_average_eval_image_metrics(0)
        shared = Evaluator(model, dm, rank=rank, world=world, regions=regions).get_average_eval_image_metrics(0)
        keys = [k for k in single if k not in ("num_rays_per_sec", "fps")]
        assert list(shared) == list(single) and all(_same(shared[k], single[k]) for k in keys), (rank, single, shared)
        mine = torch.tensor([shared[k] for k in keys], dtype=torch.float64, device="cuda")
        other = mine.clone()
        dist.broadcast(other, src=0)
        assert torch.equal(mine.isnan(), other.isnan()) and torch.equal(mine.nan_to_num(), other.nan_to_num()), "ranks disagree"
        if rank == 0:
            print("regions" if regions is not None else "whole", single)
    dist.barrier()
    if rank == 0:
        print("DEPTH_EVAL_MULTI_OK")
    sys.stdout.flush()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
