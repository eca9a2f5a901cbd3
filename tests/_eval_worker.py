"""Worker for tests/test_gpu_eval.py::test_evaluator_two_ranks_equal_one_rank (torch.distributed.run, one process per GPU):
the 2-rank average eval metrics equal the 1-rank ones bit for bit, on every rank."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main() -> None:
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    import tests.test_gpu_eval as t
    from soccernerfs_b200.engine.evaluator import Evaluator

    t.DEV = f"cuda:{torch.cuda.current_device()}"
    model = t._tiny_model()
    dm, _, _ = t._eval_setup(model, n=5)  # 5 images over 2 ranks: 3 + 2
    single = Evaluator(model, dm).get_average_eval_image_metrics(0)
    shared = Evaluator(model, dm, rank=rank, world=world).get_average_eval_image_metrics(0)
    keys = [k for k in single if k not in ("num_rays_per_sec", "fps")]
    assert keys and all(shared[k] == single[k] for k in keys), (rank, single, shared)
    assert list(shared) == list(single) and shared["num_rays_per_sec"] > 0
    mine = torch.tensor([shared[k] for k in shared], dtype=torch.float64, device="cuda")
    other = mine.clone()
    dist.broadcast(other, src=0)
    assert torch.equal(mine, other), "ranks disagree"
    dist.barrier()
    if rank == 0:
        print("EVAL_MULTI_OK", single, shared)
    sys.stdout.flush()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
