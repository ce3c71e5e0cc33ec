"""Worker of the world_size-2 gradient accumulation test (tests/test_gpu_grad_accum.py): both ranks on one device, gloo.

Rank r trains one window of runner.Trainer(accumulate_grad_batches=2) on micro-batches 2r and 2r + 1 (8 samples each)
of test_gpu_train_batch._inputs(B = 32, seed 1500), counting the all-reduces of the flat gradient, and saves the
reduced gradient the optimizer stepped on and the parameters after the step."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from test_gpu_grad_accum import _IndexDM, _drive, micro  # noqa: E402
from test_gpu_train_batch import _inputs, _module  # noqa: E402

from mcedm_b200 import runner  # noqa: E402

rank, world, out = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3]
dist.init_process_group("gloo", rank=rank, world_size=world)
dev = torch.device("cuda")
pl, _ = _module(dev)
pl.use_cuda_graph = True
inp = _inputs(pl, dev, 32, seed=1500)
rec = _drive(pl, [micro(inp, 2 * rank + k, 8) for k in range(2)])
n_params = sum(p.numel() for p in pl.model.parameters())
grad_allreduces = []
all_reduce = dist.all_reduce


def counting_all_reduce(t, *a, **k):
    if t.numel() == n_params:
        grad_allreduces.append(1)
    return all_reduce(t, *a, **k)


runner.dist.all_reduce = counting_all_reduce
tr = runner.Trainer(max_epochs=1, accumulate_grad_batches=2, check_val_every_n_epoch=100)
assert tr.world_size == world
tr.fit(pl, _IndexDM(2))
torch.cuda.synchronize()
assert len(rec["steps"]) == 1 and pl.global_step == 1
torch.save({"grad_allreduces": len(grad_allreduces), "g": rec["steps"][0][1].cpu(),
            "p": tr.optimizer.flat_params().cpu()}, os.path.join(out, f"rank{rank}.pt"))
dist.barrier()
dist.destroy_process_group()
