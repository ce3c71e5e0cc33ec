"""Worker of the world_size-2 dynamic loss scaling test (tests/test_gpu_loss_scale.py): both ranks on one device, gloo.

Each rank runs the Trainer's data-parallel step by hand: backward, flat-gradient sum all-reduce, the module's
optimizer_step hook.  Step 1: rank 1 writes inf into its gradient before the all-reduce.  Step 2: no injection."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from test_gpu_train_batch import _inputs, _module  # noqa: E402

from mcedm_b200.loss_scale import LossScaler  # noqa: E402

rank, world, out = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3]
dist.init_process_group("gloo", rank=rank, world_size=world)
dev = torch.device("cuda")
pl, _ = _module(dev)
pl.use_cuda_graph = True
opt = pl.configure_optimizers()["optimizer"]
opt.max_grad_norm = 1.0
opt.grad_scale = 1.0 / world
sc = LossScaler()
pl.model.engine().loss_scaler = sc
scales, found = [], []
for it in range(2):
    x, sigma, noise, cond, mask = _inputs(pl, dev, 8, seed=900 + 10 * it + rank)
    opt.zero_grad(set_to_none=True)
    loss = pl.forward_loss(x, sigma, noise, cond, mask, pl.get_loss_weight(sigma))
    loss.backward()
    g = opt.flat_grads()
    if it == 0 and rank == 1:
        g[12345] = float("inf")
    p0 = opt.flat_params().clone()
    dist.all_reduce(g)
    pl.optimizer_step(0, it, opt)
    torch.cuda.synchronize()
    scales.append(sc.get_scale())
    found.append(float(sc.found_inf_t))
    assert torch.equal(p0, opt.flat_params()) == (it == 0), (rank, it)
torch.save({"scales": scales, "found_inf": found, "p": opt.flat_params().cpu()}, os.path.join(out, f"rank{rank}.pt"))
dist.barrier()
dist.destroy_process_group()
