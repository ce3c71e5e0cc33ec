"""Cost of gradient accumulation on the fp16 training plan.

Graph-replayed PlMcedm training steps (forward + loss, backward, clipped Adam + EMA, as under the Trainer) on one
module: windows of N micro-batches of 32 (UNetEngine.accumulate_grads = N; N = 1 is the plain step) against one step
at B = 32 N, alternated in rounds after a warm-up and timed with CUDA events, in ms per optimizer step and samples/s.
Then the fold kernel (mcedm_grad_accumulate) alone, from CUDA events over many launches on the model's flat gradient
size: on one buffer pair (L2-resident, as right after a backward wrote the micro-batch gradient) and rotating over
buffer pairs of 2x the 126 MB L2 (HBM), with its achieved GB/s at 12 bytes per element (read g, read acc, write acc).
The fold's share of a micro-batch step is the L2-resident fold time over the B = 32 step time of the same run.  Prints
one JSON line with the card name and its power limit, read in the same run.
usage: python scripts/grad_accum_bench.py [micro-batch] [windows per round] [rounds]"""
import copy
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mcedm_b200 import _lib as L  # noqa: E402
from mcedm_b200 import data as D  # noqa: E402
from mcedm_b200.config import compose  # noqa: E402
from mcedm_b200.mcedm import PlMcedm  # noqa: E402
from mcedm_b200.utils import randomize_zero_init  # noqa: E402

MB = int(sys.argv[1]) if len(sys.argv) > 1 else 32
windows = int(sys.argv[2]) if len(sys.argv) > 2 else 10
rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 5
NS = (1, 2, 4, 8)
dev = torch.device("cuda:0")
cfg = compose("config_adm_edm_mcedm_res32", ["system=swe_per"])
st = D.field_stats("swe_per", 16)


def batch(b):
    h, tg, xg, u, mask = D.make_batch("swe_per", b, "train", seed=0)
    return tuple(t.to(dev) for t in (h, tg, xg, u, mask))


torch.manual_seed(1)
pl = PlMcedm(copy.deepcopy(cfg.model.hparams))
randomize_zero_init(pl.model, 2)
pl = pl.to(dev).train()
pl.normalizer_input.set_stats(st["input_mean"].to(dev), st["input_std"].to(dev))
pl.normalizer_target.set_stats(st["target_mean"].to(dev), st["target_std"].to(dev))
opt = pl.configure_optimizers()["optimizer"]
opt.max_grad_norm = 1.0
opt.param_groups[0]["lr"] = 1e-7                  # timing only: keep the weights where they are
eng = pl.model.engine()
batches = {b: batch(b) for b in {MB} | {MB * n for n in NS}}


def run(n_micro, b, n):
    """n optimizer steps, each on a window of n_micro micro-batches of b samples; device ms per optimizer step"""
    eng.accumulate_grads = n_micro if n_micro > 1 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        opt.zero_grad(set_to_none=True)
        for k in range(n_micro):
            pl.training_step(batches[b], k).backward()
        pl.optimizer_step(0, n_micro - 1, opt)
    e1.record()
    torch.cuda.synchronize()
    eng.accumulate_grads = None
    return e0.elapsed_time(e1) / n


configs = {f"accum {MB}x{n}": (n, MB) for n in NS} | {f"batch {MB * n}": (1, MB * n) for n in NS[1:]}
for c in configs.values():
    run(*c, 3)                                    # capture + warm-up of every shape
L.check_watchdog()
times = {k: [] for k in configs}
for _ in range(rounds):
    for k, c in configs.items():
        times[k].append(run(*c, windows))
L.check_watchdog()


def kernel_us(fn, n=500):
    assert fn(0) == 0, L.lib().mcedm_last_error()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


lib, s = L.lib(), L.stream_ptr()
n_el = eng.flat_grad().numel()
n_pairs = max(2, (2 * 126 * 2 ** 20) // (8 * n_el) + 1)
accs = [torch.zeros(n_el, device=dev) for _ in range(n_pairs)]
gs = [torch.randn(n_el, device=dev) * 1e-3 for _ in range(n_pairs)]
fold = {}
for first in (0, 1):
    tag = "write" if first else "add"
    fold[f"{tag}_l2"] = kernel_us(lambda i: lib.mcedm_grad_accumulate(L.ptr(accs[0]), L.ptr(gs[0]), n_el, 0.25, first,
                                                                      s))
    fold[f"{tag}_hbm"] = kernel_us(lambda i: lib.mcedm_grad_accumulate(L.ptr(accs[i % n_pairs]), L.ptr(gs[i % n_pairs]),
                                                                       n_el, 0.25, first, s))
L.check_watchdog()
bytes_per_el = {"add": 12, "write": 8}
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as e:  # noqa: BLE001
    power = f"unavailable ({e})"
best = {k: min(t) for k, t in times.items()}
samples = {k: c[0] * c[1] for k, c in configs.items()}
step_us = best[f"accum {MB}x1"] * 1e3
print(json.dumps({
    "gpu": torch.cuda.get_device_name(0), "power_limit": power, "micro_batch": MB, "windows_per_round": windows,
    "rounds": rounds,
    "ms_per_optimizer_step": {k: [round(t, 4) for t in ts] for k, ts in times.items()},
    "ms_per_optimizer_step_best": {k: round(v, 4) for k, v in best.items()},
    "samples_per_s_best": {k: round(samples[k] / best[k] * 1e3, 1) for k in best},
    "fold_elements": n_el, "fold_buffer_pairs_hbm": n_pairs,
    "fold_us_per_launch": {k: round(v, 2) for k, v in fold.items()},
    "fold_GBps": {k: round(bytes_per_el[k.split("_")[0]] * n_el / (v * 1e-6) / 1e9, 1) for k, v in fold.items()},
    "fold_share_of_micro_batch_step_pct": round(fold["add_l2"] / step_us * 100, 3),
}))
