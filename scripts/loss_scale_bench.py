"""Cost of dynamic loss scaling in the fp16 training plan: graph-replayed training steps of PlMcedm (forward + loss,
backward, optimizer + EMA, clipping on as under the Trainer) with the static scale and with a LossScaler, alternated in
rounds after a warm-up and timed with CUDA events, plus the per-launch time of the three kernels the dynamic step adds or
replaces (sum-of-squares partials are shared with clipping).  Prints one JSON line with the card name and its power
limit, read in the same run.
usage: python scripts/loss_scale_bench.py [B] [steps per round] [rounds]"""
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
from mcedm_b200.loss_scale import LossScaler  # noqa: E402
from mcedm_b200.mcedm import PlMcedm  # noqa: E402
from mcedm_b200.utils import randomize_zero_init  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 5
dev = torch.device("cuda:0")
cfg = compose("config_adm_edm_mcedm_res32", ["system=swe_per"])
h, tg, xg, u, mask = D.make_batch("swe_per", B, "train", seed=0)
batch = tuple(t.to(dev) for t in (h, tg, xg, u, mask))
st = D.field_stats("swe_per", 16)


def module(dynamic):
    torch.manual_seed(1)
    pl = PlMcedm(copy.deepcopy(cfg.model.hparams))
    randomize_zero_init(pl.model, 2)
    pl = pl.to(dev).train()
    pl.normalizer_input.set_stats(st["input_mean"].to(dev), st["input_std"].to(dev))
    pl.normalizer_target.set_stats(st["target_mean"].to(dev), st["target_std"].to(dev))
    opt = pl.configure_optimizers()["optimizer"]
    opt.max_grad_norm = 1.0
    if dynamic:
        pl.model.engine().loss_scaler = LossScaler()
    return pl, opt


def run(pl, opt, n):
    """n training steps; device time of the whole sequence (ms per step)"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        opt.zero_grad(set_to_none=True)
        loss = pl.training_step(batch, 0)
        loss.backward()
        pl.optimizer_step(0, 0, opt)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


mods = {name: module(name == "dynamic") for name in ("static", "dynamic")}
for pl, opt in mods.values():
    run(pl, opt, 5)                                   # capture + warm-up
L.check_watchdog()
times = {k: [] for k in mods}
for _ in range(rounds):
    for k, (pl, opt) in mods.items():
        times[k].append(run(pl, opt, steps))
L.check_watchdog()
sc = mods["dynamic"][0].model.engine().loss_scaler
skipped = float(sc.found_inf_t)


def kernel_us(fn, n=200):
    assert fn() == 0, L.lib().mcedm_last_error()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


lib = L.lib()
st_ = L.stream_ptr()
opt = mods["dynamic"][1]
p, m, v = opt.flat_params().clone(), opt._m.clone(), opt._v.clone()
g = torch.randn_like(p) * 1e-3
n = p.numel()
part = torch.empty(128, device=dev, dtype=torch.float64)
norm = torch.zeros(1, device=dev)
steps_dev = torch.zeros(1, device=dev, dtype=torch.int32)
found = torch.zeros(1, device=dev)
scale, tracker = torch.full((1,), 1024.0, device=dev), torch.zeros(1, device=dev, dtype=torch.int32)
lib.mcedm_sumsq_partial(L.ptr(g), n, L.ptr(part), 128, st_)
kern = {
    "adam_step": kernel_us(lambda: lib.mcedm_adam_step(L.ptr(p), L.ptr(g), L.ptr(m), L.ptr(v), n, 1e-9, 0.9, 0.999, 1e-8,
                                                       0.0, 10, L.ptr(part), 128, 1.0, 1.0, L.ptr(norm), st_)),
    "adam_step_dyn": kernel_us(lambda: lib.mcedm_adam_step_dyn(L.ptr(p), L.ptr(g), L.ptr(m), L.ptr(v), n, 1e-9, 0.9, 0.999,
                                                               1e-8, 0.0, L.ptr(steps_dev), L.ptr(part), 128, 1.0, 1.0,
                                                               L.ptr(norm), L.ptr(found), st_)),
    "loss_scale_update": kernel_us(lambda: lib.mcedm_loss_scale_update(L.ptr(scale), L.ptr(tracker), L.ptr(found),
                                                                       L.ptr(steps_dev), 2.0, 0.5, 2000, st_)),
    "grad_unscale": kernel_us(lambda: lib.mcedm_grad_unscale(L.ptr(g), n, L.ptr(scale), st_)),
}
L.check_watchdog()

try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as e:  # noqa: BLE001
    power = f"unavailable ({e})"
best = {k: min(t) for k, t in times.items()}
print(json.dumps({
    "gpu": torch.cuda.get_device_name(0), "power_limit": power, "B": B, "steps_per_round": steps, "rounds": rounds,
    "ms_per_step": {k: [round(t, 4) for t in ts] for k, ts in times.items()},
    "samples_per_s_best": {k: round(B / best[k] * 1e3, 1) for k in best},
    "dynamic_cost_pct": round((best["dynamic"] / best["static"] - 1) * 100, 2),
    "dynamic_last_step_skipped": skipped, "dynamic_scale": sc.get_scale(),
    "kernel_us_per_launch": {k: round(v, 2) for k, v in kern.items()},
}))
