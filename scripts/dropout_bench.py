"""Cost of dropout in the fp16 training plan: graph-replayed training steps of PlMcedm (forward + loss, backward,
optimizer + EMA) at p = 0 and p = 0.1 on one GPU, alternated in rounds after a warm-up and timed with CUDA events, plus
the per-launch time of the two dropout kernels at the shapes the B = 32 step runs them.  Prints one JSON line with the
card name and its power limit, read in the same run.
usage: python scripts/dropout_bench.py [B] [steps per round] [rounds]"""
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

B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 5
dev = torch.device("cuda:0")
cfg = compose("config_adm_edm_mcedm_res32", ["system=swe_per"])
h, tg, xg, u, mask = D.make_batch("swe_per", B, "train", seed=0)
batch = tuple(t.to(dev) for t in (h, tg, xg, u, mask))
st = D.field_stats("swe_per", 16)


def module(p):
    hp = copy.deepcopy(cfg.model.hparams)
    hp.model.dropout = p
    torch.manual_seed(1)
    pl = PlMcedm(hp)
    randomize_zero_init(pl.model, 2)
    pl = pl.to(dev).train()
    pl.normalizer_input.set_stats(st["input_mean"].to(dev), st["input_std"].to(dev))
    pl.normalizer_target.set_stats(st["target_mean"].to(dev), st["target_std"].to(dev))
    opt = pl.configure_optimizers()["optimizer"]
    opt.max_grad_norm = 1.0
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


mods = {p: module(p) for p in (0.0, 0.1)}
for p, (pl, opt) in mods.items():
    run(pl, opt, 5)                                   # capture + warm-up
L.check_watchdog()
times = {p: [] for p in mods}
for _ in range(rounds):
    for p, (pl, opt) in mods.items():
        times[p].append(run(pl, opt, steps))
L.check_watchdog()


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
eng = mods[0.1][0].model.engine()
thr, scale = eng.dropout_args()
rng = eng.dropout_rng(dev)
kern = {}
for H in (128, 64, 32):
    if H <= 64:
        import ctypes as C
        pc, bc = C.c_int(0), C.c_int(0)
        lib.mcedm_flat_geometry(H, H, C.byref(pc), C.byref(bc))
        pitch, blk = pc.value, bc.value
        x = torch.zeros(B * blk, 64, device=dev, dtype=torch.float16)
    else:
        pitch, blk = 0, 0
        x = torch.zeros(B, H, H, 64, device=dev, dtype=torch.float16)
    x.normal_()
    y = torch.zeros_like(x)
    coef = torch.cat([torch.ones(B, 64), torch.zeros(B, 64)], 1).to(dev)
    st_ = L.stream_ptr()
    kern[f"gn_apply16_dropout_{H}"] = kernel_us(lambda: lib.mcedm_gn_apply16_dropout(
        L.ptr(x), pitch, blk, L.ptr(coef), B, H, H, pitch, blk, L.ptr(y), thr, scale, 3, L.ptr(rng), 1, st_))
    kern[f"gn_apply16_{H}"] = kernel_us(lambda: lib.mcedm_gn_apply16(
        L.ptr(x), pitch, blk, L.ptr(coef), 1, 0, B, H, H, pitch, blk, L.ptr(y), None, 1, st_))
    kern[f"dropout_bwd16_{H}"] = kernel_us(lambda: lib.mcedm_dropout_bwd16(
        L.ptr(y), pitch, blk, B, H, H, thr, scale, 3, L.ptr(rng), 1, st_))
L.check_watchdog()

try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as e:  # noqa: BLE001
    power = f"unavailable ({e})"
best = {p: min(t) for p, t in times.items()}
print(json.dumps({
    "gpu": torch.cuda.get_device_name(0), "power_limit": power, "B": B, "steps_per_round": steps, "rounds": rounds,
    "ms_per_step": {str(p): [round(t, 4) for t in ts] for p, ts in times.items()},
    "samples_per_s_best": {str(p): round(B / best[p] * 1e3, 1) for p in best},
    "dropout_cost_pct": round((best[0.1] / best[0.0] - 1) * 100, 2),
    "kernel_us_per_launch": {k: round(v, 2) for k, v in kern.items()},
}))
