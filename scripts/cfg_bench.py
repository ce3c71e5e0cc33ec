"""Throughput of classifier-free-guided EDM sampling against unguided sampling, in one process.

Workload: BASELINE configs[1] (bench.py's): `--fields` rows (default 1024) of 128x128 SWE fields, `--timesteps` Heun steps
(default 50, 99 network evaluations), micro-batches of `--chunk` rows (default 256), so a guided evaluation is one network
batch of 2*chunk = 512 rows.  After one warm-up trajectory of each, w = 0 and w = `--w` (default 1.5) are timed
alternately, `--reps` times each, with CUDA events around each full sampling pass (ending in a device synchronise).
Also times one network evaluation on chunk and on 2*chunk rows (CUDA-graph replay with precomputed embedding rows, as the
sampler runs it), averaged over `--eval-reps` replays.

Guided sampling runs the network on twice the rows and the sampler kernels are a fraction of a percent of a trajectory,
so the guided rate is expected near half the unguided one.  Prints one JSON line with the card name and power limit
(read-only nvidia-smi query).  Needs a GPU: there is no CPU path.
"""
import argparse
import copy
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power = [s.strip() for s in out[0].split(",")]
        return name, power
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0), "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fields", type=int, default=1024)
    ap.add_argument("--chunk", type=int, default=256)
    ap.add_argument("--timesteps", type=int, default=50)
    ap.add_argument("--w", type=float, default=1.5)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--eval-reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cfg_bench.py needs a CUDA device")

    from mcedm_b200 import data as D
    from mcedm_b200 import dist as MD
    from mcedm_b200.config import compose
    from mcedm_b200.mcedm import PlMcedm, precond_scalars
    from mcedm_b200.utils import randomize_zero_init

    dev = torch.device("cuda", 0)
    cfg = compose("config_adm_edm_mcedm_res32", ["system=swe_per", f"diff_sampler.timesteps={args.timesteps}"])
    torch.manual_seed(1)
    pl = PlMcedm(copy.deepcopy(cfg.model.hparams))
    randomize_zero_init(pl.model, 2)
    pl.ema_model.ma_model.load_state_dict(pl.model.state_dict())
    pl = pl.to(dev).eval()
    st = D.field_stats("swe_per", 16)
    pl.normalizer_input.set_stats(st["input_mean"].to(dev), st["input_std"].to(dev))
    pl.normalizer_target.set_stats(st["target_mean"].to(dev), st["target_std"].to(dev))
    # bench.py's conditioning: 16 distinct fields repeated to `--fields` rows, u missing
    h, _, _, u, masks = D.make_batch("swe_per", 16, "eval", seed=0)
    state = pl.data_transform(h.to(dev), u.to(dev))
    mask = masks["u"].to(dev)
    torch.manual_seed(cfg.seed)
    cond = pl.get_cond_in(state, mask, None, None).permute(0, 3, 1, 2).repeat(args.fields // 16, 1, 1, 1).contiguous()
    mask = mask.permute(0, 3, 1, 2).repeat(args.fields // 16, 1, 1, 1).contiguous()
    hu = torch.empty(args.fields, 2, 128, 128, device=dev)
    sparams = {}
    for w in (0.0, args.w):
        sparams[w] = copy.deepcopy(cfg.diff_sampler)
        sparams[w].w = w

    def run(w):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        xs = MD.sample_rows(pl, hu, cond, mask, sparams[w], return_last=True, chunk=args.chunk)
        e1.record()
        torch.cuda.synchronize()
        assert torch.isfinite(xs).all()
        return e0.elapsed_time(e1) / 1e3

    for w in sparams:
        run(w)
    times = {w: [] for w in sparams}
    for _ in range(args.reps):
        for w in sparams:
            times[w].append(run(w))
    rate = {w: args.fields / (sum(t) / len(t)) for w, t in times.items()}

    # one network evaluation on chunk and 2*chunk rows, replayed as the sampler replays it
    eng = pl.ema_model.ma_model.engine()
    table = eng.embedding_table(torch.tensor([precond_scalars(1.0)[3]], device=dev))
    eval_ms = {}
    for rows in (args.chunk, 2 * args.chunk):
        g = torch.Generator(device=dev).manual_seed(rows)
        x = torch.randn(rows, 2, 128, 128, device=dev, generator=g)
        c = torch.randn(rows, 2, 128, 128, device=dev, generator=g)
        nl = torch.zeros(1, device=dev)
        out = torch.empty(rows, 2, 128, 128, device=dev)
        ss = table[:, 0] if table is not None else None
        for _ in range(3):
            eng.forward_static(x, nl, c, out, use_graph=True, ss_rows=ss)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.eval_reps):
            eng.forward_static(x, nl, c, out, use_graph=True, ss_rows=ss)
        e1.record()
        torch.cuda.synchronize()
        eval_ms[rows] = e0.elapsed_time(e1) / args.eval_reps

    name, power = card()
    print(json.dumps(dict(
        metric="edm_sampled_fields_per_sec", unit="fields/s", gpu=name, power_limit=power,
        workload=dict(fields=args.fields, chunk=args.chunk, timesteps=args.timesteps, net_evals=2 * args.timesteps - 1,
                      guided_net_batch=2 * args.chunk),
        unguided=dict(w=0.0, fields_per_s=rate[0.0], seconds=times[0.0]),
        guided=dict(w=args.w, fields_per_s=rate[args.w], seconds=times[args.w]),
        ratio_guided_over_unguided=rate[args.w] / rate[0.0],
        eval_ms={f"{r}_rows": v for r, v in eval_ms.items()},
    )))


if __name__ == "__main__":
    main()
