"""Benchmark of the m-cedm hot path on B200: EDM-sampled fields / second.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPU cores
    python bench.py ... --dump-outputs DIR                   # also writes the last timed step's fields to DIR/fields.npy

Workload (BASELINE.json configs[1]): `mcedm edm_sampler Heun sampling, n_samples=1024 of 128x128 SWE
fields` — stochastic Heun, 50 steps (99 U-Net evaluations per field), observed-state mask blending,
synthetic SWE-periodic-shaped (h,u) fields, random-init ("stress") weights of the ADM U-Net.  One STEP =
one pass of the hot path over one batch = `--fields` rows IN TOTAL (default 1024, configs[1] as written: "n_samples=1024
... sharded over 1/2/4/8 B200", STRONG scaling: 1024 / N rows per GPU) sampled through
`mcedm_b200.dist.sample_edm_sharded`: every rank runs its contiguous row block in micro-batches of `--chunk` rows and the
step ends with ONE NCCL all-gather of the final fp64 fields, inside the timed region (the only data-path collective;
models/mcedm.py:352-386 stacks the same rows on one GPU).  `value` = rows of all ranks / max-over-ranks device time with
inputs resident in HBM.  `e2e` = the same call from pinned HOST buffers, with the H2D copies of each rank's (cond, mask)
block and rank 0's D2H copy of the gathered fp64 result inside the timed region.  `--scaling weak` keeps `--fields` rows
PER GPU; under N > 1 the strong run also reports that figure as the `weak` key.

Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.
Inputs (several GB of 16-bit activations per 256-row chunk) exceed the 126 MB L2 many times over, so no
explicit L2 flush is needed between iterations (stated in config.l2).
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_PER_EVAL = 18.797e9          # per sample per U-Net forward (BASELINE.md §2)
EVALS_PER_FIELD = 99
DUMP_ROWS = 128                    # 128 fp64 fields of 2 x 128 x 128 = 32 MiB per dump


_STDOUT = sys.stdout


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--fields", type=int, default=1024, help="rows sampled per step: in total (strong) / per GPU (weak)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--no-gpu-torch-baseline", action="store_true")
    ap.add_argument("--chunk", type=int, default=256, help="micro-batch of rows per sampler launch sequence")
    ap.add_argument("--timesteps", type=int, default=50)
    ap.add_argument("--ref-fields", type=int, default=1, help="fields per step of the CPU reference arm")
    ap.add_argument("--cpu-baseline-fields", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--train-batch", type=int, default=32, help="training samples per GPU per step (config 3: 256 / 8)")
    ap.add_argument("--train-steps", type=int, default=20)
    ap.add_argument("--no-train", action="store_true", help="skip the training-throughput measurement")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the fields the last timed step returned as DIR/fields.npy "
                         f"(float64; at most {DUMP_ROWS} rows, a fixed seeded sample of them when there are more)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm only")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(tensor=float(d["bf16_tflops"]), tensor_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    hbm=float(d["hbm_gbs"]), source="measured (MEASURED_PEAKS.json)")
    return dict(tensor=1590.0, tensor_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm (oracle port) on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_sample_fields(n_fields, timesteps, seed=0):
    """Times `n_fields` full trajectories of the oracle's sample_edm on all host cores. Returns (seconds, threads)."""
    import torch

    from mcedm_b200 import data as D
    from mcedm_b200.adm_blocks import DhariwalUNet
    from mcedm_b200.config import compose
    from mcedm_b200.utils import randomize_zero_init
    from oracle import edm_oracle as O

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    cfg = compose("config_adm_edm_mcedm_res32")
    torch.manual_seed(1)
    net = DhariwalUNet(copy.deepcopy(cfg.model.hparams))
    randomize_zero_init(net, 2)
    sd = {k: v.detach() for k, v in net.state_dict().items()}
    h, tg, xg, u, masks = D.make_batch("swe_per", n_fields, "eval", seed=seed)
    st = D.field_stats("swe_per", 16)
    state = torch.cat([(h - st["input_mean"]) / st["input_std"], (u - st["target_mean"]) / st["target_std"]], -1)
    mask = masks["u"]
    g = torch.Generator().manual_seed(seed)
    cond = O.get_cond_in(state, mask, torch.randn(state.shape, generator=g)).permute(0, 3, 1, 2).contiguous()
    mask_c = mask.permute(0, 3, 1, 2).contiguous()
    sp = dict(cfg.diff_sampler)
    sp["timesteps"] = timesteps
    noise = torch.randn(mask_c.shape, generator=g)
    t0 = time.perf_counter()
    with torch.no_grad():
        O.sample_edm(sd, dict(cfg.model.hparams.model), noise, cond, mask_c, sp,
                     lambda i, x: torch.randn(x.shape, dtype=x.dtype, generator=g))
    return time.perf_counter() - t0, threads


def cpu_train_step(batch, seed=0):
    """Times one reference-algorithm training step (loss + backward through the oracle, fp32 autograd) on all host
    cores. Returns (seconds, threads)."""
    import torch

    from mcedm_b200 import data as D
    from mcedm_b200.adm_blocks import DhariwalUNet
    from mcedm_b200.config import compose
    from mcedm_b200.utils import randomize_zero_init
    from oracle import edm_oracle as O

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    cfg = compose("config_adm_edm_mcedm_res32")
    torch.manual_seed(1)
    net = DhariwalUNet(copy.deepcopy(cfg.model.hparams))
    randomize_zero_init(net, 2)
    sd = {k: v.detach().clone().requires_grad_(v.dtype.is_floating_point and "resample" not in k)
          for k, v in net.state_dict().items()}
    h, tg, xg, u, mask = D.make_batch("swe_per", batch, "train", seed=seed)
    st = D.field_stats("swe_per", 16)
    state = torch.cat([(h - st["input_mean"]) / st["input_std"], (u - st["target_mean"]) / st["target_std"]], -1)
    g = torch.Generator().manual_seed(seed)
    x = state.permute(0, 3, 1, 2).contiguous()
    mask_c = mask.permute(0, 3, 1, 2).contiguous()
    cond = O.get_cond_in(state, mask, torch.randn(state.shape, generator=g)).permute(0, 3, 1, 2).contiguous()
    noise = torch.randn(x.shape, generator=g)
    sigma = (torch.randn([batch, 1, 1, 1], generator=g) * 1.2 - 1.2).exp()
    t0 = time.perf_counter()
    loss, _ = O.training_loss(sd, dict(cfg.model.hparams.model), x, sigma, noise, cond, mask_c)
    loss.backward()
    return time.perf_counter() - t0, threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    for _ in range(min(args.warmup, 1)):
        cpu_sample_fields(1, max(2, args.timesteps // 10))
    times = []
    for _ in range(args.steps):
        dt, threads = cpu_sample_fields(args.ref_fields, args.timesteps)
        times.append(dt)
    total = sum(times)
    value = args.ref_fields * args.steps / total
    sample = f"{args.ref_fields} field(s) x {args.timesteps} Heun steps ({2 * args.timesteps - 1} net evals) per step, fp32, torch CPU"
    line = dict(impl="reference", metric="edm_sampled_fields_per_sec", value=value, unit="fields/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * total / args.steps, higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                config=dict(workload="mcedm edm_sampler Heun sampling of 128x128 SWE fields (BASELINE configs[1])",
                            timesteps=args.timesteps, fields_per_step=args.ref_fields),
                cpu_baseline=dict(value=value, unit="fields/s", cores=threads, kind="port", sample=sample),
                e2e=dict(value=value, unit="fields/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line), file=_STDOUT, flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    from mcedm_b200 import _lib as L
    from mcedm_b200 import data as D
    from mcedm_b200 import dist as MD
    from mcedm_b200.config import compose
    from mcedm_b200.mcedm import PlMcedm
    from mcedm_b200.utils import randomize_zero_init

    rank, world, local = MD.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cfg = compose("config_adm_edm_mcedm_res32", ["system=swe_per", f"diff_sampler.timesteps={args.timesteps}"])
    torch.manual_seed(1)
    pl = PlMcedm(copy.deepcopy(cfg.model.hparams))
    randomize_zero_init(pl.model, 2)
    pl.ema_model.ma_model.load_state_dict(pl.model.state_dict())
    pl = pl.to(dev).eval()
    pl.use_cuda_graph = not args.no_graph
    sp = cfg.diff_sampler
    st = D.field_stats("swe_per", 16)
    pl.normalizer_input.set_stats(st["input_mean"].to(dev), st["input_std"].to(dev))
    pl.normalizer_target.set_stats(st["target_mean"].to(dev), st["target_std"].to(dev))

    # synthetic conditioning: 16 distinct fields, each repeated rows/16 times (test_step's repeat(n_samples)); the SAME
    # rows on every rank (all ranks hold the full host-side request, each touches only its block)
    strong = args.scaling == "strong"
    rows_total = args.fields if strong else args.fields * world
    lo, hi = MD.shard_rows(rows_total, rank, world)
    rows = hi - lo
    chunk = min(args.chunk, rows)
    b = 16 if rows_total % 16 == 0 else 1
    h, tg, xg, u, masks = D.make_batch("swe_per", b, "eval", seed=0)
    state = pl.data_transform(h.to(dev), u.to(dev))
    mask = masks["u"].to(dev)
    torch.manual_seed(cfg.seed)
    cond1 = pl.get_cond_in(state, mask, None, None).permute(0, 3, 1, 2).contiguous()
    cond_all = cond1.repeat(rows_total // b, 1, 1, 1).contiguous()
    mask_all = mask.permute(0, 3, 1, 2).repeat(rows_total // b, 1, 1, 1).contiguous()
    hu_all = torch.empty(rows_total, 2, 128, 128, device=dev)          # shape-only argument of sample_edm
    host_cond = cond_all.cpu().pin_memory()
    host_mask = mask_all.cpu().pin_memory()
    host_out = torch.empty(rows_total, 1, 128, 128, 2, dtype=torch.float64).pin_memory() if rank == 0 else None
    torch.manual_seed(MD.rank_seed(cfg.seed, rank))                     # per-rank noise streams

    def one_step(e2e: bool):
        # the public multi-GPU call: this rank's block in micro-batches + ONE all-gather of the fp64 fields
        xs = MD.sample_edm_sharded(pl, hu_all, host_cond if e2e else cond_all, host_mask if e2e else mask_all, sp,
                                   return_last=True, chunk=chunk)
        if e2e and rank == 0:
            host_out.copy_(xs, non_blocking=True)
        return xs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    for _ in range(args.warmup):
        one_step(False)
    checks = multi_gpu_checks(pl, cfg, dev, rank, world) if world > 1 else None
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    launches0 = L.LAUNCHES[0]
    last = []

    def timed_step():
        last.clear()                                  # the previous step's output is freed before the next one runs
        last.append(one_step(False))

    ms = timed(timed_step, args.steps)
    launches = L.LAUNCHES[0] - launches0
    clk = clocks.stop() if rank == 0 else None
    xs = last[0]
    assert xs.shape == (rows_total, 1, 128, 128, 2) and xs.dtype == torch.float64
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, xs)          # before the e2e steps below reuse the sampler's buffers
    one_step(True)
    ms_e2e = timed(lambda: one_step(True), args.steps)
    L.check_watchdog()

    value = rows_total * args.steps / (ms / 1e3)
    e2e_value = rows_total * args.steps / (ms_e2e / 1e3)

    # weak-scaling figure next to the strong one (N > 1 only; at N = 1 they are the same run): `--fields` rows per GPU
    weak = None
    if strong and world > 1:
        wl, wh = 0, args.fields
        wc = min(args.chunk, args.fields)
        cw, mw = cond_all[:1].expand(args.fields, -1, -1, -1).contiguous(), mask_all[:1].expand(args.fields, -1, -1, -1).contiguous()
        hw = torch.empty(args.fields, 2, 128, 128, device=dev)

        def weak_step():
            MD.gather_rows(MD.sample_rows(pl, hw, cw, mw, sp, True, wc).contiguous(), args.fields * world)

        weak_step()
        n_w = max(1, min(args.steps, 2))
        ms_w = timed(weak_step, n_w)
        weak = dict(value=args.fields * world * n_w / (ms_w / 1e3), unit="fields/s", fields_per_gpu=args.fields, steps=n_w,
                    ms_per_step=ms_w / n_w, scaling="weak", collective="one NCCL all-gather of the fp64 fields per step")

    # ---- roofline of the dominant kernel: conv_igemm (3x3 implicit GEMM, N = 64), CUDA events per launch
    roof = None
    if rank == 0:
        pk = peaks()
        unet = pl.ema_model.ma_model
        x = torch.randn(chunk, 2, 128, 128, device=dev)
        prof = unet.engine().profile_kernels(x, torch.tensor([0.1], device=dev), cond_all[:chunk])
        fused = unet.engine().fused and unet.engine().infer_fmt == 1

        def grp(names, pred=lambda p: True):
            sel = [p for p in prof if p["name"] in names and pred(p)]
            return sel, sum(p["flops"] for p in sel), sum(p["bytes"] for p in sel), sum(p["ms"] for p in sel)

        # dominant kernel: the row-resident 3x3 implicit GEMM of the 128x128 level (68 % of the network's FLOPs)
        dom_name = "conv_rows_fused" if fused else "conv_rows"
        dom, fl, by, t = grp((dom_name,), lambda p: p["flops"] > 1e9 * chunk)      # N = 64 launches (not the 16-wide head)
        flat, fl_f, by_f, t_f = grp(("conv_flat_fused", "conv_flat"))
        att, fl_a, by_a, t_a = grp(("attention",))
        gn, fl_g, by_g, t_g = grp(("gn_apply16", "gn_apply"))
        cin, fl_i, by_i, t_i = grp(("conv_in_tc16", "conv_in16", "conv_in"))
        total_ms = sum(p["ms"] for p in prof)
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")    # dram bytes per launch from an `ncu --set full` capture
        if os.path.exists(tpath):
            with open(tpath) as f:
                traffic = json.load(f).get("conv_rows_kernel<64,fused>" if fused else "conv_rows_kernel<64>")
        achieved = fl / (t * 1e-3) / 1e12
        roof = dict(bound="tensor", achieved=achieved, peak=pk["tensor_sustained"], unit="TFLOP/s",
                    frac=achieved / pk["tensor_sustained"], frac_burst=achieved / pk["tensor"], peak_burst=pk["tensor"],
                    traffic=traffic,
                    traffic_note=("dram__bytes_read + dram__bytes_write of ONE launch of the variant with a 16-bit residual "
                                  "(3 tensor streams of 537 MB at 256 samples = 1.61 GB algorithmic), ncu --set full, "
                                  "profiles/r2_ncu_conv_rows.md launch 5") if fused and traffic else None,
                    kernel=("conv_rows_kernel<64, fused> (GroupNorm+SiLU-fused 3x3 implicit GEMM at 128x128, 64 input "
                            "channels -> 64 per launch, 16-bit activations)" if fused else
                            "conv_rows_kernel<64> (3x3 implicit GEMM at 128x128, 64->64 channels per launch)"),
                    launches_per_eval=len(dom), flops_per_eval=fl, bytes_per_eval=by, ms_per_eval=t,
                    achieved_gbs=by / max(1e-9, t) / 1e6, share_of_eval_ms=t / total_ms, eval_ms_sum_of_launches=total_ms,
                    launches_in_eval=len(prof),
                    peak_source=pk["source"] + ", sustained bf16 figure (kernel timed inside a long step)",
                    other_kernels=[
                        dict(kernel="conv_flat_kernel<64> (3x3 at 64x64 / 32x32, padded-flat)", bound="tensor", unit="TFLOP/s",
                             achieved=fl_f / max(1e-9, t_f) / 1e9, peak=pk["tensor_sustained"], ms_per_eval=t_f,
                             launches_per_eval=len(flat)),
                        dict(kernel="attn_kernel (softmax(QK^T/8)V at 32x32, L=1024)", bound="tensor", unit="TFLOP/s",
                             achieved=fl_a / max(1e-9, t_a) / 1e9, peak=pk["tensor_sustained"], ms_per_eval=t_a,
                             launches_per_eval=len(att)),
                        dict(kernel="gn_apply (stand-alone GroupNorm+SiLU+resample passes that remain)", bound="hbm",
                             unit="GB/s", achieved=by_g / max(1e-9, t_g) / 1e6, peak=pk["hbm"], ms_per_eval=t_g,
                             launches_per_eval=len(gn)),
                        dict(kernel="conv_in_tc (first 3x3 conv on cat([cond, x]), tensor cores, 2 MMAs per input row)", bound="hbm", unit="GB/s",
                             achieved=by_i / max(1e-9, t_i) / 1e6, peak=pk["hbm"], ms_per_eval=t_i,
                             launches_per_eval=len(cin))],
                    end_to_end_tflops=value * EVALS_PER_FIELD * FLOPS_PER_EVAL * (args.timesteps * 2 - 1) / 99 / 1e12 / world)
        roof["other_kernels"] += sampler_kernel_rooflines(dev, pk, chunk)
        roof["other_kernels"] += pde_kernel_rooflines(pl, dev, pk)
        roof["eval_frac_sustained"] = roof["end_to_end_tflops"] / pk["tensor_sustained"]
    train = None
    if not args.no_train:
        train = measure_training(args, cfg, dev, rank, world, barrier)
    cpu = None
    # the CPU baseline is a rank-0, N = 1 measurement: under torchrun the other ranks spin in the NCCL barrier on the
    # same host cores (and OMP_NUM_THREADS is forced to 1), which turned a 3 s sample into a 280 s one at N = 8
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        if train is not None:
            dt, threads = cpu_train_step(2)
            train["cpu_baseline"] = dict(value=2 / dt, unit="samples/s", cores=threads, kind="port",
                                         sample="one training step (loss + backward) of 2 samples through the oracle "
                                                f"port of the reference algorithm, torch CPU fp32 autograd, {threads} threads")
        dt, threads = cpu_sample_fields(args.cpu_baseline_fields, args.timesteps)
        cpu = dict(value=args.cpu_baseline_fields / dt, unit="fields/s", cores=threads, kind="port",
                   sample=f"{args.cpu_baseline_fields} field x {args.timesteps} Heun steps of the same workload "
                          f"(oracle port of the reference algorithm, torch CPU fp32, {threads} threads)")
    gpu_torch = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.no_gpu_torch_baseline:
        gpu_torch = gpu_torch_baseline(dev, cfg, chunk, args.timesteps)
    if rank == 0:
        line = dict(metric="edm_sampled_fields_per_sec", value=value, unit="fields/s", n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=ms / args.steps, higher_is_better=True, scaling=args.scaling,
                    vs_baseline=None, dtype="fp16" if pl.ema_model.ma_model.engine().infer_fmt else "bf16", data="synthetic",
                    config=dict(operands="fp16 tensor-core operands AND fp16 activation storage in HBM (saturating), GroupNorm+SiLU "
                                         "applied inside the convs; fp32 accumulation / statistics, fp64 sampler state; per-step "
                                         "denoiser error 1.4e-3 vs the reference (bar 1e-2)",
                                workload=(f"mcedm edm_sampler Heun sampling, n_samples={rows_total} of 128x128 SWE fields "
                                          f"sharded over {world} B200 (BASELINE configs[1])" if strong else
                                          f"mcedm edm_sampler Heun sampling, n_samples={args.fields} of 128x128 SWE fields "
                                          "per GPU (BASELINE configs[1], weak-scaling variant)"),
                                fields_total=rows_total, fields_per_gpu=rows, micro_batch=chunk,
                                timesteps=args.timesteps, net_evals_per_field=2 * args.timesteps - 1,
                                weights="random init (seed 1) + randomised zero-init tensors (seed 2)",
                                parallelism=f"independent rows sharded over {world} GPU(s) (contiguous blocks), no communication "
                                            "during the 50-step loop",
                                collective=("one NCCL all-gather of the final fp64 fields per step, inside the timed region"
                                            if world > 1 else "none (1 GPU)"),
                                cuda_graph=not args.no_graph,
                                l2="inputs per iteration (GBs of activations) exceed the 126 MB L2; no explicit flush"),
                    clocks=clk,
                    e2e=dict(value=e2e_value, unit="fields/s", h2d_bytes_per_step=int(2 * rows_total * 2 * 128 * 128 * 4),
                             d2h_bytes_per_step=int(rows_total * 2 * 128 * 128 * 8), ms_per_step=ms_e2e / args.steps,
                             api="mcedm_b200.dist.sample_edm_sharded(PlMcedm, ...) from pinned host cond / mask; rank 0 "
                                 "copies the gathered fp64 fields back to pinned host memory"),
                    gpu_launches=launches, roofline=roof, cpu_baseline=cpu, gpu_torch_baseline=gpu_torch, weak=weak,
                    checks=checks, train=train)
        print(json.dumps(line), file=_STDOUT, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(out_dir, xs):
    """Writes the fp64 fields `xs` [rows, 1, 128, 128, 2] of one sampling step as out_dir/fields.npy: every row when there
    are at most DUMP_ROWS, else DUMP_ROWS rows drawn by a fixed seed and kept in ascending order, so that two builds run
    with the same arguments write the same rows and can be compared element for element."""
    import numpy as np
    import torch

    n = xs.shape[0]
    rows = torch.arange(n)
    if n > DUMP_ROWS:
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "fields.npy"), xs[rows.to(xs.device)].cpu().numpy())


def multi_gpu_checks(pl, cfg, dev, rank, world):
    """On-box, N > 1: the rows gathered from the N ranks are bit-identical to the same rows sampled on ONE GPU with the
    same per-row noise (16 rows, 3 Heun steps; noise keyed by the GLOBAL row index, so it does not depend on the
    sharding).  Every rank takes part in the gather; rank 0 repeats the whole batch alone and compares."""
    import torch

    from mcedm_b200 import dist as MD

    n, steps = 2 * world if 2 * world >= 16 else 16, 3
    sp = copy.deepcopy(cfg.diff_sampler)
    sp.timesteps = steps
    g = torch.Generator().manual_seed(11)
    cond = torch.randn(n, 2, 128, 128, generator=g).to(dev)
    mask = torch.zeros(n, 2, 128, 128)
    mask[::2, 1] = 1.0
    mask[1::2, 0] = 1.0
    mask = mask.to(dev)
    hu = torch.zeros(n, 2, 128, 128, device=dev)

    def hook_for(row0):
        count = [0]

        def hook(kind, like):
            k = count[0]
            count[0] += 1
            out = torch.empty(like.shape, dtype=like.dtype)
            for r in range(like.shape[0]):
                gr = torch.Generator().manual_seed(100003 * (row0 + r) + k)
                out[r] = torch.randn(like.shape[1:], dtype=like.dtype, generator=gr)
            return out.to(like.device)
        return hook

    lo, hi = MD.shard_rows(n, rank, world)
    pl._noise_hook = hook_for(lo)
    try:
        gathered = MD.sample_edm_sharded(pl, hu, cond, mask, sp, return_last=True)
        ok = None
        if rank == 0:
            pl._noise_hook = hook_for(0)
            alone = pl.sample_edm(hu, cond, mask, sp, return_last=True)
            ok = bool(torch.equal(gathered, alone)) and bool(torch.isfinite(alone).all())
    finally:
        pl._noise_hook = None
    return dict(gathered_rows_equal_single_gpu_run=ok, rows=n, heun_steps=steps) if rank == 0 else None


def sampler_kernel_rooflines(dev, pk, B, n=20):
    """Achieved HBM GB/s of the sampler-state kernels (K5: churn / Euler / Heun correction with mask blending, fp64 state)
    at the bench's micro-batch: algorithmic bytes per state element = every operand read once + every result written
    once (churn 8+8+4 in, 8+4 out; euler 8+4+4 in, 8+8+4 out; correct 8+8+4+8+4 in, 8 out), CUDA events around `n`
    launches on the launching stream; operands (17-34 MB per tensor at B = 256 ... x4-6 tensors) exceed nothing but are
    streamed once per launch, as inside the sampler where 9 ms of network traffic separates two uses."""
    import torch

    from mcedm_b200 import _lib as L

    lib = L.lib()
    f64 = dict(device=dev, dtype=torch.float64)
    xa, xb, xc, xd = (torch.randn(B, 2, 128, 128, **f64) for _ in range(4))
    Fb, xin = torch.randn(B, 2, 128, 128, device=dev), torch.empty(B, 2, 128, 128, device=dev)
    mask = torch.ones(B, 2, 128, 128, device=dev)
    tot = xa.numel()
    st = L.stream_ptr()
    flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8)           # > 126 MB L2: written between launches
    out = []
    for name, fn, per in (
            ("edm_churn_kernel (x_hat = x + coef*eps*m, x_in = c_in*x_hat; fp64 state)",
             lambda: L.check(lib.mcedm_edm_churn(L.ptr(xa), L.ptr(xb), L.ptr(mask), 1.0, 0.5, tot, L.ptr(xc), L.ptr(xin), st)), 32.0),
            ("edm_euler_kernel (D = c_skip*x + c_out*F, d_cur, Euler step with mask blending)",
             lambda: L.check(lib.mcedm_edm_euler(L.ptr(xa), L.ptr(Fb), L.ptr(mask), 2.0, 1.5, 0.2, 0.9, 0.5, tot, L.ptr(xd),
                                                 L.ptr(xc), L.ptr(xin), None, st)), 36.0),
            ("edm_correct_kernel (Heun correction with mask blending)",
             lambda: L.check(lib.mcedm_edm_correct(L.ptr(xa), L.ptr(xc), L.ptr(Fb), L.ptr(xd), L.ptr(mask), 2.0, 1.5, 0.2, 0.9,
                                                   tot, L.ptr(xb), None, st)), 40.0)):
        fn()
        torch.cuda.synchronize()
        tsum = 0.0
        for _ in range(n):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            tsum += e0.elapsed_time(e1)
        ms = tsum / n
        out.append(dict(kernel=name, bound="hbm", unit="GB/s", achieved=per * tot / ms / 1e6, peak=pk["hbm"],
                        frac=per * tot / ms / 1e6 / pk["hbm"], ms_per_launch=ms, batch=B, l2="flushed between launches"))
    return out


def gpu_torch_baseline(dev, cfg, B, timesteps, n=5):
    """Library-GPU comparator (informational; NOT the reference arm and not the product path): the oracle port of the
    reference's U-Net forward (plain torch ops: cuDNN convolutions, F.group_norm, einsum attention — what the reference's
    own code runs on a GPU under this torch build) on the same device at the same micro-batch, (a) fp32 with TF32 allowed,
    (b) under bf16 autocast.  Reported as ms per evaluation and the fields/s it would bound (99 evaluations per field)."""
    import torch

    from mcedm_b200.adm_blocks import DhariwalUNet
    from mcedm_b200.utils import randomize_zero_init
    from oracle import edm_oracle as O

    torch.manual_seed(1)
    net = DhariwalUNet(copy.deepcopy(cfg.model.hparams))
    randomize_zero_init(net, 2)
    sd = {k: v.detach().to(dev) for k, v in net.state_dict().items()}
    mc = dict(cfg.model.hparams.model)
    x = torch.randn(B, 2, 128, 128, device=dev)
    cond = torch.randn(B, 2, 128, 128, device=dev)
    nl = torch.full((1,), 0.1, device=dev)
    res = {}
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.benchmark = True
    try:
        for name, ctx in (("fp32_tf32", torch.autocast("cuda", enabled=False)),
                          ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
            try:
                with torch.no_grad(), ctx:
                    for _ in range(2):
                        O.unet_forward(sd, mc, x, nl, cond)
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(n):
                        O.unet_forward(sd, mc, x, nl, cond)
                    e1.record()
                    torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / n
                res[name] = dict(ms_per_eval=ms, tflops=FLOPS_PER_EVAL * B / ms / 1e9,
                                 fields_per_s_bound=B / ((2 * timesteps - 1) * ms * 1e-3))
            except Exception as e:  # noqa: BLE001  (an informational leg must not take the bench down)
                res[name] = dict(error=f"{type(e).__name__}: {e}"[:200])
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
    res.update(batch=B, what="oracle port of DhariwalUNet.forward (models/adm_blocks.py:364-404) in torch eager on cuda:0 "
                             f"(torch {torch.__version__}, cuDNN); network evaluation only, sampler-state updates excluded")
    return res


def pde_kernel_rooflines(pl, dev, pk, B=256, n=20):
    """Achieved HBM GB/s of the PDE-residual kernels (K6) on a sampled batch in the sampler's own layout (float64 NCHW
    state): algorithmic bytes = 2 planes x 8 B read per cell (+ 8 B written per cell for the gradient), CUDA events
    around `n` launches on the launching stream; the 268 MB batch exceeds nothing but is streamed once per launch."""
    import torch

    x = torch.randn(B, 2, 128, 128, device=dev, dtype=torch.float64)
    f = pl.pde_loss
    nh, nu = pl.normalizer_input, pl.normalizer_target
    out = []
    for name, fn, byts in (
            ("swe_fv_loss_kernel (FORCE finite-volume residual + sum, fp64 NCHW state in)",
             lambda: f.residual(x[:, 0], x[:, 1], nh, nu), B * 128 * 128 * 16.0),
            ("swe_fv_grad_kernel (analytic residual gradient, one image row per CTA)",
             lambda: f.gradient(x[:, 0], x[:, 1], nh, nu, mode=0), B * 128 * 128 * 24.0)):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        out.append(dict(kernel=name, bound="hbm", unit="GB/s", achieved=byts / ms / 1e6, peak=pk["hbm"], ms_per_launch=ms,
                        batch=B))
    return out


def measure_training(args, cfg, dev, rank, world, barrier):
    """U-Net train samples/s (BASELINE metric, second half; configs[2]: masked mixed-conditioning EDM training, bf16
    tensor-core operands, data-parallel): every rank runs `--train-batch` samples per step through
    PlMcedm.training_step -> loss.backward() -> [NCCL all-reduce of the flat gradient] -> fused clip+Adam -> EMA."""
    import torch
    import torch.distributed as dist

    from mcedm_b200 import _lib as L
    from mcedm_b200 import data as D
    from mcedm_b200.mcedm import PlMcedm
    from mcedm_b200.utils import randomize_zero_init

    B = args.train_batch
    torch.manual_seed(1)
    pl = PlMcedm(copy.deepcopy(cfg.model.hparams))
    randomize_zero_init(pl.model, 2)
    pl = pl.to(dev).train()
    opt = pl.configure_optimizers()["optimizer"]
    opt.max_grad_norm = 1.0
    opt.grad_scale = 1.0 / world
    st = D.field_stats("swe_per", 16)
    pl.normalizer_input.set_stats(st["input_mean"].to(dev), st["input_std"].to(dev))
    pl.normalizer_target.set_stats(st["target_mean"].to(dev), st["target_std"].to(dev))
    host = [t.pin_memory() for t in D.make_batch("swe_per", B, "train", seed=17 + rank)]
    resident = tuple(t.to(dev) for t in host)

    # e2e: the next batch is copied host -> device on a side stream while the current step runs, and every step's loss
    # is read back through a pinned buffer one step late, so neither transfer stalls the launch queue (round 1 paid
    # ~20 % for a synchronous .item() + H2D per step)
    side = torch.cuda.Stream(device=dev)
    staged = [tuple(torch.empty_like(t, device=dev) for t in host) for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    host_loss = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_done = [torch.cuda.Event(), torch.cuda.Event()]
    losses_read = []

    def prefetch(slot):
        with torch.cuda.stream(side):
            side.wait_event(consumed[slot])                   # the step that last used this slot has finished reading it
            for d, t in zip(staged[slot], host):
                d.copy_(t, non_blocking=True)
            ready[slot].record(side)

    def step(e2e, slot=0):
        if e2e:
            torch.cuda.current_stream().wait_event(ready[slot])
            batch = staged[slot]
        else:
            batch = resident
        opt.zero_grad(set_to_none=True)
        loss = pl.training_step(batch, 0)
        loss.backward()
        if e2e:
            consumed[slot].record()
        if world > 1:
            dist.all_reduce(opt.flat_grads())                 # flat_grads() is idempotent: step() consumes this tensor
        pl.optimizer_step(0, 0, opt)
        return loss

    def timed(e2e, n):
        barrier()
        if e2e:
            for ev in consumed:
                ev.record()
            prefetch(0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            if e2e and i + 1 < n:
                prefetch((i + 1) & 1)
            loss = step(e2e, i & 1)
            if e2e:
                host_loss[i & 1].copy_(loss.detach(), non_blocking=True)      # device -> host read of the step's loss
                loss_done[i & 1].record()
                if i >= 1:
                    loss_done[(i - 1) & 1].synchronize()
                    losses_read.append(float(host_loss[(i - 1) & 1]))
        if e2e:
            loss_done[(n - 1) & 1].synchronize()
            losses_read.append(float(host_loss[(n - 1) & 1]))
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    for _ in range(5):
        step(False)
    checks = None
    if world > 1:
        # replicas saw different batches (seed 17 + rank): identical parameters after 5 steps = the gradient exchange works
        fp = opt.flat_params().double()
        cs = torch.stack([fp.sum(), (fp * torch.arange(fp.numel(), device=dev, dtype=torch.float64)).sum()])
        allc = [torch.empty_like(cs) for _ in range(world)]
        dist.all_gather(allc, cs)
        checks = dict(param_checksums_equal_across_ranks=bool(all(torch.equal(c, allc[0]) for c in allc)), after_steps=5)
    n0 = L.LAUNCHES[0]
    ms = timed(False, args.train_steps)
    launches = L.LAUNCHES[0] - n0
    ms_e2e = timed(True, args.train_steps)
    L.check_watchdog()
    assert len(losses_read) == args.train_steps and all(v == v for v in losses_read), "e2e: a step's loss was not read back"
    per = ms / args.train_steps
    bytes_in = sum(t.numel() * t.element_size() for t in host)
    return dict(metric="unet_train_samples_per_sec", value=B * world * args.train_steps / (ms / 1e3), unit="samples/s",
                ms_per_step=per, batch_per_gpu=B, global_batch=B * world, steps=args.train_steps,
                dtype="fp16" if pl.model.engine().train_plan == "fused16" else "bf16",
                plan=pl.model.engine().train_plan + (": fp16 operands and activations forward and backward, loss-scaled, "
                                                     "fp32 accumulation / statistics / master weights; weight gradients on a "
                                                     "parallel graph branch" if pl.model.engine().train_plan == "fused16" else ""),
                tflops_per_gpu=56.305e9 * B / per / 1e9,
                e2e=dict(value=B * world * args.train_steps / (ms_e2e / 1e3), unit="samples/s",
                         h2d_bytes_per_step=bytes_in, d2h_bytes_per_step=4, ms_per_step=ms_e2e / args.train_steps,
                         how="batch i+1 copied from pinned host memory on a side stream during step i; every step's "
                             "loss read back through a pinned buffer one step late"),
                gpu_launches=launches, checks=checks,
                config=dict(workload="masked mixed-conditioning EDM training step (BASELINE configs[2]): forward + loss + "
                                     "backward + grad all-reduce + clip + Adam + EMA", optimizer="Adam lr 2e-4, clip 1.0, EMA 0.999",
                            parallelism=f"data-parallel over {world} GPU(s), one NCCL all-reduce of the flat fp32 gradient",
                            cuda_graph=True))


if __name__ == "__main__":
    # stdout carries exactly ONE JSON line: anything a library prints on the way goes to stderr — at the file-descriptor
    # level, because NCCL writes its version banner to fd 1 from C (seen in front of the N = 2 line)
    sys.stdout.flush()
    _real_fd = os.dup(1)
    os.dup2(2, 1)
    _STDOUT = os.fdopen(_real_fd, "w")
    sys.stdout = sys.stderr
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
