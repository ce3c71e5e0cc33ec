"""GPU: gradient accumulation on the kernel training path (`UNetEngine.accumulate_grads`,
`Trainer(accumulate_grad_batches)`).

A window of micro-batches covering the 32 samples of test_gpu_train_batch._inputs is held to that file's bars against
its float64 reference of ONE step on all 32 (the EDM loss is a mean over samples, so Σ_k ∇L_k / N over N equal
micro-batches is the full batch's gradient).  Helpers are imported from test_gpu_train_batch."""
import gc
import math
import os
import subprocess
import sys

import pytest
import torch

from test_gpu_train_batch import TOL, _compare, _inputs, _module, _named_params, _step, reference_step, rel

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B = 32


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda")


def _release():
    gc.collect()
    torch.cuda.empty_cache()


@pytest.fixture(autouse=True)
def _release_gpu_memory():
    """Each test builds modules with captured training graphs (reference cycles: a module holds its graphs, a graph its
    module) and the float64 reference's temporaries.  Free them and return the cached blocks, so that tests later in
    the process do not capture a graph while the allocator has to release memory, which a capture does not allow."""
    yield
    _release()


def micro(inp, k, n):
    """micro-batch k of n samples of an _inputs tuple"""
    return tuple(t[k * n:(k + 1) * n].contiguous() for t in inp)


def window(pl, parts, opt=None):
    """One accumulation window over the micro-batches `parts` (N = len(parts)) through pl.forward_loss / backward, then
    the module's optimizer_step hook when `opt` is given: (mean micro-batch loss, [.grad of every parameter])."""
    eng = pl.model.engine()
    eng.accumulate_grads = len(parts)
    try:
        pl.zero_grad(set_to_none=True)
        losses = []
        for x, sigma, noise, cond, mask in parts:
            loss = pl.forward_loss(x, sigma, noise, cond, mask, pl.get_loss_weight(sigma))
            loss.backward()
            losses.append(loss.detach())
        out = torch.stack(losses).mean(), [p.grad.detach().clone() for p in pl.model.parameters()]
        if opt is not None:
            pl.optimizer_step(0, len(parts) - 1, opt)
        return out
    finally:
        eng.accumulate_grads = None


def same(a, b):
    return torch.equal(a[0], b[0]) and all(torch.equal(x, y) for x, y in zip(a[1], b[1]))


@pytest.fixture(scope="module")
def full(dev):
    pl, mcfg = _module(dev)
    inp = _inputs(pl, dev, B, seed=1100)
    yield pl, mcfg, inp, reference_step(_named_params(pl), mcfg, *inp)
    del pl
    _release()


# ------------------------------------------------------------------------------------------------ equivalence
@gpu
@pytest.mark.parametrize("mb", [8, 16])
def test_window_matches_fp64_reference_of_the_full_batch(full, mb):
    """Windows of 4 x 8 and 2 x 16 against the float64 step on all 32 samples, eager and graph-replayed; the two
    paths are bit-identical (every fold and the window fold have a fixed order)."""
    from mcedm_b200 import _lib as L

    pl, _, inp, ref = full
    parts = [micro(inp, k, mb) for k in range(B // mb)]
    pl.use_cuda_graph = False
    eager = window(pl, parts)
    _compare(pl, *eager, ref, f"{B // mb} x {mb} eager")
    pl.use_cuda_graph = True
    graph = window(pl, parts)
    again = window(pl, parts)
    L.check_watchdog()
    assert same(graph, eager) and same(again, eager)


@gpu
def test_window_on_the_fp32_stream_plan(dev):
    """The fp32-stream plan (bf16 operands): 2 x 16 against the float64 step on 32, at that plan's bars
    (test_gpu_train.py), eager and graph-replayed bit-identical."""
    pl, mcfg = _module(dev)
    pl.model.engine().train_plan = "fp32"
    inp = _inputs(pl, dev, B, seed=1200)
    ref_loss, ref_g = reference_step(_named_params(pl), mcfg, *inp)
    parts = [micro(inp, k, 16) for k in range(2)]
    pl.use_cuda_graph = False
    loss, grads = eager = window(pl, parts)
    pl.use_cuda_graph = True
    assert same(window(pl, parts), eager)
    assert pl.model.engine().train_plan == "fp32"
    names = [k for k, _ in pl.model.named_parameters()]
    lerr = abs(float(loss) - ref_loss) / abs(ref_loss)
    glob = rel(torch.cat([g.flatten() for g in grads]), torch.cat([ref_g[k].flatten() for k in names]))
    worst = max(rel(g, ref_g[k]) for k, g in zip(names, grads))
    print(f"fp32-stream 2 x 16: loss err {lerr:.2e}, global {glob:.2e}, worst tensor {worst:.2e}")
    assert lerr < 1e-2 and glob < 2e-2 and worst < 6e-2


# ------------------------------------------------------------------------------------------------ exactness
@gpu
@pytest.mark.parametrize("graph", [False, True])
def test_n1_and_a_doubled_micro_batch_are_the_plain_step_bit_for_bit(dev, graph):
    """accumulate_grads = 1 is the default path bit for bit; so is a window of N = 2 that sees the same micro-batch
    twice (halving is exact, and so is adding two equal halves)."""
    pl, _ = _module(dev)
    pl.use_cuda_graph = graph
    inp = _inputs(pl, dev, B, seed=1300)
    plain = _step(pl, inp)
    assert same(window(pl, [inp]), plain)
    assert same(window(pl, [inp, inp]), plain)


# ------------------------------------------------------------------------------------------------ Trainer loop
class _IndexDM:
    """`n` batches per epoch; a batch is an index into pre-drawn inputs (see _drive)"""

    def __init__(self, n):
        self.n = n

    def setup(self, stage):
        return None

    def train_dataloader(self):
        return list(range(self.n))

    def val_dataloader(self):
        return []


def _drive(pl, inputs):
    """pl.training_step on pre-drawn inputs[batch]; returns the records {'steps', 'ema', 'micro'} the spies fill."""
    rec = dict(steps=[], ema=0, micro=[], losses=[])
    eng = pl.model.engine()

    def training_step(batch, batch_idx):
        x, sigma, noise, cond, mask = inputs[batch]
        loss = pl.forward_loss(x, sigma, noise, cond, mask, pl.get_loss_weight(sigma))
        pl.log("train_loss", loss, on_epoch=True, sync_dist=True)
        rec["losses"].append(loss.detach())
        return loss

    fold = eng.fold_grads

    def fold_spy():
        rec["micro"].append(eng._gflat.clone())          # this backward's micro-batch gradient
        fold()

    opt_step = type(pl).optimizer_step

    def optimizer_step(epoch, batch_idx, optimizer):
        rec["steps"].append((batch_idx, optimizer.flat_grads().clone()))
        opt_step(pl, epoch, batch_idx, optimizer)

    ema_update = pl.ema_model.update

    def ema_spy(model):
        rec["ema"] += 1
        ema_update(model)

    pl.setup = lambda stage=None: None
    pl.training_step = training_step
    pl.optimizer_step = optimizer_step
    pl.ema_model.update = ema_spy
    eng.fold_grads = fold_spy
    return rec


@gpu
def test_trainer_steps_once_per_window(dev):
    """5 batches of 8 per epoch at N = 2 for 2 epochs (graph-replayed): 6 optimizer steps after batches 1, 3, 4,
    global_step 6, 6 EMA updates, each window's gradient (g_a + g_b) / 2 bit for bit and the partial window's half its
    one batch's gradient, 5 train_loss records per epoch; accumulation is off again after fit.  max_steps = 3 stops
    after the 3 windows of the first epoch."""
    from mcedm_b200 import _lib as L
    from mcedm_b200.runner import Trainer

    pl, _ = _module(dev)
    pl.use_cuda_graph = True
    inputs = [_inputs(pl, dev, 8, seed=1400 + i) for i in range(5)]
    rec = _drive(pl, inputs)
    tr = Trainer(max_epochs=2, accumulate_grad_batches=2, check_val_every_n_epoch=100)
    names = []
    record = tr._record
    tr._record = lambda name, value, kw: (names.append(name), record(name, value, kw))
    hist = tr.fit(pl, _IndexDM(5))
    L.check_watchdog()
    assert pl.global_step == 6 and rec["ema"] == 6 and tr.train_batches == 10
    assert [i for i, _ in rec["steps"]] == [1, 3, 4] * 2
    assert names.count("train_loss") == 10 and len(rec["micro"]) == 10
    for e in range(2):
        losses = torch.stack(rec["losses"][5 * e:5 * e + 5])
        assert hist[e]["train_loss"] == pytest.approx(float(losses.mean()), rel=1e-6)
        g = rec["micro"][5 * e:5 * e + 5]
        w = [s for _, s in rec["steps"][3 * e:3 * e + 3]]
        assert torch.equal(w[0], 0.5 * g[0] + 0.5 * g[1]) and torch.equal(w[1], 0.5 * g[2] + 0.5 * g[3])
        assert torch.equal(w[2], 0.5 * g[4])                   # the partial window is divided by N, not by 1
    assert pl.model.engine().accumulate_grads is None

    pl, _ = _module(dev)
    pl.use_cuda_graph = True
    rec = _drive(pl, inputs)
    tr = Trainer(max_epochs=2, max_steps=3, accumulate_grad_batches=2, check_val_every_n_epoch=100)
    hist = tr.fit(pl, _IndexDM(5))
    assert pl.global_step == 3 and rec["ema"] == 3 and len(rec["steps"]) == 3 and tr.train_batches == 5


# ------------------------------------------------------------------------------------------------ loss scaling
@gpu
@pytest.mark.parametrize("graph", [False, True])
def test_overflowing_window_skips_and_backs_off_once(full, dev, graph):
    """LossScaler(init_scale=2^40) at 2 x 16: every window until the scale is small enough overflows.  A skipped window
    leaves p, m, v unchanged bit for bit and halves the scale exactly once; the first window that applies meets the
    float64 reference's bars on the full 32."""
    from mcedm_b200.loss_scale import LossScaler

    _, _, inp, ref = full
    pl, _ = _module(dev)                         # the parameters `full`'s reference was taken at
    pl.use_cuda_graph = graph
    opt = pl.configure_optimizers()["optimizer"]
    opt.max_grad_norm = 1.0
    sc = LossScaler(init_scale=2.0 ** 40)
    pl.model.engine().loss_scaler = sc
    parts = [micro(inp, k, 16) for k in range(2)]
    scale = 2.0 ** 40
    for it in range(40):
        p0, m0, v0 = opt.flat_params().clone(), opt._m.clone(), opt._v.clone()
        loss, grads = window(pl, parts, opt)
        if float(sc.found_inf_t) == 0.0:
            break
        scale /= 2
        assert not all(torch.isfinite(g).all() for g in grads)
        assert sc.get_scale() == scale, (it, sc.get_scale())
        assert torch.equal(p0, opt.flat_params()) and torch.equal(m0, opt._m) and torch.equal(v0, opt._v)
        assert int(opt._step_dev) == 0
    else:
        pytest.fail("no window applied")
    assert it > 0
    print(f"first applied window at S = 2^{int(math.log2(scale))} after {it} skips")
    _compare(pl, loss, grads, ref, f"first applied 2 x 16 window (graph={graph})")
    assert int(opt._step_dev) == 1 and not torch.equal(p0, opt.flat_params())


# ------------------------------------------------------------------------------------------------ data-parallel
@gpu
def test_data_parallel_reduces_once_per_window(dev, tmp_path):
    """world 2 (gloo, one device), N = 2, micro-batch 8: one gradient all-reduce per window, identical parameters on
    both ranks, and those match a single-process N = 4 run over the same four micro-batches: the reduced gradient to
    the sum order, the window gradient within the bars of the float64 step on all 32 samples."""
    from mcedm_b200.runner import Trainer

    script = os.path.join(ROOT, "tests", "dist_grad_accum_worker.py")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29541", PYTHONPATH=ROOT)
    procs = [subprocess.Popen([sys.executable, script, str(r), "2", str(tmp_path)], env=env) for r in range(2)]
    codes = [p.wait(timeout=900) for p in procs]
    assert codes == [0, 0]
    res = [torch.load(os.path.join(tmp_path, f"rank{r}.pt")) for r in range(2)]
    assert res[0]["grad_allreduces"] == res[1]["grad_allreduces"] == 1
    assert torch.equal(res[0]["p"], res[1]["p"]) and torch.equal(res[0]["g"], res[1]["g"])

    pl, mcfg = _module(dev)
    pl.use_cuda_graph = True
    inp = _inputs(pl, dev, B, seed=1500)
    ref = reference_step(_named_params(pl), mcfg, *inp)
    p0 = torch.cat([p.detach().flatten() for p in pl.model.parameters()]).cpu()
    rec = _drive(pl, [micro(inp, k, 8) for k in range(4)])
    tr = Trainer(max_epochs=1, accumulate_grad_batches=4, check_val_every_n_epoch=100)
    tr.fit(pl, _IndexDM(4))
    assert len(rec["steps"]) == 1
    g = rec["steps"][0][1].cpu()
    p = tr.optimizer.flat_params().cpu()
    g_dist = res[0]["g"] / 2                   # sum over ranks of (g_a + g_b) / 2; Adam applies the 1/world
    e_g, e_p = rel(g_dist, g), rel(res[0]["p"] - p0, p - p0)
    print(f"world 2 x N 2 vs N 4: gradient {e_g:.2e}, parameter update {e_p:.2e}")
    assert e_g < 1e-5 and e_p < TOL["glob"]
    loss = torch.stack(rec["losses"]).mean()
    off, grads = 0, []
    for q in pl.model.parameters():
        grads.append(g[off:off + q.numel()].view(q.shape).to(dev))
        off += q.numel()
    _compare(pl, loss, grads, ref, "N = 4 window of 4 x 8")


# ------------------------------------------------------------------------------------------------ dropout
@gpu
def test_dropout_micro_batches_draw_their_own_masks(dev):
    """p = 0.1: the two micro-batches of a window run at dropout counters s and s + 1 - the window's gradient is half
    the sum of the plain steps at those counters, bit for bit - and the counter advances by 2."""
    from test_gpu_dropout import _pl, _set

    pl, _, _ = _pl(dev, 0.1)
    eng = pl.model.engine()
    inp = _inputs(pl, dev, B, seed=1600)
    a, b = micro(inp, 0, 16), micro(inp, 1, 16)
    for graph in (False, True):
        pl.use_cuda_graph = graph
        _set(eng, 7, 40)
        ga = _step(pl, a)
        _set(eng, 7, 41)
        gb = _step(pl, b)
        _set(eng, 7, 40)
        loss, grads = window(pl, [a, b])
        assert eng.dropout_step == 42
        assert torch.equal(loss, (ga[0] + gb[0]) / 2)
        assert all(torch.equal(w, 0.5 * x + 0.5 * y) for w, x, y in zip(grads, ga[1], gb[1])), graph
        _set(eng, 7, 40)
        same_mask = window(pl, [a, a])
        assert not all(torch.equal(w, x) for w, x in zip(same_mask[1], ga[1]))   # a's second pass drew other masks


@gpu
def test_dropout_counter_resumes_at_forwards_run(dev, tmp_path):
    """Trainer at N = 2 over 3 batches per epoch with p = 0.1: 3 forwards but 2 optimizer steps per epoch.  The
    checkpoint records 3 training batches, and a resumed run continues the dropout counter there (6 after its epoch),
    not at global_step."""
    from test_gpu_dropout import _pl

    from mcedm_b200.data import SyntheticMaskDatamodule
    from mcedm_b200.runner import ModelCheckpoint, Trainer

    def dm():
        return SyntheticMaskDatamodule(system="swe_per", n_train=12, n_test=2, batch_size=4)

    pl, _, _ = _pl(dev, 0.1)
    Trainer(max_epochs=1, accumulate_grad_batches=2, check_val_every_n_epoch=100,
            callbacks=[ModelCheckpoint(dirpath=str(tmp_path))]).fit(pl, dm())
    assert pl.global_step == 2 and pl.model.engine().dropout_step == 3
    state = torch.load(os.path.join(tmp_path, "last.ckpt"), map_location="cpu", weights_only=False)
    assert state["global_step"] == 2 and state["train_batches"] == 3
    resumed, _, _ = _pl(dev, 0.1)
    seen = []
    ts = resumed.training_step

    def spy(batch, batch_idx):
        seen.append(resumed.model.engine().dropout_step)
        return ts(batch, batch_idx)

    resumed.training_step = spy
    tr = Trainer(max_epochs=2, accumulate_grad_batches=2, check_val_every_n_epoch=100)
    tr.fit(resumed, dm(), ckpt_path=os.path.join(tmp_path, "last.ckpt"))
    assert seen == [3, 4, 5] and resumed.model.engine().dropout_step == 6
    assert resumed.global_step == 4 and tr.train_batches == 6
