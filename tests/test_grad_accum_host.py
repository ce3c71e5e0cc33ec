"""CPU: gradient accumulation's host side: `runner.accumulation_schedule`, `Trainer(accumulate_grad_batches=...)`
argument checks, and the Trainer's window loop on a torch-only module (loss / N into torch's accumulating `.grad`)."""
import pytest
import torch

from mcedm_b200.runner import ModelCheckpoint, Trainer, _ShimLightningModule, accumulation_schedule


def test_schedule_steps_after_every_nth_batch_and_the_last():
    assert accumulation_schedule(5, 2) == [(1, 0.5), (3, 0.5), (4, 0.5)]
    assert accumulation_schedule(5, 1) == [(k, 1.0) for k in range(5)]
    assert accumulation_schedule(8, 4) == [(3, 0.25), (7, 0.25)]
    assert accumulation_schedule(3, 8) == [(2, 0.125)]           # one partial window, still divided by N
    assert accumulation_schedule(0, 2) == []


@pytest.mark.parametrize("bad,exc", [(0, ValueError), (-2, ValueError), (1.5, ValueError), (2.0, ValueError),
                                     ("2", ValueError), (True, ValueError), ({0: 2}, NotImplementedError)])
def test_invalid_accumulate_grad_batches_raises(bad, exc):
    with pytest.raises(exc):
        Trainer(accumulate_grad_batches=bad)


def test_default_is_one():
    assert Trainer().accumulate_grad_batches == 1
    assert Trainer(accumulate_grad_batches=4).accumulate_grad_batches == 4


class _Tiny(_ShimLightningModule):
    def __init__(self):
        super().__init__()
        torch.manual_seed(0)
        self.lin = torch.nn.Linear(4, 3)
        self.steps = []                     # the gradient at each optimizer step
        self.losses = []

    def configure_optimizers(self):
        opt = torch.optim.SGD(self.parameters(), lr=0.1)
        orig = opt.step

        def step(*a, **k):
            self.steps.append(torch.cat([p.grad.flatten().clone() for p in self.parameters()]))
            return orig(*a, **k)

        opt.step = step
        return {"optimizer": opt}

    def training_step(self, batch, idx):
        x, y = batch
        loss = ((self.lin(x) - y) ** 2).mean()
        self.log("train_loss", loss)
        self.losses.append(float(loss.detach()))
        return loss

    def validation_step(self, batch, idx):
        return {}


class _DM:
    def __init__(self, n=5):
        self.n = n

    def setup(self, stage):
        g = torch.Generator().manual_seed(3)
        self.batches = [(torch.randn(8, 4, generator=g), torch.randn(8, 3, generator=g)) for _ in range(self.n)]

    def train_dataloader(self):
        return self.batches

    def val_dataloader(self):
        return []


def _grad(mod, batch):
    mod.zero_grad(set_to_none=True)
    x, y = batch
    ((mod.lin(x) - y) ** 2).mean().backward()
    return torch.cat([p.grad.flatten().clone() for p in mod.parameters()])


def test_trainer_steps_once_per_window_on_the_normalised_sum():
    """5 batches per epoch at N = 2 for 2 epochs: 6 optimizer steps (after batches 1, 3, 4 of each epoch), global_step
    6, every step on (sum of the window's gradients) / 2 - the partial window's is half its one batch's gradient -
    and 5 train_loss records per epoch whose mean is the epoch's logged value."""
    mod, dm = _Tiny(), _DM()
    tr = Trainer(max_epochs=2, gradient_clip_val=None, accumulate_grad_batches=2)
    seen = []
    rec = tr._record
    tr._record = lambda name, value, kw: (seen.append(name), rec(name, value, kw))
    shadow = _Tiny()                        # replays the schedule by hand on the same initial weights
    hist = tr.fit(mod, dm)
    assert mod.global_step == 6 and len(mod.steps) == 6
    assert seen.count("train_loss") == 10 and len(hist) == 2
    for e in range(2):
        assert hist[e]["train_loss"] == pytest.approx(sum(mod.losses[5 * e:5 * e + 5]) / 5, rel=1e-6)
    opt = torch.optim.SGD(shadow.parameters(), lr=0.1)
    i = 0
    for _ in range(2):
        for window in ([0, 1], [2, 3], [4]):
            g = sum(_grad(shadow, dm.batches[k]) for k in window) / 2
            torch.testing.assert_close(mod.steps[i], g, rtol=1e-6, atol=1e-7)
            off = 0
            for p in shadow.parameters():
                p.grad = g[off:off + p.numel()].view_as(p).clone()
                off += p.numel()
            opt.step()
            i += 1
    for a, b in zip(mod.parameters(), shadow.parameters()):
        torch.testing.assert_close(a, b, rtol=1e-6, atol=1e-7)


def test_trainer_n1_runs_the_plain_loop():
    mod, dm = _Tiny(), _DM()
    Trainer(max_epochs=1, gradient_clip_val=None).fit(mod, dm)
    shadow = _Tiny()
    opt = torch.optim.SGD(shadow.parameters(), lr=0.1)
    assert len(mod.steps) == 5
    for k in range(5):
        assert torch.equal(mod.steps[k], _grad(shadow, dm.batches[k]))
        opt.step()


@pytest.mark.parametrize("max_steps,batches", [(3, 5), (4, 7)])
def test_max_steps_counts_windows(max_steps, batches):
    """3 windows are epoch 0's 5 batches; the 4th ends after batch 1 of epoch 1."""
    mod = _Tiny()
    tr = Trainer(max_epochs=5, max_steps=max_steps, gradient_clip_val=None, accumulate_grad_batches=2)
    tr.fit(mod, _DM())
    assert mod.global_step == max_steps and len(mod.steps) == max_steps
    assert tr.train_batches == batches


def test_checkpoint_records_training_batches_and_resume_continues_them(tmp_path):
    mod = _Tiny()
    tr = Trainer(max_epochs=1, gradient_clip_val=None, accumulate_grad_batches=2,
                 callbacks=[ModelCheckpoint(dirpath=str(tmp_path))])
    tr.fit(mod, _DM())
    ckpt = torch.load(tmp_path / "last.ckpt", weights_only=False)
    assert ckpt["global_step"] == 3 and ckpt["train_batches"] == 5
    tr2 = Trainer(max_epochs=2, gradient_clip_val=None, accumulate_grad_batches=2)
    resumed = _Tiny()
    tr2.fit(resumed, _DM(), ckpt_path=str(tmp_path / "last.ckpt"))
    assert resumed.global_step == 6 and tr2.train_batches == 10
    old = {k: v for k, v in ckpt.items() if k != "train_batches"}   # a checkpoint written before the key existed
    torch.save(old, tmp_path / "old.ckpt")
    tr3 = Trainer(max_epochs=2, gradient_clip_val=None)
    tr3.fit(_Tiny(), _DM(), ckpt_path=str(tmp_path / "old.ckpt"))
    assert tr3.train_batches == 3 + 5
