"""CPU: dynamic loss scaling's host surface (mcedm_b200/loss_scale.py, runner.Trainer precision selection)."""
import numpy as np
import pytest
import torch

from mcedm_b200 import loss_scale as LS
from mcedm_b200.runner import Trainer


def test_update_rule_matches_torch_amp_update_scale():
    """The rule mcedm_loss_scale_update runs, restated on the host, against torch._amp_update_scale_ (CPU kernel) over
    10k random found-inf flags with growth_interval = 3."""
    rng = np.random.default_rng(0)
    flags = rng.random(10_000) < 0.3
    scale_t = torch.tensor([1024.0])
    tracker_t = torch.tensor([0], dtype=torch.int32)
    scale, tracker = 1024.0, 0
    seen = set()
    for f in flags:
        torch._amp_update_scale_(scale_t, tracker_t, torch.tensor([1.0 if f else 0.0]), 2.0, 0.5, 3)
        scale, tracker = LS.update_rule(scale, tracker, bool(f), 2.0, 0.5, 3)
        assert scale == float(scale_t[0]) and tracker == int(tracker_t[0])
        seen.add(scale)
    assert len(seen) > 20             # the walk both grew and backed off many times


def test_update_rule_never_grows_past_fp32():
    s, t = LS.update_rule(2.0 ** 127, 0, False, 2.0, 0.5, 1)
    st, tt = torch.tensor([2.0 ** 127]), torch.tensor([0], dtype=torch.int32)
    torch._amp_update_scale_(st, tt, torch.tensor([0.0]), 2.0, 0.5, 1)
    assert (s, t) == (float(st[0]), int(tt[0])) == (2.0 ** 127, 0)


def test_state_dict_layout_is_grad_scalers():
    ref = torch.amp.GradScaler("cpu", init_scale=1024.0).state_dict()
    sd = LS.LossScaler().state_dict()
    assert sd == ref
    assert [type(v) for v in sd.values()] == [type(v) for v in ref.values()]
    other = LS.LossScaler(init_scale=8.0, growth_interval=5)
    other.load_state_dict({**ref, "scale": 64.0, "_growth_tracker": 3})
    assert other.state_dict() == {**ref, "scale": 64.0, "_growth_tracker": 3}


@pytest.mark.parametrize("kw", [dict(growth_factor=3.0), dict(growth_factor=1.0), dict(growth_factor=0.5),
                                dict(backoff_factor=0.3), dict(backoff_factor=1.0), dict(backoff_factor=2.0),
                                dict(init_scale=0.0), dict(init_scale=-1024.0), dict(init_scale=float("inf")),
                                dict(growth_interval=0)])
def test_invalid_settings_raise(kw):
    with pytest.raises(ValueError):
        LS.LossScaler(**kw)


def test_valid_power_of_two_factors():
    LS.LossScaler(init_scale=3.0, growth_factor=4.0, backoff_factor=0.25, growth_interval=1)


@pytest.mark.parametrize("precision,dynamic", [(16, True), ("16", True), ("16-mixed", True), (32, False), ("32", False),
                                               ("32-true", False), ("bf16-mixed", False), (64, False), (True, False),
                                               (16.0, False)])
def test_precision_selects_dynamic_or_static(precision, dynamic):
    assert LS.dynamic_precision(precision) is dynamic
    assert Trainer(precision=precision).precision == precision


class _Eng:
    def __init__(self, plan):
        self.train_plan, self.loss_scaler = plan, None


class _Net:
    def __init__(self, plan):
        self._e = _Eng(plan)

    def engine(self):
        return self._e


class _Module:
    def __init__(self, plan):
        self.model = _Net(plan)


def test_trainer_attaches_a_scaler_on_the_fp16_plan_only():
    from mcedm_b200.optim import FusedAdam

    for precision, plan, want in [(16, "fused16", True), ("16-mixed", "fused16", True), (32, "fused16", False),
                                  (16, "fp32", False)]:
        tr, mod = Trainer(precision=precision), _Module(plan)
        tr.optimizer = FusedAdam.__new__(FusedAdam)       # selection only looks at the optimizer's type
        tr._enable_loss_scaling(mod)
        sc = mod.model.engine().loss_scaler
        assert (sc is not None) is want, (precision, plan)
        assert (tr.loss_scaler(mod) is not None) is (want and plan == "fused16")
        if want:
            assert sc.state_dict() == torch.amp.GradScaler("cpu", init_scale=1024.0).state_dict()
    tr, mod = Trainer(precision=16), _Module("fused16")
    tr.optimizer = torch.optim.SGD([torch.zeros(1, requires_grad=True)], lr=0.1)
    with pytest.raises(NotImplementedError):
        tr._enable_loss_scaling(mod)
