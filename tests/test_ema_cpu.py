"""optim.EMA without a GPU: the decay rule against diffusers' EMAModel.get_decay restated, and the
argument checks that fire before anything touches a device."""
import pytest
import torch


def diffusers_decay(optimization_step, decay, use_warmup_rule):
    """diffusers' EMAModel.get_decay with update_after_step = 0, min_decay = 0 and
    use_ema_warmup = False; without the rule, a constant decay."""
    if not use_warmup_rule:
        return decay
    step = max(0, optimization_step - 0 - 1)
    if step <= 0:
        return 0.0
    cur_decay_value = (1 + step) / (10 + step)
    cur_decay_value = min(cur_decay_value, decay)
    return max(cur_decay_value, 0.0)


@pytest.mark.parametrize("decay", [0.9999, 0.5])
@pytest.mark.parametrize("warmup", [False, True])
def test_decay_rule_matches_the_restatement(decay, warmup):
    from mri_image_generation_b200.optim import ema_decay
    for k in range(1, 1001):
        assert ema_decay(k, decay, warmup) == diffusers_decay(k, decay, warmup), k
    if warmup:
        assert ema_decay(1, decay, True) == 0.0
        # the warm-up reaches `decay` at k = 9 d / (1 - d): k = 9 for 0.5, never below 1000 for 0.9999
        assert (ema_decay(1000, decay, True) == decay) == (decay == 0.5)


@pytest.mark.parametrize("decay", [-0.1, 1.0, float("nan")])
def test_decay_outside_the_unit_interval_is_rejected(decay):
    from mri_image_generation_b200.optim import EMA
    with pytest.raises(ValueError):
        EMA(torch.nn.Linear(3, 2), decay=decay)


def test_cpu_module_raises():
    from mri_image_generation_b200._lib import MriError
    from mri_image_generation_b200.optim import EMA
    with pytest.raises(MriError):
        EMA(torch.nn.Linear(3, 2), decay=0.999)
