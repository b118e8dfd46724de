"""CPU: FusedAdam refuses what it does not implement before it touches a device, and its parameter group has
torch.optim.Adam's keys (so that the state_dict of either optimizer loads into the other)."""
import pytest
import torch
import torch.nn as nn


def _model():
    return nn.Sequential(nn.Conv2d(3, 4, 3), nn.Conv2d(4, 2, 1))


@pytest.mark.parametrize("option", ["amsgrad", "maximize", "differentiable", "fused"])
def test_unsupported_options_raise(option):
    from unet_implementations_b200.optim import FusedAdam
    m = _model()
    with pytest.raises(ValueError, match=option):
        FusedAdam(m.parameters(), model=m, **{option: True})


def test_model_is_required_and_one_group_only():
    from unet_implementations_b200.optim import FusedAdam
    m = _model()
    with pytest.raises(ValueError, match="model="):
        FusedAdam(m.parameters())
    groups = [{"params": list(m[0].parameters())}, {"params": list(m[1].parameters()), "lr": 1e-4}]
    with pytest.raises(ValueError, match="one parameter group"):
        FusedAdam(groups, model=m)


@pytest.mark.parametrize("kw", [dict(lr=-1.0), dict(eps=-1e-8), dict(betas=(1.0, 0.999)), dict(betas=(0.9, -0.1)),
                                dict(weight_decay=-1e-2)])
def test_invalid_hyperparameters_raise(kw):
    from unet_implementations_b200.optim import FusedAdam
    m = _model()
    with pytest.raises(ValueError, match="Invalid"):
        FusedAdam(m.parameters(), model=m, **kw)


def test_group_keys_are_torch_adams(monkeypatch):
    """FusedAdam's defaults are torch.optim.Adam's minus `capturable`, which in torch selects device step counts and
    a different formulation; FusedAdam always computes like torch's default (capturable=False) Adam."""
    from unet_implementations_b200 import optim

    class _NoDevice:  # stands in for the flat buffers, which need the model on its CUDA device
        def __init__(self, *args, **kwargs):
            self.count, self.master = 1, torch.zeros(1)

    monkeypatch.setattr(optim, "_FlatState", _NoDevice)
    m = _model()
    opt = optim.FusedAdam(m.parameters(), lr=3e-4, weight_decay=0.05, decoupled_weight_decay=True, model=m)
    ref = torch.optim.Adam(m.parameters(), lr=3e-4, weight_decay=0.05, decoupled_weight_decay=True)
    assert set(opt.defaults) == set(ref.defaults) - {"capturable"}
    assert all(opt.defaults[k] == ref.defaults[k] for k in opt.defaults)
