"""Developer tool: entry-point call counts of one training step with a stock loop and with FusedSGD(model=...)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
from unet_implementations_b200 import _lib
from unet_implementations_b200.models.losses import SimpleLoss
from unet_implementations_b200.models.unet import UNet
from unet_implementations_b200.optim import FusedSGD

torch.manual_seed(1234)
model = UNet().cuda().train()
x = torch.randn(2, 3, 128, 128, device="cuda")
t = torch.randint(0, 3, (2, 128, 128), device="cuda")
loss_fn = SimpleLoss()

def step():
    for p in model.parameters():
        p.grad = None
    loss_fn(model(x), t).backward()

def count(fn):
    prof = _lib.EventProfiler()
    l0 = _lib.call("b200unet_launch_count")
    _lib.PROFILER = prof
    fn()
    _lib.PROFILER = None
    torch.cuda.synchronize()
    return _lib.call("b200unet_launch_count") - l0, {k.replace("b200unet_", ""): len(v) for k, v in prof.pairs.items()}

step(); step()
print("plain step:", count(step))
opt = FusedSGD(model.parameters(), lr=1e-3, momentum=0.9, nesterov=True, model=model)
def sgd_step():
    step(); opt.step()
sgd_step(); sgd_step(); sgd_step()
print("step + FusedSGD(model):", count(sgd_step))
w = model.encoder_stages[2].block[0].weight
pk = model._packs.emitted[id(w)]
print("version", w._version, "emitted pack stamped at", pk.version, "current:", pk.valid(w, True))
