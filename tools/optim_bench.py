"""Developer tool: the flat fused optimizer steps (FusedSGD(model=...): one launch; FusedAdam(model=...): a one-block
prologue + one launch; both emit the bf16 conv packs) of the default UNet, timed alone, called eagerly and replayed
from a CUDA graph.
    python tools/optim_bench.py [--sgd-only]     (B200UNET_LIB=<other build> for an A/B)"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from unet_implementations_b200.models.unet import UNet
from unet_implementations_b200.flat import sink_of
from unet_implementations_b200.optim import FusedSGD


def median_step_us(make_opt):
    """Median over 15 steps of one optimizer step (CUDA events), the L2 flushed before each step: make_opt(model,
    capturable=False).step() called eagerly (host bookkeeping included), and make_opt(model, capturable=True).step()
    replayed from a CUDA graph of step() alone (device time only)."""
    eager, _ = _timed(make_opt, capturable=False)
    graphed, n = _timed(make_opt, capturable=True)
    return eager, graphed, n


def _timed(make_opt, capturable):
    torch.manual_seed(0)
    model = UNet().cuda().train()
    opt = make_opt(model, capturable)
    sink = sink_of(model)
    sink.flat.normal_(0, 1e-3)  # a gradient for every parameter, in place in the flat buffer (what backward leaves)
    for p in sink.params:
        p.grad = sink.dest(p)
    n = sum(p.numel() for p in sink.params)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        opt.step()
    torch.cuda.synchronize()
    fn = opt.step
    if capturable:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side), torch.cuda.graph(graph):
            opt.step()
        torch.cuda.synchronize()
        fn = graph.replay
    ts = []
    for _ in range(15):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return ts[len(ts) // 2], n


# the eager configuration is the one DESIGN section 3 records (257 us), capturable=False
us, gus, n = median_step_us(lambda m, c: FusedSGD(m.parameters(), lr=0.01, momentum=0.99, nesterov=True,
                                                  weight_decay=1e-4, model=m, capturable=c))
print(f"FusedSGD(model=...).step(): {us:.1f} us (graph-replayed: {gus:.1f} us) for {n / 1e6:.2f} M parameters "
      f"({n * 20 / 1e6:.0f} MB of fp32 traffic + {n * 4.5 / 1e6:.0f} MB of bf16 packs)")
if "--sgd-only" not in sys.argv:
    from unet_implementations_b200.optim import FusedAdam
    us, gus, n = median_step_us(lambda m, c: FusedAdam(m.parameters(), lr=1e-3, weight_decay=1e-4, model=m,
                                                       capturable=c))
    # read p, g, m, v and write p, m, v: 28 bytes per parameter
    print(f"FusedAdam(model=...).step(): {us:.1f} us (graph-replayed: {gus:.1f} us) for {n / 1e6:.2f} M parameters "
          f"({n * 28 / 1e6:.0f} MB of fp32 traffic + {n * 4.5 / 1e6:.0f} MB of bf16 packs)")
