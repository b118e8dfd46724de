"""Developer tool: the autoencoder training step (BASELINE.json configs[3]: default Autoencoder, batch 64, 512 x 512,
MSELoss) with the Adam optimizer its trainer uses (AE_pretrained/reconstruction/src/train.py:390-394), four ways:

  torch_adam_eager   forward + MSE + backward + torch.optim.Adam(foreach=True).step(), eager; the next forward re-packs
                     every conv weight Adam changed (packs.PackStore), which is part of the time
  fused_adam_eager   the same with FusedAdam(model=...): one prologue + one flat launch, packs emitted by the step
  no_opt_graph       forward + MSE + backward only, replayed as one CUDA graph
  fused_adam_graph   forward + MSE + backward + FusedAdam(capturable=True).step(), replayed as one CUDA graph

Each is timed with CUDA events over --steps steps after --warmup steps; ms per step, median of --reps windows.
    python tools/adam_step_bench.py [--batch 64] [--size 512] [--steps 10] [--warmup 3] [--reps 3]
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from unet_implementations_b200.graph import GraphedStep
from unet_implementations_b200.models.autoencoder import Autoencoder
from unet_implementations_b200.models.losses import MSELoss
from unet_implementations_b200.optim import FusedAdam


def build():
    torch.manual_seed(1234)  # bench.py's autoencoder: the trainer's dropout rates (train.py:351-370)
    return Autoencoder(encoder_dropout_rates=[0.0, 0.0, 0.05, 0.1, 0.15, 0.15],
                       decoder_dropout_rates=[0.15, 0.1, 0.1, 0.05, 0.0]).cuda().train()


def timed(fn, steps, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1) / steps)
    ms.sort()
    return ms[len(ms) // 2], ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("adam_step_bench.py needs a CUDA device")
    g = torch.Generator().manual_seed(0)
    x = torch.randn(args.batch, 3, args.size, args.size, generator=g).cuda()
    target = torch.rand(args.batch, 3, args.size, args.size, generator=g).cuda()
    loss_fn = MSELoss()
    kw = dict(lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0)
    results = {}

    def step_fn(model, opt):
        def step():
            if opt is not None:
                opt.zero_grad(set_to_none=True)
            else:
                model.zero_grad(set_to_none=True)
            loss = loss_fn(model(x), target)
            loss.backward()
            if opt is not None:
                opt.step()
            return loss
        return step

    model = build()
    n = sum(p.numel() for p in model.parameters())
    opt = torch.optim.Adam(model.parameters(), foreach=True, **kw)
    results["torch_adam_eager"] = timed(step_fn(model, opt), args.steps, args.warmup, args.reps)
    del model, opt
    torch.cuda.empty_cache()

    model = build()
    opt = FusedAdam(model.parameters(), model=model, **kw)
    results["fused_adam_eager"] = timed(step_fn(model, opt), args.steps, args.warmup, args.reps)
    del model, opt
    torch.cuda.empty_cache()

    model = build()
    gs = GraphedStep(step_fn(model, None), warmup=2)
    results["no_opt_graph"] = timed(gs.replay, args.steps, args.warmup, args.reps)
    del model, gs
    torch.cuda.empty_cache()

    model = build()
    opt = FusedAdam(model.parameters(), model=model, capturable=True, **kw)
    step = step_fn(model, opt)
    step()  # creates the optimizer state (capture needs it)
    gs = GraphedStep(step, warmup=1, optimizer=opt)
    results["fused_adam_graph"] = timed(gs.replay, args.steps, args.warmup, args.reps)

    print(f"autoencoder training step, batch {args.batch}, {args.size}x{args.size}, {n / 1e6:.2f} M parameters; "
          f"ms per step over {args.steps} steps, median of {args.reps} windows [all windows]")
    for k, (med, ms) in results.items():
        print(f"  {k:18s} {med:8.2f} ms   [{', '.join(f'{m:.2f}' for m in ms)}]")
    print(f"  optimizer share of the graphed step: {results['fused_adam_graph'][0] - results['no_opt_graph'][0]:.3f} ms")


if __name__ == "__main__":
    main()
