#!/usr/bin/env python
"""Headline benchmark: Our_UNet 512x512 training step (forward + Dice/weighted-CE loss + backward, gradient
all-reduce for N > 1), images/s, on N B200s of one box (BASELINE.json: metric / configs[1], configs[2]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload unet|ae|clip] [--impl b200|reference|torch_gpu]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Prints ONE JSON line on rank 0.  `value` = images/s with the batch resident in HBM (CUDA-event timed, max over
ranks); `e2e` = the same step through the public module API with the batch in pinned host memory: host->device
copy of image+mask and a device->host read of the loss inside the timed region, every step.
`roofline` is for the dominant kernel family (the tcgen05 implicit-GEMM convs): algorithmic conv FLOPs of the step
divided by the CUDA-event time spent inside those entry points, measured live during the timed steps.
`--impl reference` times the CPU port of the reference's step (oracle/unet_oracle.py: the reference is a pure-Python
torch project whose tree is not on the GPU box) on the host cores; `--impl torch_gpu` times the same op sequence on
stock PyTorch + cuDNN kernels ON the B200 (bf16 autocast) -- the same-box competitor of SURVEY.md 8(d).
`--workload ae` = BASELINE.json configs[3] (autoencoder reconstruction step, batch 64), `--workload clip` = configs[4]
(CLIP-conditioned UNet, batch 32 per GPU, random [B,512,16,16] features standing in for the frozen ViT's output).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "our_unet_512_train_images_per_sec"
UNIT = "img/s"
FEATS = [32, 64, 128, 256, 512, 512]


WORKLOADS = {
    # name: (metric, default batch per GPU, description)
    "unet": ("our_unet_512_train_images_per_sec", 32, "Our_UNet training step (fwd + SimpleLoss + bwd{ar})"),
    "ae": ("ae_reconstruction_512_train_images_per_sec", 64,
           "AE_pretrained reconstruction step (Autoencoder fwd + MSELoss + bwd{ar})"),
    "clip": ("clip_unet_512_train_images_per_sec", 32,
             "CLIP_UNet training step (fwd with [B,512,16,16] patch features + SimpleLoss + bwd{ar}; frozen ViT out of scope)"),
}


def extra_flops_per_image(workload, size=512):
    """Algorithmic conv FLOPs the variants add to conv_flops_per_image: (fwd, fwd+bwd)."""
    if workload == "ae":      # Conv2d(32 -> 3, 3x3) head instead of the 1x1 head (autoencoder.py:377-387)
        f = 2.0 * 3 * size * size * 32 * 9 - 2.0 * 3 * size * size * 32
        return f, 3 * f
    if workload == "clip":    # clip_fusion_conv: Conv2d(1024 -> 512, 1x1) at the bottleneck (CLIP_UNet/models/unet.py:356-364)
        hb = size >> 5
        f = 2.0 * 512 * hb * hb * 1024
        return f, 3 * f
    return 0.0, 0.0


def conv_flops_per_image(size=512):
    """Algorithmic conv FLOPs of one image (SURVEY.md A.1): returns (fwd, fwd+bwd, tensor-core-kernel share fwd+bwd).
    2*Cout*OH*OW*Cin*9 per 3x3 conv; backward = dgrad + wgrad (no dgrad for the image)."""
    fwd = bwd = tc = 0.0
    h = size
    cin = 3
    layers = []
    for s, c in enumerate(FEATS):
        if s > 0:
            h //= 2
        layers.append((cin, c, h))
        layers.append((c, c, h))
        cin = c
    for j in range(5):
        d = 4 - j
        hh = size >> d
        layers.append((FEATS[d + 1] + FEATS[d], FEATS[d], hh))
        layers.append((FEATS[d], FEATS[d], hh))
    for i, (ci, co, hh) in enumerate(layers):
        f = 2.0 * co * hh * hh * ci * 9
        fwd += f
        b = f if i == 0 else 2 * f
        bwd += b
        tc += f + b  # every 3x3 conv runs on the tcgen05 kernels (the 3-channel stem zero-padded to K = 32)
    head = 2.0 * 3 * size * size * 32
    fwd += head
    bwd += 2 * head
    return fwd, fwd + bwd, tc


class ClockSampler:
    """SM clock, power and clock-event (throttle) reasons sampled every 10 ms DURING the timed regions through NVML
    (the same counters `nvidia-smi --query-gpu=clocks.sm,...,clocks_event_reasons.*` prints, B200_PROFILING.md;
    a 200 ms nvidia-smi loop cannot see a 0.3 s timed region)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()
        self.thread = None
        self.err = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if visible:
                ids = [v for v in visible.split(",") if v.strip()]
                if index < len(ids) and ids[index].strip().isdigit():
                    phys = int(ids[index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.nv = None
            self.err = f"nvml unavailable: {e}"

    def _loop(self):
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1e3
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:  # noqa: BLE001
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((sm, pw, rs))
            except Exception as e:  # noqa: BLE001
                self.err = str(e)
                return
            time.sleep(0.01)

    def start(self):
        if self.nv is None:
            return
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self):
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [self.err or "no sampler"]}
        self.stop_flag.set()
        self.thread.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [self.err or "no samples"]}
        sm = sorted(s[0] for s in self.samples)
        reasons = set()
        for _, _, rs in self.samples:
            for bit, nm in self.REASONS.items():
                if rs & bit:
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.max_mhz,
                "power_w_max": max(s[1] for s in self.samples), "samples": len(self.samples),
                "source": "NVML, 10 ms period, during the timed regions", "reasons": sorted(reasons)}


def build_model(workload):
    """The module of the workload with the trainer's constructor arguments, seed 1234 (random init, as the trainers do)."""
    import torch
    torch.manual_seed(1234)
    if workload == "ae":
        from unet_implementations_b200.models.autoencoder import Autoencoder
        # AE_pretrained/reconstruction/src/train.py:351-370: dropout [0,0,.05,.1,.15,.15] / [.15,.1,.1,.05,0]
        return Autoencoder(encoder_dropout_rates=[0.0, 0.0, 0.05, 0.1, 0.15, 0.15],
                           decoder_dropout_rates=[0.15, 0.1, 0.1, 0.05, 0.0])
    if workload == "clip":
        from unet_implementations_b200.models.clip_unet import UNet as ClipUNet
        return ClipUNet()
    from unet_implementations_b200.models.unet import UNet
    return UNet()


def oracle_step_fn(workload, batch, size, device="cpu", autocast=False):
    """step() -> loss of the reference's op sequence (oracle/unet_oracle.py: plain torch functional ops) for the
    workload, on `device`.  Used by the CPU baseline legs and by --impl torch_gpu; never by the product path."""
    import torch

    from oracle import unet_oracle as O
    model = build_model(workload)  # construction only: weights identical to the reference's for this seed
    cfg = O.config_of(model)
    sd = {k: v.detach().clone().to(device) for k, v in model.state_dict().items()}
    x, target = O.synthetic_batch(batch, size, seed=0)
    x, target = x.to(device), target.to(device)
    g = torch.Generator().manual_seed(5)
    clip = (torch.randn(batch, 512, 1, 1, generator=g).expand(-1, -1, size >> 5, size >> 5).contiguous().to(device)
            if workload == "clip" else None)
    recon_target = torch.rand(batch, 3, size, size, generator=g).to(device) if workload == "ae" else None

    def step():
        torch.manual_seed(99)
        masks = O.draw_dropout_masks(cfg, batch, x)
        ctx = torch.autocast(device if isinstance(device, str) else device.type, dtype=torch.bfloat16, enabled=autocast)
        with ctx:
            if workload == "ae":
                return O.autoencoder_training_step(sd, x, recon_target, cfg, masks)["loss"]
            return O.training_step(sd, x, target, cfg, masks, clip_features=clip)["loss"]

    return step


def cpu_port_step_time(batch, size, steps, warmup, threads, workload="unet"):
    """Time the CPU port of the reference step (oracle) -- fp32, `threads` host threads.  Returns s/step."""
    import torch
    torch.set_num_threads(threads)
    step = oracle_step_fn(workload, batch, size)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return sum(times) / len(times)


def workload_text(workload, world, B, S):
    ar = " + grad all-reduce" if world > 1 else ""
    return (WORKLOADS[workload][2].format(ar=ar) + f", batch {B}/GPU, {S}x{S} RGB, "
            + ("3-class masks, " if workload != "ae" else "") + "random-init weights (seed 1234)")


def run_reference(args, rank, world):
    if rank != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    batch = 4  # BASELINE.json configs[0]: the reference's CPU-runnable case; a bounded sample of the per-GPU step
    steps = args.steps
    warm = 1
    s_per_step = cpu_port_step_time(batch, args.size, steps, warm, cores, args.workload)
    v = batch / s_per_step
    out = {
        "impl": "reference", "metric": WORKLOADS[args.workload][0], "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": s_per_step * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(args.workload, 1, args.batch, args.size),
                   "sample": f"each step is a {batch}-image sample of the {args.batch}-image step on the host CPU (images/s is per "
                             f"image), fp32, torch {torch.__version__} CPU ops, {cores} threads",
                   "batch": batch},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{steps} steps of batch {batch} after {warm} warm-up (oracle/unet_oracle.py, torch CPU ops)"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def run_torch_gpu(args, rank, world):
    """The same-box competitor (SURVEY.md 8d, BASELINE.md section 4 item 4): the reference's op sequence on stock
    PyTorch + cuDNN kernels on ONE B200, torch.autocast(bf16), same batch and inputs.  None of this repo's kernels run."""
    if rank != 0:
        return
    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"impl": "torch_gpu", "unavailable": "no CUDA device"}), flush=True)
        return
    torch.cuda.set_device(0)
    torch.backends.cudnn.benchmark = True
    B, S = args.batch, args.size
    step = oracle_step_fn(args.workload, B, S, device="cuda", autocast=True)
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    k = args.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(k):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / k
    v = B / (ms * 1e-3)
    out = {"impl": "torch_gpu", "metric": WORKLOADS[args.workload][0], "value": v, "unit": UNIT, "n_gpus": 1, "steps": k,
           "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "bf16", "data": "synthetic",
           "config": {"workload": workload_text(args.workload, 1, B, S),
                      "how": f"oracle/unet_oracle.py functional ops (F.conv2d / F.instance_norm / F.interpolate / SimpleLoss "
                             f"restatement) under torch.autocast(bf16), torch {torch.__version__}, cuDNN "
                             f"{torch.backends.cudnn.version()}, cudnn.benchmark on"},
           "loss": float(loss), "peak_memory_gib": round(torch.cuda.max_memory_allocated() / 2 ** 30, 2),
           "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(out), flush=True)


class Workload:
    """Model + loss + synthetic batches of one BASELINE.json configuration, behind the modules' public API."""

    def __init__(self, name, B, S, dev, rank, dense_clip=False):
        import torch

        from unet_implementations_b200 import data
        from unet_implementations_b200.models.losses import MSELoss, SimpleLoss
        self.name, self.B, self.S, self.dev = name, B, S, dev
        self.model = build_model(name).to(dev).train()
        self.loss_fn = MSELoss() if name == "ae" else SimpleLoss(weight_dice=1.0, weight_ce=1.0, ignore_index=255, smooth=1e-5,
                                                                 class_weights=None, dynamic_weights=True)
        self.data = data
        # BASELINE.md section 3 inputs, data seed 0 + rank: what the trainer hands the model (fp32 NCHW image, int64 mask)
        g = torch.Generator().manual_seed(rank)
        image = torch.randn(B, 3, S, S, generator=g)
        mask = torch.randint(0, 3, (B, S, S), generator=g)
        mask[torch.rand(B, S, S, generator=g) < 0.1] = 255
        self.resident = {"image": image.to(dev)}
        if name == "ae":   # the autoencoder's target is the un-normalised [0,1] image (AE .. src/train.py:257, :262-267)
            self.resident["target"] = torch.rand(B, 3, S, S, generator=g).to(dev)
        else:
            self.resident["mask"] = mask.to(dev)
        if name == "clip":
            # stands in for ClipPatchExtractor's output (CLIP_UNet/models/unet.py:581-617; frozen ViT, no gradient): ONE
            # pooled 512-d embedding per image, expanded over the 16x16 grid by the extractor (unet.py:611-612).  --clip-dense
            # feeds a dense [B,512,16,16] tensor instead (per-patch features, which the reference's extractor does not make)
            if dense_clip:
                self.resident["clip"] = torch.randn(B, 512, S >> 5, S >> 5, generator=g).to(dev)
            else:
                self.resident["clip"] = torch.randn(B, 512, 1, 1, generator=g).to(dev)
        # the batch as the dataset stores it (train.py:299-311 before the float conversion): uint8 HWC image, uint8 mask
        self.host = {"image": torch.randint(0, 256, (B, S, S, 3), generator=g, dtype=torch.uint8).pin_memory()}
        if name != "ae":
            m8 = mask.to(torch.uint8)
            self.host["mask"] = m8.pin_memory()
        if name == "clip":
            self.host["clip"] = (torch.randn(B, 512, S >> 5, S >> 5, generator=g) if dense_clip
                                 else torch.randn(B, 512, 1, 1, generator=g)).pin_memory()
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in self.host.values())

    def zero_grad(self):
        for p in self.model.parameters():
            p.grad = None

    def step(self, batch):
        """forward + loss + backward through the public module API; batch = dict of device tensors (either form)."""
        self.zero_grad()
        img = batch["image"]
        if self.name == "clip":
            clip = batch["clip"]
            if clip.shape[2] == 1:  # the extractor's expand over the patch grid (a view: spatial strides 0)
                clip = clip.expand(-1, -1, self.S >> 5, self.S >> 5)
            out = self.model(img, clip)
        else:
            out = self.model(img)
        if self.name == "ae":
            tgt = batch.get("target")
            if tgt is None:  # uint8 batch: the reconstruction target is the image / 255 (one kernel, no normalisation)
                tgt = self.data.preprocess_batch(img, None, mean=(0.0, 0.0, 0.0), std=(1.0, 1.0, 1.0))[0]
            loss = self.loss_fn(out, tgt)
        else:
            loss = self.loss_fn(out, batch["mask"])
        loss.backward()
        # detached: no autograd graph of an eager step stays alive into a CUDA-graph capture; under replay these are
        # the graph's static output buffers
        self.outputs = (out.detach(), loss.detach())
        return loss


def dump_outputs(path, wl):
    """What the last step of `wl` handed its caller -- loss, model output, every parameter gradient -- as float32
    DIR/loss.npy, DIR/output.npy and DIR/grad.<parameter name>.npy.  An array larger than its cap is written as a fixed
    sample: the elements at sorted indices drawn by a generator seeded with 0, the same for every build.  The caps keep
    the files under 64 MB in all (16 MB of output, at most 40 MB of gradients)."""
    import numpy as np
    import torch

    def flat_sample(t, cap):
        t = t.detach()
        if t.numel() > cap:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        return t.float().cpu().numpy()

    out, loss = wl.outputs
    grads = [(n, p.grad) for n, p in wl.model.named_parameters() if p.grad is not None]
    grad_cap = min(1 << 16, (40 << 20) // (4 * len(grads)))
    arrays = {"loss": flat_sample(loss, 1), "output": flat_sample(out, 1 << 22)}
    arrays.update(("grad." + n, flat_sample(g, grad_cap)) for n, g in grads)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="unet", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (default: the BASELINE.json configuration's)")
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch_gpu"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true", help="skip the per-entry-point CUDA-event timing")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer, optimizer and graph legs (ncu captures)")
    ap.add_argument("--no-graph", action="store_true", help="skip the CUDA-graph replay leg")
    ap.add_argument("--clip-dense", action="store_true", help="clip workload: dense per-patch features instead of the "
                    "reference extractor's pooled embedding expanded over the grid")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss, model output and parameter gradients of the "
                    "last timed step to DIR/<name>.npy (float32; large arrays as a fixed sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the b200 step computes; it does not apply to --impl " + args.impl)
    if args.batch <= 0:
        args.batch = WORKLOADS[args.workload][1]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.impl == "torch_gpu":
        run_torch_gpu(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist

    from unet_implementations_b200 import _lib, ddp

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the b200 arm has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    nccl_ctas = None
    if world > 1:
        nccl_ctas = ddp.init_process_group(dev)  # NCCL capped to a few CTAs, as many SMs left free by the conv grids

    def barrier():
        if world > 1:
            dist.barrier()

    B, S = args.batch, args.size
    wl = Workload(args.workload, B, S, dev, rank, dense_clip=args.clip_dense)
    model = wl.model
    reducer = None
    if world > 1:
        ddp.broadcast_parameters(model)
        reducer = ddp.BucketedGradAllReduce(model, bucket_bytes=16 << 20)
    torch.manual_seed(99 + rank)
    resident = wl.resident

    def step():
        return wl.step(resident)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    # clock / power sampling starts before the untimed pre-steps (NVML's first queries are slow and share driver locks
    # with kernel launches) and runs through all timed regions
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    # untimed pre-steps: the step runs at the 1 kW power cap and the SM clock it sustains drifts for the first second;
    # all timed regions below then see the same steady state (these steps are not counted in `warmup`)
    presteps = 30 if world == 1 else 60  # (8 GPUs: the first 30 steps after start-up still ran 1.5 % slower)
    for _ in range(presteps):
        step()
    torch.cuda.synchronize()

    # ---- the production form of the step: forward + loss + backward captured ONCE into a CUDA graph and replayed
    # (unet_implementations_b200.graph.GraphedStep; SURVEY.md 8d "CUDA events around a CUDA-graph-replayed step").  The
    # eager form (one Python-enqueued launch per kernel) is timed beside it.  N > 1 replays the graph too, the bucketed
    # NCCL all-reduces inside the capture (measured at 2 and 8 GPUs; B200UNET_GRAPH_DDP=0 keeps those runs eager).
    gs = None
    graph_err = None
    if not args.no_graph and (world == 1 or os.environ.get("B200UNET_GRAPH_DDP", "1") == "1"):
        try:
            from unet_implementations_b200.graph import GraphedStep
            gs = GraphedStep(step, warmup=2)
            for _ in range(3):
                gs.replay()
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001 -- the eager path stands on its own
            gs, graph_err = None, repr(e)[:300]
            torch.cuda.synchronize()
    run_step = gs.replay if gs is not None else step

    def timed(fn, k):
        barrier()
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            every = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(every, t)
            timed.per_rank_ms = [round(v.item() / k, 3) for v in every]  # per step, for the record
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    timed.per_rank_ms = None

    # ---- resident-input throughput
    # per-step events inside the region expose a one-off stall (another tenant's driver call, a host hiccup): a region
    # whose slowest step is > 1.5x its median step is measured once more and the fact is recorded in the JSON line
    remeasured = None
    for attempt in range(2):
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
        counter = [0]

        def marked_step():
            if counter[0] == 0:
                marks[0].record()
            run_step()
            counter[0] += 1
            marks[counter[0]].record()

        if sampler and attempt == 0:
            sampler.samples.clear()  # keep only what was sampled during the timed regions
        # every attempt draws the same dropout masks, so the last step's outputs depend on --steps alone
        torch.manual_seed(99 + rank)
        ms = timed(marked_step, args.steps)
        per_rank_resident = timed.per_rank_ms
        per = sorted(marks[i].elapsed_time(marks[i + 1]) for i in range(args.steps))
        worst, med = per[-1], per[len(per) // 2]
        flag = torch.tensor([1.0 if worst > 1.5 * med else 0.0], device=dev)
        if world > 1:
            dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        if flag.item() == 0.0 or attempt == 1:
            break
        remeasured = f"first attempt had a {worst:.1f} ms step against a median of {med:.1f} ms ({ms / args.steps:.2f} ms/step); measured again"
    ms_per_step = ms / args.steps
    value = world * B / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, wl)
    # the eager form of the same step (also the launch count: a graph replay launches the same kernels as graph nodes)
    l0 = _lib.call("b200unet_launch_count")
    step()
    launches_per_step = _lib.call("b200unet_launch_count") - l0
    launches = launches_per_step * args.steps
    eager_leg = None
    if gs is not None:
        ms_eager = timed(step, args.steps) / args.steps
        eager_leg = {"ms_per_step": ms_eager, "value": world * B / (ms_eager * 1e-3), "unit": UNIT}

    # ---- per-kernel-family timing for the roofline: a second timed region of the SAME step with the weight-gradient
    # kernels serialised on the main stream (in the headline region above they run on a side stream beside the next
    # layer's norm backward, where a CUDA-event pair would time two kernels sharing the SMs, not one kernel)
    prof = None
    prof_steps = min(args.steps, 10)
    if not args.no_profile:
        prof = _lib.EventProfiler()
        was = model.overlap_wgrad
        model.overlap_wgrad = False
        step()
        torch.cuda.synchronize()
        _lib.PROFILER = prof
        ms_serial = timed(step, prof_steps) / prof_steps
        _lib.PROFILER = None
        model.overlap_wgrad = was

    # ---- the same step with the gradient all-reduce switched off (N > 1): each rank's own compute time.  The spread over
    # the ranks is the lock-step cost of a synchronous step on eight power-capped GPUs (the slowest one sets the pace);
    # the difference between its maximum and the headline time is what the all-reduce itself costs.
    per_rank_no_allreduce = None
    if reducer is not None:
        reducer.enabled = False
        step()
        timed(step, min(args.steps, 10))
        per_rank_no_allreduce = timed.per_rank_ms
        reducer.enabled = True
        step()

    # ---- the gradient all-reduce alone (N > 1): the same buckets, nothing else on the GPU
    allreduce_only_ms = None
    if reducer is not None:
        def ar_only():
            for b in range(len(reducer.buckets)):
                reducer._reduce(b)
            reducer.finish()
        ar_only()
        allreduce_only_ms = timed(ar_only, 10) / 10

    # ---- end to end through the public API with host buffers (SURVEY.md 8f row 2): every step copies ITS batch from
    # pinned host memory AS THE DATASET STORES IT -- uint8 HWC image, uint8 mask (train.py:299-311 before the float
    # conversion) -- and reads its loss back to the host.  The model normalises the uint8 image inside the stem's layout
    # kernel and the loss kernels read uint8 masks.  The copies run on a side stream one step ahead of the compute stream
    # (what a pinned-memory DataLoader with non_blocking copies does); each of the K timed steps still issues and waits
    # for its own H2D copy and D2H read.
    copy_stream = torch.cuda.Stream(device=dev)
    bufs = [{k: torch.empty(v.shape, dtype=v.dtype, device=dev) for k, v in wl.host.items()} for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    state = {"i": 0}

    def prefetch(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])  # the step that last used this slot has finished with it
            for k, v in wl.host.items():
                bufs[slot][k].copy_(v, non_blocking=True)
            ready[slot].record(copy_stream)

    for sl in range(2):
        consumed[sl].record()

    # the loss of every step is read back to pinned host memory by an asynchronous copy inside the timed region; the
    # host waits for it one step later (before it reuses the slot) and for the last ones before the region ends, so
    # the CPU keeps enqueueing ahead of the GPU exactly as in the resident region
    loss_h = torch.zeros(2, dtype=torch.float32).pin_memory()
    loss_ev = [torch.cuda.Event() for _ in range(2)]
    losses = []

    # one captured step per input slot (a graph is bound to the addresses of its inputs)
    slot_graphs = None
    if gs is not None and not args.no_e2e and world == 1:
        try:
            for sl in range(2):
                for k, v in wl.host.items():
                    bufs[sl][k].copy_(v)
            from unet_implementations_b200.graph import GraphedStep
            slot_graphs = [GraphedStep(lambda sl=sl: wl.step(bufs[sl]), warmup=1) for sl in range(2)]
        except Exception as e:  # noqa: BLE001
            slot_graphs, graph_err = None, repr(e)[:300]
            torch.cuda.synchronize()

    def e2e_step():
        i = state["i"]
        slot = i & 1
        if i == 0:
            prefetch(0)
        prefetch(slot ^ 1)  # next step's batch, overlapping this step's compute
        torch.cuda.current_stream().wait_event(ready[slot])
        loss = slot_graphs[slot].replay() if slot_graphs is not None else wl.step(bufs[slot])
        consumed[slot].record()
        if i >= 2:
            loss_ev[slot].synchronize()
            losses.append(float(loss_h[slot]))
        loss_h[slot:slot + 1].copy_(loss.detach().reshape(1), non_blocking=True)
        loss_ev[slot].record()
        state["i"] = i + 1

    def e2e_drain():
        for sl in ((state["i"]) & 1, (state["i"] + 1) & 1):
            loss_ev[sl].synchronize()
            losses.append(float(loss_h[sl]))

    e2e_graphed = slot_graphs is not None
    if args.no_e2e:
        ms_e2e = float("nan")
    else:
        e2e_step()

        def e2e_region_step(counter=[0]):
            e2e_step()
            counter[0] += 1
            if counter[0] == args.steps:
                e2e_drain()  # the last losses are on the host before the closing event is recorded

        ms_e2e = timed(e2e_region_step, args.steps)
        if not all(l == l and abs(l) < 1e6 for l in losses):
            raise SystemExit(f"bench.py: non-finite loss in the end-to-end region: {losses[-4:]}")

    # ---- the same resident step followed by the trainer's optimizer step (SURVEY.md 8d: "with and without SGD step"):
    # SGD momentum 0.99, Nesterov, weight decay 1e-4 (train.py:445-451) as ONE launch over the flat master / gradient /
    # momentum buffers that also emits the bf16 conv operand packs (no repack kernels).  Last: it changes the weights.
    with_sgd = None
    gs = None
    slot_graphs = None
    run_step = step
    if not args.no_e2e:
        from unet_implementations_b200.optim import FusedSGD
        opt = FusedSGD(model.parameters(), lr=1e-6, momentum=0.99, nesterov=True, weight_decay=1e-4, model=model,
                       capturable=True)

        def sgd_step():
            step()
            opt.step()

        for _ in range(3):
            sgd_step()
        l0 = _lib.call("b200unet_launch_count")
        ms_sgd = timed(sgd_step, args.steps) / args.steps
        launches_sgd = (_lib.call("b200unet_launch_count") - l0) / args.steps
        ms_sgd_graph = None
        if world == 1 and not args.no_graph:
            try:  # the WHOLE training step (forward + loss + backward + optimizer) as one graph
                from unet_implementations_b200.graph import GraphedStep
                gso = GraphedStep(sgd_step, warmup=1, optimizer=opt)
                for _ in range(3):
                    gso.replay()
                ms_sgd_graph = timed(gso.replay, args.steps) / args.steps
                del gso
            except Exception as e:  # noqa: BLE001
                graph_err = repr(e)[:300]
                torch.cuda.synchronize()
        with_sgd = {"ms_per_step": ms_sgd, "value": world * B / (ms_sgd * 1e-3), "unit": UNIT, "step_form": "eager",
                    "graph_replay_ms_per_step": ms_sgd_graph,
                    "gpu_launches_per_step": launches_sgd,
                    "optimizer": "FusedSGD(momentum=0.99, nesterov=True, weight_decay=1e-4, model=model): one launch over the "
                                 "flat master/grad/momentum buffers, emits the bf16 weight packs (weights change every step; "
                                 "no pack kernel runs)"}
    clocks = sampler.stop() if sampler else None
    e2e_value = world * B / (ms_e2e / args.steps * 1e-3)

    fwd, fb, tc = conv_flops_per_image(S)
    xf, xfb = extra_flops_per_image(args.workload, S)
    if args.workload == "ae":  # the 3x3 reconstruction head runs on the tensor-core conv kernels; there is no 1x1 head
        tc += xfb + 3 * 2.0 * 3 * S * S * 32
    elif args.workload == "clip":
        tc += xfb
    fb += xfb
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback (B200_PROFILING.md sustained 1.4 PF)"
    roofline = None
    roofline_hbm = None
    breakdown = None
    traffic = {}
    traffic_file = None
    for cand in ("r2_traffic.json", "r1_traffic.json"):  # DRAM bytes per step and kernel family from the committed ncu
        try:                                             # launch list (tools/traffic_json.py)
            traffic = json.load(open(os.path.join(ROOT, "profiles", cand)))
            traffic_file = cand
            break
        except Exception:
            continue
    std_cfg = args.workload == "unet" and B == 32 and S == 512
    if prof is not None:
        tot = prof.totals_ms()
        conv_names = ("b200unet_conv_fprop", "b200unet_conv_dgrad", "b200unet_conv_dgrad_s2", "b200unet_conv_wgrad",
                      "b200unet_image_to_nhwc32_bf16")
        conv_ms = sum(tot.get(n, (0.0, 0))[0] for n in conv_names)
        conv_ms_step = conv_ms / prof_steps
        achieved = tc * B / (conv_ms_step * 1e-3) / 1e12 if conv_ms_step > 0 else 0.0
        tconv = traffic.get("conv")
        roofline = {"bound": "tensor", "kernel": "tcgen05 implicit-GEMM conv family (gconv/nconv/pconv fprop+dgrad, wgrad/wgradn + finalize), every 3x3 conv of the step",
                    "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                    "traffic": (tconv["dram_read_bytes"] + tconv["dram_write_bytes"]) if tconv and std_cfg else None,
                    "traffic_note": "DRAM bytes of the family per step (ncu dram__bytes_read.sum + dram__bytes_write.sum, "
                                    "profiles/%s); algorithmic conv FLOPs per step = %.3e" % (traffic_file, tc * B),
                    "peak_source": peak_src, "conv_ms_per_step": conv_ms_step,
                    "conv_share_of_step": conv_ms_step / ms_serial, "serial_ms_per_step": ms_serial,
                    "whole_step_tflops": fb * B / (ms_per_step * 1e-3) / 1e12}
        # the dominant HBM-bound family: InstanceNorm + LeakyReLU + dropout, forward apply and fused backward.
        # Algorithmic bytes (SURVEY.md 8d, bf16): forward read + write = 4 B/element, backward read dz, read y,
        # write dy = 6 B/element, 65.27 M elements per image at 512^2 (scaled by the pixel count otherwise).
        elems = 65.27e6 * (S / 512.0) ** 2 * B
        norm_ms = sum(tot.get(n, (0.0, 0))[0] for n in ("b200unet_in_apply", "b200unet_in_backward")) / prof_steps
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        if norm_ms > 0:
            ach = elems * 10.0 / (norm_ms * 1e-3) / 1e9
            tn = traffic.get("norm")
            roofline_hbm = {"bound": "hbm", "kernel": "in_apply + in_backward (InstanceNorm/LeakyReLU/dropout fwd + bwd)",
                            "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                            "traffic": (tn["dram_read_bytes"] + tn["dram_write_bytes"]) if tn and std_cfg else None,
                            "algorithmic_bytes_per_step": elems * 10.0, "ms_per_step": norm_ms,
                            "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"}
        breakdown = {k.replace("b200unet_", ""): {"ms_per_step": v[0] / prof_steps, "calls_per_step": v[1] / prof_steps}
                     for k, v in sorted(tot.items(), key=lambda kv: -kv[1][0])}
        breakdown["_note"] = ("measured in a second region of %d steps with the weight-gradient kernels serialised "
                              "(%.3f ms/step); the headline region overlaps them with the norm backward" % (prof_steps, ms_serial))

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        s_per = cpu_port_step_time(4, S, 2, 1, cores, args.workload)
        cpu = {"value": 4 / s_per, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "2 steps of batch 4 after 1 warm-up (oracle/unet_oracle.py, fp32 torch CPU ops)"}

    if rank == 0:
        out = {
            "metric": WORKLOADS[args.workload][0], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_text(args.workload, world, B, S),
                       "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"dp{world}",
                       "l2": "working set (>10 GB of activations per step) far exceeds the 126 MB L2; no flush needed",
                       "inputs": "value: fp32 NCHW image + int64 mask resident in HBM (the trainer's types, train.py:630-631); "
                                 "e2e: uint8 HWC image + uint8 mask copied from pinned host memory every step "
                                 "(the dataset's storage types, train.py:299-311), normalised on the device",
                       "optimizer_step": "not included in value / e2e (BASELINE.md: step = forward + loss + backward); measured "
                                         "beside them in with_optimizer_step; weights are constant in the value / e2e regions, so "
                                         "their cached bf16 packs are reused (no per-step repack there)",
                       "step_form": ("value: CUDA-graph replay of forward + loss + backward (graph.GraphedStep), eager form in "
                                     "`eager`" if eager_leg is not None else "eager (one host-enqueued launch per kernel)"),
                       "presteps": f"{presteps} untimed steps after the warm-up (power-cap steady state)",
                       "overlap": "weight-gradient kernels on a side stream beside the next layer's norm backward"
                                  if model.overlap_wgrad else "none (single stream)",
                       "nccl": (f"communicator capped to {nccl_ctas} CTAs; conv grids sized for "
                                f"{os.environ.get('B200UNET_RESERVED_SMS', '0')} fewer SMs") if world > 1 else None},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": wl.h2d_bytes, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps},
            "with_optimizer_step": with_sgd,
            "eager": eager_leg,
            "graph": {"value_is_graph_replay": eager_leg is not None, "e2e_is_graph_replay": e2e_graphed,
                      "error": graph_err},
            "gpu_launches": int(launches),
            "remeasured": remeasured,
            "peak_memory_gib": round(torch.cuda.max_memory_allocated(dev) / 2**30, 2),
            "per_rank_ms_per_step": per_rank_resident,
            "per_rank_ms_per_step_without_allreduce": per_rank_no_allreduce,
            "allreduce_only_ms": allreduce_only_ms,
            "clocks": clocks,
            "roofline": roofline,
            "roofline_hbm": roofline_hbm,
            "cpu_baseline": cpu,
            "breakdown_ms_per_step": breakdown,
        }
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
