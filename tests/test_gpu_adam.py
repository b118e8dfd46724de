"""GPU: FusedAdam, the flat Adam / AdamW step (optim.FusedAdam, csrc/train_aux.cu: flat_step_kernel<AdamRule>), used
WITH the model, against torch.optim.Adam (foreach on CUDA) -- the autoencoder trainer's optimizer
(AE_pretrained/reconstruction/src/train.py:390-394).

As for FusedSGD (tests/test_gpu_optim.py) the comparison is exact: two copies of a model, one stepped by torch, one
by FusedAdam; outputs, loss, every parameter and every piece of optimizer state must be bit-identical after every
step.  The kernels of the model are deterministic, FusedAdam restates torch's foreach Adam operation by operation and
the packs it emits are the round-to-nearest bf16 of the same values, so any difference is a bug.
"""
import copy

import pytest
import torch

pytestmark = pytest.mark.gpu


def _unet(kind):
    torch.manual_seed(1234)
    if kind == "full":
        from unet_implementations_b200.models.unet import UNet
        return UNet().cuda().train()
    if kind == "small":
        from unet_implementations_b200.models.unet import UNet
        return UNet(n_stages=4, features_per_stage=[32, 64, 128, 128], encoder_dropout_rates=[0, 0, 0.1, 0.2],
                    decoder_dropout_rates=[0.2, 0.1, 0]).cuda().train()
    if kind in ("ae", "ae_nodrop"):
        from unet_implementations_b200.models.autoencoder import Autoencoder
        enc, dec = ([0, 0, 0.05, 0.1], [0.1, 0.05, 0]) if kind == "ae" else ([0] * 4, [0] * 3)
        return Autoencoder(n_stages=4, features_per_stage=[32, 64, 128, 128], encoder_dropout_rates=enc,
                           decoder_dropout_rates=dec).cuda().train()
    if kind == "ae_full":
        from unet_implementations_b200.models.autoencoder import Autoencoder
        return Autoencoder(encoder_dropout_rates=[0.0, 0.0, 0.05, 0.1, 0.15, 0.15],
                           decoder_dropout_rates=[0.15, 0.1, 0.1, 0.05, 0.0]).cuda().train()
    if kind == "clip":
        from unet_implementations_b200.models.clip_unet import UNet as ClipUNet
        return ClipUNet(n_stages=4, features_per_stage=[32, 64, 128, 128], encoder_dropout_rates=[0] * 4,
                        decoder_dropout_rates=[0] * 3, clip_dim=32).cuda().train()
    raise ValueError(kind)


def _task(kind, size, b=2, seed=0):
    """(inputs, loss_fn, target) of one model kind: SimpleLoss on segmentation labels, MSELoss on an image."""
    from unet_implementations_b200.models.losses import MSELoss, SimpleLoss
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(b, 3, size, size, generator=g).cuda()
    if kind.startswith("ae"):
        return (x,), MSELoss(), torch.rand(b, 3, size, size, generator=g).cuda()
    t = torch.randint(0, 3, (b, size, size), generator=g)
    t[torch.rand(b, size, size, generator=g) < 0.1] = 255
    if kind == "clip":
        clip = torch.randn(b, 32, size >> 3, size >> 3, generator=g).cuda()
        return (x, clip), SimpleLoss(), t.cuda()
    return (x,), SimpleLoss(), t.cuda()


def _state(opt, p):
    st = opt.state[p]
    # torch keeps `step` on the CPU and advances it in place: copy it (.cpu() of a CPU tensor is the tensor itself)
    return [st["step"].to("cpu", copy=True), st["exp_avg"].clone(), st["exp_avg_sq"].clone()]


def _run(model, opt, task, steps, sched=None, scale=None, scaler=None):
    inputs, loss_fn, target = task
    out = []
    for s in range(steps):
        torch.manual_seed(100 + s)  # same dropout draw in both runs
        opt.zero_grad(set_to_none=True)
        if scaler is not None:
            with torch.autocast("cuda", dtype=torch.float16):
                y = model(*inputs)
                loss = loss_fn(y, target)
            scaler.scale(loss).backward()
            scaler.step(opt)
            scaler.update()
        else:
            y = model(*inputs)
            loss = loss_fn(y, target)
            loss.backward()
            if scale is not None:
                for p in model.parameters():
                    if p.grad is not None:
                        p.grad.mul_(scale)
            opt.step()
        if sched is not None:
            sched.step()
        ps = [p for p in model.parameters()]
        out.append((y.detach().clone(), loss.detach().clone(), [p.detach().clone() for p in ps],
                    [_state(opt, p) if p in opt.state else None for p in ps]))
    return out


def _assert_same(ra, rb):
    for s, ((ya, la, pa, sa), (yb, lb, pb, sb)) in enumerate(zip(ra, rb)):
        assert torch.equal(ya, yb), f"step {s}: outputs differ by {(ya - yb).abs().max().item():.3e} (stale packs?)"
        assert torch.equal(la, lb), f"step {s}: loss {la.item()!r} vs {lb.item()!r}"
        for i, (u, v, su, sv) in enumerate(zip(pa, pb, sa, sb)):
            assert (su is None) == (sv is None), f"step {s}: parameter {i} has state in one optimizer only"
            if su is not None:
                for name, x, z in zip(("step", "exp_avg", "exp_avg_sq"), su, sv):
                    assert torch.equal(x, z), \
                        f"step {s}: {name} of parameter {i} {tuple(u.shape)} differs by {(x - z).abs().max().item():.3e}"
            assert torch.equal(u, v), f"step {s}: parameter {i} {tuple(u.shape)} differs by {(u - v).abs().max().item():.3e}"


WD = {"none": {}, "l2": dict(weight_decay=1e-2), "adamw": dict(weight_decay=1e-2, decoupled_weight_decay=True)}


@pytest.mark.parametrize("kind,size,wd", [("small", 64, "none"), ("small", 64, "l2"), ("small", 64, "adamw"),
                                          ("full", 128, "l2"), ("ae", 64, "none"), ("ae", 64, "adamw"),
                                          ("ae_full", 128, "none")])
def test_fused_adam_is_bit_identical_to_torch_adam(kind, size, wd):
    from unet_implementations_b200.optim import FusedAdam
    ma = _unet(kind)
    mb = copy.deepcopy(ma)
    task = _task(kind, size)
    kw = dict(lr=2e-3, betas=(0.9, 0.999), eps=1e-8, **WD[wd])
    oa = torch.optim.Adam(ma.parameters(), foreach=True, **kw)
    ob = FusedAdam(mb.parameters(), model=mb, **kw)
    if kind.startswith("ae"):  # the autoencoder trainer's schedule
        sa, sb = (torch.optim.lr_scheduler.CosineAnnealingLR(o, T_max=6) for o in (oa, ob))
    else:
        sa = sb = None
    ra = _run(ma, oa, task, 4, sa)
    rb = _run(mb, ob, task, 4, sb)
    _assert_same(ra, rb)
    assert not torch.equal(ra[0][0], ra[3][0])  # the convs did see the updates


def test_fused_adam_with_beta1_at_most_one_half():
    """1 - beta1 >= 0.5 takes the other branch of ATen's lerp: end - (end - self) * (1 - weight)."""
    from unet_implementations_b200.optim import FusedAdam
    ma = _unet("small")
    mb = copy.deepcopy(ma)
    task = _task("small", 64)
    kw = dict(lr=1e-3, betas=(0.3, 0.99), eps=1e-6, weight_decay=1e-3)
    ra = _run(ma, torch.optim.Adam(ma.parameters(), foreach=True, **kw), task, 4)
    rb = _run(mb, FusedAdam(mb.parameters(), model=mb, **kw), task, 4)
    _assert_same(ra, rb)


def test_fused_adam_with_beta2_zero():
    """beta2 = 0 makes the addcmul value 1 - beta2 exactly 1, where ATen's addcmul takes its other form: one fma of
    g * g into v (DeviceAddCmulCdiv.cuh) instead of the product rounded on its own."""
    from unet_implementations_b200.optim import FusedAdam
    ma = _unet("small")
    mb = copy.deepcopy(ma)
    task = _task("small", 64)
    kw = dict(lr=1e-3, betas=(0.9, 0.0), eps=1e-8, weight_decay=1e-2, decoupled_weight_decay=True)
    ra = _run(ma, torch.optim.Adam(ma.parameters(), foreach=True, **kw), task, 4)
    rb = _run(mb, FusedAdam(mb.parameters(), model=mb, **kw), task, 4)
    _assert_same(ra, rb)


def _expected_packs(spec, conv):
    from unet_implementations_b200 import ops
    w = conv.weight.detach()
    key = spec["key"]
    if key == "stem":
        return ops.pack_stem_weights(w), None, None
    if key == "k1":
        w3 = torch.zeros((conv.out_channels, conv.in_channels, 3, 3), dtype=torch.float32, device=w.device)
        w3[:, :, 1, 1] = w[:, :, 0, 0]
        w = w3
    elif key == "head":
        wp = torch.zeros((32, conv.in_channels, 3, 3), dtype=torch.float32, device=w.device)
        wp[:conv.out_channels] = w
        w = wp
    wf, wd = ops.pack_conv_weights(w, need_dgrad=True)
    ws = ops.pack_s2_dgrad_weights(wd) if spec["ws"] is not None else None
    return wf, wd, ws


@pytest.mark.parametrize("kind,size", [("full", 64), ("clip", 64), ("ae", 64)])
def test_fused_adam_emits_the_packs_the_pack_kernels_would(kind, size):
    from unet_implementations_b200.optim import FusedAdam
    model = _unet(kind)
    opt = FusedAdam(model.parameters(), lr=1e-3, weight_decay=1e-2, decoupled_weight_decay=True, model=model)
    _run(model, opt, _task(kind, size), 2)
    ext = model._ext_packs
    convs = {id(m.weight): m for m in model.modules() if isinstance(m, torch.nn.Conv2d)}
    kinds = set()
    for wid, spec in ext.items():
        conv = convs[wid]
        assert spec["version"] == conv.weight._version
        kinds.add((spec["key"], spec["ws"] is not None))
        wf, wd, ws = _expected_packs(spec, conv)
        assert torch.equal(spec["wf"], wf), (spec["key"], conv)
        if wd is not None:
            assert torch.equal(spec["wd"], wd), (spec["key"], conv)
        if ws is not None:
            assert torch.equal(spec["ws"], ws), (spec["key"], conv)
    expected = {"full": {("stem", False), ("conv", False), ("conv", True)},
                "clip": {("stem", False), ("conv", False), ("conv", True), ("k1", False)},
                "ae": {("stem", False), ("conv", False), ("conv", True), ("head", False)}}[kind]
    assert kinds == expected
    # parameters are views of ONE flat master buffer, the moments of two more, all at the gradient offsets
    fs = opt._flat
    for p in model.parameters():
        off = fs.sink.offsets[id(p)]
        assert p.data_ptr() == fs.master.data_ptr() + 4 * off
        assert opt.state[p]["exp_avg"].data_ptr() == fs.bufs["exp_avg"].data_ptr() + 4 * off
        assert opt.state[p]["exp_avg_sq"].data_ptr() == fs.bufs["exp_avg_sq"].data_ptr() + 4 * off


def _perturbed(sd):
    sd = copy.deepcopy(sd)
    for st in sd["state"].values():
        st["exp_avg"] = st["exp_avg"] * 0.5
        st["exp_avg_sq"] = st["exp_avg_sq"] * 2.0
        st["step"] = st["step"] + 3
    return sd


@pytest.mark.parametrize("source", ["torch", "fused"])
def test_state_dict_round_trips_with_torch_adam(source):
    """Resume (train.py loads the optimizer state after building it): a state_dict of either optimizer, loaded into
    both, continues bit-identically; FusedAdam's state_dict has torch.optim.Adam's layout."""
    from unet_implementations_b200.optim import FusedAdam
    ma = _unet("ae")
    mb = copy.deepcopy(ma)
    task = _task("ae", 64)
    kw = dict(lr=1e-3, weight_decay=1e-4)
    oa = torch.optim.Adam(ma.parameters(), foreach=True, **kw)
    ob = FusedAdam(mb.parameters(), model=mb, **kw)
    _assert_same(_run(ma, oa, task, 2), _run(mb, ob, task, 2))
    sda, sdb = oa.state_dict(), ob.state_dict()
    assert set(sda["param_groups"][0]) - {"capturable"} == set(sdb["param_groups"][0])
    for k, st in sda["state"].items():
        stb = sdb["state"][k]
        assert set(st) == set(stb) == {"step", "exp_avg", "exp_avg_sq"}
        assert stb["step"].dtype == torch.float32 and stb["step"].device.type == "cpu" and stb["step"].dim() == 0
        assert all(torch.equal(st[n].cpu(), stb[n].cpu()) for n in st)
    sd = _perturbed(sda if source == "torch" else sdb)
    torch.manual_seed(7)
    msd = {k: v + 0.01 * torch.randn_like(v) for k, v in ma.state_dict().items()}
    ma.load_state_dict(msd)
    mb.load_state_dict(msd)
    oa.load_state_dict(copy.deepcopy(sd))
    ob.load_state_dict(copy.deepcopy(sd))
    _assert_same(_run(ma, oa, task, 3), _run(mb, ob, task, 3))
    assert all(float(oa.state[p]["step"]) == 8.0 for p in ma.parameters())


def test_frozen_encoder_keeps_parameters_and_step_counts():
    """Transfer learning freezes the encoder (AE_pretrained/transfer_learning/models/unet.py:452-453): its parameters
    get no gradient, so neither they nor their step counts may move; the rest trains exactly like torch."""
    from unet_implementations_b200.optim import FusedAdam
    ma = _unet("small")
    mb = copy.deepcopy(ma)
    task = _task("small", 64)
    kw = dict(lr=1e-3, weight_decay=1e-2, decoupled_weight_decay=True)
    oa = torch.optim.Adam(ma.parameters(), foreach=True, **kw)
    ob = FusedAdam(mb.parameters(), model=mb, **kw)
    _assert_same(_run(ma, oa, task, 2), _run(mb, ob, task, 2))
    for m in (ma, mb):
        for p in m.encoder_stages.parameters():
            p.requires_grad_(False)
    frozen = list(mb.encoder_stages.parameters())
    before = [p.detach().clone() for p in frozen]
    _assert_same(_run(ma, oa, task, 3), _run(mb, ob, task, 3))
    for p, q in zip(frozen, before):
        assert torch.equal(p, q)
        assert float(ob.state[p]["step"]) == 2.0
    frozen_ids = {id(p) for p in frozen}
    assert all(float(ob.state[p]["step"]) == 5.0 for p in mb.parameters() if id(p) not in frozen_ids)
    # an optimizer built over the trainable parameters only (the transfer-learning trainer's form)
    mc = _unet("small")
    for p in mc.encoder_stages[0].parameters():
        p.requires_grad_(False)
    md = copy.deepcopy(mc)
    oc = torch.optim.Adam([p for p in mc.parameters() if p.requires_grad], foreach=True, **kw)
    od = FusedAdam([p for p in md.parameters() if p.requires_grad], model=md, **kw)
    _assert_same(_run(mc, oc, task, 3), _run(md, od, task, 3))


def test_grad_scale_equals_torch_on_prescaled_gradients():
    """grad_scale (the 1 / world size of ddp.BucketedGradAllReduce) multiplies every gradient inside the step:
    exactly torch.optim.Adam on gradients pre-multiplied by the same power of two."""
    from unet_implementations_b200.optim import FusedAdam
    ma = _unet("small")
    mb = copy.deepcopy(ma)
    task = _task("small", 64)
    kw = dict(lr=1e-3, weight_decay=1e-2)
    oa = torch.optim.Adam(ma.parameters(), foreach=True, **kw)
    ob = FusedAdam(mb.parameters(), model=mb, grad_scale=0.5, **kw)
    _assert_same(_run(ma, oa, task, 4, scale=0.5), _run(mb, ob, task, 4))


def test_fp16_autocast_gradscaler_loop_matches_torch_adam():
    """train.py wraps the step in autocast + GradScaler: the scaler unscales the flat gradient views in place and
    skips steps with non-finite gradients; the loop must stay bit-identical to the same loop with torch Adam."""
    from unet_implementations_b200.optim import FusedAdam
    ma = _unet("small")
    mb = copy.deepcopy(ma)
    task = _task("small", 64)
    oa = torch.optim.Adam(ma.parameters(), lr=1e-3, foreach=True)
    ob = FusedAdam(mb.parameters(), lr=1e-3, model=mb)
    ra = _run(ma, oa, task, 5, scaler=torch.amp.GradScaler("cuda"))
    rb = _run(mb, ob, task, 5, scaler=torch.amp.GradScaler("cuda"))
    _assert_same(ra, rb)


def test_whole_autoencoder_step_with_fused_adam_in_one_graph():
    """forward + MSELoss + backward + FusedAdam(capturable=True) replayed as ONE graph (graph.GraphedStep); the
    cosine schedule is stepped between replays and reaches the kernel through the float64 device scalar.  Against an
    eager torch Adam loop on a second copy: bit-identical outputs, parameters and state."""
    from unet_implementations_b200.graph import GraphedStep
    from unet_implementations_b200.optim import FusedAdam
    ma = _unet("ae_nodrop")
    mb = copy.deepcopy(ma)
    (x,), loss_fn, t = _task("ae", 64)
    kw = dict(lr=2e-3, weight_decay=1e-2, decoupled_weight_decay=True)
    oa = torch.optim.Adam(ma.parameters(), foreach=True, **kw)
    ob = FusedAdam(mb.parameters(), model=mb, capturable=True, **kw)
    sa, sb = (torch.optim.lr_scheduler.CosineAnnealingLR(o, T_max=8) for o in (oa, ob))

    def step(model, opt):
        opt.zero_grad(set_to_none=True)
        loss = loss_fn(model(x), t)
        loss.backward()
        opt.step()
        return loss

    step(ma, oa), sa.step()
    step(mb, ob), sb.step()
    gs = GraphedStep(lambda: step(mb, ob), warmup=1, optimizer=ob)  # the warm-up step is a real training step
    step(ma, oa)
    for _ in range(4):
        sa.step(), sb.step()
        la = step(ma, oa)
        lb = gs.replay()
        assert torch.equal(la.detach(), lb.detach())
    for pa, pb in zip(ma.parameters(), mb.parameters()):
        assert torch.equal(pa, pb)
        assert all(torch.equal(u, v) for u, v in zip(_state(oa, pa), _state(ob, pb)))
    assert float(ob.state[next(mb.parameters())]["step"]) == 6.0


def test_capturing_before_the_first_eager_step_is_a_clear_error():
    from unet_implementations_b200.optim import FusedAdam
    model = _unet("ae_nodrop")
    opt = FusedAdam(model.parameters(), model=model, capturable=True)
    graph = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError, match="capturable=True and after one eager step"):
        with torch.cuda.graph(graph):
            opt.step()
