"""GPU: the fused optimizer step used WITH the model (SURVEY.md 8f row 1; Our_UNet/src/train.py:431-453, :650, :664).

The round-1 bug these tests exist for: `FusedSGD` updates parameters through raw pointers, `UNet` caches its bf16
operand packs per parameter version, so the convs kept running on the initial weights.  The gate is the strongest
one available: two copies of the same `UNet`, one stepped by `torch.optim.SGD`, one by `FusedSGD` -- logits, loss and
EVERY parameter must be bit-identical after every step (the kernels are deterministic, the optimizer arithmetic is
torch's operation by operation, and the packs the optimizer emits are the round-to-nearest bf16 of the same values).
"""
import copy

import pytest
import torch

pytestmark = pytest.mark.gpu


def _model(full=False):
    from unet_implementations_b200.models.unet import UNet
    torch.manual_seed(1234)
    if full:
        return UNet().cuda().train()
    return UNet(n_stages=4, features_per_stage=[32, 64, 128, 128], encoder_dropout_rates=[0, 0, 0.1, 0.2],
                decoder_dropout_rates=[0.2, 0.1, 0]).cuda().train()


def _batch(size, b=2, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(b, 3, size, size, generator=g).cuda()
    t = torch.randint(0, 3, (b, size, size), generator=g)
    t[torch.rand(b, size, size, generator=g) < 0.1] = 255
    return x, t.cuda()


def _run(model, opt, x, t, steps, sched=None):
    from unet_implementations_b200.models.losses import SimpleLoss
    loss_fn = SimpleLoss()
    out = []
    for s in range(steps):
        torch.manual_seed(100 + s)  # same dropout draw in both runs
        opt.zero_grad(set_to_none=True)
        logits = model(x)
        loss = loss_fn(logits, t)
        loss.backward()
        opt.step()
        if sched is not None:
            sched.step()
        out.append((logits.detach().clone(), loss.detach().clone(), [p.detach().clone() for p in model.parameters()]))
    return out


@pytest.mark.parametrize("flat", [False, True])
@pytest.mark.parametrize("full,size", [(False, 64), (True, 128)])
def test_fused_sgd_with_unet_is_bit_identical_to_torch_sgd(flat, full, size):
    from unet_implementations_b200.optim import FusedSGD
    ma = _model(full)
    mb = copy.deepcopy(ma)
    x, t = _batch(size)
    kw = dict(lr=0.005, momentum=0.99, nesterov=True, weight_decay=1e-4)  # train.py:445-451
    oa = torch.optim.SGD(ma.parameters(), **kw)
    ob = FusedSGD(mb.parameters(), model=mb if flat else None, **kw)
    lam = lambda e: (1 - e / 10) ** 0.9  # noqa: E731  (train.py:466-475)
    ra = _run(ma, oa, x, t, 4, torch.optim.lr_scheduler.LambdaLR(oa, lam))
    rb = _run(mb, ob, x, t, 4, torch.optim.lr_scheduler.LambdaLR(ob, lam))
    for s, ((la, lossa, pa), (lb, lossb, pb)) in enumerate(zip(ra, rb)):
        assert torch.equal(la, lb), f"step {s}: logits differ by {(la - lb).abs().max().item():.3e} (stale weight packs?)"
        assert torch.equal(lossa, lossb)
        for i, (u, v) in enumerate(zip(pa, pb)):
            assert torch.equal(u, v), f"step {s}: parameter {i} {tuple(u.shape)} differs by {(u - v).abs().max().item():.3e}"
    # the convs did see the updates: step-3 logits are not step-0 logits
    assert not torch.equal(ra[0][0], ra[3][0])
    sa, sb = oa.state_dict(), ob.state_dict()
    assert sa["state"].keys() == sb["state"].keys()
    for k in sa["state"]:
        assert torch.equal(sa["state"][k]["momentum_buffer"], sb["state"][k]["momentum_buffer"])


@pytest.mark.parametrize("size", [32, 64])
def test_flat_sgd_with_a_single_channel_unet_is_bit_identical_to_torch_sgd(size):
    """The flat step emits a stem pack (input channels padded to 32) for a 1-channel first conv.  Images narrower than
    64 px take the plain first-conv route, which must get its own pack, not the emitted stem pack."""
    from unet_implementations_b200.models.unet import UNet
    from unet_implementations_b200.optim import FusedSGD
    torch.manual_seed(1234)
    ma = UNet(in_channels=1, n_stages=4, features_per_stage=[32, 64, 128, 128]).cuda().train()
    mb = copy.deepcopy(ma)
    x, t = _batch(size)
    x = x[:, :1].contiguous()
    kw = dict(lr=0.005, momentum=0.99, nesterov=True, weight_decay=1e-4)
    ra = _run(ma, torch.optim.SGD(ma.parameters(), **kw), x, t, 2)
    rb = _run(mb, FusedSGD(mb.parameters(), model=mb, **kw), x, t, 2)
    for s, ((la, lossa, pa), (lb, lossb, pb)) in enumerate(zip(ra, rb)):
        assert torch.equal(la, lb), f"step {s}: logits differ by {(la - lb).abs().max().item():.3e}"
        assert torch.equal(lossa, lossb)
        assert all(torch.equal(u, v) for u, v in zip(pa, pb))


def test_flat_step_emits_the_packs_the_pack_kernels_would():
    from unet_implementations_b200 import ops
    from unet_implementations_b200.optim import FusedSGD
    model = _model(full=True)
    x, t = _batch(64)
    opt = FusedSGD(model.parameters(), lr=0.05, momentum=0.9, nesterov=True, weight_decay=1e-4, model=model)
    _run(model, opt, x, t, 2)
    ext = model._ext_packs
    convs = [m for m in model.modules() if isinstance(m, torch.nn.Conv2d) and m.kernel_size == (3, 3)]
    assert len(ext) == len(convs) == 22
    kinds = set()
    for conv in convs:
        spec = ext[id(conv.weight)]
        assert spec["version"] == conv.weight._version
        kinds.add((spec["key"], spec["ws"] is not None))
        if spec["key"] == "stem":
            assert torch.equal(spec["wf"], ops.pack_stem_weights(conv.weight))
            continue
        wf, wd = ops.pack_conv_weights(conv.weight, need_dgrad=True)
        assert torch.equal(spec["wf"], wf) and torch.equal(spec["wd"], wd), conv
        if spec["ws"] is not None:
            assert torch.equal(spec["ws"], ops.pack_s2_dgrad_weights(wd))
    assert kinds == {("stem", False), ("conv", False), ("conv", True)}
    # parameters are views of ONE flat master buffer, gradients of ONE flat gradient buffer, same offsets
    fs = opt._flat
    for p in model.parameters():
        off = fs.sink.offsets[id(p)]
        assert p.data_ptr() == fs.master.data_ptr() + 4 * off
        assert p.grad is not None and p.grad.data_ptr() == fs.sink.flat.data_ptr() + 4 * off


def test_flat_step_survives_load_state_dict_and_frozen_parameters():
    """train.py:888-902 resumes by load_state_dict AFTER the optimizer exists; transfer learning freezes the encoder
    (AE_pretrained/transfer_learning/models/unet.py:452-453)."""
    from unet_implementations_b200.models.losses import SimpleLoss
    from unet_implementations_b200.optim import FusedSGD
    ma = _model()
    mb = copy.deepcopy(ma)
    for m in (ma, mb):
        for p in m.encoder_stages[0].parameters():
            p.requires_grad_(False)
    kw = dict(lr=0.01, momentum=0.99, nesterov=True, weight_decay=1e-4)
    oa = torch.optim.SGD([p for p in ma.parameters() if p.requires_grad], **kw)
    ob = FusedSGD([p for p in mb.parameters() if p.requires_grad], model=mb, **kw)
    x, t = _batch(64)
    _run(ma, oa, x, t, 2)
    _run(mb, ob, x, t, 2)
    # "resume": new weights and optimizer state arrive through the public loaders
    torch.manual_seed(7)
    sd = {k: v + 0.01 * torch.randn_like(v) for k, v in ma.state_dict().items()}
    osd = copy.deepcopy(oa.state_dict())
    for st in osd["state"].values():
        st["momentum_buffer"] = st["momentum_buffer"] * 0.5
    ma.load_state_dict(sd)
    mb.load_state_dict(sd)
    oa.load_state_dict(copy.deepcopy(osd))
    ob.load_state_dict(copy.deepcopy(osd))
    ra = _run(ma, oa, x, t, 3)
    rb = _run(mb, ob, x, t, 3)
    for (la, _, pa), (lb, _, pb) in zip(ra, rb):
        assert torch.equal(la, lb)
        assert all(torch.equal(u, v) for u, v in zip(pa, pb))
    loss = SimpleLoss()(mb(x), t)
    assert torch.isfinite(loss)


def test_flat_sink_rejects_an_aliased_stale_grad():
    from unet_implementations_b200.flat import FlatGradSink
    from unet_implementations_b200.models.losses import SimpleLoss
    model = _model()
    FlatGradSink(model)
    x, t = _batch(64)
    SimpleLoss()(model(x), t).backward()
    w = model.segmentation_output.weight
    assert w.grad is not None
    if w.grad.data_ptr() == model._grad_sink.flat.data_ptr() + 4 * model._grad_sink.offsets[id(w)]:
        with pytest.raises(RuntimeError, match="set_to_none=True"):
            SimpleLoss()(model(x), t).backward()  # gradients kept from the first backward alias the buffer
    model.zero_grad(set_to_none=True)
    SimpleLoss()(model(x), t).backward()


# ------------------------------------------------------------------------------------------------ f2: uint8 inputs
def test_uint8_batch_feeds_the_stem_and_the_loss_bit_identically():
    """SURVEY.md 8f row 2 (train.py:299-311, :630-631): uint8 HWC images -> bf16 NHWC(32) in one kernel, uint8 masks
    read by the loss kernels.  Everything downstream must be bit-identical to the fp32 NCHW + int64 route."""
    from unet_implementations_b200 import data, ops
    from unet_implementations_b200.models.losses import SimpleLoss
    model = _model(full=True)
    g = torch.Generator().manual_seed(3)
    img = torch.randint(0, 256, (2, 128, 128, 3), generator=g, dtype=torch.uint8).cuda()
    msk = torch.randint(0, 3, (2, 128, 128), generator=g, dtype=torch.uint8)
    msk[torch.rand(2, 128, 128, generator=g) < 0.1] = 255
    msk = msk.cuda()
    x32, t64 = data.preprocess_batch(img, msk)
    assert torch.equal(ops.preprocess_u8_nhwc32(img, data.IMAGENET_MEAN, data.IMAGENET_STD), ops.image_to_nhwc32(x32))
    res = []
    for xin, tin in ((x32, t64), (img, msk)):
        model.zero_grad(set_to_none=True)
        torch.manual_seed(11)
        logits = model(xin)
        loss = SimpleLoss()(logits, tin)
        loss.backward()
        res.append((logits.detach().clone(), loss.detach().clone(), [p.grad.clone() for p in model.parameters()]))
    (la, lossa, ga), (lb, lossb, gb) = res
    assert torch.equal(la, lb) and torch.equal(lossa, lossb)
    assert all(torch.equal(u, v) for u, v in zip(ga, gb))
    # ragged sizes take the scalar path of the loss kernels and the tail of the layout kernel
    img2 = torch.randint(0, 256, (3, 37, 53, 3), generator=g, dtype=torch.uint8).cuda()
    x2, _ = data.preprocess_batch(img2, None)
    assert torch.equal(ops.preprocess_u8_nhwc32(img2, data.IMAGENET_MEAN, data.IMAGENET_STD), ops.image_to_nhwc32(x2))
    lg = torch.randn(3, 3, 37, 53, generator=g).cuda().requires_grad_(True)
    t8 = torch.randint(0, 3, (3, 37, 53), generator=g, dtype=torch.uint8)
    t8[torch.rand(3, 37, 53, generator=g) < 0.2] = 255
    t8 = t8.cuda()
    l8 = SimpleLoss()(lg, t8)
    g8, = torch.autograd.grad(l8, lg)
    l64 = SimpleLoss()(lg, t8.long())
    g64, = torch.autograd.grad(l64, lg)
    assert torch.equal(l8, l64) and torch.equal(g8, g64)


def test_upblock_standalone_matches_the_reference_ops():
    """UpBlock.forward (unet.py:203-231) outside UNet.forward: bilinear 2x, cat([up, skip]), ConvBlock."""
    import torch.nn.functional as F
    from oracle import unet_oracle as O
    from unet_implementations_b200.models.unet import UpBlock
    torch.manual_seed(3)
    up = UpBlock(64, 32, 32, 3, spatial_dropout_rate=0.0).cuda().train()
    x = torch.randn(2, 64, 16, 16, device="cuda", requires_grad=True)
    skip = torch.randn(2, 32, 32, 32, device="cuda", requires_grad=True)
    out = up(x, skip)
    out.square().mean().backward()
    # oracle: the reference's op sequence in fp32 on the CPU with the same parameters
    xc, sc = x.detach().cpu().requires_grad_(True), skip.detach().cpu().requires_grad_(True)
    cat = torch.cat([F.interpolate(xc, size=sc.shape[2:], mode="bilinear", align_corners=False), sc], 1)
    h = cat
    mods = list(up.conv_block.block)
    ws = []
    for i in range(0, len(mods), 3):
        conv, norm = mods[i], mods[i + 1]
        w = conv.weight.detach().cpu().requires_grad_(True)
        gam, bet = norm.weight.detach().cpu().requires_grad_(True), norm.bias.detach().cpu().requires_grad_(True)
        ws.append((conv, w))
        h = F.leaky_relu(F.instance_norm(F.conv2d(h, w, conv.bias.detach().cpu(), 1, 1), weight=gam, bias=bet, eps=1e-5), 0.01)
    h.square().mean().backward()
    assert O.rel_l2(out.detach().cpu(), h.detach()) < 2e-2
    assert O.rel_l2(x.grad.cpu(), xc.grad) < 5e-2 and O.rel_l2(skip.grad.cpu(), sc.grad) < 5e-2
    for conv, w in ws:
        assert O.rel_l2(conv.weight.grad.cpu(), w.grad) < 5e-2
