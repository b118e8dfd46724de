"""CPU: the conv weight packs the flat optimizers emit (optim.flat_pack_kinds, packs.layout), and when packs.PackStore
reuses a pack.  No device: the store test swaps packs.build for a stand-in that records what it was asked to build."""
import torch

from unet_implementations_b200 import packs
from unet_implementations_b200.optim import flat_pack_kinds

BF16 = torch.bfloat16


def _layouts(model, dtype=BF16):
    return [packs.layout(conv, kind, dtype) for conv, kind in flat_pack_kinds(model)]


def test_default_unet_emits_one_stem_and_21_plain_packs():
    from unet_implementations_b200.models.unet import UNet
    lays = _layouts(UNet())
    assert len(lays) == 22
    assert lays[0] == packs.Layout("stem", cout=32, cin=3, cout_pad=32, cin_pad=32, ksize=3, dtype=BF16)
    assert all(lay.kind == "conv" and lay.cin_pad == lay.cin and lay.cout_pad == lay.cout and lay.ksize == 3
               for lay in lays[1:])


def test_clip_unet_adds_one_centre_tap_pack():
    from unet_implementations_b200.models.clip_unet import UNet
    lays = _layouts(UNet())
    k1 = [lay for lay in lays if lay.kind == "k1"]
    assert len(lays) == 23 and len(k1) == 1
    assert k1[0] == packs.Layout("k1", cout=512, cin=1024, cout_pad=512, cin_pad=1024, ksize=1, dtype=BF16)


def test_autoencoder_head_pads_its_output_channels():
    from unet_implementations_b200.models.autoencoder import Autoencoder
    model = Autoencoder()
    kinds = flat_pack_kinds(model)
    assert [kind for _, kind in kinds].count("head") == 1 and kinds[-1] == (model.reconstruction_output[0], "head")
    assert packs.layout(model.reconstruction_output[0], "head") == \
        packs.Layout("head", cout=3, cin=32, cout_pad=32, cin_pad=32, ksize=3, dtype=BF16)
    assert packs.layout(model.reconstruction_output[0], "head", torch.float32).cout_pad == 8


def test_single_channel_stem_pack_serves_only_stem_requests(monkeypatch):
    from unet_implementations_b200.models.unet import UNet
    model = UNet(in_channels=1)
    conv, kind = flat_pack_kinds(model)[0]
    assert kind == "stem" and conv is model.encoder_stages[0].block[0]
    assert (packs.layout(conv, "stem").cin, packs.layout(conv, "stem").cin_pad) == (1, 32)
    assert packs.layout(conv, "conv") != packs.layout(conv, "stem")

    built = []

    def fake_build(w, lay, need_dgrad):
        built.append((lay.kind, need_dgrad))
        return torch.empty(0), torch.empty(0) if need_dgrad else None

    monkeypatch.setattr(packs, "build", fake_build)
    store = model._packs
    emitted = store.emit(conv, "stem")
    assert built == [("stem", False)] and store.emit(conv, "stem") is emitted
    view = model._ext_packs[id(conv.weight)]  # the read-only view tests and tools read
    assert view["key"] == "stem" and view["wf"] is emitted.wf and view["version"] == conv.weight._version
    assert store.get(conv, "stem", BF16, False)[0] is emitted.wf
    wf, _ = store.get(conv, "conv", BF16, False)  # the plain first-conv route of images narrower than 64 px
    assert wf is not emitted.wf and built[-1] == ("conv", False)
    assert store.get(conv, "conv", BF16, False)[0] is wf and len(built) == 2
    _, wd = store.get(conv, "conv", BF16, True)  # a dgrad pack is needed: rebuilt
    assert wd is not None and len(built) == 3
    with torch.no_grad():
        conv.weight.add_(1.0)  # someone else wrote the weight: every pack of it is stale
    assert store.get(conv, "stem", BF16, False)[0] is not emitted.wf and len(built) == 4
    store.stamp([conv.weight])  # a flat step rewrote the emitted pack from the current values
    assert store.get(conv, "stem", BF16, False)[0] is emitted.wf and len(built) == 4
