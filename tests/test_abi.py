"""CPU: the C-ABI shared library loads and exports every symbol include/b200unet.h declares; the ctypes table in
_lib.py covers the same set.  No compute entry point is called (there is no GPU here)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "b200unet.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b200unet_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from unet_implementations_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = declared_symbols()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/b200unet.h but not exported"
    assert set(_lib.SIGNATURES) == set(names), set(_lib.SIGNATURES) ^ set(names)


def test_version_and_sizing_calls_need_no_gpu():
    from unet_implementations_b200 import _lib
    assert _lib.call("b200unet_version") == 100
    assert _lib.call("b200unet_conv_fprop_partials", 32, 512, 512, 32) >= 4
    assert _lib.call("b200unet_loss_workspace", 4, 512 * 512) > 0


def test_statistics_slots_cover_the_cta_pair_layout():
    """The fprop epilogue writes one partial-sum slot per (image, CTA, TMEM lane quarter); as CTA pairs (cta_group::2)
    a cluster owns 8 slots per image it touches.  The sizing call the caller allocates from must cover that layout
    for every streamed-weight layer of the model at the benchmark batch (conv_fprop_dgrad.cu: gconv_grid)."""
    from unet_implementations_b200 import _lib
    sms = 148  # without a device the library sizes for 148 SMs
    for n, hw, cout, bn, mt in [(32, 128, 128, 128, 2), (32, 64, 256, 256, 1), (32, 32, 512, 256, 1), (32, 256, 64, 64, 4),
                                (4, 128, 128, 128, 2), (1, 64, 256, 256, 1)]:
        per_img_pairs = -(-hw // 8) * -(-hw // (16 * mt)) // 2 * (cout // bn)
        total = per_img_pairs * n
        tiles_per_cluster = max(1, -(-total // (sms // 2)))
        need = 8 * (-(-per_img_pairs // tiles_per_cluster) + 1)
        assert _lib.call("b200unet_conv_fprop_partials", n, hw, hw, cout) >= need, (n, hw, cout)


def test_product_path_fails_loudly_without_a_device():
    # a child process with every GPU hidden, so that a GPU host checks the CPU-only case too
    code = (
        "import pytest, torch\n"
        "assert not torch.cuda.is_available()\n"
        "from unet_implementations_b200.models.losses import SimpleLoss\n"
        "from unet_implementations_b200.models.unet import UNet\n"
        "m = UNet(n_stages=2, features_per_stage=[32, 32], encoder_dropout_rates=[0, 0], decoder_dropout_rates=[0])\n"
        "with pytest.raises(RuntimeError, match='no CPU path'):\n"
        "    m(torch.zeros(1, 3, 16, 16))\n"
        "with pytest.raises(RuntimeError, match='no CPU path'):\n"
        "    SimpleLoss()(torch.zeros(1, 3, 8, 8), torch.zeros(1, 8, 8, dtype=torch.long))\n"
        "print('ok')\n"
    )
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout[-2000:] + r.stderr[-4000:]


def test_missing_library_is_an_error(monkeypatch, tmp_path):
    from unet_implementations_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(RuntimeError, match="not built"):
        _lib.load()
