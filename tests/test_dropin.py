"""CPU: the drop-in shim (dropin/sitecustomize.py) makes the reference's trainer import this implementation
(SURVEY.md 8b "import paths").  The reference tree is not part of this repository, so the test writes a stand-in of
the layout the shim serves: `src/train.py` with the trainer's model / loss imports (train.py:28-29) and its
`create_optimizer` (SGD, Nesterov, train.py:431-451), and the reference's own `models/` and `utils/` packages.  The
stand-in `models.unet` / `models.losses` cannot be imported, so the shim must take precedence over the tree."""
import os
import subprocess
import sys

from conftest import ROOT

_SHADOWED = "raise ImportError('the reference model module was imported: the drop-in shim did not take precedence')\n"
REFERENCE_LAYOUT = {
    "models/__init__.py": "",
    "models/unet.py": _SHADOWED,
    "models/losses.py": _SHADOWED,
    "utils/__init__.py": "",
    "utils/metrics.py": "def dice_per_class(*args, **kwargs):\n    raise NotImplementedError\n",
    "src/__init__.py": "",
    "src/train.py": (
        "import torch.optim as optim\n"
        "\n"
        "from models.losses import SimpleLoss\n"
        "from models.unet import UNet\n"
        "\n"
        "\n"
        "def create_optimizer(model, lr, weight_decay, momentum):\n"
        "    return optim.SGD(model.parameters(), lr=lr, momentum=momentum, weight_decay=weight_decay, nesterov=True)\n"
    ),
}


def test_reference_trainer_imports_the_b200_model_through_the_shim(tmp_path):
    ref = tmp_path / "Our_UNet"
    for rel, text in REFERENCE_LAYOUT.items():
        (ref / rel).parent.mkdir(parents=True, exist_ok=True)
        (ref / rel).write_text(text)
    code = (
        "import models.unet as mu, models.losses as ml\n"
        "assert mu.UNet.__module__ == 'unet_implementations_b200.models.unet', mu.UNet.__module__\n"
        "assert ml.SimpleLoss.__module__ == 'unet_implementations_b200.models.losses'\n"
        "import src.train as T\n"                       # the trainer (train.py:28-29)
        "assert T.UNet is mu.UNet and T.SimpleLoss is ml.SimpleLoss\n"
        "assert T.create_optimizer.__module__ == 'src.train'\n"
        "import src.models.unet as smu\n"               # evaluate.py:32
        "assert smu.UNet is mu.UNet\n"
        "import src.utils.metrics as sm, utils.metrics as um\n"   # evaluate.py:33-41
        "assert sm is um\n"
        "m = T.UNet()\n"
        "opt = T.create_optimizer(m, 0.01, 1e-4, 0.99)\n"
        "assert len(opt.param_groups[0]['params']) == len(m.state_dict()) == 90\n"
        "print('ok')\n"
    )
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "dropin"), ROOT, str(ref)])
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=str(tmp_path),
                       timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout[-2000:] + r.stderr[-4000:]
