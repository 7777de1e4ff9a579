"""The drop-in overlay: with `seg_b200.launch` ordering sys.path as [overlay, reference root], the
reference's own registries resolve DeepLab / PSPNet / CrossEntropyLoss2d to the B200-native classes and everything else
to the reference's.  The reference tree is stood in for by a tree with its layout, package files and public names, built
from tests/golden/overlay_registries.json (recorded from the reference by oracle/make_golden_overlay.py, with a snapshot of
where each name resolved there)."""
import json
import os
import subprocess
import sys

import pytest

from oracle.make_golden_overlay import resolve

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "overlay_registries.json")
OVERLAID = ("models", "utils.losses", "utils.metrics", "utils.sync_batchnorm")  # modules the overlay replaces
MODULE_FILE = {"utils.losses": "utils/losses.py", "utils.metrics": "utils/metrics.py", "utils.lr_scheduler": "utils/lr_scheduler.py",
               "utils.helpers": "utils/helpers.py", "utils.lovasz_losses": "utils/lovasz_losses.py",
               "utils.sync_batchnorm": "utils/sync_batchnorm/__init__.py", "base": "base/__init__.py"}
# stand-ins whose behaviour the walk-through below relies on; every other name is an inert stub
SPECIAL = {
    ("base/base_model.py", "BaseModel"): "class BaseModel(nn.Module):\n    def __init__(self):\n        super().__init__()\n"
                                         "        self.logger = logging.getLogger(self.__class__.__name__)\n",
    ("utils/sync_batchnorm/batchnorm.py", "SynchronizedBatchNorm2d"): "class SynchronizedBatchNorm2d(nn.BatchNorm2d):\n    pass\n",
    ("utils/sync_batchnorm/replicate.py", "DataParallelWithCallback"): "class DataParallelWithCallback(nn.DataParallel):\n    pass\n",
    ("utils/sync_batchnorm/__init__.py", "convert_model"):
        "def convert_model(module):\n    for name, m in module.named_children():\n        if isinstance(m, nn.BatchNorm2d):\n"
        "            setattr(module, name, SynchronizedBatchNorm2d(m.num_features))\n    return module\n",
}


def _stub(name):
    if name[0].isupper():
        return f"class {name}:\n    def __init__(self, *args, **kwargs):\n        pass\n"
    return f"def {name}(*args, **kwargs):\n    return None\n"


def build_stand_in(root, golden):
    """Files at the reference's paths defining the reference's names, importing across files the way the reference does."""
    resolved = golden["resolved"]
    imports, defs = {}, {}
    for mod, names in resolved.items():
        own = MODULE_FILE.get(mod)
        for name, where in names.items():
            if where == "engine":
                if own and mod in OVERLAID:  # the reference defines it too; the overlay must win
                    defs.setdefault(own, {})[name] = None
                elif own:
                    src = next(m for m in OVERLAID if resolved.get(m, {}).get(name) == "engine")
                    imports.setdefault(own, []).append(f"from {src} import {name}")
                continue
            defs.setdefault(where, {})[name] = None
            if own and where != own:
                dotted = where[:-3].replace("/", ".")
                parent = dotted.rsplit(".", 1)[0]
                if own.endswith("__init__.py") and os.path.dirname(where) == os.path.dirname(own):
                    line = f"from .{os.path.basename(where)[:-3]} import {name}"
                else:
                    line = f"from {parent if parent in OVERLAID else dotted} import {name}"
                imports.setdefault(own, []).append(line)
    # the reference's own models/ and utils/ are regular packages (their __init__.py import the registries); the overlay's
    # must shadow them, which only the sys.path order of launch.setup_paths decides
    for init, entries in golden["packages"].items():
        for mod, names in entries:
            imports.setdefault(init, []).append(f"from {mod} import {', '.join(names)}")
            target = os.path.join(os.path.dirname(init), mod.lstrip(".").replace(".", "/") + ".py")
            for n in names:
                defs.setdefault(target, {}).setdefault(n, None)
    for path in set(imports) | set(defs):
        body = ["import logging", "import torch.nn as nn"] + imports.get(path, []) + [""]
        body += [SPECIAL.get((path, n)) or _stub(n) for n in defs.get(path, {})]
        os.makedirs(os.path.join(root, os.path.dirname(path)), exist_ok=True)
        with open(os.path.join(root, path), "w") as f:
            f.write("\n".join(body))
    with open(os.path.join(root, "config.json"), "w") as f:
        json.dump(golden["config"], f)


CODE = r"""
import sys
from seg_b200 import launch
launch.setup_paths(sys.argv[1])
import models, seg_b200
from utils import losses, lr_scheduler, helpers, metrics
assert metrics.eval_metrics is seg_b200.eval_metrics and metrics.AverageMeter is seg_b200.AverageMeter
assert hasattr(metrics, 'batch_pix_accuracy') and losses.LovaszSoftmax is seg_b200.LovaszSoftmax
assert models.DeepLab is seg_b200.DeepLab and models.PSPNet is seg_b200.PSPNet, (models.DeepLab, models.PSPNet)
assert models.UNet.__module__.endswith('unet') and 'reference' in models.UNet.__init__.__code__.co_filename
assert losses.CrossEntropyLoss2d is seg_b200.CrossEntropyLoss2d
assert hasattr(losses, 'DiceLoss') and hasattr(losses, 'LovaszSoftmax') and hasattr(lr_scheduler, 'Poly')
from base import BaseModel
m = models.DeepLab(19, backbone='resnet50', pretrained=False, freeze_bn=False, freeze_backbone=False, output_stride=16)
assert isinstance(m, BaseModel)
# exactly what train.py:14-16,26,30 and base_trainer.py:46-57 do
import json
cfg = json.load(open(sys.argv[1] + '/config.json'))
cfg['arch']['args']['pretrained'] = False
cfg['arch']['type'], cfg['arch']['args']['backbone'] = 'PSPNet', 'resnet50'
model = getattr(models, cfg['arch']['type'])(21, **cfg['arch']['args'])
loss = getattr(losses, cfg['loss'])(ignore_index=cfg['ignore_index'])
groups = [{'params': model.get_decoder_params()}, {'params': model.get_backbone_params(), 'lr': 0.001}]
import torch
opt = torch.optim.SGD(groups, lr=0.01, momentum=0.9, weight_decay=1e-4)
assert sum(len(g['params']) for g in opt.param_groups) == len(list(model.parameters()))
# base/base_trainer.py:11-12,33-35: config['use_synch_bn'] -> convert_model + DataParallelWithCallback from utils.sync_batchnorm
from utils.sync_batchnorm import convert_model, DataParallelWithCallback, SynchronizedBatchNorm2d
assert model.use_sync_bn is False and convert_model(model) is model and model.use_sync_bn is True   # engine model: marked, BN holders kept
assert all(not isinstance(mm, SynchronizedBatchNorm2d) for mm in model.modules())
import torch.nn as nn
plain = convert_model(nn.Sequential(nn.Conv2d(3, 4, 1), nn.BatchNorm2d(4)))                         # anything else: the reference's conversion
assert isinstance(plain[1], SynchronizedBatchNorm2d)
assert issubclass(DataParallelWithCallback, nn.DataParallel)
print(str(model).splitlines()[-1])
print('OVERLAY_OK')
"""


def test_overlay_resolves_registries(tmp_path):
    with open(GOLD) as f:
        golden = json.load(f)
    ref = str(tmp_path / "reference")
    build_stand_in(ref, golden)
    env = dict(os.environ)
    env.pop("SEG_REFERENCE_ROOT", None)
    env["PYTHONPATH"] = os.path.join(ROOT, "pytorch-segmentation_b200")
    r = subprocess.run([sys.executable, "-W", "ignore", "-c", CODE, ref], env=env, cwd=ref, capture_output=True, text=True, timeout=600)
    assert "OVERLAY_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
    assert "Nbr of trainable parameters: 51446762" in r.stdout
    assert resolve(ref) == golden["resolved"]


def test_constructor_defaults_match_the_reference():
    """A config that omits `backbone` must build the architecture the reference would (models/deeplabv3_plus.py:337,
    models/pspnet.py:42, models/upernet.py:121); `pretrained` cannot be honoured offline: the default only warns."""
    import inspect
    import logging
    import seg_b200
    want = {"DeepLab": "xception", "PSPNet": "resnet152", "UperNet": "resnet101"}
    for name, backbone in want.items():
        sig = inspect.signature(getattr(seg_b200, name).__init__)
        assert sig.parameters["backbone"].default == backbone, name
        assert sig.parameters["pretrained"].default is None, name
        assert list(sig.parameters)[1:3] == ["num_classes", "in_channels"], name
    records = []
    h = logging.Handler()
    h.emit = records.append
    logging.getLogger("DeepLab").addHandler(h)
    try:
        seg_b200.DeepLab(5, backbone="resnet50")                    # default pretrained -> warning, random init
        n = len(records)
        seg_b200.DeepLab(5, backbone="resnet50", pretrained=False)  # explicit False -> silent
    finally:
        logging.getLogger("DeepLab").removeHandler(h)
    assert n >= 1 and len(records) == n and "ImageNet" in records[0].getMessage()
    with pytest.raises(RuntimeError, match="network"):
        seg_b200.DeepLab(5, backbone="resnet50", pretrained=True)
