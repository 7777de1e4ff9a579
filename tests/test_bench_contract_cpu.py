"""bench.py's bookkeeping, checked without a GPU: the per-image work figures behind `roofline` are re-counted from the oracle's
own convolution calls (BASELINE.md §3: conv MACs x 2, fwd + dgrad + wgrad, no dgrad for the convolution that reads the image), and
both arms of the bench describe the same workload."""
import argparse
import importlib.util
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import models as om
from oracle import weights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("seg_bench_module", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _count_conv_flops(fn):
    """Run fn() with F.conv2d intercepted; returns (forward flop, flop of the convs that read a tensor needing no gradient)."""
    real = F.conv2d
    tot = {"fwd": 0.0, "no_dgrad": 0.0}

    def counted(x, w, b=None, stride=1, padding=0, dilation=1, groups=1):
        y = real(x, w, b, stride, padding, dilation, groups)
        K, Cg, R, S = w.shape
        fl = 2.0 * y.shape[0] * y.shape[2] * y.shape[3] * K * Cg * R * S
        tot["fwd"] += fl
        if x.shape[1] == 3:  # the image: no input gradient
            tot["no_dgrad"] += fl
        return y
    F.conv2d = counted
    try:
        with torch.no_grad():
            fn()
    finally:
        F.conv2d = real
    return tot["fwd"], tot["no_dgrad"]


@pytest.mark.parametrize("tag", ["C3", "C2", "C4", "C5"])
def test_train_gflop_per_image_matches_a_recount(tag):
    b = _bench()
    cfg = b.CONFIGS[tag]
    x = torch.randn(2, 3, cfg["size"], cfg["size"])  # batch 2: train-mode BatchNorm of the 1x1 pooled maps needs > 1 value
    if cfg["arch"] == "DeepLab" and cfg["kw"]["backbone"] == "xception":
        sd = weights.deeplab_xception_state_dict(cfg["nc"], seed=0)
        run = lambda: om.deeplab_forward(sd, x, backbone="xception", train=True)  # noqa: E731
    elif cfg["arch"] == "DeepLab":
        sd = weights.deeplab_resnet_state_dict(cfg["nc"], cfg["kw"]["backbone"], seed=0)
        run = lambda: om.deeplab_forward(sd, x, backbone=cfg["kw"]["backbone"], train=True)  # noqa: E731
    elif cfg["arch"] == "PSPNet":
        sd = weights.pspnet_state_dict(cfg["nc"], cfg["kw"]["backbone"], seed=0)
        run = lambda: om.pspnet_forward(sd, x, backbone=cfg["kw"]["backbone"], train=True, use_aux=True)  # noqa: E731
    else:
        sd = weights.upernet_state_dict(cfg["nc"], cfg["kw"]["backbone"], seed=0)
        run = lambda: om.upernet_forward(sd, x, backbone=cfg["kw"]["backbone"], train=True)  # noqa: E731
    sd = {k: v.to("meta") for k, v in sd.items()}  # shapes only: the count needs no arithmetic
    x = x.to("meta")
    fwd, no_dgrad = _count_conv_flops(run)
    train = (3.0 * fwd - no_dgrad) / 2 / 1e9
    assert abs(train - cfg["gflop"]) < 2e-3 * cfg["gflop"], f"{tag}: recount {train:.2f} GFLOP/img vs bench.py's {cfg['gflop']}"


def test_both_arms_describe_the_same_workload():
    b = _bench()
    for tag in b.CONFIGS:
        b.CFG = b.CONFIGS[tag]
        args = argparse.Namespace(batch=b.CFG["batch"], gpus=1)
        mine = b.config_dict(args, 1, use_graph=True, last_loss=1.0)
        ref = b.config_dict(args, 1)
        for k in ("workload", "per_gpu_batch", "global_batch", "parallelism"):
            assert mine[k] == ref[k]
        assert tag in mine["workload"] and b.CFG["name"] in b.metric_name()
    b.CFG = b.CONFIGS["C3"]
    assert b.metric_name() == "images/sec DeepLabV3+/ResNet101 513x513 train step (fwd+CE+bwd+SGD)"  # BASELINE.json's metric


def test_dump_outputs_files(tmp_path):
    import numpy as np
    b = _bench()
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Conv2d(3, 4, 3), torch.nn.BatchNorm2d(4), torch.nn.Conv2d(4, 2, 1))
    model[2].bias.requires_grad_(False)
    b.dump_outputs(str(tmp_path / "d"), torch.tensor(2.5), model)
    got = {f: np.load(tmp_path / "d" / f) for f in sorted(os.listdir(tmp_path / "d"))}
    assert sorted(got) == ["buffers.npy", "loss.npy", "params.npy"]
    assert got["loss.npy"].dtype == np.float64 and got["loss.npy"].tolist() == [2.5]
    params = torch.cat([p.detach().reshape(-1) for p in model.parameters() if p.requires_grad])
    assert got["params.npy"].dtype == np.float32 and np.array_equal(got["params.npy"], params.numpy())
    assert np.array_equal(got["buffers.npy"], torch.cat([model[1].running_mean, model[1].running_var]).numpy())
    big = torch.arange(1000, dtype=torch.float32)
    s = b._dump_sample(big, 100, seed=1)
    assert s.shape == (100,) and torch.equal(s, b._dump_sample(big, 100, seed=1)) and bool((s[1:] > s[:-1]).all())  # distinct
    assert (b.DUMP_PARAMS + b.DUMP_BUFFERS) * 4 + 8 <= 64e6


def test_bench_input_recipe_is_the_oracles():
    from oracle import synth
    b = _bench()
    for tag in ("C3", "C5"):
        b.CFG = b.CONFIGS[tag]
        cfg = b.CFG
        x, y = b.synthetic_batch(2, 1234)
        xr, yr = synth.make_batch(2, cfg["size"], cfg["size"], cfg["nc"], cfg["ignore"], seed=1234)
        assert torch.equal(x, xr) and torch.equal(y, yr)
    b.CFG = b.CONFIGS["C3"]
