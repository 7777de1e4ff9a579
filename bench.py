#!/usr/bin/env python
"""bench.py — images/sec of one TRAINING step (forward + per-pixel CE + backward [+ SyncBN exchange + gradient
all-reduce] + SGD update) of DeepLabV3+/ResNet-101, 513x513, 19 classes (BASELINE.json metric, SURVEY.md §8d config C3)
on N B200s of one node, synthetic data, random-init weights.

    python bench.py --gpus 1 --steps 10 --warmup 3                     # this engine (hand-written sm_100a kernels)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference --gpus 1 --steps 2 --warmup 1     # reference algorithm on the host CPU cores
    python bench.py --gpus 1 --steps 10 --warmup 3 --dump-outputs DIR  # + the last timed step's results as DIR/*.npy

One JSON line on stdout (rank 0).  `value` = device-resident throughput through the fused train step; `e2e` = the same
step driven through the reference-facing plugin surface (model(x) -> CrossEntropyLoss2d -> backward -> torch.optim.SGD,
i.e. what train.py/trainer.py:55-71 call) with the batch copied from pinned host memory every step and the loss read
back; `roofline` = algorithmic conv FLOPs / CUDA-event time of the tcgen05 implicit-GEMM launches inside the timed
region, against the measured dense-bf16 peak; `cpu_baseline` = the CPU oracle port timed on this box's host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "pytorch-segmentation_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

# BASELINE.json configs (SURVEY.md §8d).  train GFLOP/img = conv fwd + dgrad + wgrad, measured on the reference with hooks
# (BASELINE.md §3).  C3 is the headline (the metric string below is BASELINE.json's); the others are reported the same way.
CONFIGS = {
    "C3": dict(name="DeepLabV3+/ResNet101 513x513", arch="DeepLab", kw=dict(backbone="resnet101", output_stride=16), nc=19, size=513, batch=16,
               loss="CE", ignore=255, gflop=555.63, sync_bn=True, recipe="CE, SGD m0.9 wd1e-4, lr .01/.001"),
    "C2": dict(name="PSPNet/ResNet50 473x473", arch="PSPNet", kw=dict(backbone="resnet50"), nc=21, size=473, batch=16,
               loss="CE", ignore=255, gflop=1071.78, sync_bn=False, recipe="CE + 0.4 CE(aux), SGD m0.9 wd1e-4, lr .01/.001"),
    "C4": dict(name="DeepLabV3+/Xception 769x769", arch="DeepLab", kw=dict(backbone="xception", output_stride=16), nc=19, size=769, batch=8,
               loss="CE", ignore=255, gflop=1150.90, sync_bn=False, recipe="CE, SGD m0.9 wd1e-4, lr .01/.001"),
    "C5": dict(name="UperNet/ResNet101 512x512", arch="UperNet", kw=dict(backbone="resnet101"), nc=150, size=512, batch=8,
               loss="LovaszSoftmax", ignore=-1, gflop=1123.96, sync_bn=False, recipe="Lovasz-softmax (ignore -1), SGD m0.9 wd1e-4, lr .01/.001"),
}
CFG = CONFIGS["C3"]  # replaced in main() by --config


def metric_name():
    if CFG is CONFIGS["C3"]:
        return "images/sec DeepLabV3+/ResNet101 513x513 train step (fwd+CE+bwd+SGD)"
    return f"images/sec {CFG['name']} train step (fwd+{CFG['loss']}+bwd+SGD)"


def workload(backbone=None, world=1, sync_bn=False):
    tag = [k for k, v in CONFIGS.items() if v is CFG][0]
    return f"{CFG['name']} {CFG['nc']}cls train step ({tag}: {CFG['recipe']}" + (", SyncBN" if (world > 1 and sync_bn) else "") + ")"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.lines, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def synthetic_batch(B, seed):
    """Synthetic inputs of SURVEY.md §8(d): randn images; 16x16-block-constant labels with a 4-pixel ignore border.  Stated here
    (not imported from oracle/, which only the CPU legs may touch); tests/test_bench_contract_cpu.py pins it to the oracle's."""
    H = W = CFG["size"]
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, 3, H, W, generator=g)
    blocks = torch.randint(0, CFG["nc"], (B, (H + 15) // 16, (W + 15) // 16), generator=g)
    y = blocks.repeat_interleave(16, 1).repeat_interleave(16, 2)[:, :H, :W].contiguous()
    for sl in ((slice(None), slice(0, 4)), (slice(None), slice(-4, None)), (slice(None), slice(None), slice(0, 4)), (slice(None), slice(None), slice(-4, None))):
        y[sl] = CFG["ignore"]
    return x, y


# elements kept of the dumped parameters (48 MiB of float32) and buffers (8 MiB): with the loss, under 64 MB in all
DUMP_PARAMS, DUMP_BUFFERS = 12 << 20, 2 << 20


def _dump_sample(flat, n, seed):
    """`flat` whole if it has at most n elements, else n distinct elements at sorted positions drawn from a fixed seed (the
    same positions in every run of the same config, so two builds are compared element for element)."""
    if flat.numel() <= n:
        return flat
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(seed))[:n].sort().values
    return flat[idx.to(flat.device)]


def dump_outputs(out_dir, loss, model):
    """What a caller of the timed step holds after its last step: the loss (loss.npy, float64), the updated trainable
    parameters (params.npy) and the updated floating-point buffers such as BatchNorm running statistics (buffers.npy), each
    flattened in module order and sampled by _dump_sample, float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    with torch.no_grad():
        params = torch.cat([p.detach().reshape(-1).float() for p in model.parameters() if p.requires_grad])
        bufs = torch.cat([b.detach().reshape(-1).float() for b in model.buffers() if b.is_floating_point()])
        arrays = {"loss": np.array([float(loss)], dtype=np.float64),
                  "params": _dump_sample(params, DUMP_PARAMS, seed=1).cpu().numpy(),
                  "buffers": _dump_sample(bufs, DUMP_BUFFERS, seed=2).cpu().numpy()}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return arrays


def host_threads():
    """Threads for the CPU arm: all cores up to 32 — ATen/oneDNN at batch 2 gets SLOWER beyond that on the 128-core
    GPU hosts (measured: 0.09 img/s at 128 threads vs ~0.5 at 8-32); override with SEG_CPU_THREADS."""
    env = os.environ.get("SEG_CPU_THREADS")
    if env:
        return int(env)
    return min(os.cpu_count() or 1, 32)


def _oracle_model(device):
    """(state_dict with requires_grad, forward fn, backbone-parameter predicate) of the oracle port of CFG's network."""
    from oracle import models as om
    from oracle import weights
    a, kw, nc = CFG["arch"], CFG["kw"], CFG["nc"]
    if a == "DeepLab" and kw["backbone"] == "xception":
        sd0 = weights.deeplab_xception_state_dict(nc, seed=0)
        fwd = lambda sd, x: (om.deeplab_forward(sd, x, backbone="xception", train=True, dropout=True),)
    elif a == "DeepLab":
        sd0 = weights.deeplab_resnet_state_dict(nc, kw["backbone"], seed=0)
        fwd = lambda sd, x: (om.deeplab_forward(sd, x, backbone=kw["backbone"], train=True, dropout=True),)
    elif a == "PSPNet":
        sd0 = weights.pspnet_state_dict(nc, kw["backbone"], seed=0)
        fwd = lambda sd, x: om.pspnet_forward(sd, x, backbone=kw["backbone"], train=True, dropout=True)
    else:
        sd0 = weights.upernet_state_dict(nc, kw["backbone"], seed=0)
        fwd = lambda sd, x: (om.upernet_forward(sd, x, backbone=kw["backbone"], train=True, dropout=True),)
    sd = om.clone_sd({k: v.to(device) for k, v in sd0.items()}, requires_grad=True)
    names = om.param_names(sd)
    is_bb = (lambda n: n.startswith("backbone.")) if a != "PSPNet" else (lambda n: n.startswith("initial.") or n.startswith("layer"))
    seen, bb, dec = set(), [], []
    for n in names:  # aliased tensors (UperNet's shared smooth conv) once
        if id(sd[n]) in seen:
            continue
        seen.add(id(sd[n]))
        (bb if is_bb(n) else dec).append(sd[n])
    return sd, fwd, bb, dec


def _oracle_loss(outs, y):
    from oracle import losses as ol
    if CFG["loss"] == "LovaszSoftmax":
        return ol.lovasz_softmax(outs[0], y, CFG["ignore"])
    loss = ol.cross_entropy2d(outs[0], y, CFG["ignore"])
    if len(outs) > 1:
        loss = loss + 0.4 * ol.cross_entropy2d(outs[1], y, CFG["ignore"])
    return loss


def cpu_port_step_time(batch, steps, warmup, threads):
    """Reference algorithm on the host cores: oracle model + loss + autograd backward + torch.optim.SGD (fp32)."""
    torch.set_num_threads(threads)
    sd, fwd, bb, dec = _oracle_model("cpu")
    opt = torch.optim.SGD([{"params": dec}, {"params": bb, "lr": 0.001}], lr=0.01, momentum=0.9, weight_decay=1e-4)
    x, y = synthetic_batch(batch, 1234)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad()
        loss = _oracle_loss(fwd(sd, x), y)
        loss.backward()
        opt.step()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return sum(times) / len(times)


def _import_reference_tree():
    """The UNMODIFIED reference tree, packed by baseline/install_ref.sh into baseline/_ref/reference.zip (git-ignored; built in
    the build container where /root/reference exists, shipped to the GPU box like a built .so).  Returns its `models` package or
    None.  Shims: SURVEY.md §8c (skimage stub; UperNet's undefined module globals)."""
    z = os.path.join(ROOT, "baseline", "_ref", "reference.zip")
    if not os.path.exists(z):
        return None
    import types
    import warnings
    warnings.filterwarnings("ignore")
    for n in ("skimage", "skimage.filters"):
        sys.modules.setdefault(n, types.ModuleType(n))
    if not hasattr(sys.modules["skimage.filters"], "gaussian"):
        sys.modules["skimage.filters"].gaussian = None
    for name in list(sys.modules):  # this process may hold the overlay's / nothing's `models`, `utils`, `base`
        if name.split(".")[0] in ("models", "utils", "base"):
            del sys.modules[name]
    sys.path.insert(0, z)
    import models as ref_models
    from utils import helpers
    import models.upernet as up
    up.freeze_backbone, up.set_trainable = False, helpers.set_trainable
    return ref_models


def reference_gpu_step_time(batch, steps, warmup, n_gpus, budget_s=None):
    """BASELINE.md §4 "Reference GPU path (cuDNN)" — the denominator of north_star's ">= 6x": the UNMODIFIED reference model,
    wrapped exactly as BaseTrainer does it (base/base_trainer.py:33-38: convert_model + DataParallelWithCallback when
    use_synch_bn, else nn.DataParallel; device_ids = range(n_gpu)), fp32 NCHW, cudnn.benchmark = True (trainer.py:35), the
    reference's own loss class and torch.optim.SGD with the differential learning rates of base_trainer.py:46-57, the same
    per-GPU batch, ONE process over n_gpus devices.  Falls back to the oracle port (single GPU) if the tree is not shipped.
    `budget_s` bounds the leg by wall clock (the reference's threaded DataParallel + SyncBN step takes seconds at N > 1): after 3
    warm-up steps one step is timed and the number of timed steps is cut to fit.  Returns (s/step, how, timed steps, warm-up)."""
    torch.backends.cudnn.benchmark = True
    dev = torch.device("cuda", 0)
    x, y = synthetic_batch(batch * n_gpus, 1234)
    ref_models = _import_reference_tree()
    how = None
    if ref_models is not None:
        from utils import losses as ref_losses
        from utils.sync_batchnorm import DataParallelWithCallback, convert_model
        torch.manual_seed(0)
        kw = dict(CFG["kw"])
        model = getattr(ref_models, CFG["arch"])(CFG["nc"], pretrained=False, **kw)
        ids = list(range(n_gpus))
        if CFG["sync_bn"]:
            model = DataParallelWithCallback(convert_model(model), device_ids=ids)
        else:
            model = torch.nn.DataParallel(model, device_ids=ids)
        model.to(dev).train()
        crit = getattr(ref_losses, CFG["loss"] if CFG["loss"] != "CE" else "CrossEntropyLoss2d")(ignore_index=CFG["ignore"])
        opt = torch.optim.SGD([{"params": [p for p in model.module.get_decoder_params() if p.requires_grad]},
                               {"params": [p for p in model.module.get_backbone_params() if p.requires_grad], "lr": 0.001}],
                              lr=0.01, momentum=0.9, weight_decay=1e-4)

        def step(xd, yd):
            opt.zero_grad()
            out = model(xd)
            if isinstance(out, tuple):  # trainer.py:57-62: PSP* returns (out, aux)
                loss = crit(out[0], yd) + 0.4 * crit(out[1], yd)
            else:
                loss = crit(out, yd)
            if isinstance(model, torch.nn.DataParallel):
                loss = loss.mean()
            loss.backward()
            opt.step()
        how = (f"UNMODIFIED reference tree (baseline/_ref/reference.zip): models.{CFG['arch']} wrapped as base/base_trainer.py:33-38 "
               f"({'convert_model + DataParallelWithCallback' if CFG['sync_bn'] else 'nn.DataParallel'}, device_ids=range({n_gpus})), fp32 NCHW, "
               f"cudnn.benchmark, utils.losses.{'CrossEntropyLoss2d' if CFG['loss'] == 'CE' else CFG['loss']}, torch.optim.SGD; one process")
    else:
        if n_gpus > 1:
            raise RuntimeError("reference tree not shipped (run baseline/install_ref.sh in the build container)")
        sd, fwd, bb, dec = _oracle_model(dev)
        opt = torch.optim.SGD([{"params": dec}, {"params": bb, "lr": 0.001}], lr=0.01, momentum=0.9, weight_decay=1e-4)

        def step(xd, yd):
            opt.zero_grad()
            _oracle_loss(fwd(sd, xd), yd).backward()
            opt.step()
        how = "oracle port (same ATen/cuDNN calls as the reference; the reference tree was not shipped), fp32 NCHW, cudnn.benchmark"
    xd, yd = x.to(dev), y.to(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if budget_s is not None:
        warmup = min(warmup, 3)
        t0 = time.time()
        for _ in range(warmup):
            step(xd, yd)
            for d in range(n_gpus):
                torch.cuda.synchronize(d)
            if time.time() - t0 > 0.5 * budget_s:  # autotuning 8 threaded replicas can already eat the budget
                break
        t1 = time.time()
        step(xd, yd)
        for d in range(n_gpus):
            torch.cuda.synchronize(d)
        one = max(time.time() - t1, 1e-4)
        left = budget_s - (time.time() - t0)
        steps = int(max(2, min(steps, left / one)))
        warmup = 0  # already done (warmup + 1 steps)
    for i in range(warmup + steps):
        if i == warmup:
            for d in range(n_gpus):
                torch.cuda.synchronize(d)
            e0.record()
        step(xd, yd)
    e1.record()
    for d in range(n_gpus):
        torch.cuda.synchronize(d)
    return e0.elapsed_time(e1) * 1e-3 / steps, how, steps, warmup


def config_dict(args, world, use_graph=None, last_loss=None):
    """`config` of the JSON line — the SAME dict for this engine's arm and for `--impl reference` (the driver compares them)."""
    B = args.batch
    c = {"workload": workload(world=world, sync_bn=CFG["sync_bn"]), "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
         "l2": "per-step working set (activations ~GBs) far exceeds the 126 MB L2; no explicit flush needed",
         "dropout": "on (the reference's nn.Dropout / nn.Dropout2d sites)"}
    if use_graph is not None:
        c["cuda_graph"] = use_graph
    if last_loss is not None:
        c["last_loss"] = last_loss
    return c


def run_reference(args):
    """Reference arm: the reference's algorithm for this path on the host cores (CPU oracle port, pinned bit-exactly to the
    reference by tests/golden) on THIS arm's config; every timed step is a bounded sample of the configured step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    B = args.cpu_batch
    t = cpu_port_step_time(B, args.steps, args.warmup, threads)
    v = B / t
    sample = (f"{args.steps} timed steps (after {args.warmup} warm-up) of batch {B} — a bounded sample of the {args.batch}-image step of the same "
              f"workload; the CPU path's images/sec does not depend on the batch at these sizes (conv-bound) — fp32, {threads} threads")
    print(json.dumps({
        "impl": "reference", "metric": metric_name(), "value": v, "unit": "images/sec", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config_dict(args, max(args.gpus, 1)),
        "cpu_baseline": {"value": v, "unit": "images/sec", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    global CFG
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C3", choices=list(CONFIGS), help="BASELINE.json config (C3 = the headline)")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (0 = the config's: 16 for C2/C3, 8 for C4/C5)")
    ap.add_argument("--cpu-batch", type=int, default=4, help="per-step sample of the CPU legs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-gpu-ref", "--no-gpu-aten", dest="no_gpu_ref", action="store_true",
                    help="skip the reference-GPU leg (unmodified reference tree through ATen/cuDNN on the same GPUs)")
    ap.add_argument("--gpu-ref-steps", type=int, default=int(os.environ.get("SEG_GPU_REF_STEPS", "30")),
                    help="timed steps of the reference-GPU leg (BASELINE.md §4 asks 10 warm-up + 50; default 10 + 30 keeps the run short)")
    ap.add_argument("--graph", type=int, default=int(os.environ.get("SEG_CUDA_GRAPH", "1")), help="replay the fused step from a CUDA graph")
    ap.add_argument("--plugin-graph", type=int, default=int(os.environ.get("SEG_PLUGIN_GRAPH", "1")),
                    help="e2e leg: replay model(x)/backward from CUDA graphs (seg_b200 model.cuda_graphs())")
    ap.add_argument("--plugin-optim", default=os.environ.get("SEG_PLUGIN_OPTIM", "fused"), choices=["fused", "torch"],
                    help="e2e leg optimiser: seg_b200.optim.SGD (torch.optim.SGD subclass, one kernel per group) or stock torch.optim.SGD")
    ap.add_argument("--ref-only", action="store_true", help="run ONLY the reference-GPU leg (single process, nn.DataParallel over --ref-gpus devices) and print its JSON")
    ap.add_argument("--ref-gpus", type=int, default=1)
    ap.add_argument("--ref-sync-bn", type=int, default=-1, help="reference-GPU leg: 1 = convert_model + DataParallelWithCallback, 0 = nn.DataParallel, -1 = the config's")
    ap.add_argument("--bucket-mb", type=float, default=float(os.environ.get("SEG_BUCKET_MB", "0")),
                    help="N > 1: gradient all-reduce bucket size of the fused step in MB; 0 (default) = one all-reduce after the backward — "
                         "measured faster than 25 MB buckets overlapped on a side stream at N = 2 (28.6 vs 29.3 ms) and N = 8 (29.3 vs 30.1 ms): "
                         "the NCCL kernels take SMs from the backward they overlap (profiles/scale_r02.txt)")
    ap.add_argument("--trace", default=None, help="after the timed runs, trace 2 steps per C-ABI call and write a table here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last of them computed (loss, parameters, BN statistics) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.ref_only):
        ap.error("--dump-outputs writes this engine's outputs: not with --impl reference or --ref-only")
    CFG = CONFIGS[args.config]
    if args.batch <= 0:
        args.batch = CFG["batch"]
    if args.impl == "reference":
        return run_reference(args)
    if args.ref_only:
        if args.ref_sync_bn >= 0:
            CFG = dict(CFG, sync_bn=bool(args.ref_sync_bn))
        tg, how, _, _ = reference_gpu_step_time(args.batch, args.steps, args.warmup, args.ref_gpus)
        print(json.dumps({"impl": "reference-gpu", "metric": metric_name(), "value": args.batch * args.ref_gpus / tg, "unit": "images/sec",
                          "n_gpus": args.ref_gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": tg * 1e3, "per_gpu_batch": args.batch,
                          "sync_bn": CFG["sync_bn"], "how": how}))
        return

    import torch.distributed as dist
    import seg_b200
    from seg_b200 import comm, lib, ops
    from seg_b200.train import FusedTrainStep

    rank, world, local = comm.init_distributed()
    torch.cuda.set_device(local)
    lib.require_device()
    dev = torch.device("cuda", local)
    B, K, W = args.batch, args.steps, max(args.warmup, 0)
    NC, IGNORE = CFG["nc"], CFG["ignore"]

    torch.manual_seed(0)
    model = getattr(seg_b200, CFG["arch"])(NC, pretrained=False, **CFG["kw"]).to(dev).train()
    if world > 1 and CFG["sync_bn"]:
        model.use_sync_bn = True      # what the overlay's convert_model does for config["use_synch_bn"]
        model._attach_sync_bn()
    x_cpu, y_cpu = synthetic_batch(B, 1234 + rank)
    x_pin, y_pin = x_cpu.pin_memory(), y_cpu.pin_memory()
    x_dev, y_dev = x_pin.to(dev), y_pin.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    crit_cls = seg_b200.CrossEntropyLoss2d if CFG["loss"] == "CE" else getattr(seg_b200, CFG["loss"])
    from seg_b200.optim import SGD as FusedSGD

    def plugin_objects():
        """What train.py / BaseTrainer build: loss from the registry, SGD with differential learning rates."""
        crit = crit_cls(ignore_index=IGNORE)
        opt_cls = FusedSGD if args.plugin_optim == "fused" else torch.optim.SGD
        opt = opt_cls([{"params": list(model.get_decoder_params())}, {"params": list(model.get_backbone_params()), "lr": 0.001}],
                      lr=0.01, momentum=0.9, weight_decay=1e-4)
        return crit, opt

    def plugin_loss(crit, out, yd):
        if isinstance(out, tuple):  # trainer.py:57-62: PSP* returns (out, aux)
            return crit(out[0], yd) + 0.4 * crit(out[1], yd)
        return crit(out, yd)

    # ------------------------------------------------------------ device-resident step  -> `value`
    # CE configs: the fused train step (fused upsample+CE, multi-tensor SGD, the whole step one CUDA graph).  Lovasz (C5): the
    # plugin-surface step (model(x) -> LovaszSoftmax -> backward -> SGD) on device-resident inputs.
    use_graph = bool(args.graph)
    fused = CFG["loss"] == "CE"
    if fused:
        stepper = FusedTrainStep(model, ignore_index=IGNORE, lr=0.01, backbone_lr_scale=0.1, momentum=0.9, weight_decay=1e-4, world=world,
                                 cuda_graph=use_graph, bucket_mb=args.bucket_mb)
        dev_step = lambda: stepper.step(x_dev, y_dev)
        eager_step = lambda: stepper._step_impl(x_dev, y_dev)
    else:
        stepper = None
        crit_v, opt_v = plugin_objects()
        if use_graph:
            model.cuda_graphs(True, warmup=2)

        def dev_step():
            opt_v.zero_grad(set_to_none=True)
            l = plugin_loss(crit_v, model(x_dev), y_dev)
            l.backward()
            opt_v.step()
            return l
        eager_step = dev_step
    for _ in range(max(W, 4 if not fused else 0)):
        dev_step()
    barrier()
    # kernel launches of ONE step (counted on an eager step; a graph replay issues the same kernels)
    if not fused and use_graph:
        model.cuda_graphs(False)
    lib.reset_launch_count()
    eager_step()
    launches_per_step = lib.launch_count()
    if not fused and use_graph:
        model.cuda_graphs(True, warmup=0)
        for _ in range(2):
            dev_step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ops.PROFILE = None if use_graph else []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        loss = dev_step()
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    if args.dump_outputs and rank == 0:
        # here, right after the K timed steps: the profiling and e2e legs below train the same model further
        assert stepper is None or stepper.steps == W + 1 + K, (stepper.steps, W, K)  # warm-up, launch count, timed
        dump_outputs(args.dump_outputs, loss.item(), model)
    launches = launches_per_step * K
    prof, ops.PROFILE = ops.PROFILE, None
    if prof is None:  # graph replay: measure the conv launches on two extra eager steps (same kernels, same shapes)
        if not fused:
            model.cuda_graphs(False)
        ops.PROFILE = []
        for _ in range(2):
            eager_step()
        torch.cuda.synchronize()
        prof, ops.PROFILE = ops.PROFILE, None
        conv_steps = 2
    else:
        conv_steps = K
    clocks = sampler.stop() if rank == 0 else None
    last_loss = float(loss.item())
    value = world * B * K / (ms_total * 1e-3)

    # roofline of the dominant kernel family (tcgen05 implicit-GEMM conv: fprop + dgrad + wgrad launches)
    conv_ms = sum(a.elapsed_time(b) for _, _, a, b, _ in prof)
    conv_flops = sum(f for _, f, _, _, _ in prof)
    conv_bytes = sum(nb for _, _, _, _, nb in prof)
    by_kind = {}
    for kind, f, a, b, _ in prof:
        d = by_kind.setdefault(kind, [0.0, 0.0, 0])
        d[0] += f
        d[1] += a.elapsed_time(b)
        d[2] += 1
    peak_tf, peak_hbm, peak_src = measured_peaks()
    achieved = conv_flops / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
    traffic, traffic_src = None, None
    for tname in ("roofline_traffic_r02.json", "roofline_traffic_r01.json"):
        tpath = os.path.join(ROOT, "profiles", tname)
        if args.config == "C3" and os.path.exists(tpath):  # dram bytes per conv launch from the committed ncu launch list of this workload
            with open(tpath) as f:
                tj = json.load(f)
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), f"profiles/{tname} (ncu dram__bytes_read.sum + dram__bytes_write.sum, mean over %d conv launches)" % tj.get("launches", 0)
            break
    roofline = {
        "bound": "tensor", "kernel": "conv_gemm_tc<BN,KIND> / conv_gemm_tc2 (tcgen05 implicit GEMM; fprop+dgrad+wgrad launches)",
        "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf, "peak_source": peak_src,
        "traffic": traffic, "traffic_unit": "bytes/launch (DRAM)", "traffic_source": traffic_src,
        "algorithmic_bytes_per_launch": conv_bytes / max(len(prof), 1), "algorithmic_flops_per_launch": conv_flops / max(len(prof), 1),
        "launches": len(prof), "conv_share_of_step": (conv_ms / conv_steps) / (ms_total / K) if ms_total else None,
        "timed_on": "the timed steps" if not use_graph else "2 eager steps after the graph-replayed timed region (identical kernels)",
        "by_kind_tflops": {k: (v[0] / (v[1] * 1e-3) / 1e12 if v[1] > 0 else 0.0) for k, v in by_kind.items()},
        "whole_step_frac_of_peak": value / world * CFG["gflop"] / 1e3 / peak_tf,
    }

    # ------------------------------------------------------------ plugin surface with host buffers -> `e2e`
    # The repo's public API, nothing bench-local: model(x) -> loss -> backward -> optimizer.step().  At N > 1 the gradient
    # all-reduce, the global-mean loss and the SyncBN exchange all happen INSIDE those calls (seg_b200/nets.py, losses.py).
    e2e = None
    if not args.no_e2e:
        if fused:
            crit, opt = plugin_objects()
        else:
            crit, opt = crit_v, opt_v

        # the reference's DataPrefetcher (base/base_dataloader.py:49-85) copies the NEXT batch on a side stream while the
        # current step computes; same here: every step's batch still crosses PCIe once, inside the timed region
        copy_stream = torch.cuda.Stream()
        slots = [(torch.empty_like(x_dev), torch.empty_like(y_dev), torch.cuda.Event()) for _ in range(2)]
        state = {"i": 0}

        def prefetch(slot):
            xd, yd, ev = slots[slot]
            copy_stream.wait_stream(torch.cuda.current_stream())  # the slot's previous consumer has been enqueued
            with torch.cuda.stream(copy_stream):
                xd.copy_(x_pin, non_blocking=True)
                yd.copy_(y_pin, non_blocking=True)
                ev.record(copy_stream)

        prefetch(0)

        def plugin_step():
            cur = state["i"] & 1
            state["i"] += 1
            xd, yd, ev = slots[cur]
            torch.cuda.current_stream().wait_event(ev)
            prefetch(cur ^ 1)  # next step's batch, overlapped with this step's kernels
            opt.zero_grad(set_to_none=True)
            l = plugin_loss(crit, model(xd), yd)
            l.backward()
            opt.step()
            return l.item()  # device -> host read of the step's result (trainer.py:72)

        # graph replay of the plugin path: model(x) and loss.backward() replay captured forward / backward tapes (two
        # eager calls warm up, the third captures).  If the capture fails the leg is measured eagerly and says so.
        plugin_graph, plugin_graph_err = bool(args.plugin_graph), None
        if plugin_graph:
            model.cuda_graphs(True, warmup=2)
            try:
                for _ in range(4):
                    plugin_step()
            except Exception as e:  # noqa: BLE001 — reported in the JSON line, the eager leg below still measures e2e
                plugin_graph, plugin_graph_err = False, repr(e)[:300]
                model.cuda_graphs(False)
                torch.cuda.synchronize()
                state["i"] = 0
                prefetch(0)
        if not plugin_graph:
            model.cuda_graphs(False)
            for _ in range(min(W, 2)):
                plugin_step()
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        Ke = K
        t0.record()
        for _ in range(Ke):
            plugin_step()
        t1.record()
        barrier()
        ms_e2e = max_over_ranks(t0.elapsed_time(t1))
        e2e = {"value": world * B * Ke / (ms_e2e * 1e-3), "unit": "images/sec",
               "h2d_bytes_per_step": int(x_pin.numel() * 4 + y_pin.numel() * 8), "d2h_bytes_per_step": 4,
               "api": f"seg_b200.{CFG['arch']}.forward -> seg_b200.{crit_cls.__name__} -> backward -> " + ("seg_b200.optim.SGD" if args.plugin_optim == "fused" else "torch.optim.SGD") +
                      ".step (train.py plugin surface; at N > 1 gradient all-reduce, global-mean loss and SyncBN exchange happen inside these calls); batch prefetched on a side stream like the reference's DataPrefetcher",
               "optimizer": args.plugin_optim,
               "ms_per_step": ms_e2e / Ke, "cuda_graph": plugin_graph, "cuda_graph_error": plugin_graph_err}
        if world > 1:
            model.release_graphs()

    if args.trace and fused:  # every rank runs the traced steps (they contain the exchanges); rank 0 writes the table
        lib.TRACE = []
        for _ in range(2):
            stepper._step_impl(x_dev, y_dev)  # eager: every C-ABI call is timed with its own event pair
        torch.cuda.synchronize()
        tr, lib.TRACE = lib.TRACE, None
        agg = {}
        for name, meta, a, b in tr:
            key = (name, meta[:8] if meta else None)
            d = agg.setdefault(key, [0.0, 0, 0.0])
            d[0] += a.elapsed_time(b) / 2
            d[1] += 1
            d[2] += (meta[8] if meta else 0.0) / 2
        tot = sum(v[0] for v in agg.values())
        by_name = {}
        for (name, _), v in agg.items():
            by_name[name] = by_name.get(name, 0.0) + v[0]
        with open(args.trace if rank == 0 else os.devnull, "w") as f:
            f.write(f"# per-step totals over 2 traced steps (eager, every C-ABI call timed with its own CUDA-event pair), {world} rank(s); sum of call times {tot:.2f} ms\n")
            for name, ms in sorted(by_name.items(), key=lambda kv: -kv[1]):
                f.write(f"{name:28s} {ms:9.3f} ms  {100 * ms / tot:5.1f}%\n")
            f.write("\n# name (N,H,W,C,K,R,stride,dil | rows,C,flag) ms/step calls/2steps TFLOP/s (conv) or TB/s algorithmic (streaming)\n")
            for (name, meta), v in sorted(agg.items(), key=lambda kv: -kv[1][0])[:110]:
                tf = v[2] / (v[0] * 1e-3) / 1e12 if v[0] > 0 and v[2] > 0 else 0.0
                f.write(f"{name:22s} {str(meta):48s} {v[0]:8.3f} {v[1]:4d} {tf:8.1f}\n")

    # ------------------------------------------------------------ baselines: the reference's algorithm on this box
    if stepper is not None and world > 1:
        stepper.release_graph()  # a live graph holding NCCL kernels blocks the communicator's destruction
    del stepper
    model.release_graphs()
    del model
    torch.cuda.empty_cache()
    barrier()
    cpu_baseline = None
    if rank == 0:
        cpu_baseline = {}
        if world == 1 and not args.no_cpu_baseline:
            threads = host_threads()
            t = cpu_port_step_time(args.cpu_batch, 5, 1, threads)
            cpu_baseline = {"value": args.cpu_batch / t, "unit": "images/sec", "cores": threads, "kind": "port",
                            "sample": f"5 timed steps (after 1 warm-up) of batch {args.cpu_batch} of the same train step, fp32 oracle port, {threads} threads"}
        # at N > 1 the reference's one-process DataParallelWithCallback + threaded SyncBN step takes SECONDS (measured: 4.9 s at
        # N = 2, profiles/bench_r02_n2.json) — informational, so opt-in there (SEG_GPU_REF_MULTI=1) to keep scaling runs short
        if not args.no_gpu_ref and (world == 1 or os.environ.get("SEG_GPU_REF_MULTI", "0") == "1"):
            try:  # the reference's OWN GPU path on the same GPUs: the denominator of north_star's ">= 6x" (BASELINE.md §4)
                budget = float(os.environ.get("SEG_GPU_REF_BUDGET_S", "60")) if world > 1 else None
                tg, how, ref_steps, ref_warm = reference_gpu_step_time(B, args.gpu_ref_steps, 10, world, budget)
                cpu_baseline["reference_gpu_path"] = {"value": B * world / tg, "unit": "images/sec", "ms_per_step": tg * 1e3, "per_gpu_batch": B,
                                                      "n_gpus": world, "timed_steps": ref_steps, "warmup": ref_warm if budget is None else 4, "how": how,
                                                      "engine_over_reference_gpu": {"value": value / (B * world / tg), "e2e": (e2e["value"] / (B * world / tg)) if e2e else None}}
            except Exception as e:  # informational only
                cpu_baseline["reference_gpu_path"] = {"unavailable": repr(e)[:300]}
        if not cpu_baseline:
            cpu_baseline = None
    if world > 1:
        # the other ranks wait on the HOST (TCPStore key) while rank 0 drives nn.DataParallel over all the GPUs: an NCCL barrier
        # would park a spinning kernel on every GPU the reference is about to use
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            store.set("seg_bench_reference_leg_done", "1")
        else:
            store.wait(["seg_bench_reference_leg_done"])

    if rank == 0:
        print(json.dumps({
            "metric": metric_name(), "value": value, "unit": "images/sec", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": config_dict(args, world, use_graph, last_loss),
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline,
        }))
    sys.stdout.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
