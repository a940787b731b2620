#!/usr/bin/env python
"""Generate the golden fixtures by EXECUTING THE UNMODIFIED REFERENCE ($TURBOPRUNE_REFERENCE) on CPU.

The reference has no tests / golden vectors of its own (SURVEY.md §4), so parity is pinned by
outputs of the reference code itself, produced here once and committed:

  ops_small.npz        ConvMask / Conv1dMask / LinearMask forward + autograd backward (fp32)
  prune_small.npz      prune_mag / prune_snip / prune_synflow / prune_random_* on a small conv net
  probs.json           ERK / balanced keep-probabilities for ResNet-18/50, VGG-16 layer shapes (hex fp32 / repr)
  densities.json       generate_densities schedules
  imp_hashes.json      seed-0 ResNet-18 (CIFAR) IMP levels: SHA-256 of weights, thresholds, masks
  sgd_small.npz        torch.optim.SGD(momentum, wd) trajectory used by the reference harness
  reference_models.json  seed-0 ResNet-18 (CIFAR) state-dict digests at init, after prune_er_erk / prune_er_balanced
                       and after prune_mag(0.8); the reference's conf/ files the config composer is tested on
  reference_run.npz    that model's eval logits on a fixed batch, and a batch_crop at translate = 3

Run with the reference checked out:  TURBOPRUNE_REFERENCE=<dir> python tests/golden/make_golden.py
"""
import contextlib
import hashlib
import json
import os
import sys

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import refshim  # noqa: E402

ml, pu, cm = refshim.load_reference()
torch.set_num_threads(8)


def sha(arrs):
    h = hashlib.sha256()
    for a in arrs:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


@contextlib.contextmanager
def cuda_as_cpu():
    """The reference hard-codes 'cuda' in prune_snip / prune_synflow (pruning_utils.py:178-179,254-257);
    map those placements to the CPU while the reference code runs (fixture generation only)."""
    real_to, real_device = torch.Tensor.to, torch.device

    def to(self, *a, **k):
        a = tuple("cpu" if (isinstance(x, str) and x.startswith("cuda")) else x for x in a)
        a = tuple(real_device("cpu") if (isinstance(x, real_device) and x.type == "cuda") else x for x in a)
        return real_to(self, *a, **k)

    class _Dev:
        def __call__(self, *a, **k):
            a = tuple("cpu" if (isinstance(x, str) and x.startswith("cuda")) else x for x in a)
            return real_device(*a, **k)

        def __instancecheck__(self, obj):
            return isinstance(obj, real_device)

    torch.Tensor.to = to
    pu.torch.device = real_device  # keep type; handled through Tensor.to above
    try:
        yield
    finally:
        torch.Tensor.to = real_to


def small_net():
    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.c1 = ml.ConvMask(in_channels=3, out_channels=8, kernel_size=3, padding=1, bias=True)
            self.bn = nn.BatchNorm2d(8)
            self.c2 = ml.ConvMask(in_channels=8, out_channels=16, kernel_size=3, stride=2, padding=1, bias=False)
            self.fc = ml.Conv1dMask(16, 10, bias=True)
            self.ln = ml.LinearMask(in_features=10, out_features=10, bias=True)

        def forward(self, x):
            x = torch.relu(self.bn(self.c1(x)))
            x = torch.relu(self.c2(x)).mean((2, 3))
            return self.ln(self.fc(x))
    return Net()


def masked(net):
    return [m for m in net.modules() if isinstance(m, (ml.ConvMask, ml.Conv1dMask, ml.LinearMask))]


def gen_ops():
    out = {}
    g = torch.Generator().manual_seed(0)
    cases = {
        "conv3x3": dict(n=2, cin=8, cout=16, k=3, s=1, p=1, hw=9, bias=True),
        "conv3x3s2": dict(n=2, cin=16, cout=8, k=3, s=2, p=1, hw=10, bias=False),
        "conv1x1s2": dict(n=3, cin=16, cout=24, k=1, s=2, p=0, hw=8, bias=False),
        "conv7x7s2": dict(n=1, cin=3, cout=8, k=7, s=2, p=3, hw=20, bias=False),
    }
    for name, c in cases.items():
        layer = ml.ConvMask(in_channels=c["cin"], out_channels=c["cout"], kernel_size=c["k"], stride=c["s"],
                            padding=c["p"], bias=c["bias"])
        layer.set_er_mask(0.5)
        x = torch.randn(c["n"], c["cin"], c["hw"], c["hw"], generator=g, requires_grad=True)
        y = layer(x)
        dy = torch.randn(y.shape, generator=g)
        y.backward(dy)
        out.update({f"{name}.x": x.detach().numpy(), f"{name}.w": layer.weight.detach().numpy(),
                    f"{name}.m": layer.mask.numpy(), f"{name}.dy": dy.numpy(), f"{name}.y": y.detach().numpy(),
                    f"{name}.dx": x.grad.numpy(), f"{name}.dw": layer.weight.grad.numpy(),
                    f"{name}.cfg": np.array([c["s"], c["p"]])})
        if c["bias"]:
            out[f"{name}.b"] = layer.bias.detach().numpy(); out[f"{name}.db"] = layer.bias.grad.numpy()
    for name, layer, shape in [("conv1d", ml.Conv1dMask(12, 7, bias=True), (5, 12)),
                               ("linear", ml.LinearMask(in_features=12, out_features=7, bias=True), (2, 3, 12))]:
        layer.set_er_mask(0.5)
        x = torch.randn(*shape, generator=g, requires_grad=True)
        y = layer(x); dy = torch.randn(y.shape, generator=g); y.backward(dy)
        out.update({f"{name}.x": x.detach().numpy(), f"{name}.w": layer.weight.detach().numpy(),
                    f"{name}.m": layer.mask.numpy(), f"{name}.b": layer.bias.detach().numpy(),
                    f"{name}.dy": dy.numpy(), f"{name}.y": y.detach().numpy(), f"{name}.dx": x.grad.numpy(),
                    f"{name}.dw": layer.weight.grad.numpy(), f"{name}.db": layer.bias.grad.numpy()})
    np.savez_compressed(os.path.join(HERE, "ops_small.npz"), **out)


def gen_prune():
    out = {}
    cfg = refshim.make_cfg(precision="float32")
    torch.manual_seed(0)
    net = small_net()
    g = torch.Generator().manual_seed(1)
    images = torch.randn(4, 3, 8, 8, generator=g); labels = torch.randint(0, 10, (4,), generator=g)
    loader = [(images, labels)]
    layers = masked(net)
    init = {k: v.clone() for k, v in net.state_dict().items()}
    out["images"] = images.numpy(); out["labels"] = labels.numpy()
    for i, m in enumerate(layers):
        out[f"w{i}"] = m.weight.detach().numpy().copy()

    def snap(tag):
        for i, m in enumerate(layers):
            out[f"{tag}.m{i}"] = m.mask.numpy().copy()

    # iterative magnitude pruning 1.0 -> 0.8 -> 0.64 (masks feed forward)
    for lvl, d in enumerate([0.8, 0.64, 0.3]):
        pu.prune_mag(net, d); snap(f"mag{lvl}")
    # density increase on an already sparse net: threshold falls inside the zeros
    pu.prune_mag(net, 0.9); snap("mag_up")
    # snip / synflow from a fresh dense state, and from a masked state
    for tag, fn in [("snip", pu.prune_snip), ("synflow", pu.prune_synflow)]:
        net.load_state_dict(init); net.zero_grad()
        for m in layers:
            m.mask = torch.ones_like(m.weight)
        net.train()
        # prune_synflow calls model.zero_grad() after scoring (pruning_utils.py:270): wrap THIS instance's method (the
        # reference source stays untouched) so the gradients and the linearised |w| it scored are captured first
        captured = {}
        real_zero_grad = net.zero_grad

        def capturing_zero_grad(*a, **k):
            if all(m.weight.grad is not None for m in layers):
                captured["g"] = [m.weight.grad.detach().numpy().copy() for m in layers]
                captured["w"] = [m.weight.detach().numpy().copy() for m in layers]
            return real_zero_grad(*a, **k)
        net.zero_grad = capturing_zero_grad
        with cuda_as_cpu():
            fn(cfg, net, loader, 0.5)
        del net.zero_grad
        for i, m in enumerate(layers):
            if tag == "synflow":
                out[f"{tag}.g{i}"] = captured["g"][i]
                out[f"{tag}.absw{i}"] = captured["w"][i]          # |w| at scoring time (signs restored afterwards)
            else:
                out[f"{tag}.g{i}"] = (m.weight.grad.numpy().copy() if m.weight.grad is not None else np.zeros(m.weight.shape, np.float32))
        snap(tag)
    # random criteria (torch generator stream is part of the contract)
    for tag, fn in [("rand_erk", pu.prune_random_erk), ("rand_bal", pu.prune_random_balanced)]:
        net.load_state_dict(init)
        for m in layers:
            m.mask = torch.ones_like(m.weight)
        torch.manual_seed(7)
        fn(net, 0.4); snap(tag)
    for tag, fn in [("er_erk", pu.prune_er_erk), ("er_bal", pu.prune_er_balanced)]:
        torch.manual_seed(9)
        fn(net, 0.3); snap(tag)
    np.savez_compressed(os.path.join(HERE, "prune_small.npz"), **out)


def layer_shapes(model_name, dataset):
    torch.manual_seed(0)
    m = cm.TorchVisionModel(refshim.make_cfg(model_name, dataset))
    return m, [tuple(l.weight.shape) for l in masked(m)]


def gen_probs_and_hashes():
    probs = {}
    for name, ds in [("resnet18", "cifar10"), ("resnet50", "imagenet"), ("vgg16", "cifar100")]:
        model, shapes = layer_shapes(name, ds)
        entry = {"shapes": [list(s) for s in shapes]}
        for d in (0.2, 0.05):
            torch.manual_seed(0)
            sl, npl, tot = [], [], 0
            for l in masked(model):                     # reference arithmetic, pruning_utils.py:357-371
                sl.append(torch.tensor(l.weight.shape).sum() / l.weight.numel()); npl.append(l.weight.numel()); tot += l.weight.numel()
            kept = (torch.tensor(sl) * torch.tensor(npl)).sum()
            C = (tot * d) / kept
            erk = [torch.clamp(C * s, 0, 1) for s in sl]
            entry[f"erk@{d}"] = [float(p).hex() for p in erk]
            # balanced: replay reference loop (:388-407)
            L = len(npl); X = d * tot / L; bal = []
            for l, n in enumerate(npl):
                if X / n < 1.0:
                    bal.append(X / n)
                else:
                    bal.append(1); X = X + (X - n) / (L - l)
            entry[f"balanced@{d}"] = [float(b).hex() for b in bal]
        probs[f"{name}/{ds}"] = entry
    json.dump(probs, open(os.path.join(HERE, "probs.json"), "w"), indent=0)

    # IMP hashes on seed-0 ResNet-18 / CIFAR-10
    torch.manual_seed(0)
    model = cm.TorchVisionModel(refshim.make_cfg("resnet18", "cifar10"))
    layers = masked(model)
    rec = {"weights_sha256": sha([l.weight.detach().numpy() for l in layers]), "levels": []}
    density = 1.0
    for _ in range(4):
        density *= 0.8
        n = sum(l.weight.numel() for l in layers)
        k = int((1 - density) * n)
        scores = torch.cat([(l.mask * l.weight).detach().abs().flatten() for l in layers])
        thr = torch.kthvalue(scores, k)[0]
        pu.prune_mag(model, density)
        rec["levels"].append({"density": density, "k": k, "thr_bits": int(np.float32(thr.item()).view(np.uint32)),
                              "masks_sha256": sha([l.mask.numpy() for l in layers]),
                              "sparsity_percent": model.get_overall_sparsity()})
    json.dump(rec, open(os.path.join(HERE, "imp_hashes.json"), "w"), indent=1)


def gen_densities():
    sys.modules.setdefault("wandb", type(sys)("wandb"))
    import importlib
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "utils" or k.startswith("utils.")}
    sys.path.insert(0, refshim.REFERENCE_ROOT)
    try:
        hu = importlib.import_module("utils.harness_utils")
    finally:
        sys.path.remove(refshim.REFERENCE_ROOT)
        for k in list(sys.modules):
            if k == "utils" or k.startswith("utils."):
                sys.modules.pop(k)
        sys.modules.update(saved)
    out = {}
    for method, target, rate in [("mag", 0.999, 0.2), ("mag", 0.988, 0.2), ("mag", 0.2, 0.2), ("random_erk", 0.9, 0.3),
                                 ("er_erk", 0.8, 0.2), ("snip", 0.5, 0.2), ("synflow", 0.95, 0.2), ("just dont", 0.5, 0.2)]:
        cfg = refshim.Cfg({"pruning_params": {"prune_method": method, "target_sparsity": target, "prune_rate": rate}})
        out[f"{method}|{target}|{rate}"] = [float(x).hex() for x in hu.generate_densities(cfg, 0.0)]
    json.dump(out, open(os.path.join(HERE, "densities.json"), "w"), indent=0)


def gen_sgd():
    g = torch.Generator().manual_seed(3)
    w = torch.randn(257, generator=g).requires_grad_(True)
    opt = torch.optim.SGD([w], lr=0.2, momentum=0.9, weight_decay=5e-4)
    out = {"w0": w.detach().numpy().copy()}
    for step in range(3):
        w.grad = torch.randn(257, generator=g)
        out[f"g{step}"] = w.grad.numpy().copy()
        opt.step()
        out[f"w{step + 1}"] = w.detach().numpy().copy()
    np.savez_compressed(os.path.join(HERE, "sgd_small.npz"), **out)


def gen_aug():
    """aug_small.npz: the reference's batch_crop / batch_flip_lr / batch_cutout (utils/dataset.py:38-98) run on CPU; the
    draws each call made are re-drawn from the same seed and stored next to its output."""
    ds = refshim.load_reference_dataset()
    g = torch.Generator().manual_seed(11)
    imgs = torch.randn(7, 3, 12, 12, generator=g)
    padded = torch.nn.functional.pad(imgs, (2,) * 4, "reflect")                  # translate = 2 -> 16 x 16, r <= 2 branch
    padded4 = torch.nn.functional.pad(imgs, (4,) * 4, "reflect")                 # translate = 4 -> the two-pass branch
    out = {"imgs": imgs.numpy(), "padded": padded.numpy(), "padded4": padded4.numpy()}
    for tag, src, r in (("crop2", padded, 2), ("crop4", padded4, 4)):
        torch.manual_seed(21); out[f"{tag}.out"] = ds.batch_crop(src, 12).numpy()
        torch.manual_seed(21); out[f"{tag}.shifts"] = torch.randint(-r, r + 1, size=(7, 2)).numpy()
    torch.manual_seed(22); out["flip.out"] = ds.batch_flip_lr(imgs).numpy()
    torch.manual_seed(22); out["flip.mask"] = (torch.rand(7) < 0.5).numpy()
    torch.manual_seed(23); out["cut.out"] = ds.batch_cutout(imgs, 5).numpy()
    torch.manual_seed(23); out["cut.y"] = torch.randint(0, 12 - 5 + 1, size=(7,)).numpy(); out["cut.x"] = torch.randint(0, 12 - 5 + 1, size=(7,)).numpy()
    # the epoch pipeline of CifarLoader.__iter__ (:204-221): translate -> flip -> cutout
    torch.manual_seed(24)
    x = ds.batch_crop(padded4, 12); x = ds.batch_flip_lr(x); x = ds.batch_cutout(x, 3)
    out["epoch.out"] = x.numpy()
    torch.manual_seed(24)
    out["epoch.shifts"] = torch.randint(-4, 5, size=(7, 2)).numpy(); out["epoch.mask"] = (torch.rand(7) < 0.5).numpy()
    out["epoch.y"] = torch.randint(0, 12 - 3 + 1, size=(7,)).numpy(); out["epoch.x"] = torch.randint(0, 12 - 3 + 1, size=(7,)).numpy()
    np.savez_compressed(os.path.join(HERE, "aug_small.npz"), **out)


REFERENCE_CONF_FILES = [          # what compose() reads for the three compositions in test_config_composer_and_densities
    "cifar10_er_erk.yaml", "imagenet_er_balanced.yaml",
    "dataset_params/dp_cifar10.yaml", "optimizer_params/sgd_cifar10.yaml", "experiment_params/ep_cifar10.yaml",
    "model_params/mp_resnet18.yaml", "dataset_params/dp_imagenet_ffcv.yaml", "optimizer_params/sgd_imagenet.yaml",
    "experiment_params/ep_imagenet.yaml", "model_params/mp_resnet50.yaml", "cyclic_training/ct_no_cyclic.yaml",
    "pruning_params/iterative_imp.yaml", "pruning_params/pai_er_erk.yaml", "pruning_params/iterative_wr.yaml",
]


def gen_reference_checks():
    """reference_models.json / reference_run.npz: the reference's model construction, ER masks, magnitude pruning,
    eval forward, batch_crop and conf/ tree, for the CPU tests that check the oracle and the product against them."""
    import yaml
    cfg = refshim.make_cfg("resnet18", "cifar10")
    rec, run = {}, {}
    torch.manual_seed(0)
    r = cm.TorchVisionModel(cfg)
    rec["init"] = refshim.state_digests(r.state_dict())
    for fn in ("prune_er_erk", "prune_er_balanced"):
        torch.manual_seed(5); getattr(pu, fn)(r, 0.2)
        rec[fn] = {"state": refshim.state_digests(r.state_dict()), "sparsity_percent": r.get_overall_sparsity()}
    torch.manual_seed(0)
    r = cm.TorchVisionModel(cfg)
    x = torch.randn(4, 3, 32, 32, generator=torch.Generator().manual_seed(4))
    r.eval()
    with torch.no_grad():
        run["logits.x"], run["logits.y"] = x.numpy(), r(x).numpy()
    pu.prune_mag(r, 0.8)
    rec["prune_mag_0.8_masks"] = refshim.state_digests({n: m.mask for n, m in r.model.named_modules() if isinstance(m, (ml.ConvMask, ml.Conv1dMask, ml.LinearMask))})
    conf = {f: yaml.safe_load(open(os.path.join(refshim.REFERENCE_ROOT, "conf", f))) for f in REFERENCE_CONF_FILES}
    json.dump({"resnet18_cifar10": rec, "conf": conf}, open(os.path.join(HERE, "reference_models.json"), "w"), indent=0)

    ds = refshim.load_reference_dataset()
    imgs = torch.randn(5, 3, 10, 10, generator=torch.Generator().manual_seed(3))
    pad = torch.nn.functional.pad(imgs, (3,) * 4, "reflect")                   # translate = 3
    torch.manual_seed(8); run["crop3.out"] = ds.batch_crop(pad, 10).numpy()
    torch.manual_seed(8); run["crop3.shifts"] = torch.randint(-3, 4, size=(5, 2)).numpy()
    run["crop3.padded"] = pad.numpy()
    np.savez_compressed(os.path.join(HERE, "reference_run.npz"), **run)


if __name__ == "__main__":
    gen_ops(); gen_prune(); gen_probs_and_hashes(); gen_densities(); gen_sgd(); gen_aug(); gen_reference_checks()
    for f in sorted(os.listdir(HERE)):
        print(f, os.path.getsize(os.path.join(HERE, f)))
