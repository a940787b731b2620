#!/usr/bin/env python
"""Generate cifar_loader_small.npz by EXECUTING THE UNMODIFIED REFERENCE CifarLoader (utils/dataset.py:101-226) on CPU.

  cifar_loader_small.npz   a tiny uint8 data set written in the reference's .pt cache format, every batch the reference's
                           loader yields for it (train: flip + translate 2 + altflip, three epochs, drop_last; a second
                           train loader with random flip + translate 2 + cutout 4 for two epochs; the test loader), and the
                           random draws each run made, re-drawn from the same seed in the order the loader made them.

The loader loads its data with torch.load(map_location="cuda"); that placement is mapped to the CPU while it runs, so
the fixture holds the CPU arithmetic (images / 255 as a true division).  Kept apart from make_golden.py so that
regenerating this file leaves the other fixtures untouched.

Run with the reference checked out:  TURBOPRUNE_REFERENCE=<dir> python tests/golden/make_cifar_golden.py
"""
import contextlib
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import refshim  # noqa: E402


@contextlib.contextmanager
def load_to_cpu():
    real = torch.load

    def load(*a, **k):
        k["map_location"] = "cpu"
        return real(*a, **k)
    torch.load = load
    try:
        yield
    finally:
        torch.load = real


def write_pt(root, dataset, split, images, labels, classes):
    d = os.path.join(root, "cifar10" if dataset == "CIFAR10" else "cifar100")
    os.makedirs(d, exist_ok=True)
    torch.save({"images": torch.from_numpy(images), "labels": torch.from_numpy(labels), "classes": classes},
               os.path.join(d, f"{dataset}_{split}.pt"))


def run(ds, root, seed, epochs, **kw):
    torch.manual_seed(seed)
    with load_to_cpu():
        loader = ds.CifarLoader(root, **kw)
    return [[(x.numpy().copy(), t.numpy().copy()) for x, t in loader] for _ in range(epochs)], len(loader)


def gen_cifar_loader():
    ds = refshim.load_reference_dataset()
    g = np.random.default_rng(5)
    out = {}
    cases = [  # tag, dataset, n, seed, epochs, loader arguments, draws in the loader's order
        ("a", "CIFAR10", 16, 41, 3, dict(train=True, batch_size=5, aug={"flip": True, "translate": 2}, altflip=True)),
        ("b", "CIFAR100", 10, 42, 2, dict(train=True, batch_size=4, aug={"flip": True, "translate": 2, "cutout": 4})),
        ("t", "CIFAR10", 16, 43, 1, dict(train=False, batch_size=5)),
    ]
    with tempfile.TemporaryDirectory() as root:
        for tag, dataset, n, seed, epochs, kw in cases:
            images = g.integers(0, 256, size=(n, 32, 32, 3), dtype=np.uint8)
            labels = g.integers(0, 10, size=(n,)).astype(np.int64)
            split = "train" if kw["train"] else "test"
            write_pt(root, dataset, split, images, labels, [f"c{i}" for i in range(10)])
            batches, nb = run(ds, root, seed, epochs, dataset=dataset, **kw)
            out[f"{tag}.images"], out[f"{tag}.labels"], out[f"{tag}.len"] = images, labels, np.array(nb)
            for e, ep in enumerate(batches):
                for b, (x, t) in enumerate(ep):
                    out[f"{tag}.e{e}.b{b}.x"], out[f"{tag}.e{e}.b{b}.y"] = x, t
            # the same draws again from the same seed, in the order CifarLoader.__iter__ makes them
            torch.manual_seed(seed)
            aug, draws = kw.get("aug", {}), []
            for e in range(epochs):
                if e == 0 and aug.get("flip"):
                    draws.append(torch.rand(n).numpy())
                if aug.get("translate", 0):
                    r = aug["translate"]
                    draws.append(torch.randint(-r, r + 1, size=(n, 2)).numpy())
                if aug.get("flip") and not kw.get("altflip"):
                    draws.append(torch.rand(n).numpy())
                if aug.get("cutout", 0):
                    s = aug["cutout"]
                    draws.append(torch.randint(0, 32 - s + 1, size=(n,)).numpy())
                    draws.append(torch.randint(0, 32 - s + 1, size=(n,)).numpy())
                if kw["train"]:
                    draws.append(torch.randperm(n).numpy())
            out[f"{tag}.ndraws"] = np.array(len(draws))
            for k, d in enumerate(draws):
                out[f"{tag}.draw{k}"] = d
    np.savez_compressed(os.path.join(HERE, "cifar_loader_small.npz"), **out)


if __name__ == "__main__":
    gen_cifar_loader()
    f = os.path.join(HERE, "cifar_loader_small.npz")
    print(f, os.path.getsize(f))
