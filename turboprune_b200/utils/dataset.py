"""The loaders: the reference's CIFAR loader on the real data set, and a synthetic on-device generator
(reference utils/dataset.py: CifarLoader / AirbenchLoaders :101-256, FFCVImagenet :347-430).

``make_loaders(cfg, device, world, rank)`` picks one per config:

  CIFAR, ``dataset_params.dataloader_type`` absent or ``synthetic``   SyntheticLoaders
  CIFAR, any other ``dataloader_type`` (the reference ships ``torch``) AirbenchLoaders: the data set from
                                                                      ``dataset_params.data_root_dir``
  ImageNet                                                            SyntheticLoaders (FFCV / webdataset out of scope)

``CifarLoader`` keeps the data set on the GPU as stored (uint8 NHWC) and builds each epoch — normalisation, pre-flip,
translate, flip, cutout and the shuffle, with the reference's random draws — in one ``tp_cifar_epoch`` launch.  It reads
``<data_root_dir>/cifar10|cifar100/<DATASET>_train|test.pt`` (the reference's cache), or converts torchvision's extracted
archive next to it; nothing is downloaded.

Same batch contract for all: an iterable of ``(images fp32 [B,3,H,W], labels int64 [B])`` with ``len()``; ImageNet-shaped
synthetic batches come channels_last like FFCV's ToTorchImage.  The synthetic generator is seeded per rank; either a
fixed number of distinct batches is generated once and cycled (an epoch costs no host work), or
(``dataset_params.synthetic_fresh``) every step draws a new batch on the device.  ``DevicePrefetcher`` is the
host->device leg for loaders that produce pinned host batches.
"""
import os
import pickle
from ctypes import c_float, c_void_p
from math import ceil

import numpy as np
import torch

from .. import _cabi, ops


# ---- airbench-style GPU augmentation (reference utils/dataset.py:38-98): same names, same draws, one fused kernel ------
def _ptr(t):
    return c_void_p(t.data_ptr()) if t is not None else None


def _augment(src, out_hw, r, shifts=None, flip=None, corner_y=None, corner_x=None, cut_size=0):
    if not src.is_cuda:
        raise RuntimeError("turboprune_b200 augmentation kernels need CUDA tensors (B200 / sm_100a); there is no CPU path")
    lib = _cabi.load()
    src = src.contiguous().float()
    n, c = src.shape[:2]
    h, w = out_hw
    out = torch.empty(n, c, h, w, dtype=torch.float32, device=src.device)
    f8 = flip.to(torch.uint8).contiguous() if flip is not None else None
    sh = shifts.to(torch.int64).contiguous() if shifts is not None else None
    cy = corner_y.to(torch.int64).contiguous() if corner_y is not None else None
    cx = corner_x.to(torch.int64).contiguous() if corner_x is not None else None
    with torch.cuda.device(src.device):
        rc = lib.tp_cifar_augment(_ptr(src), _ptr(out), _ptr(sh), _ptr(f8), _ptr(cy), _ptr(cx), int(cut_size), n, c, h, w, int(r),
                                  _cabi.stream_ptr(src.device))
    _cabi.check(rc, "tp_cifar_augment")
    ops._count()
    return out


def batch_flip_lr(inputs):
    """reference :38-40 — the flip mask is drawn with torch's generator on the inputs' device, like upstream."""
    flip_mask = torch.rand(len(inputs), device=inputs.device) < 0.5
    return _augment(inputs, inputs.shape[-2:], 0, flip=flip_mask)


def batch_crop(images, crop_size):
    """reference :43-69 — random translation: a crop_size window of the padded images at a per-image shift."""
    r = (images.size(-1) - crop_size) // 2
    shifts = torch.randint(-r, r + 1, size=(len(images), 2), device=images.device)
    return _augment(images, (crop_size, crop_size), r, shifts=shifts)


def batch_cutout(inputs, size):
    """reference :72-98 — one size x size square per image zeroed."""
    n, c, h, w = inputs.shape
    corner_y = torch.randint(0, h - size + 1, size=(n,), device=inputs.device)
    corner_x = torch.randint(0, w - size + 1, size=(n,), device=inputs.device)
    return _augment(inputs, (h, w), 0, corner_y=corner_y, corner_x=corner_x, cut_size=size)


def augment_epoch(padded, crop_size, flip=True, cutout=0):
    """CifarLoader.__iter__ (:204-221, random-flip branch) for one epoch in ONE pass: the draws are made in the
    reference's order (crop shifts, flip mask, cutout corners), the pixels move once instead of three times."""
    n = len(padded)
    r = (padded.size(-1) - crop_size) // 2
    shifts = torch.randint(-r, r + 1, size=(n, 2), device=padded.device) if r > 0 else None
    flip_mask = (torch.rand(n, device=padded.device) < 0.5) if flip else None
    cy = cx = None
    if cutout > 0:
        cy = torch.randint(0, crop_size - cutout + 1, size=(n,), device=padded.device)
        cx = torch.randint(0, crop_size - cutout + 1, size=(n,), device=padded.device)
    return _augment(padded, (crop_size, crop_size), r, shifts=shifts, flip=flip_mask, corner_y=cy, corner_x=cx, cut_size=cutout)


def synth_normal_(out, seed, counter_offset=0, raw_words=False):
    """Fill ``out`` (fp32, dense memory) with the Philox4x32-10 / Box-Muller stream (element order = memory order)."""
    lib = _cabi.load()
    with torch.cuda.device(out.device):
        rc = lib.tp_synth_normal(_ptr(out), out.numel(), int(seed), int(counter_offset), int(bool(raw_words)), _cabi.stream_ptr(out.device))
    _cabi.check(rc, "tp_synth_normal")
    ops._count()
    return out


def synth_labels_(out, num_classes, seed, counter_offset=0):
    lib = _cabi.load()
    with torch.cuda.device(out.device):
        rc = lib.tp_synth_labels(_ptr(out), out.numel(), int(num_classes), int(seed), int(counter_offset), _cabi.stream_ptr(out.device))
    _cabi.check(rc, "tp_synth_labels")
    ops._count()
    return out


class SyntheticLoader:
    """``fresh=True``: every iteration draws a new batch on the device (Philox, seeded per rank — SURVEY.md §8(d));
    otherwise ``distinct`` batches are generated once and cycled."""

    def __init__(self, batch_size, steps, shape, num_classes, device, seed=0, distinct=4, channels_last=False, fresh=False):
        self.gen = torch.Generator(device=device).manual_seed(seed)
        self.seed, self._ctr = int(seed), 0
        self.steps = steps
        self.batch_size, self.shape, self.num_classes, self.device = batch_size, tuple(shape), num_classes, device
        self.channels_last = channels_last
        self.fresh = fresh
        self.batches = [] if fresh else [self._draw() for _ in range(min(distinct, steps))]

    def _draw(self):
        c, h, w = self.shape
        dev = torch.device(self.device)
        if dev.type == "cuda":
            # our generator: Philox4x32-10 -> Box-Muller straight into the batch buffer, a fresh counter range per batch
            shp = (self.batch_size, h, w, c) if self.channels_last else (self.batch_size, c, h, w)
            x = torch.empty(shp, dtype=torch.float32, device=dev)
            t = torch.empty(self.batch_size, dtype=torch.int64, device=dev)
            synth_normal_(x, self.seed, self._ctr)
            synth_labels_(t, self.num_classes, self.seed ^ 0x5DEECE66D, self._ctr)
            self._ctr += (x.numel() + 3) // 4
            return (x.permute(0, 3, 1, 2) if self.channels_last else x), t
        if self.channels_last:       # NHWC memory, logical NCHW (what FFCV's ToTorchImage hands over, dataset.py:391)
            x = torch.randn(self.batch_size, h, w, c, device=self.device, generator=self.gen).permute(0, 3, 1, 2)
        else:
            x = torch.randn(self.batch_size, c, h, w, device=self.device, generator=self.gen)
        return x, torch.randint(0, self.num_classes, (self.batch_size,), device=self.device, generator=self.gen)

    def __len__(self):
        return self.steps

    def __iter__(self):
        for i in range(self.steps):
            yield self._draw() if self.fresh else self.batches[i % len(self.batches)]


class DevicePrefetcher:
    """Wraps an iterable of HOST batches (pinned ``(images, labels)``) and yields device batches: batch i+1 crosses PCIe
    on a copy stream while step i computes (two staging slots, guarded by events).  Stands where the reference's
    loaders hand over device tensors (FFCV ``ToDevice(non_blocking=True)``, dataset.py:385-430)."""

    def __init__(self, host_loader, device):
        self.loader, self.device = host_loader, device
        self.copy_stream = torch.cuda.Stream(device)
        self.slots = [None, None]
        self.ready = [torch.cuda.Event(), torch.cuda.Event()]
        self.consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def __len__(self):
        return len(self.loader)

    def _issue(self, j, batch):
        x, t = batch
        if self.slots[j] is None or self.slots[j][0].shape != x.shape:
            self.slots[j] = (torch.empty_strided(x.shape, x.stride(), dtype=x.dtype, device=self.device),
                             torch.empty(t.shape, dtype=t.dtype, device=self.device))
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.consumed[j])
            self.slots[j][0].copy_(x, non_blocking=True); self.slots[j][1].copy_(t, non_blocking=True)
            self.ready[j].record(self.copy_stream)

    def __iter__(self):
        cur = torch.cuda.current_stream(self.device)
        for ev in self.consumed:
            ev.record(cur)
        it = iter(self.loader)
        nxt = next(it, None)
        if nxt is None:
            return
        self._issue(0, nxt)
        i = 0
        while nxt is not None:
            j = i % 2
            nxt = next(it, None)
            if nxt is not None:
                self._issue(1 - j, nxt)              # overlaps with the step consuming slot j
            cur = torch.cuda.current_stream(self.device)
            cur.wait_event(self.ready[j])
            yield self.slots[j]
            self.consumed[j].record(torch.cuda.current_stream(self.device))
            i += 1


# ---- the CIFAR data sets (reference :101-256) --------------------------------------------------------------------------
CIFAR10_MEAN = (0.4914, 0.4822, 0.4465)
CIFAR10_STD = (0.2470, 0.2435, 0.2616)
CIFAR100_MEAN = (0.5071, 0.4867, 0.4408)
CIFAR100_STD = (0.2675, 0.2565, 0.2761)


def cifar_paths(path, train=True, dataset="CIFAR10"):
    """(.pt cache, torchvision's extracted archive directory).  The dataset name is compared case-sensitively, as in
    the reference: anything but "CIFAR10" is CIFAR-100."""
    d = os.path.join(path, "cifar10" if dataset == "CIFAR10" else "cifar100")
    pt = os.path.join(d, f"{dataset}_{'train' if train else 'test'}.pt")
    return pt, os.path.join(d, "cifar-10-batches-py" if dataset == "CIFAR10" else "cifar-100-python")


def _read_archive(archive, train, cifar10):
    """torchvision's extracted python-pickle archive -> (uint8 [N,32,32,3], int64 [N], class names), read directly."""
    def unpickle(name):
        with open(os.path.join(archive, name), "rb") as f:
            return pickle.load(f, encoding="latin1")
    if cifar10:
        files, key, meta, names = ([f"data_batch_{k}" for k in range(1, 6)] if train else ["test_batch"]), "labels", "batches.meta", "label_names"
    else:
        files, key, meta, names = (["train"] if train else ["test"]), "fine_labels", "meta", "fine_label_names"
    parts = [unpickle(f) for f in files]
    images = np.concatenate([np.asarray(p["data"], np.uint8).reshape(-1, 3, 32, 32) for p in parts]).transpose(0, 2, 3, 1)
    labels = np.concatenate([np.asarray(p[key], np.int64) for p in parts])
    return np.ascontiguousarray(images), labels, list(unpickle(meta)[names])


def load_cifar(path, train=True, dataset="CIFAR10", map_location="cpu"):
    """The data set as the reference caches it: {"images": uint8 [N,32,32,3], "labels": int64 [N], "classes": [...]}.

    Reads the .pt cache; failing that converts torchvision's extracted archive in the same directory and writes the
    cache (atomically, under a file lock, like the reference).  Raises FileNotFoundError naming both when neither exists.
    """
    pt, archive = cifar_paths(path, train, dataset)
    if not os.path.exists(pt):
        if not os.path.isdir(archive):
            raise FileNotFoundError(f"{dataset} {'train' if train else 'test'} set not found: neither {pt} nor the "
                                    f"extracted torchvision archive {archive} exists (nothing is downloaded)")
        from filelock import FileLock
        with FileLock(pt + ".lock"):
            if not os.path.exists(pt):
                images, labels, classes = _read_archive(archive, train, dataset == "CIFAR10")
                tmp = pt + ".tmp"
                torch.save({"images": torch.from_numpy(images), "labels": torch.from_numpy(labels), "classes": classes}, tmp)
                os.rename(tmp, pt)
    return torch.load(pt, map_location=map_location)


class CifarLoader:
    """The reference's CifarLoader (:101-226), same constructor, draws and batches, with one epoch = one kernel launch.

    The random draws are torch's, on the data's device and in the reference's order (first epoch: the pre-flip mask;
    every epoch: translate shifts, the per-epoch flip mask unless altflip, cutout corners y then x, the permutation), and
    they happen at the first ``next()`` like the reference's generator, so a caller that takes one batch and stops (SNIP,
    SynFlow) leaves the same CUDA random stream behind.  Each epoch is written into a fresh buffer; batches are slices of
    it.  One difference: ``.images`` is the uint8 NHWC data set on the device, not a normalised fp32 copy.
    """

    def __init__(self, path, train=True, batch_size=500, aug=None, drop_last=None, shuffle=None, altflip=False,
                 dataset="CIFAR10", device=None):
        self.epoch = 0
        data = load_cifar(path, train, dataset)
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.images = data["images"].to(dev).contiguous()
        self.labels = data["labels"].to(dev, torch.int64).contiguous()
        self.classes = data["classes"]
        self.mean, self.std = (CIFAR10_MEAN, CIFAR10_STD) if dataset == "CIFAR10" else (CIFAR100_MEAN, CIFAR100_STD)
        self.aug = aug or {}
        for k in self.aug.keys():
            assert k in ["flip", "translate", "cutout"], "Unrecognized key: %s" % k
        self.batch_size = batch_size
        self.drop_last = train if drop_last is None else drop_last
        self.shuffle = train if shuffle is None else shuffle
        self.altflip = altflip
        self._preflip = None

    def __len__(self):
        return len(self.images) // self.batch_size if self.drop_last else ceil(len(self.images) / self.batch_size)

    def __setattr__(self, k, v):
        if k in ("images", "labels"):
            assert self.epoch == 0, "Changing images or labels is only unsupported before iteration."
        super().__setattr__(k, v)

    def __iter__(self):
        n, h, w, _ = self.images.shape
        dev = self.images.device
        flip = self.aug.get("flip", False)
        if self.epoch == 0 and flip:
            self._preflip = torch.rand(n, device=dev) < 0.5
        r = self.aug.get("translate", 0)
        shifts = torch.randint(-r, r + 1, size=(n, 2), device=dev) if r > 0 else None
        flip_mask, flip_all = None, False
        if flip:
            if self.altflip:
                flip_all = self.epoch % 2 == 1
            else:
                flip_mask = torch.rand(n, device=dev) < 0.5
        cut = self.aug.get("cutout", 0)
        cy = cx = None
        if cut > 0:
            cy = torch.randint(0, h - cut + 1, size=(n,), device=dev)
            cx = torch.randint(0, w - cut + 1, size=(n,), device=dev)
        self.epoch += 1
        perm = torch.randperm(n, device=dev) if self.shuffle else None
        images, labels = cifar_epoch(self.images, self.labels, self.mean, self.std, perm=perm, shifts=shifts, r=r,
                                     preflip=self._preflip, flip=flip_mask, flip_all=flip_all, cut_y=cy, cut_x=cx,
                                     cut_size=cut)
        for i in range(len(self)):
            yield images[i * self.batch_size:(i + 1) * self.batch_size], labels[i * self.batch_size:(i + 1) * self.batch_size]


def cifar_epoch(u8, labels, mean, std, perm=None, shifts=None, r=0, preflip=None, flip=None, flip_all=False,
                cut_y=None, cut_x=None, cut_size=0):
    """One epoch of the uint8 NHWC data set ``u8`` as fp32 NCHW images and int64 labels, in the order of ``perm``
    (tp_cifar_epoch; every draw optional)."""
    if not u8.is_cuda or u8.dtype != torch.uint8:
        raise RuntimeError("turboprune_b200 CIFAR epoch kernel needs a CUDA uint8 tensor (B200 / sm_100a); there is no CPU path")
    lib = _cabi.load()
    u8 = u8.contiguous()
    n, h, w, c = u8.shape
    out = torch.empty(n, c, h, w, dtype=torch.float32, device=u8.device)
    lab = labels.to(torch.int64).contiguous() if labels is not None else None
    lab_out = torch.empty(n, dtype=torch.int64, device=u8.device) if labels is not None else None
    i64 = lambda t: t.to(torch.int64).contiguous() if t is not None else None
    b8 = lambda t: t.to(torch.uint8).contiguous() if t is not None else None
    pm, sh, cy, cx, pf, fl = i64(perm), i64(shifts), i64(cut_y), i64(cut_x), b8(preflip), b8(flip)
    m, s = (c_float * c)(*mean), (c_float * c)(*std)
    with torch.cuda.device(u8.device):
        rc = lib.tp_cifar_epoch(_ptr(u8), _ptr(lab), _ptr(out), _ptr(lab_out), _ptr(pm), _ptr(sh), int(r), _ptr(pf), _ptr(fl),
                                int(bool(flip_all)), _ptr(cy), _ptr(cx), int(cut_size), m, s, n, c, h, w,
                                _cabi.stream_ptr(u8.device))
    _cabi.check(rc, "tp_cifar_epoch")
    ops._count()
    return out, lab_out


class AirbenchLoaders:
    """train_loader / test_loader on the CIFAR data set under ``dataset_params.data_root_dir`` (reference :229-256):
    train with flip + translate 2 + altflip, test unaugmented, both at ``dataset_params.total_batch_size``."""

    def __init__(self, cfg, device=None):
        dp = cfg.dataset_params
        print(f"[turboprune_b200] {dp.dataset_name} from {dp.data_root_dir} (CifarLoader: one tp_cifar_epoch launch per epoch)")
        self.train_loader = CifarLoader(path=dp.data_root_dir, batch_size=dp.total_batch_size, train=True,
                                        aug={"flip": True, "translate": 2}, altflip=True, dataset=dp.dataset_name, device=device)
        self.test_loader = CifarLoader(path=dp.data_root_dir, batch_size=dp.total_batch_size, train=False,
                                       dataset=dp.dataset_name, device=device)


def uses_real_cifar(cfg):
    """True when the config asks for the CIFAR data set: a CIFAR dataset_name and a dataloader_type other than
    "synthetic" (absent counts as synthetic)."""
    kind = getattr(cfg.dataset_params, "dataloader_type", None)
    return cfg.dataset_params.dataset_name.lower().startswith("cifar") and kind is not None and str(kind) != "synthetic"


def make_loaders(cfg, device, world_size=1, rank=0):
    """The loader pair a config asks for (module docstring): AirbenchLoaders or SyntheticLoaders."""
    if uses_real_cifar(cfg):
        return AirbenchLoaders(cfg, device)
    return SyntheticLoaders(cfg, device, world_size, rank)


class SyntheticLoaders:
    """train_loader / test_loader pair sized from the config (dataset_params.total_batch_size // world_size,
    reference dataset.py:411)."""

    def __init__(self, cfg, device, world_size=1, rank=0):
        name = cfg.dataset_params.dataset_name.lower()
        ncls = 1000 if name.startswith("imagenet") else (100 if name.startswith("cifar100") else 10)
        shape = (3, 224, 224) if name.startswith("imagenet") else (3, 32, 32)
        bs = max(1, cfg.dataset_params.total_batch_size // world_size)
        steps = int(getattr(cfg.dataset_params, "synthetic_steps_per_epoch", 8))
        seed = cfg.experiment_params.seed * world_size + rank
        fresh = bool(getattr(cfg.dataset_params, "synthetic_fresh", False))
        self.train_loader = SyntheticLoader(bs, steps, shape, ncls, device, seed, channels_last=name.startswith("imagenet"),
                                            fresh=fresh)
        self.test_loader = SyntheticLoader(bs, max(1, steps // 4), shape, ncls, device, seed + 7919,
                                           channels_last=name.startswith("imagenet"))
