"""Oracle for the CIFAR loader (test infrastructure only): the reference's CifarLoader (utils/dataset.py:101-226)
restated on numpy arrays for GIVEN random draws.

  cifar_normalize   images / 255 -> T.Normalize(mean, std), uint8 [N,H,W,C] -> fp32 [N,C,H,W].  ``cuda_arith`` picks
                    the rounding of the first step: ATen's CUDA true-divide by a CPU scalar multiplies by the fp32
                    reciprocal, the CPU kernel divides.  sub_ / div_ by the per-channel tensors are true fp32 ops on both.
  cifar_epoch       one epoch: normalise -> pre-flip -> reflect pad -> crop at the shifts -> flip -> cutout -> gather by
                    the permutation, each step the reference's own, written as numpy slicing.
  replay_loader     the loader's iteration for several epochs, asking ``draw`` for each random draw in the reference's
                    order (first epoch: pre-flip mask; every epoch: shifts, flip mask, cutout y, cutout x, permutation).
"""
from math import ceil

import numpy as np

CIFAR10_MEAN = np.array((0.4914, 0.4822, 0.4465), np.float32)
CIFAR10_STD = np.array((0.2470, 0.2435, 0.2616), np.float32)
CIFAR100_MEAN = np.array((0.5071, 0.4867, 0.4408), np.float32)
CIFAR100_STD = np.array((0.2675, 0.2565, 0.2761), np.float32)


def constants(dataset):
    """The reference picks the CIFAR-10 constants only for the exact name "CIFAR10" (dataset.py:113-120)."""
    return (CIFAR10_MEAN, CIFAR10_STD) if dataset == "CIFAR10" else (CIFAR100_MEAN, CIFAR100_STD)


def cifar_normalize(u8, mean, std, cuda_arith):
    x = np.asarray(u8).astype(np.float32).transpose(0, 3, 1, 2)
    x = x * (np.float32(1.0) / np.float32(255.0)) if cuda_arith else x / np.float32(255.0)
    c = x.shape[1]
    m = np.asarray(mean, np.float32).reshape(1, c, 1, 1)
    s = np.asarray(std, np.float32).reshape(1, c, 1, 1)
    return np.ascontiguousarray((x - m) / s, dtype=np.float32)


def cifar_epoch(u8, labels, mean, std, cuda_arith, perm=None, shifts=None, r=0, preflip=None, flip=None, flip_all=False,
                cut_y=None, cut_x=None, cut_size=0):
    """Images fp32 [N,C,H,W] and labels of one epoch; every draw optional (None: that step is skipped)."""
    x = cifar_normalize(u8, mean, std, cuda_arith)
    n, _, h, w = x.shape
    if preflip is not None:
        x = np.where(np.asarray(preflip, bool).reshape(-1, 1, 1, 1), x[..., ::-1], x)
    if shifts is not None:
        pad = np.pad(x, ((0, 0), (0, 0), (r, r), (r, r)), mode="reflect")
        out = np.empty_like(x)
        for i in range(n):
            sy, sx = int(shifts[i][0]), int(shifts[i][1])
            out[i] = pad[i, :, r + sy:r + sy + h, r + sx:r + sx + w]
        x = out
    if flip_all:
        x = x[..., ::-1]
    elif flip is not None:
        x = np.where(np.asarray(flip, bool).reshape(-1, 1, 1, 1), x[..., ::-1], x)
    if cut_y is not None:
        yy = np.arange(h).reshape(1, 1, h, 1) - np.asarray(cut_y).reshape(-1, 1, 1, 1)
        xx = np.arange(w).reshape(1, 1, 1, w) - np.asarray(cut_x).reshape(-1, 1, 1, 1)
        x = np.where((yy >= 0) & (yy < cut_size) & (xx >= 0) & (xx < cut_size), np.float32(0), x)
    idx = np.arange(n) if perm is None else np.asarray(perm)
    return np.ascontiguousarray(x[idx], dtype=np.float32), np.asarray(labels)[idx]


def replay_loader(u8, labels, mean, std, cuda_arith, draw, epochs, batch_size, aug=None, train=True, drop_last=None,
                  shuffle=None, altflip=False):
    """[[(images, labels) per batch] per epoch].  ``draw(kind, *args)`` returns the next draw as a numpy array:
    ("rand", n) -> the uniforms of torch.rand(n); ("randint", lo, hi, size); ("randperm", n)."""
    aug = aug or {}
    drop_last = train if drop_last is None else drop_last
    shuffle = train if shuffle is None else shuffle
    n, h, w = len(u8), u8.shape[1], u8.shape[2]
    nb = n // batch_size if drop_last else ceil(n / batch_size)
    pad, cut = aug.get("translate", 0), aug.get("cutout", 0)
    preflip, out = None, []
    for epoch in range(epochs):
        if epoch == 0 and aug.get("flip", False):
            preflip = draw("rand", n) < 0.5
        shifts = draw("randint", -pad, pad + 1, (n, 2)) if pad > 0 else None
        flip, flip_all = None, False
        if aug.get("flip", False):
            if altflip:
                flip_all = epoch % 2 == 1
            else:
                flip = draw("rand", n) < 0.5
        cy = cx = None
        if cut > 0:
            cy = draw("randint", 0, h - cut + 1, (n,))
            cx = draw("randint", 0, w - cut + 1, (n,))
        perm = draw("randperm", n) if shuffle else None
        x, t = cifar_epoch(u8, labels, mean, std, cuda_arith, perm=perm, shifts=shifts, r=pad, preflip=preflip, flip=flip,
                           flip_all=flip_all, cut_y=cy, cut_x=cx, cut_size=cut)
        out.append([(x[i * batch_size:(i + 1) * batch_size], t[i * batch_size:(i + 1) * batch_size]) for i in range(nb)])
    return out


def recorded(draws):
    """A ``draw`` for replay_loader that hands out stored draws in sequence (the kinds are the caller's business)."""
    it = iter(draws)
    return lambda kind, *args: np.asarray(next(it))
