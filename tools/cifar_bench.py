#!/usr/bin/env python
"""The CIFAR loader on one GPU, at CIFAR-10 train size (N = 50 000, 32 x 32 x 3):

  1. tp_cifar_epoch (pre-flip + translate 2 + altflip + shuffle, the AirbenchLoaders train epoch): CUDA events over
     repeated launches; achieved GB/s over the algorithmic bytes N*H*W*C read + 4*N*C*H*W + 16*N written.
  2. the same epoch done with the reference's torch expressions (normalise, pre-flip and reflect-pad once; then per epoch
     the masked-assignment crop over the 25 shifts, the altflip flip and one images[idxs] gather per batch), checked
     bit-identical to 1. with the same draws.
  3. one ResNet-18 CIFAR-10 epoch through PruningHarness.train_epoch at batch 512 (97 steps), on the real loader over a
     generated full-size data set and on the synthetic loader.

    python tools/cifar_bench.py [--reps 50]

Inputs are generated from fixed seeds.  Prints the card's name and power limit first; every time is measured here.
"""
import argparse
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

N, NTEST, H, W, C, R, BS = 50_000, 10_000, 32, 32, 3, 2, 512


def card():
    i = torch.cuda.current_device()
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(i), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        q = f"nvidia-smi unavailable ({e})"
    return f"{torch.cuda.get_device_name(i)}, power limit / max SM clock: {q}"


def event_times(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts), min(ts)


def reference_setup(u8, mean, std, preflip):
    """Epoch 0 of the reference loader: images / 255 -> NCHW channels_last -> Normalize -> pre-flip -> reflect pad."""
    x = (u8 / 255).permute(0, 3, 1, 2).to(memory_format=torch.channels_last)
    x = (x - mean.view(1, -1, 1, 1)) / std.view(1, -1, 1, 1)
    x = torch.where(preflip.view(-1, 1, 1, 1), x.flip(-1), x)
    return F.pad(x, (R,) * 4, "reflect")


def reference_epoch(padded, labels, shifts, flip_all, perm):
    """The reference's per-epoch torch work: crop by masked assignment per shift pair, flip, then one gather per batch."""
    out = torch.empty((len(padded), C, H, W), device=padded.device, dtype=padded.dtype)
    for sy in range(-R, R + 1):
        for sx in range(-R, R + 1):
            m = (shifts[:, 0] == sy) & (shifts[:, 1] == sx)
            out[m] = padded[m, :, R + sy:R + sy + H, R + sx:R + sx + W]
    if flip_all:
        out = out.flip(-1)
    return [(out[perm[i * BS:(i + 1) * BS]], labels[perm[i * BS:(i + 1) * BS]]) for i in range(len(padded) // BS)]


def harness_epoch_times(overrides, base_dir, epochs):
    from turboprune_b200.harness_definitions.standard_pruning_harness import PruningHarness
    from turboprune_b200.utils import config as tp_config
    cfg = tp_config.compose("synthetic_rn18_imp", [f"dataset_params.total_batch_size={BS}", f"experiment_params.base_dir={base_dir}",
                                                   *overrides], os.path.join(ROOT, "conf_b200"))
    torch.manual_seed(0)
    h = PruningHarness(cfg=cfg, gpu_id=0, expt_dir=("cifar_bench", base_dir))
    h._setup_optimizer()
    h._setup_scheduler(epochs + 1)
    assert len(h.train_loader) == N // BS, len(h.train_loader)
    h.train_epoch()                                   # warm-up: eager steps, graph capture
    ts = []
    for _ in range(epochs):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        h.train_epoch()                               # ends in a host sync (loss / accuracy .item())
        torch.cuda.synchronize(); ts.append((time.perf_counter() - t0) * 1e3)
    return type(h.train_loader).__name__, ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--train-epochs", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cifar_bench needs a CUDA device")
    from turboprune_b200.utils import dataset as ds
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    print(f"[card] {card()}")

    g = torch.Generator().manual_seed(0)
    u8 = torch.randint(0, 256, (N, H, W, C), dtype=torch.uint8, generator=g).to(dev)
    labels = torch.randint(0, 10, (N,), generator=g).to(dev)
    mean_t, std_t = torch.tensor(ds.CIFAR10_MEAN, device=dev), torch.tensor(ds.CIFAR10_STD, device=dev)
    torch.manual_seed(1)
    preflip = torch.rand(N, device=dev) < 0.5
    shifts = torch.randint(-R, R + 1, (N, 2), device=dev)
    perm = torch.randperm(N, device=dev)

    # 1. the kernel, odd epoch (altflip flips every image)
    kernel = lambda: ds.cifar_epoch(u8, labels, ds.CIFAR10_MEAN, ds.CIFAR10_STD, perm=perm, shifts=shifts, r=R, preflip=preflip,
                                    flip_all=True)
    med, best = event_times(kernel, args.reps)
    nbytes = N * H * W * C + 4 * N * C * H * W + 16 * N
    print(f"[tp_cifar_epoch] N={N} {H}x{W}x{C}: median {med:.3f} ms, min {best:.3f} ms over {args.reps} launches; "
          f"{nbytes / 1e6:.1f} MB algorithmic -> {nbytes / med / 1e6:.0f} GB/s (median), {nbytes / best / 1e6:.0f} GB/s (min); "
          "source 154 MB + output 615 MB exceed the 126 MB L2")

    # 2. the reference's torch expressions on the same card, same draws
    padded = reference_setup(u8, mean_t, std_t, preflip)
    setup_med, _ = event_times(lambda: reference_setup(u8, mean_t, std_t, preflip), max(5, args.reps // 5))
    ref_med, ref_best = event_times(lambda: reference_epoch(padded, labels, shifts, True, perm), max(5, args.reps // 5))
    ref = reference_epoch(padded, labels, shifts, True, perm)
    x, t = kernel()
    nb = N // BS
    same = torch.equal(torch.cat([b for b, _ in ref]), x[:nb * BS]) and torch.equal(torch.cat([l for _, l in ref]), t[:nb * BS])
    print(f"[reference torch] epoch-0 setup (normalise, pre-flip, pad): median {setup_med:.3f} ms; per epoch (crop over "
          f"{(2 * R + 1) ** 2} shifts, flip, {nb} batch gathers): median {ref_med:.3f} ms, min {ref_best:.3f} ms; "
          f"kernel speed-up per epoch {ref_med / med:.1f}x; batches bit-identical to tp_cifar_epoch: {same}")
    if not same:
        raise SystemExit("tp_cifar_epoch differs from the reference's torch expressions")
    del padded, ref, x, t

    # 3. ResNet-18 / CIFAR-10 epochs through the harness: real loader on a generated full-size set vs synthetic
    with tempfile.TemporaryDirectory() as tmp:
        os.makedirs(os.path.join(tmp, "cifar10"))
        gt = torch.Generator().manual_seed(2)
        for split, n in (("train", N), ("test", NTEST)):
            torch.save({"images": torch.randint(0, 256, (n, H, W, C), dtype=torch.uint8, generator=gt),
                        "labels": torch.randint(0, 10, (n,), generator=gt), "classes": [str(k) for k in range(10)]},
                       os.path.join(tmp, "cifar10", f"CIFAR10_{split}.pt"))
        loader = ds.CifarLoader(tmp, train=True, batch_size=BS, aug={"flip": True, "translate": 2}, altflip=True, device=dev)
        it_med, _ = event_times(lambda: [b for b in loader], max(5, args.reps // 5))
        print(f"[CifarLoader] one train epoch iterated (draws + tp_cifar_epoch + {len(loader)} slices): median {it_med:.3f} ms")
        del loader
        rows = []
        for tag, ov in (("real", ["dataset_params.dataloader_type=torch", f"+dataset_params.data_root_dir={tmp}"]),
                        ("synthetic", [f"dataset_params.synthetic_steps_per_epoch={N // BS}"])):
            kind, ts = harness_epoch_times(ov, os.path.join(tmp, "ex"), args.train_epochs)
            rows.append((tag, kind, ts))
            print(f"[train_epoch {tag}] ResNet-18 bf16, batch {BS}, {N // BS} steps, loader {kind}: "
                  f"{', '.join(f'{v:.1f}' for v in ts)} ms (median {statistics.median(ts):.1f} ms)")
        real, syn = statistics.median(rows[0][2]), statistics.median(rows[1][2])
        print(f"[loader share] real - synthetic = {real - syn:.1f} ms per epoch ({100 * (real - syn) / real:.1f} % of the real-data epoch)")


if __name__ == "__main__":
    main()
