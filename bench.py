#!/usr/bin/env python
"""Headline benchmark: images/sec of the masked data-parallel train step, ResNet-50 @ 80 % unstructured
(ERK) sparsity, ImageNet-shaped synthetic data, bf16 autocast — BASELINE.json's metric and config.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference ...                      (the reference's CPU path = oracle port, host cores)

One "step" = one ``PruningHarness.train_step`` call over one batch (the product's own step, not a copy of it):
H2D (e2e only) -> zero_grad -> autocast forward through the sm_100a masked-conv kernels -> CE loss -> backward
(dgrad/wgrad kernels, mask fused in wgrad) -> P2P gradient mean over NVLink under the backward pass (N>1) -> fused SGD
-> LR scheduler step.  Nothing is skipped in the timed region.

Output: ONE JSON line (see the task contract): value = whole-job images/s with inputs resident in HBM,
e2e = the same through the public API with pinned-host inputs copied every step and the loss read back,
roofline = the masked implicit-GEMM kernels' achieved TFLOP/s (CUDA events on the launching stream, live in the
timed region) against the measured sustained bf16 peak, cpu_baseline = the oracle port timed on host cores.
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
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "images_per_sec_resnet50_erk80_train_step"
GFLOP_PER_IMG = 24.30           # SURVEY.md §8(d): fwd 8.178 + dgrad 7.942 + wgrad 8.178 (masked layers, dense)
ROOFLINE_IMG_S = 39.8e3         # SURVEY.md §8(d): per-layer max(tensor, HBM) masked-GEMM roofline per GPU


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf=d["bf16_tflops_sustained"], tf_burst=d["bf16_tflops"], src="measured")
    return dict(hbm=6650.0, tf=1400.0, tf_burst=1590.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []
        self.nv = []            # in-process NVML samples (sm MHz, max MHz, reasons bitmask): every 10 ms, so even a
        self._stop = False      # 0.2 s timed region (8 GPUs x batch 64) is sampled; nvidia-smi -lms stays as the fallback

    def _nvml_loop(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(self.index).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            while not self._stop:
                self.nv.append((pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM), mx,
                                int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))))
                time.sleep(0.01)
        except Exception:
            pass

    def start(self):
        try:
            self.tn = threading.Thread(target=self._nvml_loop, daemon=True); self.tn.start()
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True); self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        self._stop = True
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        if self.nv:
            # NVML throttle-reason bits: 0x4 sw_power_cap, 0x8 hw_slowdown, 0x20 sw_thermal_slowdown, 0x40 hw_thermal_slowdown
            bits = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
            sm_sorted = sorted(v[0] for v in self.nv)
            loaded = sm_sorted[len(sm_sorted) // 3:] or sm_sorted
            allbits = 0
            for v in self.nv:
                allbits |= v[2]
            return {"sm_mhz": float(statistics.median(loaded)), "sm_max_mhz": float(self.nv[0][1]),
                    "reasons": sorted(n for b, n in bits.items() if allbits & b), "samples": len(self.nv), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm_sorted = sorted(sm)
        loaded = sm_sorted[len(sm_sorted) // 3:] or sm_sorted       # drop idle samples at the edges
        return {"sm_mhz": statistics.median(loaded) if loaded else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_SAMPLE = 1 << 18           # --dump-outputs: elements kept per tensor (ResNet-50: 267 tensors, 35 MiB of float32)


def dump_outputs(out_dir, loss, model):
    """What the last timed step hands its caller: the loss ``train_step`` returned and the parameters / BatchNorm
    statistics it left in the model, as ``<out_dir>/<name>.npy`` (float32; float64 stays float64).  A tensor of more
    than DUMP_SAMPLE elements is flattened and sampled at positions drawn from a fixed seed, the same in every run."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss}
    arrays.update((k, v) for k, v in model.model.state_dict().items() if v.is_floating_point() and not k.endswith(".mask"))
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_SAMPLE, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        t = t.double() if t.dtype == torch.float64 else t.float()
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy())


def triangular_lr(total_steps, warmup_fraction=0.2):
    """LR multiplier schedule of the reference (utils/schedulers.py:79-117): interp [0.2, 1, 0]."""
    import numpy as np
    return np.interp(np.arange(1 + total_steps), [0, int(warmup_fraction * total_steps), total_steps], [0.2, 1, 0])


def host_threads():
    """Thread count of the CPU arm: set explicitly (torchrun exports OMP_NUM_THREADS=1, and torch's default differs
    between boxes), physical cores = logical CPUs // 2, capped at 64."""
    n = os.cpu_count() or 2
    return max(1, min(64, n // 2))


def cpu_train_step_rate(batch, steps, warmup, threads=None):
    """The reference's CPU path (oracle port): RN50 ERK-80 train step, bf16 autocast, on host cores."""
    import torch
    import oracle.model as om
    from oracle import prune as OP
    from oracle.train import train_step
    torch.set_num_threads(threads or host_threads())
    torch.manual_seed(0)
    net = om.build("resnet50", "imagenet")
    torch.manual_seed(1)
    probs = OP.erk_keep_probabilities([tuple(m.weight.shape) for _, m in om.masked_layers(net)], 0.2)
    om.set_er_masks(net, probs)
    opt = torch.optim.SGD(net.parameters(), lr=0.2, momentum=0.9, weight_decay=1e-4)
    g = torch.Generator().manual_seed(2)
    x = torch.randn(batch, 3, 224, 224, generator=g); t = torch.randint(0, 1000, (batch,), generator=g)
    net.train()
    for _ in range(warmup):
        train_step(net, opt, x, t)
    t0 = time.perf_counter()
    for _ in range(steps):
        train_step(net, opt, x, t)
    dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ.pop("OMP_NUM_THREADS", None)          # torchrun sets it to 1 for every rank; the CPU arm owns the box
    batch = 16
    steps = max(1, min(args.steps, 40))
    warm = max(3, min(args.warmup, 3))
    rate, s_per_step, threads = cpu_train_step_rate(batch, steps, warm, host_threads())
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "images/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": s_per_step * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "resnet50 imagenet-shape ERK-80% masked train step (reference CPU path, oracle port)",
                   "global_batch": batch, "sample": f"batch {batch} per step on host cores", "threads": threads},
        "cpu_baseline": {"value": rate, "unit": "images/s", "cores": threads, "kind": "port",
                         "sample": f"{steps} steps of batch {batch} after {warm} warm-up steps (torch CPU, bf16 autocast), "
                                   f"torch.set_num_threads({threads}), os.cpu_count()={os.cpu_count()}"},
        "e2e": {"value": rate, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def gpu_eager_reference(dev, B, steps, world):
    """The kernels to beat (BASELINE.md §5): the reference's own GPU execution model — cuDNN convs on mask*w, ATen
    BatchNorm / ReLU, torch.optim.SGD under bf16 autocast (the oracle's module graph moved to cuda), ATen kthvalue on
    the concatenated scores (pruning_utils.py:75-79), NCCL all_reduce of the 102 MB gradient (world > 1)."""
    import torch
    import torch.distributed as dist
    from oracle import model as OM, prune as OP
    out = {}
    torch.manual_seed(0)
    ref = OM.build("resnet50", "imagenet")
    probs = OP.erk_keep_probabilities([tuple(m.weight.shape) for _, m in OM.masked_layers(ref)], 0.2)
    torch.manual_seed(1)
    OM.set_er_masks(ref, probs)
    ref = ref.to(dev).to(memory_format=torch.channels_last).train()
    opt = torch.optim.SGD(ref.parameters(), lr=0.2, momentum=0.9, weight_decay=1e-4)
    g = torch.Generator(device=dev).manual_seed(2)
    x = torch.randn(B, 3, 224, 224, device=dev, generator=g).contiguous(memory_format=torch.channels_last)
    t = torch.randint(0, 1000, (B,), device=dev, generator=g)
    prev = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True

    def ref_step():
        opt.zero_grad()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = torch.nn.functional.cross_entropy(ref(x), t)
        loss.backward()
        opt.step()
    for _ in range(3):
        ref_step()
    torch.cuda.synchronize(dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        ref_step()
    b.record(); torch.cuda.synchronize(dev)
    ms = a.elapsed_time(b) / steps
    out["cudnn_eager_train_step"] = {"ms_per_step": ms, "images_per_s": B / ms * 1e3, "batch": B,
                                     "what": "F.conv2d(x, mask*w) on cuDNN + ATen BN/ReLU + torch.optim.SGD, bf16 autocast, channels_last, cudnn.benchmark"}
    # ATen kthvalue + where on the same 25.5 M scores (reference prune_mag, pruning_utils.py:73-87)
    layers = [m for _, m in OM.masked_layers(ref)]
    n = sum(m.weight.numel() for m in layers); k = int((1 - 0.2) * n)
    ones = [torch.ones_like(m.weight) for m in layers]

    def aten_prune():
        scores = torch.cat([(mk * m.weight).detach().abs().flatten() for m, mk in zip(layers, ones)])
        thr, _ = torch.kthvalue(scores, k)
        return [torch.where((mk * m.weight).detach().abs() <= thr, 0.0, 1.0) for m, mk in zip(layers, ones)]
    aten_prune(); torch.cuda.synchronize(dev)
    ts = []
    for _ in range(3):
        a.record(); aten_prune(); b.record(); torch.cuda.synchronize(dev)
        ts.append(a.elapsed_time(b))
    out["aten_prune_mag"] = {"us": statistics.median(ts) * 1e3, "elements": n,
                             "GBps_on_12B_per_elem": 12.0 * n / (statistics.median(ts) / 1e3) / 1e9,
                             "what": "per-layer abs(mask*w), torch.cat, torch.kthvalue, per-layer torch.where"}
    del ref, opt, layers, ones
    torch.backends.cudnn.benchmark = prev
    torch.cuda.empty_cache()
    if world > 1:
        buf = torch.randn(25_557_032, device=dev)
        for _ in range(3):
            dist.all_reduce(buf)
        torch.cuda.synchronize(dev); dist.barrier()
        a.record()
        for _ in range(10):
            dist.all_reduce(buf)
        b.record(); torch.cuda.synchronize(dev)
        us = torch.tensor([a.elapsed_time(b) / 10 * 1e3], device=dev)
        dist.all_reduce(us, op=dist.ReduceOp.MAX)
        out["nccl_allreduce_102MB"] = {"us": float(us.item()), "busbw_GBps": 2 * 25_557_032 * 4 * (world - 1) / world / (float(us.item()) / 1e6) / 1e9}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--global-batch", type=int, default=512, help="reference semantics: total_batch_size split over ranks")
    ap.add_argument("--per-gpu-batch", type=int, default=0, help="override: fixed per-GPU batch (weak scaling)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-topk", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the cuDNN / ATen / NCCL 'kernels to beat' sub-record")
    ap.add_argument("--no-graph", action="store_true", help="do not capture the train step into a CUDA graph")
    ap.add_argument("--no-overlap", action="store_true", help="launch the gradient exchange after the backward pass")
    ap.add_argument("--no-wgrad-side-stream", action="store_true", help="keep the weight-gradient GEMMs on the compute stream")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last timed step's loss and the "
                    "model state it left as DIR/<name>.npy (same arguments, same inputs: compares two builds)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import tempfile
    import torch
    import torch.distributed as dist
    from turboprune_b200 import ops
    from turboprune_b200.harness_definitions.standard_pruning_harness import PruningHarness
    from turboprune_b200.utils import config as tp_config, custom_models as cm, pruning_utils as pu
    from turboprune_b200.utils.dataset import DevicePrefetcher, SyntheticLoader

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(3, args.warmup)
    K = args.steps
    B = args.per_gpu_batch or max(1, args.global_batch // world)
    scaling = "weak" if args.per_gpu_batch else "strong"
    use_graph = not args.no_graph

    # ---- BASELINE.json config 2 through the product surface: the composed config, TorchVisionModel, prune_er_erk,
    # ---- PruningHarness (its train_step owns gradient arena / weight shadow / P2P reducer / CUDA graph) ----
    total_steps = 3 * (W + K) + 16
    cfg = tp_config.compose("synthetic_rn50_erk80", [
        f"dataset_params.total_batch_size={B * world}", f"dataset_params.synthetic_steps_per_epoch={total_steps}",
        "+dataset_params.synthetic_fresh=true", "optimizer_params.weight_decay=1e-4",
        f"experiment_params.distributed={'true' if world > 1 else 'false'}",
        f"+experiment_params.cuda_graph={'true' if use_graph else 'false'}",
        f"+experiment_params.wgrad_side_stream={'false' if args.no_wgrad_side_stream else 'true'}",
        f"experiment_params.base_dir={tempfile.gettempdir()}"], os.path.join(ROOT, "conf_b200"))
    torch.manual_seed(0)
    model = cm.TorchVisionModel(cfg)             # seed-0 ResNet-50
    torch.manual_seed(1)
    pu.prune_er_erk(model, 0.2)                  # ERK-80 % Bernoulli masks (identical on every rank by construction)
    harness = PruningHarness(cfg=cfg, gpu_id=rank, expt_dir=("bench", tempfile.gettempdir()), model=model)
    model = harness.model
    model.train()
    sparsity = model.get_overall_sparsity()
    harness._setup_optimizer()
    harness._setup_scheduler(1)                  # TriangularSchedule over total_steps, stepped per iteration like train_epoch
    if harness.distributed and args.no_overlap:
        harness._ensure_reducer(); harness.reducer.overlap = False
    loss_acc = torch.zeros((), device=dev)
    batches = iter(harness.train_loader)         # fresh Philox batch per step, generated on the device

    def step(batch):
        out = harness.train_step(batch)["loss"]
        harness.scheduler.step()
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(nsteps, fn):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(nsteps):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- warm-up: W steps through harness.train_step (the third one captures the CUDA graph) ----
    l0 = ops.launch_count()
    step(next(batches))
    launches_per_step = ops.launch_count() - l0  # kernel-launching C-ABI calls of one (eager) step; the graph replays the same kernels
    for i in range(max(W, 4) - 1):
        step(next(batches))
    assert (harness._graph is not None) == use_graph

    # ---- device-resident run (value) ----
    clocks = ClockSampler(local_rank); clocks.start()

    last_loss = [None]

    def dev_step(i):
        last_loss[0] = step(next(batches))
        loss_acc.add_(last_loss[0])
    ms_total = timed(K, dev_step)
    launches = launches_per_step * K
    clk = clocks.stop()
    if harness.reducer is not None:
        harness.reducer.check_status()
    img_s = world * B * K / (ms_total / 1e3)
    if args.dump_outputs and rank == 0:             # before the eager / e2e steps below train the model further
        dump_outputs(args.dump_outputs, last_loss[0], model)

    # ---- per-kernel timing of the masked GEMMs: CUDA events around every C-ABI conv call on the launching stream
    # (eager steps of the same workload through the same harness — events cannot be read back from inside a replayed graph) ----
    timer = ops.KernelTimer()
    KT = min(K, 5)
    cfg.experiment_params["cuda_graph"] = False
    side_wgrad = cfg.experiment_params.get("wgrad_side_stream", True)
    cfg.experiment_params["wgrad_side_stream"] = False      # per-kernel durations: every GEMM alone on the device, on ONE stream
    ops.set_timer(timer)
    ms_eager = timed(KT, lambda i: step(next(batches)))
    ops.set_timer(None)
    cfg.experiment_params["cuda_graph"] = use_graph
    cfg.experiment_params["wgrad_side_stream"] = side_wgrad
    tot = timer.totals()
    gemm_ms = sum(v[0] for v in tot.values()) * (K / KT)
    pk = peaks()
    flops = GFLOP_PER_IMG * 1e9 * B * K
    achieved_tf = flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    # Algorithmic bytes of the masked convs/linears (SURVEY.md §8(d): bf16 activations in + out per op):
    # fprop x+y, dgrad dy+dx (the stem has no dgrad), wgrad x+dy.  Shapes taken from the live model.
    io = {}
    hooks = []
    for name, m in model._masked():
        hooks.append(m.register_forward_hook(lambda mod, inp, out, name=name: io.__setitem__(name, (inp[0].numel(), (out[0] if isinstance(out, tuple) else out).numel()))))
    probe = torch.randn(2, 3, 224, 224, device=dev).contiguous(memory_format=torch.channels_last)
    model.eval()
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        model(probe)
    model.train()
    for h in hooks:
        h.remove()
    first = next(iter(io))
    per_img = sum(3 * (a + b) for a, b in io.values()) - sum(io[first])          # elements per 2 images
    alg_bytes_step = 2.0 * per_img / 2 * B
    achieved_gbs = alg_bytes_step * K / (gemm_ms / 1e3) / 1e9 if gemm_ms > 0 else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_igemm_traffic.json")
    if not os.path.isfile(tpath):
        tpath = os.path.join(ROOT, "profiles", "r01_igemm_traffic.json")
    if os.path.isfile(tpath) and B == 512:
        traffic = json.load(open(tpath))["dram_bytes_per_launch"]
    n_launch = sum(v[2] for v in tot.values()) / KT
    roofline = {"bound": "hbm", "achieved": achieved_gbs, "peak": pk["hbm"], "unit": "GB/s",
                "frac": achieved_gbs / pk["hbm"], "traffic": traffic,
                "traffic_note": f"dram read+write per igemm kernel launch, ncu over one eager step at B=512 ({os.path.relpath(tpath, ROOT)})" if traffic else None,
                "peak_source": pk["src"] + " HBM copy bandwidth",
                "kernel": "k_igemm_fwd (fprop+dgrad) / k_igemm_wgrad — masked implicit GEMM, tcgen05 + TMA",
                "why_hbm": "sum over the 54 layers: conv I/O bytes / HBM peak (11.4 ms at B=512) exceeds FLOPs / tensor peak (8.5 ms); 30 of 54 layers are HBM-bound",
                "algorithmic_bytes_per_step": alg_bytes_step, "algorithmic_bytes_per_launch": alg_bytes_step / n_launch,
                "launches_per_step": n_launch,
                "timing": f"CUDA events around each masked-GEMM C-ABI call over {KT} eager harness.train_step calls ({ms_eager / KT:.2f} ms/step eager); step rate from the harness's CUDA-graph replay" if use_graph else "CUDA events, eager",
                "ms_per_step_in_kernel": gemm_ms / K,
                "by_op_ms_per_step": {k: v[0] / KT for k, v in tot.items()},
                "share_of_step": gemm_ms / ms_total,
                "tensor": {"achieved_tflops": achieved_tf, "peak_tflops": pk["tf"], "frac": achieved_tf / pk["tf"],
                           "flops_per_step": GFLOP_PER_IMG * 1e9 * B, "peak_source": pk["src"] + " sustained bf16"},
                "frac_of_masked_gemm_roofline_img_s": (img_s / world) / ROOFLINE_IMG_S}

    # ---- end-to-end run: pinned host batches -> DevicePrefetcher (copy stream, double-buffered) -> harness.train_step,
    # ---- loss read back every step like the reference's loss.item() (base_harness.py:134) ----
    e2e = None
    if not args.no_e2e:
        hg = torch.Generator().manual_seed(7 + rank)
        hpool = [(torch.randn(B, 224, 224, 3, generator=hg).pin_memory().permute(0, 3, 1, 2),
                  torch.randint(0, 1000, (B,), generator=hg).pin_memory()) for _ in range(2)]
        h2d = hpool[0][0].numel() * 4 + hpool[0][1].numel() * 8

        class HostLoader:
            def __init__(self, n): self.n = n
            def __len__(self): return self.n
            def __iter__(self):
                for i in range(self.n):
                    yield hpool[i % 2]

        def run_e2e(n):
            for batch in DevicePrefetcher(HostLoader(n), dev):
                float(step(batch).item())
        run_e2e(2)
        torch.cuda.synchronize(dev)
        ms_e2e = timed(1, lambda i: run_e2e(K))
        e2e = {"value": world * B * K / (ms_e2e / 1e3), "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
               "ms_per_step": ms_e2e / K, "api": "DevicePrefetcher(pinned host batches) -> PruningHarness.train_step -> loss.item()"}

    # ---- mask top-k (second half of the metric): prune_mag over the model's 25.5 M masked weights, and the
    # ---- VGG-16-sized SynFlow select (134.7 M elements, 16 B/elem) ----
    topk = None
    if not args.no_topk and rank == 0:
        def time_plan(plan, k, reps=10, clean=False):
            for _ in range(3):
                plan.run(k)
            flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)
            other = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device=dev) if clean else None
            tms, info = [], None
            for _ in range(reps):
                flush.zero_()                                  # 256 MiB write: evicts the 126 MB L2
                if clean:                                      # ... and leaves it full of DIRTY lines whose write-back competes with the
                    other.sum()                                # timed kernel for DRAM; reading another 256 MiB leaves clean, unrelated lines
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); plan.enqueue(k); b.record(); torch.cuda.synchronize(dev)
                tms.append(a.elapsed_time(b))
                _, _, info = plan.finish(k)                    # status read-back (+ exact fallback if the bracket missed)
                if info["path"] != 0:                          # fast path did not hold: the honest time includes the fallback
                    a.record(); plan.run(k); b.record(); torch.cuda.synchronize(dev)
                    tms[-1] = a.elapsed_time(b)
            del flush, other
            return statistics.median(tms), info
        layers = [m for _, m in model._masked()]
        ws = [m.weight.detach() for m in layers]; ms_ = [torch.ones_like(m.mask) for m in layers]
        n = sum(w.numel() for w in ws); k = int((1 - 0.2) * n)
        tmed, info = time_plan(ops.TopKPlan(ws, ms_), k)      # pointer tables marshalled once: the timed call is the C-ABI call
        gbs = 12.0 * n / (tmed / 1e3) / 1e9
        tclean, _ = time_plan(ops.TopKPlan(ws, ms_), k, clean=True)
        topk = {"metric": "mask_topk_GBps", "elements": n, "k": k, "algorithmic_bytes": 12 * n, "ms": tmed, "GBps": gbs,
                "roofline": {"bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"], "traffic": None},
                "path": info["path"], "candidates": info["candidates"], "l2": "flushed between reps (256 MiB write: the L2 is full of dirty lines when the timed call starts)",
                "clean_l2": {"ms": tclean, "GBps": 12.0 * n / (tclean / 1e3) / 1e9, "frac": 12.0 * n / (tclean / 1e3) / 1e9 / pk["hbm"],
                             "how": "same, plus a 256 MiB read of another buffer after the flush: the L2 holds clean unrelated lines"},
                "timed": "tp_topk_enqueue: one memset + one cooperative kernel (sample, bracket, sweep, resolve, patch); the 100-byte status read-back (tp_topk_finish) follows outside the events"}
        del ms_
        n2, nseg = 134_657_728, 16
        sizes = [n2 // nseg] * (nseg - 1); sizes.append(n2 - sum(sizes))
        g2 = torch.Generator(device=dev).manual_seed(11)
        w2 = [torch.randn(s_, device=dev, generator=g2).abs_() * 0.02 for s_ in sizes]
        gr2 = [torch.randn(s_, device=dev, generator=g2) * 1e-3 for s_ in sizes]
        m2 = [torch.ones(s_, device=dev) for s_ in sizes]
        t2, info2 = time_plan(ops.TopKPlan(w2, m2, gs=gr2, kind=2), int(0.95 * n2), reps=5)
        gbs2 = 16.0 * n2 / (t2 / 1e3) / 1e9
        topk["synflow_vgg16_size"] = {"elements": n2, "k": int(0.95 * n2), "algorithmic_bytes": 16 * n2, "ms": t2, "GBps": gbs2,
                                      "frac_of_hbm_peak": gbs2 / pk["hbm"], "path": info2["path"], "candidates": info2["candidates"]}
        del w2, gr2, m2
        torch.cuda.empty_cache()

    gpu_eager = None
    if not args.no_gpu_eager:
        try:
            gpu_eager = gpu_eager_reference(dev, B, min(K, 5), world)
        except Exception as e:           # the comparison arm must never take the bench line down
            gpu_eager = {"error": repr(e)[:200]}
        if gpu_eager and "cudnn_eager_train_step" in gpu_eager:
            gpu_eager["speedup_vs_cudnn_eager"] = gpu_eager["cudnn_eager_train_step"]["ms_per_step"] / (ms_total / K)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rate, s_per_step, threads = cpu_train_step_rate(16, 6, 2, host_threads())
        cpu = {"value": rate, "unit": "images/s", "cores": threads, "kind": "port",
               "sample": f"6 steps of batch 16 of the same workload after 2 warm-up steps (oracle port, torch CPU bf16 autocast, {s_per_step:.2f} s/step), "
                         f"torch.set_num_threads({threads}), os.cpu_count()={os.cpu_count()}"}

    # data-parallel invariant: after all these steps every rank holds bit-identical weights (same seed, bit-identical
    # gradient mean, deterministic kernels) — one checksum per rank, compared
    replicas_identical = None
    if world > 1:
        with torch.no_grad():
            mine = torch.stack([p.detach().double().sum() for p in model.parameters()]).sum().reshape(1)
        allv = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allv, mine)
        replicas_identical = all(torch.equal(allv[0], v) for v in allv)
    if rank == 0:
        line = {
            "metric": METRIC, "value": img_s, "unit": "images/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "resnet50 imagenet-shape [B,3,224,224] ERK-80% unstructured masks, SGD(0.9, wd 1e-4), CE loss, TriangularSchedule",
                       "global_batch": B * world, "per_gpu_batch": B, "parallelism": f"dp{world}",
                       "api": "PruningHarness.train_step (conf_b200/synthetic_rn50_erk80.yaml)",
                       "inputs": "fresh Philox batch generated on the device every step (generation inside the timed region)",
                       "sparsity_percent": sparsity, "cuda_graph": bool(use_graph), "l2": "inputs (308 MB/batch at B=512) and activations exceed the 126 MB L2",
                       "grad_exchange": "none (1 GPU)" if world == 1 else
                       ("tp_p2p_allreduce over symmetric memory (NVLink), per-bucket on a side stream under the backward pass, mask applied in the kernel; no NCCL on the data path"
                        + ("" if not args.no_overlap else " [overlap disabled]"))},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clk,
            "topk": topk, "reference_gpu_eager": gpu_eager, "loss_mean": float(loss_acc.item()) / K,
            "replicas_identical": replicas_identical,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
