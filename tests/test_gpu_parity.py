"""GPU (B200) parity tests: every call goes through the C-ABI; the checker is the oracle / golden fixtures.

Bars: pruning = bit-exact masks and thresholds; masked conv/linear = bf16 tensor-core arithmetic with fp32
accumulation, compared with the oracle evaluated on the same bf16-rounded operands: forward / dX outputs are
bf16 (rel. error <= 2^-8 of the tensor's max), dW / db are fp32 (<= 1e-4); losses <= 1e-3 relative
(BASELINE.json north_star)."""
import hashlib
import json
import ctypes
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")


def _rel(a, b):
    a = a.detach().float().cpu(); b = b.detach().float().cpu()
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device: the gpu-marked parity tests run on the B200 box")
    from turboprune_b200 import _cabi
    _cabi.load()          # fails loudly if the extension is missing
    return torch.device("cuda", 0)


# ---------------------------------------------------------------- pruning -----------------------------------
def _run_prune(ws, ms, k, gs=None, kind=0):
    from turboprune_b200 import ops
    from oracle import prune as P
    tw = [torch.from_numpy(w).cuda() for w in ws]; tm = [torch.from_numpy(m).cuda() for m in ms]
    tg = None if gs is None else [torch.from_numpy(g).cuda() for g in gs]
    outs, thr, info = ops.topk_threshold_mask(tw, tm, k, gs=tg, kind=kind)
    sc = P.layer_scores(ws, ms, gs, kind)
    ref_thr = P.kth_smallest(np.concatenate([s.ravel() for s in sc]), k)
    ref = [P.apply_threshold(s, ref_thr) for s in sc]
    got_thr = np.float32(thr.item())
    assert (np.isnan(ref_thr) and np.isnan(got_thr)) or got_thr.view(np.uint32) == np.float32(ref_thr).view(np.uint32)
    for o, r in zip(outs, ref):
        assert np.array_equal(o.cpu().numpy(), r)
    return info


def test_topk_bit_exact_vs_oracle(dev):
    rng = np.random.RandomState(0)
    sizes = [1, 1000, 4096 * 3 + 17, 300000, 1_000_003]          # ragged, unaligned tails, single element
    ws = [rng.randn(n).astype(np.float32) * 0.05 for n in sizes]
    ones = [np.ones(n, np.float32) for n in sizes]
    half = [(rng.rand(n) < 0.5).astype(np.float32) for n in sizes]
    gs = [rng.randn(n).astype(np.float32) * 1e-3 for n in sizes]
    N = sum(sizes)
    for k in (1, 2, int(0.2 * N), int(0.9 * N), N - 1, N):
        _run_prune(ws, ones, k)
    _run_prune(ws, half, int(0.6 * N))                            # tie-heavy: half the scores are exact zeros
    _run_prune(ws, half, int(0.3 * N))                            # threshold inside the zeros
    _run_prune(ws, half, int(0.7 * N), gs=gs, kind=1)
    _run_prune(ws, half, int(0.7 * N), gs=gs, kind=2)


def test_topk_adversarial_inputs(dev):
    rng = np.random.RandomState(1)
    n = 500_000
    ones = [np.ones(n, np.float32)]
    info = _run_prune([np.full(n, 0.3, np.float32)], ones, n // 2)                # all equal (not a bin edge)
    _run_prune([np.zeros(n, np.float32)], ones, n // 3)                            # all zero
    w = rng.randn(n).astype(np.float32); w[:1000] = np.nan; w[1000:1100] = np.inf; w[1100:1200] = 1e-42   # NaN, inf, subnormals
    _run_prune([w], ones, n - 50)                                                  # NaN threshold -> masks all ones
    _run_prune([w], ones, n // 2)
    _run_prune([np.sort(rng.randn(n).astype(np.float32))], ones, n // 5)          # sorted input (sampling stress)
    _run_prune([-np.abs(w[1200:])], [np.ones(n - 1200, np.float32)], 17)          # negative weights, -0.0 handled by |.|


def test_topk_k_out_of_range_raises(dev):
    from turboprune_b200 import ops
    w = [torch.randn(100, device=dev)]; m = [torch.ones(100, device=dev)]
    with pytest.raises(RuntimeError):
        ops.topk_threshold_mask(w, m, 0)          # the reference raises here too (pruning_utils.py:78-79)
    with pytest.raises(RuntimeError):
        ops.topk_threshold_mask(w, m, 101)


def test_topk_full_size_properties(dev):
    """ResNet-50 / VGG-16 sized inputs (too big for the numpy oracle in seconds): size-independent properties."""
    from turboprune_b200 import ops
    for n, nseg in ((25_502_912, 54), (134_657_728, 16)):
        g = torch.Generator(device=dev).manual_seed(n % 1000)
        sizes = [n // nseg] * (nseg - 1); sizes.append(n - sum(sizes))
        ws = [torch.randn(s, device=dev, generator=g) * 0.03 for s in sizes]
        ms = [torch.ones(s, device=dev) for s in sizes]
        k = int((1 - 0.2) * n)
        outs, thr, info = ops.topk_threshold_mask(ws, ms, k)
        flat = torch.cat([w.abs() for w in ws])
        assert thr == torch.kthvalue(flat, k)[0]                                   # same order statistic as ATen
        zeros = sum(int((o == 0).sum()) for o in outs)
        assert zeros == int((flat <= thr).sum()) and zeros >= k
        cz = ops.count_zeros(outs).tolist()
        assert cz[-1] == zeros
        # idempotence: pruning the pruned model to the same density changes nothing
        outs2, thr2, _ = ops.topk_threshold_mask(ws, outs, k)
        assert all(torch.equal(a, b) for a, b in zip(outs, outs2))
        del flat, ws, ms, outs, outs2


def test_prune_small_net_matches_reference_fixture(dev):
    """prune_mag / snip on the small conv net of the golden fixture through the product's pruning_utils."""
    z = np.load(os.path.join(G, "prune_small.npz"))
    from turboprune_b200 import ops, _cabi
    ws = [torch.from_numpy(z[f"w{i}"]).cuda() for i in range(4)]
    ms = [torch.ones_like(w) for w in ws]
    for lvl, d in enumerate([0.8, 0.64, 0.3]):
        n = sum(w.numel() for w in ws); k = int((1 - d) * n)
        ms, thr, _ = ops.topk_threshold_mask(ws, ms, k)
        for i in range(4):
            assert np.array_equal(ms[i].cpu().numpy(), z[f"mag{lvl}.m{i}"])
    gs = [torch.from_numpy(z[f"snip.g{i}"]).cuda() for i in range(4)]
    n = sum(w.numel() for w in ws)
    new, _, _ = ops.topk_threshold_mask(ws, [torch.ones_like(w) for w in ws], int(0.5 * n), gs=gs, kind=_cabi.TP_SCORE_SNIP)
    for i in range(4):
        assert np.array_equal(new[i].cpu().numpy(), z[f"snip.m{i}"])
    # SynFlow: |w| and the gradients captured from the running reference just before its model.zero_grad()
    aw = [torch.from_numpy(z[f"synflow.absw{i}"]).cuda() for i in range(4)]
    gs = [torch.from_numpy(z[f"synflow.g{i}"]).cuda() for i in range(4)]
    new, _, _ = ops.topk_threshold_mask(aw, [torch.ones_like(w) for w in aw], int(0.5 * n), gs=gs, kind=_cabi.TP_SCORE_SYNFLOW)
    for i in range(4):
        assert np.array_equal(new[i].cpu().numpy(), z[f"synflow.m{i}"])


def test_imp_levels_hashes_match_reference(dev):
    """Seed-0 ResNet-18/CIFAR-10 through the product wrappers: IMP levels reproduce the reference's mask hashes."""
    import refshim
    from turboprune_b200.utils import custom_models as cm, pruning_utils as pu
    h = json.load(open(os.path.join(G, "imp_hashes.json")))
    torch.manual_seed(0)
    model = cm.TorchVisionModel(refshim.make_cfg("resnet18", "cifar10"))
    layers = [m for _, m in model._masked()]
    hh = hashlib.sha256()
    for m in layers:
        hh.update(m.weight.detach().numpy().tobytes())
    if hh.hexdigest() != h["weights_sha256"]:
        pytest.skip("torch initialisation stream differs from the fixture's (other torch build)")
    model = model.cuda()
    density = 1.0
    for lvl in h["levels"]:
        density *= 0.8
        pu.prune_mag(model, density)
        hm = hashlib.sha256()
        for m in layers:
            hm.update(m.mask.cpu().numpy().tobytes())
        assert hm.hexdigest() == lvl["masks_sha256"]
        assert abs(model.get_overall_sparsity() - lvl["sparsity_percent"]) < 1e-9


def test_random_and_er_criteria_match_reference_fixture(dev):
    """RNG-stream parity: Bernoulli (er_*) masks are drawn on the CPU model exactly like the reference."""
    z = np.load(os.path.join(G, "prune_small.npz"))
    from turboprune_b200.utils import mask_layers as ml, pruning_utils as pu
    import torch.nn as nn

    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.c1 = ml.ConvMask(in_channels=3, out_channels=8, kernel_size=3, padding=1, bias=True)
            self.bn = nn.BatchNorm2d(8)
            self.c2 = ml.ConvMask(in_channels=8, out_channels=16, kernel_size=3, stride=2, padding=1, bias=False)
            self.fc = ml.Conv1dMask(16, 10, bias=True)
            self.ln = ml.LinearMask(in_features=10, out_features=10, bias=True)
    torch.manual_seed(0)
    net = Net()
    layers = [net.c1, net.c2, net.fc, net.ln]
    for i, m in enumerate(layers):
        assert np.array_equal(m.weight.detach().numpy(), z[f"w{i}"])        # same init stream as the fixture
    # er_*: Bernoulli keep-masks drawn on the CPU model with seed 9, exactly as make_golden.py drove the reference
    # (set_er_mask keeps torch's generator: the RNG stream is part of mask parity, mask_layers.py:36-43)
    for tag, fn in (("er_erk", pu.prune_er_erk), ("er_bal", pu.prune_er_balanced)):
        torch.manual_seed(9)
        fn(net, 0.3)
        for i, m in enumerate(layers):
            assert np.array_equal(m.mask.numpy(), z[f"{tag}.m{i}"]), (tag, i)
    # the fixture drew rand_erk / rand_bal first (seed 7) and er_* afterwards (seed 9), each from fresh masks
    net_gpu = net.cuda()
    for tag, fn in (("rand_erk", pu.prune_random_erk), ("rand_bal", pu.prune_random_balanced)):
        for m in layers:
            m.mask = torch.ones_like(m.weight)
        torch.manual_seed(7)
        # the reference draws randn_like on the weight's device; the fixture was generated on CPU, so draw there
        noises = [torch.randn_like(m.weight.cpu()) for m in layers]
        fr = pu._erk_fracs(layers, 0.4)[1] if tag == "rand_erk" else pu._balanced_fracs(layers, 0.4)
        pu._per_layer_random(net_gpu, fr, [nz.cuda() for nz in noises])
        for i, m in enumerate(layers):
            assert np.array_equal(m.mask.cpu().numpy(), z[f"{tag}.m{i}"]), (tag, i)


# ---------------------------------------------------------------- masked operators ---------------------------
@pytest.mark.parametrize("name", ["conv3x3", "conv3x3s2", "conv1x1s2", "conv7x7s2"])
def test_small_golden_convs(dev, name):
    """Tiny odd-shaped cases from the reference fixture (channel counts far below a tile: padding paths)."""
    z = np.load(os.path.join(G, "ops_small.npz"))
    from turboprune_b200.utils import mask_layers as ml
    from oracle import mask_ops as R
    s, p = (int(v) for v in z[f"{name}.cfg"])
    x, w, m, dy = (torch.from_numpy(z[f"{name}.{k}"]) for k in ("x", "w", "m", "dy"))
    cout, cin, kh, kw = w.shape
    layer = ml.ConvMask(in_channels=cin, out_channels=cout, kernel_size=kh, stride=s, padding=p, bias=f"{name}.b" in z).cuda()
    with torch.no_grad():
        layer.weight.copy_(w); layer.mask.copy_(m)
        if layer.bias is not None:
            layer.bias.copy_(torch.from_numpy(z[f"{name}.b"]))
    xg = x.cuda()
    y = layer(xg)
    b = torch.from_numpy(z[f"{name}.b"]) if layer.bias is not None else None
    yr = R.masked_conv2d(x, w, m, b, s, p, bf16_operands=True)
    assert _rel(y, yr) < 4e-3
    y.backward(dy.cuda().to(y.dtype))
    _, dwr, dbr = R.masked_conv2d_grads(x, w, m, dy, s, p, bf16_operands=True, has_bias=b is not None)
    assert _rel(layer.weight.grad, dwr) < 1e-4
    assert bool((layer.weight.grad[layer.mask == 0] == 0).all())
    if b is not None:
        assert _rel(layer.bias.grad, dbr) < 1e-4


CASES = [  # n, h, w, cin, cout, k, stride, pad, bias
    (2, 8, 8, 64, 64, 1, 1, 0, False), (3, 7, 7, 128, 256, 1, 1, 0, True), (2, 14, 14, 128, 128, 3, 1, 1, False),
    (2, 14, 14, 128, 128, 3, 2, 1, True), (2, 14, 14, 256, 512, 1, 2, 0, False), (3, 7, 7, 512, 512, 3, 1, 1, False),
    (5, 9, 11, 64, 192, 3, 1, 1, False), (2, 15, 15, 64, 64, 3, 2, 1, False),
    # input channels that are not a TMA-friendly multiple (the reference wraps ANY nn.Conv2d): zero-padded to 64 / 8
    (2, 9, 9, 16, 24, 3, 1, 1, True), (2, 10, 10, 12, 20, 3, 2, 1, False), (3, 8, 8, 24, 40, 1, 1, 0, False),
    (2, 8, 8, 3, 16, 3, 1, 1, False), (2, 7, 7, 100, 72, 3, 1, 1, False), (2, 6, 6, 20, 16, 1, 2, 0, True),
    # a partial last M tile (980 pixels), a stride-2 3x3 with a partial N tile (Cout 96), N = 1000
    (5, 14, 14, 64, 64, 3, 1, 1, False), (3, 20, 20, 128, 512, 1, 1, 0, False), (4, 16, 16, 64, 96, 3, 2, 1, False),
    (2, 9, 9, 256, 1000, 1, 1, 0, False),
]


@pytest.mark.parametrize("case", CASES)
def test_masked_conv_fwd_bwd_vs_oracle(dev, case):
    n, h, w, cin, cout, k, s, p, bias = case
    from turboprune_b200 import ops
    from oracle import mask_ops as R
    g = torch.Generator().manual_seed(sum(case[:8]))
    x = torch.randn(n, cin, h, w, generator=g).to(torch.bfloat16)
    wt = torch.randn(cout, cin, k, k, generator=g) / (cin * k * k) ** 0.5
    mk = (torch.rand(cout, cin, k, k, generator=g) < 0.3).float()
    b = torch.randn(cout, generator=g) if bias else None
    xg = x.cuda().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    wg = wt.cuda().requires_grad_(True)
    bg = b.cuda().requires_grad_(True) if bias else None
    y = ops.masked_conv2d(xg, wg, mk.cuda(), bg, (s, s), (p, p))
    yr = R.masked_conv2d(x.float(), wt, mk, b, s, p, bf16_operands=True)
    assert y.dtype == torch.bfloat16 and y.shape == yr.shape
    assert _rel(y, yr) < 4e-3
    dy = torch.randn(yr.shape, generator=g).to(torch.bfloat16)
    y.backward(dy.cuda())
    dxr, dwr, dbr = R.masked_conv2d_grads(x.float(), wt, mk, dy.float(), s, p, bf16_operands=True, has_bias=bias)
    assert _rel(xg.grad, dxr) < 4e-3
    assert _rel(wg.grad, dwr) < 1e-4
    assert bool((wg.grad[mk.cuda() == 0] == 0).all())           # masked weights receive exactly zero gradient
    if bias:
        assert _rel(bg.grad, dbr) < 1e-4


def test_linear_layers_vs_oracle(dev):
    from turboprune_b200.utils.mask_layers import Conv1dMask, LinearMask
    from oracle import mask_ops as R
    torch.manual_seed(0)
    for fc, shape in ((Conv1dMask(2048, 1000, bias=True), (64, 2048)), (Conv1dMask(512, 10, bias=True), (96, 512)),
                      (LinearMask(in_features=384, out_features=1152, bias=True), (4, 197, 384))):
        fc = fc.cuda(); fc.set_er_mask(0.3)
        x = torch.randn(*shape, device=dev, dtype=torch.bfloat16, requires_grad=True)
        y = fc(x); dy = torch.randn_like(y); y.backward(dy)
        w2 = fc.weight.detach().cpu().reshape(fc.weight.shape[0], -1); m2 = fc.mask.cpu().reshape(w2.shape)
        yr = R.masked_linear(x.detach().cpu(), w2, m2, fc.bias.detach().cpu(), bf16_operands=True)
        gx, gw, gb = R.masked_linear_grads(x.detach().cpu(), w2, m2, dy.cpu(), True, True)
        assert _rel(y, yr) < 4e-3 and _rel(x.grad, gx) < 4e-3
        assert _rel(fc.weight.grad.reshape(w2.shape), gw) < 1e-4 and _rel(fc.bias.grad, gb) < 1e-4


def test_conv_full_size_linearity_property(dev):
    """BASELINE-size layer (ResNet-50 layer2 3x3, B=64): linearity in the input, conv(a*x1 + x2) = a*conv(x1) + conv(x2)."""
    from turboprune_b200 import ops
    g = torch.Generator(device=dev).manual_seed(3)
    w = torch.randn(128, 128, 3, 3, device=dev, generator=g) / 34.0
    m = (torch.rand(128, 128, 3, 3, device=dev, generator=g) < 0.17).float()
    x1 = torch.randn(64, 128, 28, 28, device=dev, generator=g).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    x2 = torch.randn(64, 128, 28, 28, device=dev, generator=g).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    y1 = ops.masked_conv2d(x1, w, m).float(); y2 = ops.masked_conv2d(x2, w, m).float()
    y3 = ops.masked_conv2d((2 * x1 + x2).to(torch.bfloat16), w, m).float()
    xs = (2 * x1 + x2).to(torch.bfloat16).float() - (2 * x1.float() + x2.float())      # rounding of the summed input
    assert float((y3 - (2 * y1 + y2)).abs().max()) < 0.05 * float(y3.abs().max()) + float(xs.abs().max())
    # zero mask -> exactly zero output, all-ones mask == unmasked
    assert float(ops.masked_conv2d(x1, w, torch.zeros_like(m)).abs().max()) == 0.0


# ---------------------------------------------------------------- optimizer / train step ---------------------
def test_fused_sgd_matches_oracle_and_torch(dev):
    from turboprune_b200.optim import FusedSGD
    from oracle.train import sgd_momentum_step
    z = np.load(os.path.join(G, "sgd_small.npz"))
    p = torch.nn.Parameter(torch.from_numpy(z["w0"]).cuda())
    opt = FusedSGD([p], lr=0.2, momentum=0.9, weight_decay=5e-4)
    for step in range(3):
        p.grad = torch.from_numpy(z[f"g{step}"]).cuda()
        opt.step()
        assert np.allclose(p.detach().cpu().numpy(), z[f"w{step + 1}"], rtol=5e-7, atol=1e-7)   # torch.optim.SGD trajectory


def test_train_step_loss_and_grads_vs_oracle(dev):
    """Config #1 shape (ResNet-18 / CIFAR-10, bf16 autocast): one step from identical weights.

    loss <= 1e-3 relative vs the oracle (CPU bf16 autocast) AND vs the reference's eager GPU path (the oracle
    modules moved to cuda: mask*w -> cuDNN, ATen BN).  Gradients through 18 bf16 layers are noisy in ANY bf16
    implementation (ReLU gates flip), so each gradient is judged against an fp32 run of the oracle: our error
    must not exceed twice the eager-bf16 path's own error (+2 % of the tensor max).  Masked weights: exactly
    zero gradient; post-step weights close (masked ones decay identically)."""
    import copy
    import refshim
    import oracle.model as om
    from oracle.train import train_step
    from turboprune_b200.utils import custom_models as cm, pruning_utils as pu
    torch.manual_seed(0)
    mine = cm.TorchVisionModel(refshim.make_cfg("resnet18", "cifar10"))
    torch.manual_seed(1)
    pu.prune_er_erk(mine, 0.2)
    ref = om.build("resnet18", "cifar10")
    ref.load_state_dict(mine.model.state_dict())
    ref32 = copy.deepcopy(ref)
    eager = copy.deepcopy(ref).cuda()
    mine = mine.cuda()
    g = torch.Generator().manual_seed(5)
    x = torch.randn(128, 3, 32, 32, generator=g); t = torch.randint(0, 10, (128,), generator=g)
    mk = lambda m: torch.optim.SGD(m.parameters(), lr=0.01, momentum=0.9, weight_decay=5e-4)
    for m in (ref, ref32, eager, mine):
        m.train()
    l_ref, _ = train_step(ref, mk(ref), x, t)
    l_32, _ = train_step(ref32, mk(ref32), x, t, use_amp=False)
    l_eager, _ = train_step(eager, mk(eager), x.cuda(), t.cuda(), device_type="cuda")
    l_mine, _ = train_step(mine, mk(mine), x.cuda(), t.cuda(), device_type="cuda")
    assert abs(l_ref - l_mine) / abs(l_ref) <= 1e-3
    assert abs(l_eager - l_mine) / abs(l_eager) <= 1e-3
    for (n1, p32), (_, pe), (n2, pm) in zip(ref32.named_parameters(), eager.named_parameters(), mine.model.named_parameters()):
        assert n1 == n2
        if p32.grad.abs().max() > 0:
            e_mine, e_eager = _rel(pm.grad, p32.grad), _rel(pe.grad, p32.grad)
            assert e_mine <= 2 * e_eager + 0.02, (n1, e_mine, e_eager)
    for (_, m), (_, r) in zip(mine._masked(), om.masked_layers(ref)):
        assert bool((m.weight.grad[m.mask == 0] == 0).all())
        assert _rel(m.weight, r.weight) < 1e-2      # lr * (bf16 gradient noise of two different bf16 paths) on top of identical decay


def test_run_experiment_level_loop(dev, tmp_path):
    """Config #1 (ResNet-18 / CIFAR-10-shape, IMP, 1 prune cycle) through run_experiment.main on synthetic data:
    levels [1.0, 0.8], checkpoints in the reference's layout, 20 % sparsity after the cycle, weights rewound to init."""
    import csv
    import run_experiment
    from turboprune_b200.utils import config as C
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cfg = C.compose("synthetic_rn18_imp", ["dataset_params.total_batch_size=64", "dataset_params.synthetic_steps_per_epoch=3",
                                           f"experiment_params.base_dir={tmp_path}"], os.path.join(root, "conf_b200"))
    prefix, expt = run_experiment.main(cfg)
    ck = os.path.join(expt, "checkpoints")
    for name in ("model_init.pt", "model_level_0.pt", "model_level_1.pt"):
        assert os.path.isfile(os.path.join(ck, name)), name
    assert os.path.isfile(os.path.join(expt, "artifacts", "optimizer_init.pt"))
    rows = list(csv.DictReader(open(os.path.join(expt, f"{prefix}_summary.csv"))))
    assert [r["Level"] for r in rows] == ["0", "1"]
    assert float(rows[0]["Sparsity"]) == 0.0 and abs(float(rows[1]["Sparsity"]) - 20.0) < 1e-3
    init = torch.load(os.path.join(ck, "model_init.pt")); lvl0 = torch.load(os.path.join(ck, "model_level_0.pt"))
    lvl1 = torch.load(os.path.join(ck, "model_level_1.pt"))
    assert set(init) == set(lvl1) and init["fc.weight"].shape == (10, 512, 1) and "conv1.mask" in init
    # the level-1 mask is the magnitude mask of the level-0 weights (global threshold, ties pruned)
    from oracle import prune as P
    names = [k[:-5] for k in lvl0 if k.endswith(".mask")]
    ws = [lvl0[n + ".weight"].cpu().numpy() for n in names]; ms = [lvl0[n + ".mask"].cpu().numpy() for n in names]
    ref_masks, _, _ = P.prune_global(ws, ms, 0.8)
    for n, rm in zip(names, ref_masks):
        assert np.array_equal(lvl1[n + ".mask"].cpu().numpy(), rm), n


# ---------------------------------------------------------------- fused BN / pooling / graph / other configs -----
BN_CASES = [(4, 64, 9, 7, True, False), (8, 256, 14, 14, True, True), (3, 2048, 7, 7, False, False), (16, 64, 56, 56, True, False),
            (2, 192, 5, 5, False, True)]


@pytest.mark.parametrize("case", BN_CASES)
def test_fused_batchnorm_vs_torch(dev, case):
    """BatchNorm2dB200 (+residual)(+ReLU) vs torch's BatchNorm2d evaluated in fp32 on the same bf16 inputs:
    outputs / input grads are bf16 (<= 1e-2 of max), parameter grads and running statistics fp32 (<= 1e-4)."""
    from turboprune_b200.fused_norm import BatchNorm2dB200
    n, c, h, w, relu, res = case
    g = torch.Generator().manual_seed(c + n)
    x = (torch.randn(n, c, h, w, generator=g) * 1.7 + 0.3).to(dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    r = torch.randn(n, c, h, w, generator=g).to(dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last) if res else None
    bn = BatchNorm2dB200(c).to(dev); ref = torch.nn.BatchNorm2d(c).to(dev)
    with torch.no_grad():
        bn.weight.copy_(torch.rand(c, generator=g) + 0.5); bn.bias.copy_(torch.randn(c, generator=g) * 0.1)
    ref.load_state_dict(bn.state_dict())
    xa = x.clone().requires_grad_(True); xb = x.clone().float().requires_grad_(True)
    ra = r.clone().requires_grad_(True) if res else None; rb = r.clone().float().requires_grad_(True) if res else None
    z = bn(xa, residual=ra, relu=relu)
    zr = ref(xb)
    zr = zr + rb if res else zr
    zr = torch.relu(zr) if relu else zr
    dz = torch.randn(z.shape, generator=g).to(dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    z.backward(dz); zr.backward(dz.float())
    assert _rel(z, zr) < 1e-2 and _rel(xa.grad, xb.grad) < 1e-2
    assert _rel(bn.weight.grad, ref.weight.grad) < 1e-4 and _rel(bn.bias.grad, ref.bias.grad) < 1e-4
    assert _rel(bn.running_mean, ref.running_mean) < 1e-4 and _rel(bn.running_var, ref.running_var) < 1e-4
    assert int(bn.num_batches_tracked) == 1
    if res:
        assert _rel(ra.grad, rb.grad) < 1e-2
    bn.eval(); ref.eval()
    with torch.no_grad():
        assert _rel(bn(x, relu=relu), torch.relu(ref(x.float())) if relu else ref(x.float())) < 1e-2


@pytest.mark.parametrize("case", [(6, 64, 128, 3, 1, 1, 19, True), (5, 128, 256, 1, 1, 0, 14, False), (4, 64, 64, 3, 2, 1, 30, False),
                                  (3, 3, 64, 7, 2, 3, 40, False)])
def test_conv_epilogue_batchnorm_statistics(dev, case):
    """The conv epilogue's per-channel (sum, sum of squares) of the bf16 outputs equal a direct reduction of the
    stored activation, and conv -> BatchNorm with the statistics handed over through the epilogue matches the
    two-pass path (outputs, running statistics, all gradients)."""
    import copy
    from turboprune_b200 import fused_norm as fn
    from turboprune_b200.utils import mask_layers as ml
    b, cin, cout, k, s, p, hw, bias = case
    g = torch.Generator(device=dev).manual_seed(sum(case[:7]))
    conv = ml.ConvMask(in_channels=cin, out_channels=cout, kernel_size=k, stride=s, padding=p, bias=bias).to(dev)
    with torch.no_grad():
        conv.mask.copy_((torch.rand(conv.weight.shape, device=dev, generator=g) < 0.4).float())
        if bias:
            conv.bias.copy_(torch.randn(cout, device=dev, generator=g) * 3)         # |mean| >> std for some channels
    bn = fn.BatchNorm2dB200(cout).to(dev).train()
    with torch.no_grad():
        bn.weight.copy_(torch.rand(cout, device=dev, generator=g) + 0.5); bn.bias.copy_(torch.randn(cout, device=dev, generator=g))
    x = torch.randn(b, cin, hw, hw, device=dev, generator=g).to(torch.bfloat16 if cin >= 8 else torch.float32)
    x = x.contiguous(memory_format=torch.channels_last)
    y, stats = conv(x, want_stats=True)
    yf = y.detach().float()
    ref1 = yf.sum(dim=(0, 2, 3)); ref2 = (yf * yf).sum(dim=(0, 2, 3))
    got = stats.sum(dim=0)
    assert float((got[0] - ref1).abs().max()) <= 1e-4 * float(ref2.sqrt().max()) * (y.numel() / cout) ** 0.5 + 1e-3
    assert _rel(got[1], ref2) < 1e-5
    res = []
    for fused in (False, True):
        c2, b2 = copy.deepcopy(conv), copy.deepcopy(bn)
        xx = x.clone().requires_grad_(cin >= 8)
        if fused:
            z, _ = fn._conv_bn(c2, b2, xx, relu=True)
        else:
            z = b2(c2(xx), relu=True)
        gz = torch.Generator(device=dev).manual_seed(11)
        z.backward(torch.randn(z.shape, device=dev, generator=gz).to(z.dtype).contiguous(memory_format=torch.channels_last))
        res.append((z.detach().float(), b2.running_mean.clone(), b2.running_var.clone(), c2.weight.grad.clone(),
                    b2.weight.grad.clone(), b2.bias.grad.clone(), xx.grad.float() if cin >= 8 else None))
    a_, b_ = res
    assert _rel(b_[0], a_[0]) < 1e-2                                    # bf16 outputs: a last-bit flip of scale/shift at most
    assert _rel(b_[1], a_[1]) < 1e-5 and _rel(b_[2], a_[2]) < 1e-4
    for i in (3, 4, 5):
        assert _rel(b_[i], a_[i]) < 2e-2
    if a_[6] is not None:
        assert _rel(b_[6], a_[6]) < 2e-2


def test_maxpool_vs_torch(dev):
    from turboprune_b200.fused_norm import MaxPool2dB200
    g = torch.Generator().manual_seed(3)
    x = torch.randn(6, 64, 23, 17, generator=g).to(dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    for k, s, p in ((3, 2, 1), (2, 2, 0), (3, 1, 1)):
        xa = x.clone().requires_grad_(True); xb = x.clone().float().requires_grad_(True)
        ya = MaxPool2dB200(k, s, p)(xa); yb = torch.nn.functional.max_pool2d(xb, k, s, p)
        assert torch.equal(ya.float(), yb)                                    # selection is exact
        dy = torch.randn(ya.shape, generator=g).to(dev).to(torch.bfloat16)
        ya.backward(dy); yb.backward(dy.float())
        assert _rel(xa.grad, xb.grad) < 1e-2                                  # sums of <= 4 bf16 values, rounded once


def test_cuda_graph_step_is_bit_identical_to_eager(dev, tmp_path):
    """PruningHarness.train_step owns the captured step (persistent gradient arena, one-launch weight shadow,
    device-scalar LR, cached SGD table): six steps with the capture (3 eager + 3 replays, LR changed every step by the
    scheduler) give bit-identical weights, buffers and losses to six eager steps from the same state; replacing a
    mask tensor (pruning) drops the capture."""
    import copy
    import refshim
    from turboprune_b200.utils import custom_models as cm, pruning_utils as pu
    torch.manual_seed(0)
    base = cm.TorchVisionModel(refshim.make_cfg("resnet18", "cifar10", precision="bfloat16"))
    torch.manual_seed(1)
    pu.prune_er_erk(base, 0.2)
    g = torch.Generator().manual_seed(2)
    xs = [torch.randn(64, 3, 32, 32, generator=g).to(dev) for _ in range(6)]
    ts = [torch.randint(0, 10, (64,), generator=g).to(dev) for _ in range(6)]
    runs = []
    for use_graph in (False, True):
        cfg = refshim.make_cfg("resnet18", "cifar10", precision="bfloat16")
        cfg["experiment_params"]["cuda_graph"] = use_graph
        cfg["experiment_params"]["epochs_per_level"] = 1
        h = refshim.make_harness(cfg, copy.deepcopy(base), 64, str(tmp_path))
        h.model.train()
        losses = []
        for i in range(6):
            for grp in h.optimizer.param_groups:
                grp["lr"] = 0.05 * (1 + i)                       # a per-iteration schedule: nothing may be baked in
            losses.append(float(h.train_step((xs[i], ts[i]))["loss"].item()))
        assert (h._graph is not None) == use_graph
        runs.append((h, losses))
    (h1, l1), (h2, l2) = runs
    assert l1 == l2
    for (n1, p1), (n2, p2) in zip(h1.model.named_parameters(), h2.model.named_parameters()):
        assert torch.equal(p1, p2), n1
    for (n1, b1), (n2, b2) in zip(h1.model.named_buffers(), h2.model.named_buffers()):
        assert torch.equal(b1, b2), n1
    assert torch.equal(h1.train_accuracy.stat, h2.train_accuracy.stat)
    # pruning assigns new mask tensors: the capture must be dropped and rebuilt, never replayed on stale pointers
    pu.prune_mag(h2.model, 0.5)
    pu.prune_mag(h1.model, 0.5)
    for i in range(4):
        a = float(h1.train_step((xs[i], ts[i]))["loss"].item()); b = float(h2.train_step((xs[i], ts[i]))["loss"].item())
        assert a == b
    assert h2._graph is not None
    for (_, m1), (_, m2) in zip(h1.model._masked(), h2.model._masked()):
        assert torch.equal(m1.weight, m2.weight) and bool((m2.weight.grad[m2.mask == 0] == 0).all())


def test_batched_weight_staging_matches_per_layer(dev):
    """WeightStager: one launch writes the bf16(mask*w) fprop / dgrad operands of every layer (stem conv with 3
    channels, 3x3 and 1x1 convs, the fc) — bit-identical to the per-layer staging kernel; the pairs are consumed
    exactly once; a train step with the stager gives bit-identical weights to one without."""
    import copy
    import refshim
    from turboprune_b200 import ops
    from turboprune_b200.optim import FusedSGD
    from turboprune_b200.utils import custom_models as cm, pruning_utils as pu
    from turboprune_b200.utils.mask_layers import MASKED_LAYER_TYPES
    torch.manual_seed(0)
    base = cm.TorchVisionModel(refshim.make_cfg("resnet18", "cifar10"))
    torch.manual_seed(1)
    pu.prune_er_erk(base, 0.3)
    model = copy.deepcopy(base).to(dev).train()
    layers = [m for m in model.modules() if isinstance(m, MASKED_LAYER_TYPES)]
    stager = ops.WeightStager(layers)
    stager.stage()
    for l in layers:
        w = l.weight.detach(); m = l.mask
        if w.dim() != 4:
            w = w.reshape(w.shape[0], w.shape[1], 1, 1); m = m.reshape(w.shape)
        cout, cin, r, s = w.shape
        cin_p, cout_p, has_wd, wf_ld = ops._operand_plan(cout, cin, r, s)
        wf, wd = ops.stage_weights(w.contiguous(), m.contiguous(), cin_p, has_wd, cout_p, wf_ld=wf_ld)
        got = ops.take_staged(l)
        assert got is not None and ops.take_staged(l) is None            # consumed exactly once
        assert torch.equal(got[0], wf)
        if has_wd:
            assert torch.equal(got[1][:, :wd.shape[1]], wd)
    # pruning replaces mask tensors: the table follows
    pu.prune_mag(model, 0.5)
    stager.stage()
    l = layers[3]
    wf, _ = ops.stage_weights(l.weight.detach(), l.mask, l.weight.shape[1], False)
    assert torch.equal(ops.take_staged(l)[0], wf)
    for l in layers:
        ops.take_staged(l)
    # same step with / without the stager
    g = torch.Generator().manual_seed(5)
    x = torch.randn(32, 3, 32, 32, generator=g).to(dev); t = torch.randint(0, 10, (32,), generator=g).to(dev)
    res = []
    for use in (False, True):
        m2 = copy.deepcopy(base).to(dev).train()
        opt = FusedSGD(m2.parameters(), lr=0.05, momentum=0.9, weight_decay=5e-4)
        st = ops.WeightStager([q for q in m2.modules() if isinstance(q, MASKED_LAYER_TYPES)])
        for _ in range(2):
            opt.zero_grad()
            if use:
                st.stage()
            with torch.autocast("cuda", dtype=torch.bfloat16):
                torch.nn.functional.cross_entropy(m2(x), t).backward()
            opt.step()
        res.append([p.detach().clone() for p in m2.parameters()])
    assert all(torch.equal(a, b) for a, b in zip(*res))


@pytest.mark.parametrize("arch", ["resnet18", "vgg16"])
def test_arena_direct_gradient_writes_equal_autograd_accumulation(dev, arch):
    """(vgg16: convolutions WITH a bias — its gradient goes to the slot too, once.)
    With a GradArena attached, wgrad / BN backward write dW, db, dgamma, dbeta straight into the slots (no
    AccumulateGrad kernel); the values must be the ones autograd would have accumulated into a fresh .grad, and a
    model whose grads were detached (zero_grad(set_to_none=True)) must fall back to the ordinary path."""
    import copy
    import refshim
    from turboprune_b200.grad_exchange import GradArena
    from turboprune_b200.utils import custom_models as cm, pruning_utils as pu
    torch.manual_seed(0)
    base = cm.TorchVisionModel(refshim.make_cfg(arch, "cifar10"))
    torch.manual_seed(1)
    pu.prune_er_erk(base, 0.3)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(32, 3, 32, 32, generator=g).to(dev); t = torch.randint(0, 10, (32,), generator=g).to(dev)

    def run(m):
        torch.manual_seed(7)                   # vgg16's classifier has dropout: the same draw for every run
        with torch.autocast("cuda", dtype=torch.bfloat16):
            torch.nn.functional.cross_entropy(m(x), t).backward()

    plain = copy.deepcopy(base).to(dev).train()
    run(plain)
    direct = copy.deepcopy(base).to(dev).train()
    arena = GradArena(list(direct.parameters()))
    assert all(hasattr(p, "_tp_grad_slot") for p in direct.parameters())
    arena.zero()
    run(direct)
    for (n, a), (_, b) in zip(plain.named_parameters(), direct.named_parameters()):
        assert b.grad.data_ptr() == b._tp_grad_slot.data_ptr(), n
        assert torch.equal(a.grad, b.grad), n
    # detached grads: the ordinary autograd path must be used and the arena left alone
    direct.zero_grad(set_to_none=True)
    before = arena.flat.clone()
    run(direct)
    assert torch.equal(arena.flat, before)
    for (n, a), (_, b) in zip(plain.named_parameters(), direct.named_parameters()):
        assert torch.equal(a.grad, b.grad), n


def test_config4_vgg16_synflow_and_config5_deit_snip(dev):
    """BASELINE.json configs 4 and 5 as parity-test cases: VGG-16 / CIFAR-100 shape with one-shot SynFlow to 95 %,
    DeiT-small with SNIP to 50 % (masked Linear path): pruning hits the target sparsity, masks are {0,1}, a train
    step through the kernels gives a finite loss."""
    import refshim
    from turboprune_b200.utils import custom_models as cm, pruning_utils as pu
    from turboprune_b200.utils.dataset import SyntheticLoader
    for model, cfg, shape, ncls, method, density in (
            (None, refshim.make_cfg("vgg16", "cifar100", precision="bfloat16", prune_method="synflow"), (3, 32, 32), 100, pu.prune_synflow, 0.05),
            ("deit", refshim.make_cfg("local_deit_small_patch16_224", "imagenet", mask_layer_type="LinearMask", precision="bfloat16",
                                      prune_method="snip"), (3, 224, 224), 1000, pu.prune_snip, 0.5)):
        torch.manual_seed(0)
        net = (cm.CustomModel(cfg) if model == "deit" else cm.TorchVisionModel(cfg)).to(dev).train()
        loader = SyntheticLoader(8, 2, shape, ncls, dev, seed=1)
        method(cfg, net, loader, density)
        sp = net.get_overall_sparsity()
        assert abs(sp - (1 - density) * 100) < 0.01, sp
        for _, m in net._masked():
            assert bool(((m.mask == 0) | (m.mask == 1)).all())
        opt = torch.optim.SGD(net.parameters(), lr=0.01, momentum=0.9)
        xb, tb = next(iter(loader))
        opt.zero_grad()                                   # prune_snip leaves its scoring gradients in .grad (like the reference)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = torch.nn.functional.cross_entropy(net(xb), tb)
        loss.backward(); opt.step()
        assert bool(torch.isfinite(loss))
        for _, m in net._masked():
            assert bool((m.weight.grad[m.mask == 0] == 0).all())


# ---------------------------------------------------------------- loss parity through the product's train step ----
def _zero_dropout(net):
    for m in net.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0


@pytest.mark.parametrize("name", ["resnet50", "vgg16", "deit_small"])
def test_harness_train_step_loss_vs_oracle(dev, tmp_path, name):
    """BASELINE.json configs 2 / 4 / 5 (ResNet-50 ImageNet-shape B=32, VGG-16 CIFAR-100-shape B=64, DeiT-S B=8), ERK masks
    at 80 % sparsity, bf16 autocast: ONE ``PruningHarness.train_step`` (the call run_experiment.py makes, reference
    base_harness.py:115-134) against the CPU oracle's train step from identical weights — loss <= 1e-3 relative
    (north_star), every masked weight gets exactly zero gradient.  Dropout (VGG classifier) is set to p = 0 on both
    sides: its random stream is not part of the parity contract."""
    import refshim
    import oracle.model as om
    from oracle import vit as ov
    from oracle.train import train_step
    from turboprune_b200.utils import custom_models as cm, pruning_utils as pu
    if name == "deit_small":
        cfg = refshim.make_cfg("local_deit_small_patch16_224", "imagenet", mask_layer_type="LinearMask", precision="bfloat16")
        B, shape, ncls = 8, (3, 224, 224), 1000
        torch.manual_seed(0)
        mine = cm.CustomModel(cfg)
        ref = ov.build("local_deit_small_patch16_224")
    else:
        ds = "imagenet" if name == "resnet50" else "cifar100"
        cfg = refshim.make_cfg(name, ds, precision="bfloat16")
        B, shape, ncls = (32, (3, 224, 224), 1000) if name == "resnet50" else (64, (3, 32, 32), 100)
        torch.manual_seed(0)
        mine = cm.TorchVisionModel(cfg)
        ref = om.build(name, ds)
    cfg["optimizer_params"]["lr"] = 0.01
    torch.manual_seed(1)
    pu.prune_er_erk(mine, 0.2)
    ref.load_state_dict(mine.model.state_dict())
    _zero_dropout(mine); _zero_dropout(ref)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, *shape, generator=g); t = torch.randint(0, ncls, (B,), generator=g)
    o = cfg.optimizer_params
    opt_ref = torch.optim.SGD(ref.parameters(), lr=o.lr, momentum=o.momentum, weight_decay=o.weight_decay)
    ref.train()
    l_ref, _ = train_step(ref, opt_ref, x, t)
    h = refshim.make_harness(cfg, mine, B, str(tmp_path))
    h.model.train()
    l_mine = float(h.train_step((x.to(dev), t.to(dev)))["loss"].item())
    assert abs(l_ref - l_mine) / abs(l_ref) <= 1e-3, (name, l_ref, l_mine)
    for _, m in h.model._masked():
        assert bool((m.weight.grad[m.mask == 0] == 0).all())
    # two more steps: the third captures the CUDA graph; the loss stays finite and keeps following the oracle loosely
    for _ in range(3):
        l_ref, _ = train_step(ref, opt_ref, x, t)
        l_mine = float(h.train_step((x.to(dev), t.to(dev)))["loss"].item())
    assert h._graph is not None
    assert abs(l_ref - l_mine) / abs(l_ref) <= 2e-2, (name, l_ref, l_mine)


# ---------------------------------------------------------------- gradient exchange over NVLink (2 ranks) ---------
def test_p2p_allreduce_two_ranks(dev):
    """tp_p2p_allreduce_mask (one-shot, two-shot, NVLS when the fabric offers a multicast address) with a mask, on 2
    GPUs: bit-exact against oracle.train.allreduce_mean_mask, replicas bit-identical; then the overlapped reducer
    inside two PruningHarness ranks (level-loop smoke).  Needs >= 2 GPUs (skipped on the 1-GPU test box)."""
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    port = 29500 + os.getpid() % 400
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "tools", "p2p_check.py"), "--no-timing"]
    r = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "P2P CHECK PASS" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def test_level_loop_two_ranks(dev, tmp_path):
    """run_experiment.py under torchrun on 2 GPUs (reference README.md:85-91): ResNet-18 on ImageNet-shaped synthetic
    batches, IMP one cycle — the harness's captured step with the overlapped P2P reducer (created once per process,
    reused by the second level's harness), rank-0 mask broadcast, replica checksum after every level."""
    import csv
    import glob
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    port = 29900 + os.getpid() % 90
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "run_experiment.py"), "--config-name=synthetic_rn50_erk80",
           f"--config-path={os.path.join(root, 'conf_b200')}", "model_params=resnet18_convmask", "pruning_params=imp_one_cycle",
           "dataset_params.total_batch_size=32", "dataset_params.synthetic_steps_per_epoch=5", f"experiment_params.base_dir={tmp_path}"]
    r = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    (summary,) = glob.glob(os.path.join(str(tmp_path), "*", "*_summary.csv"))
    rows = list(csv.DictReader(open(summary)))
    assert [row["Level"] for row in rows] == ["0", "1"] and abs(float(rows[1]["Sparsity"]) - 20.0) < 1e-3


# ---------------------------------------------------------------- tile skipping (north_star) ----------------------
@pytest.mark.parametrize("case", [(2, 14, 256, 192, 3, 1, 1), (3, 12, 512, 320, 1, 1, 0), (2, 15, 128, 128, 3, 2, 1), (2, 9, 192, 64, 3, 1, 1)])
def test_kblock_skipping_bit_identical_to_dense_walk(dev, case):
    """Masks with dead filters, dead input-channel blocks and dead taps (what structured sparsity in the IMP tail /
    SynFlow produces): the staging kernel's occupancy bits equal a direct computation from mask*w, a positive number of
    64x64 blocks is skipped, and fprop / dgrad / wgrad results are BIT-IDENTICAL to the dense walk over the same
    operands (a skipped block only ever adds zeros)."""
    from turboprune_b200 import ops
    n, hw, cin, cout, k, s_, p_ = case
    g = torch.Generator(device=dev).manual_seed(sum(case))
    x = torch.randn(n, cin, hw, hw, device=dev, generator=g).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    w = torch.randn(cout, cin, k, k, device=dev, generator=g) / (cin * k * k) ** 0.5
    m = (torch.rand(cout, cin, k, k, device=dev, generator=g) < 0.3).float()
    m[:, 64:128] = 0                       # a dead 64-channel input block (every tap)
    m[64:128] = 0                          # 64 dead filters: a whole row group of the fprop operand
    m[:, :64, 0, 0] = 0                    # one dead tap for the first channel block
    if cout > 128:
        m[128:, :, k - 1, k - 1] = 0
    if cout > 128:
        m[128:192] = 0                     # a whole 128-channel wgrad tile row without a single kept weight
    if k > 1:
        m[:, :, 0, 0:2] = 0                # taps (0,0), (0,1) dead everywhere: whole 256-column wgrad tiles are empty
    # occupancy bits vs a direct computation
    cout_p = ops._round_up(cout, 64 if k > 1 else 8)
    wf, wd = ops.stage_weights(w, m, cin, True, cout_p)
    eff = (m * w).to(torch.bfloat16).float()
    ref_f = eff.permute(0, 2, 3, 1).reshape(cout, k * k * cin)                       # [co][tap*cin + ci]
    padr = (-cout) % 64
    ref_f = torch.nn.functional.pad(ref_f, (0, 0, 0, padr)).reshape((cout + padr) // 64, 64, k * k * cin // 64, 64)
    occ_f = (ref_f != 0).any(dim=3).any(dim=1).cpu()
    words = ops.kmask_rows(wf.kmask, wf.shape[1]).cpu().to(torch.int64) & 0xFFFFFFFF
    got_f = torch.tensor([[(int(words[r, b // 32]) >> (b % 32)) & 1 for b in range(occ_f.shape[1])] for r in range(occ_f.shape[0])]).bool()
    assert torch.equal(got_f, occ_f)
    empty, total = ops.kblock_occupancy(wf.kmask, wf.shape[1])
    assert empty > 0 and empty == int((~occ_f).sum())
    ed, td = ops.kblock_occupancy(wd.kmask, wd.shape[1])
    assert ed > 0
    outs = {}
    for skip in (True, False):
        ops.set_kblock_skip(skip)
        try:
            xx = x.clone().requires_grad_(True); ww = w.clone().requires_grad_(True)
            y = ops.masked_conv2d(xx, ww, m, None, (s_, s_), (p_, p_))
            gy = torch.Generator(device=dev).manual_seed(7)
            dy = torch.randn(y.shape, device=dev, generator=gy).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
            y.backward(dy)
            outs[skip] = (y.detach().clone(), xx.grad.detach().clone(), ww.grad.detach().clone())
        finally:
            ops.set_kblock_skip(True)
    for a, b in zip(outs[True], outs[False]):
        assert torch.equal(a, b)
    if cout >= 128:
        assert float(outs[True][0][:, 64:128].abs().max()) == 0.0      # dead filters: exactly zero outputs


@pytest.mark.parametrize("case", [(2, 14, 128, 256, 3), (4, 8, 256, 384, 1), (2, 10, 64, 128, 3)])
def test_wgrad_skips_tiles_under_empty_mask_blocks(dev, case):
    """tp_conv_wgrad with the occupancy mask: 128-channel x 256-column output tiles whose mask blocks are all zero are
    neither computed nor read back.  The split-K workspace is poisoned with NaN first: a skipped tile that was read
    anyway would show; the result equals the dense walk bit for bit and is exactly zero under the dead blocks.  A kept
    weight that is exactly 0.0 keeps its block alive (the occupancy follows the MASK there, not mask * w)."""
    from turboprune_b200 import ops
    n, hw, cin, cout, k = case
    g = torch.Generator(device=dev).manual_seed(sum(case))
    x = torch.randn(n, hw, hw, cin, device=dev, generator=g).to(torch.bfloat16)
    w = torch.randn(cout, cin, k, k, device=dev, generator=g) * 0.05
    m = (torch.rand(cout, cin, k, k, device=dev, generator=g) < 0.3).float()
    m[:128, :, 0, 0] = 0                                   # first tile row: tap (0,0) dead (a whole 256-column tile for cin >= 256 ...)
    if k > 1:
        m[:128, :, 0, 1] = 0                               # ... and tap (0,1) too: chunks 0..3 empty for cin = 128 as well
    if cout > 128:
        m[128:256] = 0                                     # second tile row completely dead
    w[130:140] = 0.0                                       # zero weights under a zero mask: still empty
    if cout > 128:
        m[130, 3, k - 1, k - 1] = 1.0                      # ONE kept weight in the dead tile row, and its value is exactly 0.0:
                                                           # mask * w is zero everywhere in that block, the block must stay occupied
    desc = ops.make_desc(n, hw, hw, cin, cout, k, k, (1, 1), (k // 2, k // 2))
    wf, _ = ops.stage_weights(w, m, cin, False, cout, want_kmask=True)
    empty, total = ops.kblock_occupancy(wf.kmask, wf.shape[1])
    assert empty > 0
    y = ops.conv_fprop(desc, x, wf)
    dy = torch.randn(y.shape, device=dev, generator=g).to(torch.bfloat16)
    dense, _ = ops.conv_wgrad(desc, x, dy, m, cin)
    dense = dense.clone()
    nbytes = ops._cabi.load().tp_conv_workspace_bytes(ctypes.byref(desc), 2)
    wsb = ops._workspace(nbytes, x.device, "wgrad")
    wsb[: wsb.numel() // 4 * 4].view(torch.float32).fill_(float("nan"))
    skip, _ = ops.conv_wgrad(desc, x, dy, m, cin, kmask=wf.kmask)
    assert torch.isfinite(skip).all()
    assert torch.equal(skip, dense)
    assert float(skip[m == 0].abs().max()) == 0.0
    if cout > 128:
        assert float(dense[130, 3, k - 1, k - 1]) != 0.0    # the zero-valued kept weight has a gradient


def test_skipped_block_report_on_structured_and_iid_masks(dev):
    """Honest accounting: iid ERK-80 masks on ResNet-18 leave (almost) no 64x64 block empty; killing filters does."""
    import refshim
    from turboprune_b200 import ops
    from turboprune_b200.utils import custom_models as cm, pruning_utils as pu
    from turboprune_b200.utils.mask_layers import MASKED_LAYER_TYPES
    torch.manual_seed(0)
    model = cm.TorchVisionModel(refshim.make_cfg("resnet18", "cifar10"))
    torch.manual_seed(1)
    pu.prune_er_erk(model, 0.2)
    model = model.to(dev)
    st = ops.WeightStager([m for m in model.modules() if isinstance(m, MASKED_LAYER_TYPES)])
    st.stage()
    rep = ops.skipped_block_report(st)
    assert rep["total_blocks"] > 1000 and rep["fraction"] < 0.01
    for _, m in model._masked():
        if m.weight.dim() == 4 and m.weight.shape[0] >= 128:
            m.mask[: m.weight.shape[0] // 2] = 0                      # half of the filters dead (in place: same tensors)
    st.stage()
    rep2 = ops.skipped_block_report(st)
    assert rep2["fraction"] > 0.3
    for l in st.layers:
        ops.take_staged(l)


def test_harness_train_epoch_vs_oracle(dev, tmp_path):
    """``PruningHarness.train_epoch`` (reference base_harness.py:151-202) over a 5-step epoch of ResNet-18 / CIFAR-shape
    batches with the TriangularSchedule stepped every iteration: the learning rate seen by every step equals the oracle's,
    the epoch loss (mean of the per-step losses, read once at the end) and the accuracy follow the CPU oracle's epoch;
    the last three steps are CUDA-graph replays whose LR comes from the device scalar."""
    import refshim
    import oracle.model as om
    from oracle.train import train_epoch, triangular_schedule
    from turboprune_b200.utils import custom_models as cm, pruning_utils as pu
    cfg = refshim.make_cfg("resnet18", "cifar10", precision="bfloat16")
    cfg["optimizer_params"]["lr"] = 0.02
    cfg["experiment_params"]["epochs_per_level"] = 1
    torch.manual_seed(0)
    mine = cm.TorchVisionModel(cfg)
    torch.manual_seed(1)
    pu.prune_er_erk(mine, 0.2)
    ref = om.build("resnet18", "cifar10")
    ref.load_state_dict(mine.model.state_dict())
    g = torch.Generator().manual_seed(3)
    batches = [(torch.randn(64, 3, 32, 32, generator=g), torch.randint(0, 10, (64,), generator=g)) for _ in range(5)]
    o = cfg.optimizer_params
    opt_ref = torch.optim.SGD(ref.parameters(), lr=o.lr, momentum=o.momentum, weight_decay=o.weight_decay)
    sch_ref = triangular_schedule(opt_ref, len(batches), 1, o.warmup_fraction)
    loss_ref, acc_ref, lrs_ref, losses_ref = train_epoch(ref, opt_ref, sch_ref, batches)
    h = refshim.make_harness(cfg, mine, 64, str(tmp_path))
    h.train_loader = [(x.to(dev), t.to(dev)) for x, t in batches]
    h._setup_scheduler(1)
    seen_lr = []
    real_step = h.train_step

    def spy(batch):
        seen_lr.append(h.optimizer.param_groups[0]["lr"])
        return real_step(batch)
    h.train_step = spy
    out = h.train_epoch()
    assert h._graph is not None
    assert np.allclose(seen_lr, lrs_ref, rtol=1e-12)
    dev_lr = float(next(iter(h.optimizer._lr_dev.values())).item())
    assert abs(dev_lr - lrs_ref[-1]) <= 1e-6 * lrs_ref[-1]                   # the scalar the last replay consumed
    assert abs(out["train_loss"] - loss_ref) / loss_ref <= 5e-3, (out, loss_ref, losses_ref)
    assert abs(out["train_acc"] - acc_ref) <= 100.0 * 8 / 320                # a handful of argmax flips between two bf16 paths


# ---------------------------------------------------------------- data path (SURVEY §8(f) row 3) --------------------
def test_cifar_augmentation_kernel_matches_reference_fixture(dev):
    """tp_cifar_augment with the draws the reference made (fixture written by running utils/dataset.py:38-98): every op
    alone and the fused translate -> flip -> cutout epoch pass are bit-exact; the public batch_* wrappers (same names,
    draws made with torch's generator in the reference's order) equal the oracle fed with the re-drawn values."""
    from oracle import data as D
    from turboprune_b200.utils import dataset as ds
    z = np.load(os.path.join(G, "aug_small.npz"))
    T = lambda k: torch.from_numpy(z[k]).to(dev)
    imgs, pad2, pad4 = T("imgs"), T("padded"), T("padded4")
    assert np.array_equal(ds._augment(pad2, (12, 12), 2, shifts=T("crop2.shifts")).cpu().numpy(), z["crop2.out"])
    assert np.array_equal(ds._augment(pad4, (12, 12), 4, shifts=T("crop4.shifts")).cpu().numpy(), z["crop4.out"])
    assert np.array_equal(ds._augment(imgs, (12, 12), 0, flip=T("flip.mask")).cpu().numpy(), z["flip.out"])
    assert np.array_equal(ds._augment(imgs, (12, 12), 0, corner_y=T("cut.y"), corner_x=T("cut.x"), cut_size=5).cpu().numpy(), z["cut.out"])
    fused = ds._augment(pad4, (12, 12), 4, shifts=T("epoch.shifts"), flip=T("epoch.mask"), corner_y=T("epoch.y"), corner_x=T("epoch.x"), cut_size=3)
    assert np.array_equal(fused.cpu().numpy(), z["epoch.out"])
    # public wrappers: same draw order as the reference on the images' device
    g = torch.Generator().manual_seed(4)
    big = torch.randn(33, 3, 32, 32, generator=g).to(dev)
    padb = torch.nn.functional.pad(big, (4,) * 4, "reflect")
    torch.manual_seed(31); a = ds.batch_crop(padb, 32)
    torch.manual_seed(31); sh = torch.randint(-4, 5, size=(33, 2), device=dev)
    assert np.array_equal(a.cpu().numpy(), D.batch_crop(padb.cpu().numpy(), 32, sh.cpu().numpy()))
    torch.manual_seed(32); b = ds.batch_flip_lr(big)
    torch.manual_seed(32); fm = torch.rand(33, device=dev) < 0.5
    assert np.array_equal(b.cpu().numpy(), D.batch_flip_lr(big.cpu().numpy(), fm.cpu().numpy()))
    torch.manual_seed(33); c = ds.batch_cutout(big, 8)
    torch.manual_seed(33); cy = torch.randint(0, 25, size=(33,), device=dev); cx = torch.randint(0, 25, size=(33,), device=dev)
    assert np.array_equal(c.cpu().numpy(), D.batch_cutout(big.cpu().numpy(), 8, cy.cpu().numpy(), cx.cpu().numpy()))
    torch.manual_seed(34); e = ds.augment_epoch(padb, 32, flip=True, cutout=6)
    torch.manual_seed(34)
    sh = torch.randint(-4, 5, size=(33, 2), device=dev); fm = torch.rand(33, device=dev) < 0.5
    cy = torch.randint(0, 27, size=(33,), device=dev); cx = torch.randint(0, 27, size=(33,), device=dev)
    ref = D.augment(padb.cpu().numpy(), 32, sh.cpu().numpy(), fm.cpu().numpy(), 6, cy.cpu().numpy(), cx.cpu().numpy())
    assert np.array_equal(e.cpu().numpy(), ref)


def test_synthetic_generator_matches_oracle(dev):
    """Philox4x32-10 words bit-exact against the oracle (pinned by Random123's known-answer vector), Box-Muller normals to
    float rounding, labels exact; the loader draws a fresh, reproducible batch every step."""
    from oracle import data as D
    from turboprune_b200.utils import dataset as ds
    n = 100_003
    raw = torch.empty(n, dtype=torch.float32, device=dev)
    ds.synth_normal_(raw, seed=12345678901, counter_offset=77, raw_words=True)
    assert np.array_equal(raw.cpu().numpy().view(np.uint32), D.synth_words(n, 12345678901, 77))
    x = torch.empty(n, dtype=torch.float32, device=dev)
    ds.synth_normal_(x, seed=9, counter_offset=5)
    ref = D.synth_normal(n, 9, 5)
    assert float(np.abs(x.cpu().numpy() - ref).max()) < 2e-5
    t = torch.empty(4099, dtype=torch.int64, device=dev)
    ds.synth_labels_(t, 1000, seed=9, counter_offset=3)
    assert np.array_equal(t.cpu().numpy(), D.synth_labels(4099, 1000, 9, 3))
    a = ds.SyntheticLoader(8, 3, (3, 32, 32), 10, dev, seed=5, fresh=True)
    b = ds.SyntheticLoader(8, 3, (3, 32, 32), 10, dev, seed=5, fresh=True)
    xa = [x.clone() for x, _ in a]; xb = [x.clone() for x, _ in b]
    assert all(torch.equal(p, q) for p, q in zip(xa, xb)) and not torch.equal(xa[0], xa[1])
    cl = ds.SyntheticLoader(4, 1, (3, 16, 16), 10, dev, seed=1, channels_last=True, fresh=True)
    xc, tc = next(iter(cl))
    assert xc.shape == (4, 3, 16, 16) and xc.is_contiguous(memory_format=torch.channels_last) and tc.dtype == torch.int64


@pytest.mark.parametrize("case", [(3, 3, 224, 224, 7, 2, 3, torch.float32, True), (5, 3, 32, 32, 3, 1, 1, torch.float32, False),
                                  (2, 1, 37, 29, 5, 2, 2, torch.float32, False), (2, 4, 20, 300, 3, 1, 1, torch.bfloat16, True),
                                  (1, 8, 9, 9, 3, 2, 0, torch.float32, False)])
def test_stem_im2col_strip_kernel_equals_cell_kernel(dev, case, monkeypatch):
    """The strip kernel (input rows staged once in shared memory, division-free gathers) writes the same bf16 matrix as the
    per-cell kernel, bit for bit: RGB 7x7/2 ImageNet stem, CIFAR stem, odd sizes, output rows wider than one strip, bf16 and
    channels_last / NCHW-strided inputs."""
    from turboprune_b200 import ops
    n, c, h, w, k, s_, p_, dt, cl = case
    g = torch.Generator(device=dev).manual_seed(sum(case[:7]))
    x = torch.randn(n, c, h, w, device=dev, generator=g).to(dt)
    if cl:
        x = x.contiguous(memory_format=torch.channels_last)
    desc = ops.make_desc(n, h, w, c, 16, k, k, (s_, s_), (p_, p_))
    cg, kp = ops.stem_geometry(c, k, k)
    outs = []
    for mode in ("cell", "rows"):
        monkeypatch.setenv("TP_STEM_IM2COL", mode)
        outs.append(ops.im2col_stem(x, desc, kp, cg))
    assert torch.equal(outs[0].view(torch.int16), outs[1].view(torch.int16))
    # and against a direct unfold of the bf16-rounded input (column = tap * cg + channel)
    cols = torch.nn.functional.unfold(x.float().to(torch.bfloat16).float().contiguous(), k, padding=p_, stride=s_)   # [n, c*k*k, L]
    cols = cols.view(n, c, k * k, -1).permute(0, 3, 2, 1).reshape(n * desc.p * desc.q, k * k * c)
    assert torch.equal(outs[1][:, :k * k * c].float(), cols)
    assert float(outs[1][:, k * k * c:].abs().max()) == 0.0 if kp > k * k * c else True


@pytest.mark.parametrize("case", [(6, 64, 128, 3, 18), (4, 128, 256, 1, 14), (3, 64, 64, 3, 23)])
def test_bn_backward_reduction_in_dgrad_epilogue(dev, case):
    """conv_a -> BatchNorm+ReLU -> conv_b: with the fusion conv_b's dgrad writes g = dz * [z > 0] and the partial sums
    (sum g, sum g*xhat) so that the BatchNorm backward runs no reduction pass; against the unfused path: identical gate
    (exactly the same zeros), dgamma / dbeta to fp32 summation-order accuracy, input and weight gradients to bf16 accuracy;
    a BatchNorm whose output has two consumers falls back transparently."""
    import copy
    from turboprune_b200 import fused_norm as fn, ops
    from turboprune_b200.utils import mask_layers as ml
    b, c1, c2, k, hw = case
    g = torch.Generator(device=dev).manual_seed(sum(case))
    conv_a = ml.ConvMask(in_channels=64, out_channels=c1, kernel_size=3, padding=1, bias=False).to(dev)
    bn = fn.BatchNorm2dB200(c1).to(dev).train()
    conv_b = ml.ConvMask(in_channels=c1, out_channels=c2, kernel_size=k, padding=k // 2, bias=False).to(dev)
    with torch.no_grad():
        conv_a.mask.copy_((torch.rand(conv_a.weight.shape, device=dev, generator=g) < 0.5).float())
        conv_b.mask.copy_((torch.rand(conv_b.weight.shape, device=dev, generator=g) < 0.5).float())
        bn.weight.copy_(torch.rand(c1, device=dev, generator=g) + 0.5); bn.bias.copy_(torch.randn(c1, device=dev, generator=g) * 0.3)
    x = torch.randn(b, 64, hw, hw, device=dev, generator=g).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    res = []
    for fused in (False, True):
        ops.set_bn_bwd_fusion(fused)
        try:
            ca, bb, cb = copy.deepcopy(conv_a), copy.deepcopy(bn), copy.deepcopy(conv_b)
            xx = x.clone().requires_grad_(True)
            z, _ = fn._conv_bn(ca, bb, xx, relu=True)
            assert (getattr(z, "_tp_bn_src", None) is not None) == fused
            out = cb(z)
            gz = torch.Generator(device=dev).manual_seed(5)
            out.backward(torch.randn(out.shape, device=dev, generator=gz).to(out.dtype).contiguous(memory_format=torch.channels_last))
            assert not fn._PARTIALS                                   # the offer was consumed by the BatchNorm's backward
            res.append((xx.grad.float(), ca.weight.grad.clone(), bb.weight.grad.clone(), bb.bias.grad.clone(), cb.weight.grad.clone()))
        finally:
            ops.set_bn_bwd_fusion(True)
    u, f = res
    assert _rel(f[2], u[2]) < 1e-4 and _rel(f[3], u[3]) < 1e-4        # dgamma, dbeta: same terms, different summation order
    assert _rel(f[4], u[4]) == 0.0                                     # conv_b's wgrad does not depend on the fusion
    assert _rel(f[0], u[0]) < 2e-2 and _rel(f[1], u[1]) < 2e-2         # through bf16 dy: a last-bit flip of the coefficients at most
    # two consumers of the BatchNorm output: autograd sums the gradients, the hint cannot match, results stay right
    ca, bb, cb = copy.deepcopy(conv_a), copy.deepcopy(bn), copy.deepcopy(conv_b)
    xx = x.clone().requires_grad_(True)
    z, _ = fn._conv_bn(ca, bb, xx, relu=True)
    (cb(z).float().sum() + (z.float() * 0.5).sum()).backward()
    fn.drop_partials()
    ops.set_bn_bwd_fusion(False)
    try:
        ca2, bb2, cb2 = copy.deepcopy(conv_a), copy.deepcopy(bn), copy.deepcopy(conv_b)
        x2 = x.clone().requires_grad_(True)
        z2, _ = fn._conv_bn(ca2, bb2, x2, relu=True)
        (cb2(z2).float().sum() + (z2.float() * 0.5).sum()).backward()
    finally:
        ops.set_bn_bwd_fusion(True)
    assert _rel(bb.weight.grad, bb2.weight.grad) < 1e-4 and _rel(xx.grad, x2.grad) < 2e-2
