"""CPU: the oracle (numpy / torch-CPU restatement) against the golden fixtures produced by the
unmodified reference (tests/golden/make_golden.py)."""
import json
import os

import numpy as np
import pytest
import torch

import oracle
from oracle import prune as P
from oracle import mask_ops as M

G = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def ops_npz():
    return np.load(os.path.join(G, "ops_small.npz"))


@pytest.fixture(scope="module")
def prune_npz():
    return np.load(os.path.join(G, "prune_small.npz"))


def T(a):
    return torch.from_numpy(np.asarray(a))


@pytest.mark.parametrize("name", ["conv3x3", "conv3x3s2", "conv1x1s2", "conv7x7s2"])
def test_masked_conv_matches_reference(ops_npz, name):
    z = ops_npz
    s, p = (int(v) for v in z[f"{name}.cfg"])
    b = T(z[f"{name}.b"]) if f"{name}.b" in z else None
    y = M.masked_conv2d(T(z[f"{name}.x"]), T(z[f"{name}.w"]), T(z[f"{name}.m"]), b, s, p)
    assert torch.allclose(y, T(z[f"{name}.y"]), rtol=1e-5, atol=1e-6)
    dx, dw, db = M.masked_conv2d_grads(T(z[f"{name}.x"]), T(z[f"{name}.w"]), T(z[f"{name}.m"]), T(z[f"{name}.dy"]), s, p,
                                       has_bias=b is not None)
    assert torch.allclose(dx, T(z[f"{name}.dx"]), rtol=1e-4, atol=1e-5)
    assert torch.allclose(dw, T(z[f"{name}.dw"]), rtol=1e-4, atol=1e-5)
    # the gradient of a masked weight is exactly zero
    assert (dw[T(z[f"{name}.m"]) == 0] == 0).all()
    if b is not None:
        assert torch.allclose(db, T(z[f"{name}.db"]), rtol=1e-4, atol=1e-5)


def test_masked_linear_and_conv1d_match_reference(ops_npz):
    z = ops_npz
    y = M.masked_conv1d_k1(T(z["conv1d.x"]), T(z["conv1d.w"]), T(z["conv1d.m"]), T(z["conv1d.b"]))
    assert torch.allclose(y, T(z["conv1d.y"]), rtol=1e-5, atol=1e-6)
    dx, dw, db = M.masked_linear_grads(T(z["conv1d.x"]), T(z["conv1d.w"])[:, :, 0], T(z["conv1d.m"])[:, :, 0], T(z["conv1d.dy"]),
                                       has_bias=True)
    assert torch.allclose(dx, T(z["conv1d.dx"]), rtol=1e-4, atol=1e-5)
    assert torch.allclose(dw, T(z["conv1d.dw"])[:, :, 0], rtol=1e-4, atol=1e-5)
    assert torch.allclose(db, T(z["conv1d.db"]), rtol=1e-4, atol=1e-5)
    y = M.masked_linear(T(z["linear.x"]), T(z["linear.w"]), T(z["linear.m"]), T(z["linear.b"]))
    assert torch.allclose(y, T(z["linear.y"]), rtol=1e-5, atol=1e-6)
    dx, dw, db = M.masked_linear_grads(T(z["linear.x"]), T(z["linear.w"]), T(z["linear.m"]), T(z["linear.dy"]), has_bias=True)
    assert torch.allclose(dx, T(z["linear.dx"]), rtol=1e-4, atol=1e-5)
    assert torch.allclose(dw, T(z["linear.dw"]), rtol=1e-4, atol=1e-5)


def _ws(z):
    return [z[f"w{i}"] for i in range(4)]


def test_prune_mag_levels_bit_exact(prune_npz):
    z = prune_npz
    ws = _ws(z)
    ms = [np.ones_like(w) for w in ws]
    for lvl, d in enumerate([0.8, 0.64, 0.3]):
        ms, thr, k = P.prune_global(ws, ms, d)
        for i in range(4):
            assert np.array_equal(ms[i], z[f"mag{lvl}.m{i}"]), (lvl, i)
    # density goes UP on a sparse net: threshold falls inside the zeros, masks unchanged
    ms2, thr, k = P.prune_global(ws, ms, 0.9)
    assert thr == 0.0
    for i in range(4):
        assert np.array_equal(ms2[i], z[f"mag_up.m{i}"])
        assert np.array_equal(ms2[i], ms[i])


@pytest.mark.parametrize("tag,kind", [("snip", P.SCORE_SNIP), ("synflow", P.SCORE_SYNFLOW)])
def test_prune_grad_scores_bit_exact(prune_npz, tag, kind):
    z = prune_npz
    # synflow scores the linearised |w| with the gradients the reference held right before its model.zero_grad()
    # (pruning_utils.py:263-270); make_golden.py captures both from the running reference
    ws = [z[f"synflow.absw{i}"] for i in range(4)] if tag == "synflow" else _ws(z)
    gs = [z[f"{tag}.g{i}"] for i in range(4)]
    ms = [np.ones_like(w) for w in ws]
    new, thr, k = P.prune_global(ws, ms, 0.5, gs=gs, kind=kind)
    for i in range(4):
        assert np.array_equal(new[i], z[f"{tag}.m{i}"])


def test_ties_are_pruned_and_k0_raises():
    w = [np.array([[1, 1, 1, 2], [2, 3, 4, 5]], np.float32)]
    m = [np.ones_like(w[0])]
    new, thr, k = P.prune_global(w, m, 0.75)          # k = 2 -> thr = 1 -> all three 1s go
    assert k == 2 and thr == 1.0 and int((new[0] == 0).sum()) == 3
    with pytest.raises(RuntimeError):
        P.prune_global(w, m, 1.0)                     # k == 0: torch.kthvalue raises in the reference


def test_kth_smallest_matches_torch_including_nan_and_negzero():
    rng = np.random.RandomState(0)
    x = rng.randn(5000).astype(np.float32)
    x[:7] = np.nan; x[7:20] = 0.0; x[20:25] = -0.0; x[25] = np.inf; x[26] = -np.inf
    for k in (1, 2, 13, 2500, 4990, 4993, 4994, 5000):
        a = P.kth_smallest(x, k); b = torch.kthvalue(torch.from_numpy(x), k)[0].item()
        assert (np.isnan(a) and np.isnan(b)) or a == b, k


def test_keep_probabilities_match_reference():
    probs = json.load(open(os.path.join(G, "probs.json")))
    for key, e in probs.items():
        shapes = [tuple(s) for s in e["shapes"]]
        for d in (0.2, 0.05):
            erk = P.erk_keep_probabilities(shapes, d)
            assert [float(p).hex() for p in erk] == e[f"erk@{d}"], key
            bal = P.balanced_keep_probabilities([int(np.prod(s)) for s in shapes], d)
            assert [float(b).hex() for b in bal] == e[f"balanced@{d}"], key


def test_generate_densities_match_reference():
    dens = json.load(open(os.path.join(G, "densities.json")))
    for key, vals in dens.items():
        method, target, rate = key.split("|")
        got = P.generate_densities(method, float(target), float(rate), 0.0)
        assert [float(x).hex() for x in got] == vals, key
    assert len(P.generate_densities("mag", 0.988, 0.2)) == 21      # "20 prune cycles" + the dense level


def test_sgd_matches_torch_trajectory():
    z = np.load(os.path.join(G, "sgd_small.npz"))
    w, buf = z["w0"], None
    for step in range(3):
        w, buf = oracle.sgd_momentum_step(w, z[f"g{step}"], buf, 0.2, 0.9, 5e-4, step == 0)
        # torch fuses g + wd*w and w - lr*buf into FMAs, numpy rounds each product: <= 4 ulp apart
        assert np.allclose(w, z[f"w{step + 1}"], rtol=5e-7, atol=1e-7)


def test_allreduce_mean_mask_fixed_order():
    rng = np.random.RandomState(1)
    gs = [rng.randn(1000).astype(np.float32) for _ in range(4)]
    m = (rng.rand(1000) < 0.5).astype(np.float32)
    out = oracle.allreduce_mean_mask(gs, m)
    ref = (gs[0] / 4 + gs[1] / 4 + gs[2] / 4 + gs[3] / 4) * m      # DDP: divide first, then sum (power of two: identical)
    assert np.array_equal(out, ref.astype(np.float32))


def test_oracle_matches_reference_fixture():
    """Seed-0 ResNet-18 / CIFAR-10 of the oracle against the reference's (reference_models.json, reference_run.npz):
    bit-identical state dict, eval logits and masks after magnitude pruning to 80 % density."""
    import refshim
    import oracle.model as om
    ref = json.load(open(os.path.join(G, "reference_models.json")))["resnet18_cifar10"]
    run = np.load(os.path.join(G, "reference_run.npz"))
    torch.manual_seed(0); mine = om.build("resnet18", "cifar10")
    assert refshim.state_digests({"model." + k: v for k, v in mine.state_dict().items()}) == ref["init"]
    mine.eval()
    assert torch.equal(mine(T(run["logits.x"])), T(run["logits.y"]))
    layers = om.masked_layers(mine)
    new, thr, k = P.prune_global([m.weight.detach().numpy() for _, m in layers], [m.mask.numpy() for _, m in layers], 0.8)
    assert refshim.state_digests({n: T(a) for (n, _), a in zip(layers, new)}) == ref["prune_mag_0.8_masks"]
    h = json.load(open(os.path.join(G, "imp_hashes.json")))
    import hashlib
    hh = hashlib.sha256()
    for a in new:
        hh.update(np.ascontiguousarray(a).tobytes())
    assert hh.hexdigest() == h["levels"][0]["masks_sha256"]
    assert int(np.float32(thr).view(np.uint32)) == h["levels"][0]["thr_bits"]


# ---------------------------------------------------------------- data path (SURVEY §8(f) row 3) --------------------
def test_augmentation_oracle_matches_reference_fixtures():
    """oracle.data.batch_crop / batch_flip_lr / batch_cutout / augment against outputs of the reference's own functions
    (utils/dataset.py:38-98, fixtures written by make_golden.py)."""
    from oracle import data as D
    z = np.load(os.path.join(G, "aug_small.npz"))
    assert np.array_equal(D.batch_crop(z["padded"], 12, z["crop2.shifts"]), z["crop2.out"])
    assert np.array_equal(D.batch_crop(z["padded4"], 12, z["crop4.shifts"]), z["crop4.out"])
    assert np.array_equal(D.batch_flip_lr(z["imgs"], z["flip.mask"]), z["flip.out"])
    assert np.array_equal(D.batch_cutout(z["imgs"], 5, z["cut.y"], z["cut.x"]), z["cut.out"])
    assert np.array_equal(D.augment(z["padded4"], 12, z["epoch.shifts"], z["epoch.mask"], 3, z["epoch.y"], z["epoch.x"]), z["epoch.out"])
    r = np.load(os.path.join(G, "reference_run.npz"))                  # translate = 3
    assert np.array_equal(D.batch_crop(r["crop3.padded"], 10, r["crop3.shifts"]), r["crop3.out"])


def test_philox_known_answer_and_generator_statistics():
    """Philox4x32-10 pinned by Random123's known-answer vector (counter 0, key 0); the derived normals / labels behave."""
    from oracle import data as D
    w = D.philox4x32_10(np.array([0], dtype=np.uint64), 0)[0]
    assert [int(x) for x in w] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    x = D.synth_normal(200_000, seed=7)
    assert abs(float(x.mean())) < 0.01 and abs(float(x.std()) - 1.0) < 0.01 and np.isfinite(x).all()
    t = D.synth_labels(100_000, 10, seed=7)
    assert t.min() == 0 and t.max() == 9 and abs(np.bincount(t, minlength=10) / 1e5 - 0.1).max() < 0.01
    assert not np.array_equal(D.synth_words(64, 7, 0), D.synth_words(64, 7, 16))       # counter offset moves the stream
    assert np.array_equal(D.synth_words(64, 7, 16)[:32], D.synth_words(128, 7, 0)[64:96])
