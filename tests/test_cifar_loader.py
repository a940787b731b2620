"""The CIFAR loader: data set readers, the loader choice, the epoch oracle against the reference's own batches
(cifar_loader_small.npz, written by running its CifarLoader), and on the GPU the tp_cifar_epoch kernel, CifarLoader and a
CIFAR-10 run of run_experiment on a generated data set."""
import csv
import json
import os
import pickle

import numpy as np
import pytest
import torch

import cifar_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


# ---------------------------------------------------------------- fixtures written into tmp_path --------------------
def write_pt(root, dataset, train, images, labels, classes=None):
    from turboprune_b200.utils.dataset import cifar_paths
    pt, _ = cifar_paths(str(root), train, dataset)
    os.makedirs(os.path.dirname(pt), exist_ok=True)
    torch.save({"images": torch.from_numpy(images), "labels": torch.from_numpy(labels),
                "classes": classes or [f"class{i}" for i in range(int(labels.max()) + 1)]}, pt)


def write_archive(root, dataset, images_by_file, labels_by_file, classes):
    """torchvision's extracted layout: pickled dicts with CHW-flattened uint8 rows."""
    from turboprune_b200.utils.dataset import cifar_paths
    _, archive = cifar_paths(str(root), True, dataset)
    os.makedirs(archive, exist_ok=True)
    key = "labels" if dataset == "CIFAR10" else "fine_labels"
    for name, imgs in images_by_file.items():
        with open(os.path.join(archive, name), "wb") as f:
            pickle.dump({"data": imgs.transpose(0, 3, 1, 2).reshape(len(imgs), -1),
                         key: [int(v) for v in labels_by_file[name]]}, f)
    meta, names = ("batches.meta", "label_names") if dataset == "CIFAR10" else ("meta", "fine_label_names")
    with open(os.path.join(archive, meta), "wb") as f:
        pickle.dump({names: classes}, f)


def learnable_set(n, seed, templates, noise=24.0):
    """Class k = a fixed random low-frequency template plus per-image noise: learnable in a few epochs only if the
    images keep their labels."""
    g = np.random.default_rng(seed)
    labels = g.integers(0, len(templates), size=n).astype(np.int64)
    x = templates[labels] + g.normal(0.0, noise, size=(n, 32, 32, 3))
    return np.clip(np.rint(x), 0, 255).astype(np.uint8), labels


def class_templates(k, seed=0):
    g = np.random.default_rng(seed)
    low = g.uniform(30, 225, size=(k, 4, 4, 3))
    return np.repeat(np.repeat(low, 8, axis=1), 8, axis=2)


# ---------------------------------------------------------------- CPU ------------------------------------------------
def test_pt_and_archive_readers_agree_and_cache(tmp_path):
    from turboprune_b200.utils.dataset import cifar_paths, load_cifar
    g = np.random.default_rng(1)
    for dataset, files in (("CIFAR10", [f"data_batch_{k}" for k in range(1, 6)]), ("CIFAR100", ["train"])):
        imgs = {f: g.integers(0, 256, size=(3, 32, 32, 3), dtype=np.uint8) for f in files}
        labs = {f: g.integers(0, 10, size=3).astype(np.int64) for f in files}
        classes = [f"k{i}" for i in range(10)]
        arch_root, pt_root = tmp_path / f"a_{dataset}", tmp_path / f"p_{dataset}"
        write_archive(arch_root, dataset, imgs, labs, classes)
        all_i = np.concatenate([imgs[f] for f in files]); all_l = np.concatenate([labs[f] for f in files])
        write_pt(pt_root, dataset, True, all_i, all_l, classes)
        pt_cache, _ = cifar_paths(str(arch_root), True, dataset)
        assert not os.path.exists(pt_cache)
        a = load_cifar(str(arch_root), True, dataset)              # converts the archive, leaves the cache
        assert os.path.isfile(pt_cache) and not os.path.exists(pt_cache + ".tmp")
        c = load_cifar(str(arch_root), True, dataset)              # now read from the cache
        p = load_cifar(str(pt_root), True, dataset)
        for d in (a, c):
            assert d["images"].dtype == torch.uint8 and d["images"].shape == (len(all_i), 32, 32, 3)
            assert np.array_equal(d["images"].numpy(), p["images"].numpy()) and np.array_equal(d["images"].numpy(), all_i)
            assert d["labels"].dtype == torch.int64 and np.array_equal(d["labels"].numpy(), all_l)
            assert d["classes"] == p["classes"] == classes


def test_missing_data_set_names_both_paths(tmp_path):
    from turboprune_b200.utils.dataset import CifarLoader, cifar_paths, load_cifar
    for dataset, train in (("CIFAR10", True), ("CIFAR100", False), ("cifar10", True)):
        pt, archive = cifar_paths(str(tmp_path), train, dataset)
        with pytest.raises(FileNotFoundError) as e:
            load_cifar(str(tmp_path), train, dataset)
        assert pt in str(e.value) and archive in str(e.value)
    assert cifar_paths("r", True, "cifar10")[0] == os.path.join("r", "cifar100", "cifar10_train.pt")   # case-sensitive, like upstream
    with pytest.raises(FileNotFoundError):
        CifarLoader(str(tmp_path), device="cpu")


def test_make_loaders_table(tmp_path):
    from turboprune_b200.utils.config import Cfg
    from turboprune_b200.utils.dataset import AirbenchLoaders, CifarLoader, SyntheticLoaders, make_loaders, uses_real_cifar
    write_pt(tmp_path, "CIFAR10", True, np.zeros((6, 32, 32, 3), np.uint8), np.arange(6, dtype=np.int64) % 3)
    write_pt(tmp_path, "CIFAR10", False, np.zeros((4, 32, 32, 3), np.uint8), np.arange(4, dtype=np.int64) % 3)

    def cfg(name, kind="absent"):
        dp = {"dataset_name": name, "total_batch_size": 4, "data_root_dir": str(tmp_path), "synthetic_steps_per_epoch": 1}
        if kind != "absent":
            dp["dataloader_type"] = kind
        return Cfg({"dataset_params": Cfg(dp), "experiment_params": Cfg({"seed": 0})})
    rows = [("CIFAR10", "absent", False), ("CIFAR10", "synthetic", False), ("CIFAR100", "synthetic", False),
            ("CIFAR10", "torch", True), ("cifar100", "torch", True), ("ImageNet", "absent", False),
            ("ImageNet", "ffcv", False), ("imagenet", "torch", False)]
    for name, kind, real in rows:
        assert uses_real_cifar(cfg(name, kind)) is real, (name, kind)
    for name, kind, real in rows:
        if real and name != "CIFAR10":
            continue                                    # no CIFAR-100 files written: the choice itself is checked above
        if real:
            loaders = make_loaders(cfg(name, kind), "cpu")
            assert isinstance(loaders, AirbenchLoaders) and isinstance(loaders.train_loader, CifarLoader)
            tr, te = loaders.train_loader, loaders.test_loader
            assert (tr.drop_last, tr.shuffle, tr.altflip, tr.aug) == (True, True, True, {"flip": True, "translate": 2})
            assert (te.drop_last, te.shuffle, te.aug) == (False, False, {})
            assert (len(tr), len(te), tr.batch_size) == (1, 1, 4)
            assert tr.images.dtype == torch.uint8 and tr.images.shape == (6, 32, 32, 3)
        else:
            assert isinstance(make_loaders(cfg(name, kind), "cpu"), SyntheticLoaders), (name, kind)


def test_oracle_matches_reference_loader_fixture():
    """The oracle's epochs, fed the draws the reference's CifarLoader made, equal every batch it yielded (CPU arithmetic)."""
    z = np.load(os.path.join(GOLDEN, "cifar_loader_small.npz"))
    cases = {"a": ("CIFAR10", 3, dict(batch_size=5, aug={"flip": True, "translate": 2}, altflip=True, train=True)),
             "b": ("CIFAR100", 2, dict(batch_size=4, aug={"flip": True, "translate": 2, "cutout": 4}, train=True)),
             "t": ("CIFAR10", 1, dict(batch_size=5, train=False))}
    for tag, (dataset, epochs, kw) in cases.items():
        mean, std = O.constants(dataset)
        draws = O.recorded([z[f"{tag}.draw{k}"] for k in range(int(z[f"{tag}.ndraws"]))])
        got = O.replay_loader(z[f"{tag}.images"], z[f"{tag}.labels"], mean, std, False, draws, epochs, **kw)
        assert len(got[0]) == int(z[f"{tag}.len"])
        for e, ep in enumerate(got):
            for b, (x, t) in enumerate(ep):
                assert np.array_equal(x, z[f"{tag}.e{e}.b{b}.x"]), (tag, e, b)
                assert np.array_equal(t, z[f"{tag}.e{e}.b{b}.y"]), (tag, e, b)
            assert f"{tag}.e{e}.b{len(ep)}.x" not in z
    assert [len(z[f"t.e0.b{b}.y"]) for b in range(4)] == [5, 5, 5, 1]          # the partial last test batch


def test_normalize_oracle_cpu_arithmetic_is_torch_cpu():
    """cuda_arith=False is the reference's expressions as torch evaluates them on the CPU; the CUDA form differs from it
    only by the rounding of images / 255 (one ulp of a value in [0, 1])."""
    import torchvision.transforms as T
    u = np.arange(256, dtype=np.uint8).reshape(1, 16, 16, 1).repeat(3, axis=3)
    for dataset in ("CIFAR10", "CIFAR100"):
        mean, std = O.constants(dataset)
        a, b = O.cifar_normalize(u, mean, std, False), O.cifar_normalize(u, mean, std, True)
        want = T.Normalize(torch.tensor(mean), torch.tensor(std))(torch.from_numpy(u).permute(0, 3, 1, 2) / 255)
        assert np.array_equal(a, want.contiguous().numpy())
        assert (a != b).any() and np.abs(a - b).max() <= 1e-6


# ---------------------------------------------------------------- GPU ------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device: the gpu-marked CIFAR loader tests run on the B200 box")
    from turboprune_b200 import _cabi
    _cabi.load()
    return torch.device("cuda", 0)


def torch_reference_normalize(u8_dev, mean, std):
    """The reference's expressions, evaluated by torch on the device: T.Normalize(mean, std)(u8 / 255 -> NCHW)."""
    import torchvision.transforms as T
    return T.Normalize(torch.tensor(mean), torch.tensor(std))(u8_dev.permute(0, 3, 1, 2) / 255)


@pytest.mark.gpu
def test_normalization_bit_exact_vs_torch_cuda(dev):
    from turboprune_b200.utils import dataset as ds
    u = torch.arange(256, dtype=torch.uint8).reshape(1, 16, 16, 1).repeat(1, 1, 1, 3)
    for dataset in ("CIFAR10", "CIFAR100"):
        mean, std = O.constants(dataset)
        want = torch_reference_normalize(u.to(dev), mean, std).contiguous().cpu().numpy()
        assert np.array_equal(O.cifar_normalize(u.numpy(), mean, std, True), want), dataset
        got, _ = ds.cifar_epoch(u.to(dev), None, tuple(map(float, mean)), tuple(map(float, std)))
        assert np.array_equal(got.cpu().numpy(), want), dataset


def _epoch_args(n, h, w, r, g, preflip=False, flip=False, flip_all=False, cut=0, perm=True):
    t = lambda a: torch.from_numpy(np.asarray(a))
    a = {}
    if perm:
        a["perm"] = t(g.permutation(n).astype(np.int64))
    if r:
        a["shifts"], a["r"] = t(g.integers(-r, r + 1, size=(n, 2)).astype(np.int64)), r
    if preflip:
        a["preflip"] = t(g.random(n) < 0.5)
    if flip:
        a["flip"] = t(g.random(n) < 0.5)
    a["flip_all"] = flip_all
    if cut:
        a["cut_y"] = t(g.integers(0, h - cut + 1, size=n).astype(np.int64))
        a["cut_x"] = t(g.integers(0, w - cut + 1, size=n).astype(np.int64))
        a["cut_size"] = cut
    return a


EPOCH_CASES = [  # n, c, h, w, r, preflip, flip, flip_all, cut, perm
    (37, 3, 32, 32, 2, True, False, True, 0, True),
    (37, 3, 32, 32, 2, True, True, False, 8, True),
    (20, 3, 32, 32, 0, False, False, False, 0, False),
    (300, 3, 32, 32, 4, False, True, False, 5, True),
    (11, 3, 12, 20, 3, True, False, True, 4, True),          # non-square, float4 rows
    (13, 3, 9, 10, 2, True, True, False, 9, True),           # non-square, rows not a multiple of 4, cutout = h
    (7, 1, 31, 29, 30 - 2, False, True, False, 0, True),     # one channel, r = h-3 (deep reflection)
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", EPOCH_CASES)
def test_epoch_kernel_vs_oracle(dev, case):
    from turboprune_b200.utils import dataset as ds
    n, c, h, w, r, preflip, flip, flip_all, cut, perm = case
    r = min(r, h - 1, w - 1)
    g = np.random.default_rng(n * 131 + h)
    u8 = g.integers(0, 256, size=(n, h, w, c), dtype=np.uint8)
    labels = g.integers(0, 100, size=n).astype(np.int64)
    mean, std = g.uniform(0.3, 0.6, size=c).astype(np.float32), g.uniform(0.2, 0.3, size=c).astype(np.float32)
    a = _epoch_args(n, h, w, r, g, preflip, flip, flip_all, cut, perm)
    want_x, want_t = O.cifar_epoch(u8, labels, mean, std, True, **{k: (v.numpy() if torch.is_tensor(v) else v) for k, v in a.items()})
    got_x, got_t = ds.cifar_epoch(torch.from_numpy(u8).to(dev), torch.from_numpy(labels).to(dev), tuple(map(float, mean)),
                                  tuple(map(float, std)), **{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in a.items()})
    assert got_x.shape == (n, c, h, w) and got_x.is_contiguous()
    assert np.array_equal(got_x.cpu().numpy(), want_x) and np.array_equal(got_t.cpu().numpy(), want_t)


@pytest.mark.gpu
def test_epoch_kernel_with_reference_fixture_draws(dev):
    """Fixture case a (the AirbenchLoaders train augmentation): the kernel reproduces the reference's batches up to the
    CPU/CUDA rounding of images / 255, and equals the oracle's CUDA arithmetic bit for bit."""
    from turboprune_b200.utils import dataset as ds
    z = np.load(os.path.join(GOLDEN, "cifar_loader_small.npz"))
    u8, labels = z["a.images"], z["a.labels"]
    mean, std = O.constants("CIFAR10")
    pre = z["a.draw0"] < 0.5
    k = 1
    for e in range(3):
        sh, perm = z[f"a.draw{k}"], z[f"a.draw{k + 1}"]; k += 2
        args = dict(perm=perm, shifts=sh, r=2, preflip=pre, flip_all=e % 2 == 1)
        want_x, want_t = O.cifar_epoch(u8, labels, mean, std, True, **args)
        got_x, got_t = ds.cifar_epoch(torch.from_numpy(u8).to(dev), torch.from_numpy(labels).to(dev), tuple(map(float, mean)),
                                      tuple(map(float, std)), **{a: (torch.from_numpy(np.asarray(v)).to(dev) if isinstance(v, np.ndarray) else v)
                                                                 for a, v in args.items()})
        got_x, got_t = got_x.cpu().numpy(), got_t.cpu().numpy()
        assert np.array_equal(got_x, want_x) and np.array_equal(got_t, want_t)
        ref_x = np.concatenate([z[f"a.e{e}.b{b}.x"] for b in range(3)])
        assert np.array_equal(got_t[:15], np.concatenate([z[f"a.e{e}.b{b}.y"] for b in range(3)]))
        assert np.abs(got_x[:15] - ref_x).max() <= 1e-6


@pytest.mark.gpu
def test_epoch_kernel_rejects_invalid_arguments(dev):
    from ctypes import c_float, c_void_p
    from turboprune_b200 import _cabi
    lib = _cabi.load()
    u8 = torch.zeros(4, 32, 32, 3, dtype=torch.uint8, device=dev)
    out = torch.empty(4, 3, 32, 32, device=dev)
    i64 = torch.zeros(8, dtype=torch.int64, device=dev)
    P = lambda t: c_void_p(t.data_ptr())
    m, s = (c_float * 4)(0.5, 0.5, 0.5, 0.5), (c_float * 4)(0.25, 0.25, 0.25, 0.25)
    st = _cabi.stream_ptr(dev)

    def call(src=P(u8), shifts=None, r=0, flip=None, flip_all=0, cy=None, cx=None, cut=0, c=3, h=32, w=32, mean=m, labels=None,
             labels_out=None):
        return lib.tp_cifar_epoch(src, labels, P(out), labels_out, None, shifts, r, None, flip, flip_all, cy, cx, cut, mean, s,
                                  4, c, h, w, st)
    assert call() == 0
    torch.cuda.synchronize()
    bad = [dict(src=None), dict(mean=None), dict(c=5), dict(c=0), dict(h=0), dict(r=32, shifts=P(i64)), dict(r=-1),
           dict(h=4, r=4, shifts=P(i64)), dict(shifts=P(i64), r=0), dict(cy=P(i64), cx=None, cut=2), dict(cy=P(i64), cx=P(i64), cut=0),
           dict(cy=P(i64), cx=P(i64), cut=33), dict(flip=P(u8), flip_all=1), dict(labels=P(i64)),
           dict(h=84, w=84)]                                                    # 20.7 KiB: over the staging limit
    for kw in bad:
        assert call(**kw) == -1, kw


def _remake_draws(dev, n, h, w, epochs, aug, altflip, shuffle):
    """The reference CifarLoader.__iter__'s draws, in its order, from the current CUDA generator state."""
    out = []
    for e in range(epochs):
        if e == 0 and aug.get("flip"):
            out.append(torch.rand(n, device=dev))
        if aug.get("translate", 0):
            r = aug["translate"]
            out.append(torch.randint(-r, r + 1, size=(n, 2), device=dev))
        if aug.get("flip") and not altflip:
            out.append(torch.rand(n, device=dev))
        if aug.get("cutout", 0):
            out.append(torch.randint(0, h - aug["cutout"] + 1, size=(n,), device=dev))
            out.append(torch.randint(0, w - aug["cutout"] + 1, size=(n,), device=dev))
        if shuffle:
            out.append(torch.randperm(n, device=dev))
    return [d.cpu().numpy() for d in out]


@pytest.mark.gpu
@pytest.mark.parametrize("dataset,aug,altflip,bs", [
    ("CIFAR10", {"flip": True, "translate": 2}, True, 64),
    ("CIFAR100", {"flip": True, "translate": 3, "cutout": 6}, False, 50),
])
def test_cifar_loader_end_to_end_vs_oracle(dev, tmp_path, dataset, aug, altflip, bs):
    from turboprune_b200.utils.dataset import CifarLoader
    g = np.random.default_rng(7)
    ntr, nte = 300, 130
    tr_u8, tr_l = g.integers(0, 256, size=(ntr, 32, 32, 3), dtype=np.uint8), g.integers(0, 100, size=ntr).astype(np.int64)
    te_u8, te_l = g.integers(0, 256, size=(nte, 32, 32, 3), dtype=np.uint8), g.integers(0, 100, size=nte).astype(np.int64)
    classes = [f"class{k}" for k in range(100)]
    write_pt(tmp_path, dataset, True, tr_u8, tr_l, classes)
    write_pt(tmp_path, dataset, False, te_u8, te_l, classes)
    mean, std = O.constants(dataset)
    torch.manual_seed(123)
    tr = CifarLoader(str(tmp_path), train=True, batch_size=bs, aug=aug, altflip=altflip, dataset=dataset, device=dev)
    te = CifarLoader(str(tmp_path), train=False, batch_size=bs, dataset=dataset, device=dev)
    assert len(tr) == ntr // bs and len(te) == -(-nte // bs) and tr.classes == te.classes
    assert tr.images.device == dev and tr.images.dtype == torch.uint8
    state = torch.cuda.get_rng_state(dev)
    it = iter(tr)
    assert torch.equal(torch.cuda.get_rng_state(dev), state) and tr.epoch == 0       # nothing drawn before next()
    got = []
    for e in range(3):
        got.append([(x.cpu().numpy(), t.cpu().numpy()) for x, t in (it if e == 0 else tr)])
        assert tr.epoch == e + 1
    with pytest.raises(AssertionError):
        tr.images = tr.images
    after = torch.cuda.get_rng_state(dev)
    torch.manual_seed(123)
    draws = _remake_draws(dev, ntr, 32, 32, 3, aug, altflip, True)
    assert torch.equal(torch.cuda.get_rng_state(dev), after)                        # same stream consumed, same order
    want = O.replay_loader(tr_u8, tr_l, mean, std, True, O.recorded(draws), 3, bs, aug=aug, train=True, altflip=altflip)
    for e in range(3):
        assert len(got[e]) == len(want[e]) == len(tr)
        for (gx, gt), (wx, wt) in zip(got[e], want[e]):
            assert gx.shape == (bs, 3, 32, 32) and np.array_equal(gx, wx) and np.array_equal(gt, wt)
    # the test loader: stored order, no draws, the partial last batch
    state = torch.cuda.get_rng_state(dev)
    tb = [(x.cpu().numpy(), t.cpu().numpy()) for x, t in te]
    assert torch.equal(torch.cuda.get_rng_state(dev), state)
    assert [len(t) for _, t in tb] == [bs] * (nte // bs) + [nte % bs]
    wx, wt = O.cifar_epoch(te_u8, te_l, mean, std, True)
    assert np.array_equal(np.concatenate([x for x, _ in tb]), wx) and np.array_equal(np.concatenate([t for _, t in tb]), wt)


@pytest.mark.gpu
def test_batches_survive_the_next_epoch_and_one_batch_leaves_upstreams_rng(dev, tmp_path):
    """Every epoch gets a fresh buffer (a held batch is not overwritten); taking one batch and stopping, as prune_snip /
    prune_synflow do, consumes exactly the draws of the reference's first next()."""
    from turboprune_b200.utils.dataset import CifarLoader
    g = np.random.default_rng(9)
    write_pt(tmp_path, "CIFAR10", True, g.integers(0, 256, size=(40, 32, 32, 3), dtype=np.uint8), g.integers(0, 10, size=40).astype(np.int64))
    torch.manual_seed(5)
    tr = CifarLoader(str(tmp_path), train=True, batch_size=8, aug={"flip": True, "translate": 2}, altflip=True, device=dev)
    for x, _ in tr:
        break
    first = x.clone()
    after = torch.cuda.get_rng_state(dev)
    torch.manual_seed(5)
    _remake_draws(dev, 40, 32, 32, 1, {"flip": True, "translate": 2}, True, True)
    assert torch.equal(torch.cuda.get_rng_state(dev), after)
    for _ in tr:
        pass
    assert torch.equal(x, first)


@pytest.mark.gpu
def test_run_experiment_trains_on_a_cifar10_file(dev, tmp_path):
    """The reference's cifar10_er_erk config (dataloader_type: torch) through run_experiment.main reads the data set
    from data_root_dir and learns it: a generated 10-class set whose classes are noisy copies of fixed templates."""
    import yaml
    import run_experiment
    from turboprune_b200.utils import config as C
    conf = tmp_path / "conf"
    for rel, data in json.load(open(os.path.join(GOLDEN, "reference_models.json")))["conf"].items():
        (conf / rel).parent.mkdir(parents=True, exist_ok=True)
        (conf / rel).write_text(yaml.safe_dump(data))
    tpl = class_templates(10)
    data = tmp_path / "data"
    write_pt(data, "CIFAR10", True, *learnable_set(4000, 1, tpl))
    write_pt(data, "CIFAR10", False, *learnable_set(1000, 2, tpl))
    cfg = C.compose("cifar10_er_erk", [f"dataset_params.data_root_dir={data}", f"experiment_params.base_dir={tmp_path / 'ex'}",
                                       "dataset_params.total_batch_size=128", "experiment_params.epochs_per_level=3",
                                       "+pruning_params.target_sparsity=0.8"], str(conf))
    assert cfg.dataset_params.dataloader_type == "torch"
    prefix, expt = run_experiment.main(cfg)
    rows = list(csv.DictReader(open(os.path.join(expt, f"{prefix}_summary.csv"))))
    acc = float(rows[-1]["Last_Test_Acc"])
    print(f"[cifar10_er_erk on the generated set] sparsity {rows[-1]['Sparsity']} last test acc {acc:.2f} %")
    assert 75.0 < float(rows[-1]["Sparsity"]) < 90.0                          # ER-ERK draws around the 80 % target
    assert acc >= 50.0, acc                                                   # 100 % measured on a B200; chance is 10 %
    # without the file the run stops with the missing path
    cfg = C.compose("cifar10_er_erk", [f"dataset_params.data_root_dir={tmp_path / 'nowhere'}", f"experiment_params.base_dir={tmp_path / 'ex'}",
                                       "+pruning_params.target_sparsity=0.8"], str(conf))
    with pytest.raises(FileNotFoundError, match="CIFAR10_train.pt"):
        run_experiment.main(cfg)
