"""CPU: the C-ABI library builds for sm_100a, loads, exports every symbol the header declares; host-side
mirrors keep the reference's surface; the product refuses to run without CUDA."""
import json
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def test_library_exports_every_declared_symbol(built_lib):
    from turboprune_b200 import _cabi
    header = open(os.path.join(ROOT, "include", "turboprune_b200.h")).read()
    declared = set(re.findall(r"\b(tp_[a-z0-9_]+)\s*\(", header)) - {"tp_conv_desc"}
    lib = _cabi.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
        assert name in _cabi.SIGNATURES, f"{name} has no ctypes signature"
    assert set(_cabi.SIGNATURES) <= declared
    assert lib.tp_abi_version() >= 1
    assert b"range" in lib.tp_strerror(-4)


def test_sass_contains_blackwell_tensor_and_tma_instructions(built_lib):
    import shutil, subprocess
    cu = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.isfile(cu):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cu, "-sass", built_lib], stdout=subprocess.PIPE, text=True).stdout
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, mnemonic


def test_no_cpu_fallback():
    from turboprune_b200.utils.mask_layers import ConvMask, Conv1dMask
    with pytest.raises(RuntimeError):
        ConvMask(in_channels=8, out_channels=8, kernel_size=3, padding=1)(torch.randn(1, 8, 4, 4))
    with pytest.raises(RuntimeError):
        Conv1dMask(8, 4)(torch.randn(2, 8))


def test_mask_layer_surface():
    from turboprune_b200.utils import mask_layers as ml
    c = ml.ConvMask(in_channels=4, out_channels=6, kernel_size=3, stride=2, padding=1, bias=False)
    assert c.mask.dtype == torch.float32 and c.mask.shape == c.weight.shape and bool((c.mask == 1).all())
    assert "mask" in dict(c.named_buffers()) and "mask" in c.state_dict()
    torch.manual_seed(0); c.set_er_mask(0.3)
    torch.manual_seed(0); ref = torch.zeros_like(c.weight).bernoulli_(0.3)
    assert torch.equal(c.mask, ref) and "mask" in dict(c.named_buffers())      # re-assignment keeps the buffer registered
    f = ml.Conv1dMask(10, 3, bias=True)
    assert f.weight.shape == (3, 10, 1) and f.mask.shape == (3, 10, 1)
    l = ml.LinearMask(in_features=10, out_features=3, bias=True)
    assert l.mask.shape == (3, 10)


def test_custom_models_build_like_the_reference():
    import refshim
    from turboprune_b200.utils import custom_models as cm, pruning_utils as pu
    torch.manual_seed(0)
    m = cm.TorchVisionModel(refshim.make_cfg("resnet18", "cifar10"))
    names = [n for n, _ in m._masked()]
    assert len(names) == 21 and names[0] == "conv1" and names[-1] == "fc"
    assert m.get_overall_sparsity() == 0
    sd = m.model.state_dict()
    assert sd["fc.weight"].shape == (10, 512, 1) and sd["conv1.mask"].dtype == torch.float32
    # the reference's seed-0 model and its ER masks (tests/golden/make_golden.py): bit-identical state dicts
    ref = json.load(open(os.path.join(GOLDEN, "reference_models.json")))["resnet18_cifar10"]
    assert refshim.state_digests(m.state_dict()) == ref["init"]
    for fn in ("prune_er_erk", "prune_er_balanced"):
        torch.manual_seed(5); getattr(pu, fn)(m, 0.2)
        assert refshim.state_digests(m.state_dict()) == ref[fn]["state"]
        assert m.get_overall_sparsity() == ref[fn]["sparsity_percent"]       # percent
    # vgg16 / cifar100 surgery
    v = cm.TorchVisionModel(refshim.make_cfg("vgg16", "cifar100"))
    assert len(v._masked()) == 16 and v.model.state_dict()["classifier.6.weight"].shape == (100, 4096, 1)


def test_prune_dispatcher_semantics():
    import refshim
    from turboprune_b200.utils import pruning_utils as pu

    class Console:
        def __init__(self): self.lines = []
        def print(self, *a, **k): self.lines.append(" ".join(str(x) for x in a))

    class H:
        distributed = False
        console = Console()
        train_loader = None
        class model:
            @staticmethod
            def get_overall_sparsity(): return 0.0
    cfg = refshim.make_cfg(prune_method="does_not_exist")
    assert pu.prune_the_model(cfg, H, 0.5) is None              # unknown method: message, no exception
    assert any("Unknown pruning method" in l for l in H.console.lines)
    assert pu.get_dtype_amp(refshim.make_cfg(precision="bfloat16")) == (torch.bfloat16, True)
    assert pu.get_dtype_amp(refshim.make_cfg(precision="float32")) == (torch.float32, False)


def test_fused_sgd_state_dict_is_torch_compatible():
    from turboprune_b200.optim import FusedSGD
    p = torch.nn.Parameter(torch.randn(5))
    a = FusedSGD([p], lr=0.2, momentum=0.9, weight_decay=1e-4)
    b = torch.optim.SGD([p], lr=0.2, momentum=0.9, weight_decay=1e-4)
    ga, gb = a.state_dict()["param_groups"][0], b.state_dict()["param_groups"][0]
    for key in ("lr", "momentum", "weight_decay", "dampening", "nesterov"):
        assert ga[key] == gb[key]
    sched = torch.optim.lr_scheduler.LambdaLR(a, lambda i: 0.5)
    assert a.param_groups[0]["lr"] == pytest.approx(0.1)


def test_config_composer_and_densities(tmp_path):
    import yaml
    from turboprune_b200.utils import config as C
    from turboprune_b200.utils.harness_utils import generate_densities
    c = C.compose("synthetic_rn18_imp", ["experiment_params.epochs_per_level=3"], os.path.join(ROOT, "conf_b200"))
    assert c.pruning_params.prune_method == "mag" and c.experiment_params.epochs_per_level == 3
    assert isinstance(c.optimizer_params.weight_decay, float)             # '5e-4' is a float like under hydra
    assert generate_densities(c, 0.0) == [1.0, 0.8]
    with pytest.raises(KeyError):
        C.compose("synthetic_rn18_imp", ["pruning_params.rewind_epoch=1"], os.path.join(ROOT, "conf_b200"))   # needs '+'
    c = C.compose("synthetic_rn18_imp", ["+pruning_params.rewind_epoch=1", "pruning_params=er_erk_80"], os.path.join(ROOT, "conf_b200"))
    assert c.pruning_params.prune_method == "er_erk" and c.pruning_params.rewind_epoch == 1
    # the reference's own conf/ files, consumed unchanged (SURVEY Appendix D, configs 1-3), restored from the fixture
    ref_conf = tmp_path / "conf"
    for rel, data in json.load(open(os.path.join(GOLDEN, "reference_models.json")))["conf"].items():
        (ref_conf / rel).parent.mkdir(parents=True, exist_ok=True)
        (ref_conf / rel).write_text(yaml.safe_dump(data))
    c = C.compose("cifar10_er_erk", ["pruning_params=iterative_imp", "pruning_params.target_sparsity=0.2"], str(ref_conf))
    assert generate_densities(c, 0.0) == [1.0, 0.8] and c.model_params.model_name == "resnet18"
    c = C.compose("imagenet_er_balanced", ["pruning_params=pai_er_erk", "+pruning_params.target_sparsity=0.8"], str(ref_conf))
    assert c.dataset_params.total_batch_size == 512 and generate_densities(c, 0.0) == [1 - 0.8]
    c = C.compose("imagenet_er_balanced", ["pruning_params=iterative_wr", "pruning_params.target_sparsity=0.988"], str(ref_conf))
    assert len(generate_densities(c, 0.0)) == 21


def test_cli_override_floats_parse_like_hydra():
    """'5e-4' / '1e-1' on the command line are floats for hydra; PyYAML alone would hand the harness strings."""
    from turboprune_b200.utils import config as C
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cfg = C.compose("synthetic_rn18_imp", ["optimizer_params.weight_decay=5e-4", "optimizer_params.lr=1e-1",
                                           "+pruning_params.rewind_epoch=2", "model_params.model_name=resnet50"],
                    os.path.join(root, "conf_b200"))
    assert cfg.optimizer_params.weight_decay == 5e-4 and isinstance(cfg.optimizer_params.weight_decay, float)
    assert cfg.optimizer_params.lr == 0.1 and cfg.pruning_params.rewind_epoch == 2 and cfg.model_params.model_name == "resnet50"


def test_mask_epoch_counts_new_mask_tensors():
    """Captured graphs / pointer tables key on it: assigning a mask bumps it, in-place edits and other attributes do not."""
    from turboprune_b200.utils import mask_layers as ml
    m = ml.ConvMask(in_channels=8, out_channels=8, kernel_size=1)
    e0 = ml.mask_epoch()
    m.mask.fill_(0.0); m.weight.data.mul_(2); m.foo = 1
    assert ml.mask_epoch() == e0
    m.set_er_mask(0.5)
    assert ml.mask_epoch() == e0 + 1
    m.mask = torch.ones_like(m.weight)
    assert ml.mask_epoch() == e0 + 2 and "mask" in dict(m.named_buffers())


def test_operand_planning_of_the_weight_shadow():
    """Host-side layout decisions shared by the per-layer staging and the one-launch WeightStager."""
    from turboprune_b200 import ops
    assert ops.stem_geometry(3, 7, 7) == (3, 152)            # RGB 7x7 stem: 147 real columns, K padded to 8
    assert ops.stem_geometry(3, 3, 3) == (3, 32)             # CIFAR stem
    assert ops.stem_geometry(8, 3, 3) == (8, 72)
    assert ops._operand_plan(64, 3, 7, 7) == (3, 64, False, 152)          # stem: no dgrad operand
    assert ops._operand_plan(64, 64, 3, 3) == (64, 64, True, 576)
    assert ops._operand_plan(96, 64, 3, 3) == (64, 128, True, 576)        # multi-tap backward walks Cout in 64-blocks
    assert ops._operand_plan(1000, 2048, 1, 1) == (2048, 1000, True, 2048)
    assert ops._operand_plan(10, 512, 1, 1) == (512, 16, True, 512)
    assert ops._operand_plan(32, 12, 3, 3) == (64, 64, True, 576)         # 9..63 channels with k > 1: zero-padded to 64
    assert ops._operand_plan(24, 16, 1, 1) == (16, 24, True, 16)
    assert ops._operand_plan(10, 10, 1, 1) == (16, 16, True, 16)          # a 1x1 / linear needs 16-byte rows only
    assert ops.padded_cin(3, 1, 1) == 8 and ops.padded_cin(65, 3, 3) == 128 and ops.padded_cin(256, 3, 3) == 256


def test_device_resident_checkpoint_cache(tmp_path, monkeypatch):
    """save_model keeps a clone of what it wrote; load_model / reset_weights are served from it while the file on
    disk is still the one written (format on disk unchanged), and fall back to torch.load otherwise."""
    import refshim
    from turboprune_b200.utils import custom_models as cm, harness_utils as hu
    torch.manual_seed(0)
    model = cm.TorchVisionModel(refshim.make_cfg("resnet18", "cifar10"))
    ck = tmp_path / "checkpoints"; ck.mkdir()
    path = str(ck / "model_init.pt")
    hu.save_model(model, path)
    on_disk = torch.load(path)
    want = {k: v.clone() for k, v in model.model.state_dict().items()}
    assert set(on_disk) == set(want) and all(torch.equal(on_disk[k], want[k]) for k in want)      # same file format / content
    with torch.no_grad():
        for p_ in model.parameters():
            p_.add_(1.0)
    calls = []
    real_load = torch.load
    monkeypatch.setattr(torch, "load", lambda *a, **k: (calls.append(a), real_load(*a, **k))[1])
    model.load_model(path)
    assert not calls                                                     # served from the cache
    assert all(torch.equal(v, want[k]) for k, v in model.model.state_dict().items())
    cfg = refshim.make_cfg("resnet18", "cifar10"); cfg.pruning_params.training_type = "imp"
    with torch.no_grad():
        for p_ in model.parameters():
            p_.mul_(0.5)
    model.reset_weights(cfg, str(tmp_path))
    assert not calls
    assert all(torch.equal(v, want[k]) for k, v in model.model.state_dict().items() if not k.endswith("mask"))
    # a file rewritten behind our back is not served from the cache
    other = {k: torch.zeros_like(v) for k, v in want.items()}
    real_save = torch.save
    real_save(other, path)
    os.utime(path, ns=(1, 1))
    model.load_model(path)
    assert len(calls) == 1
    assert all(float(v.abs().sum()) == 0 for v in model.model.state_dict().values())
