"""Import the UNMODIFIED reference (TurboPrune, directory given by $TURBOPRUNE_REFERENCE) for fixture generation.

Test/fixture infrastructure only.  The reference needs a handful of packages that
are not installed with this project (fastargs, omegaconf, timm, ...); we inject empty
stand-ins for them into ``sys.modules`` so that ``utils.mask_layers``,
``utils.pruning_utils`` and ``utils.custom_models`` import unchanged.

Only ``tests/golden/make_golden.py`` calls :func:`load_reference`: the tests compare
against the fixtures it wrote and never need the reference itself.
"""
import importlib
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("TURBOPRUNE_REFERENCE", "")


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "utils", "mask_layers.py"))


def _stub(name, **attrs):
    mod = types.ModuleType(name)
    mod.__dict__.update(attrs)
    mod.__path__ = []  # behave like a package so sub-imports resolve
    sys.modules[name] = mod
    return mod


class _Anything:
    """Permissive placeholder class (type hints / never-instantiated bases)."""

    def __init__(self, *a, **k):
        pass

    def __class_getitem__(cls, item):
        return cls


def _install_stubs():
    if "fastargs" not in sys.modules:
        _stub("fastargs", get_current_config=lambda: None)
    if "omegaconf" not in sys.modules:
        _stub("omegaconf", DictConfig=_Anything, OmegaConf=_Anything, MISSING="???")
    if "timm" not in sys.modules:
        _stub("timm")
        _stub("timm.models", register_model=lambda f: f)
        _stub("timm.models.vision_transformer", VisionTransformer=_Anything, _cfg=lambda **k: {})
        _stub("timm.models.registry", register_model=lambda f: f)
        _stub("timm.models.layers", trunc_normal_=lambda *a, **k: None)


_loaded = {}


def load_reference():
    """Return (mask_layers, pruning_utils, custom_models) of the real reference."""
    if _loaded:
        return _loaded["ml"], _loaded["pu"], _loaded["cm"]
    if not reference_available():
        raise FileNotFoundError(REFERENCE_ROOT)
    _install_stubs()
    # the reference uses the top-level package name ``utils``; make sure ours (or
    # anything else called utils) is not shadowing it while we import.
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "utils" or k.startswith("utils.")}
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        ml = importlib.import_module("utils.mask_layers")
        pu = importlib.import_module("utils.pruning_utils")
        cm = importlib.import_module("utils.custom_models")
    finally:
        sys.path.remove(REFERENCE_ROOT)
        ref_mods = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "utils" or k.startswith("utils.")}
        sys.modules.update(saved)
    _loaded.update(ml=ml, pu=pu, cm=cm, mods=ref_mods)
    return ml, pu, cm


def load_reference_dataset():
    """The reference's utils/dataset.py (airbench-style GPU augmentation helpers) — needs a webdataset stand-in."""
    if "dataset" in _loaded:
        return _loaded["dataset"]
    if not reference_available():
        raise FileNotFoundError(REFERENCE_ROOT)
    _install_stubs()
    if "webdataset" not in sys.modules:
        _stub("webdataset")
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "utils" or k.startswith("utils.")}
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        ds = importlib.import_module("utils.dataset")
    finally:
        sys.path.remove(REFERENCE_ROOT)
        for k in list(sys.modules):
            if k == "utils" or k.startswith("utils."):
                sys.modules.pop(k)
        sys.modules.update(saved)
    _loaded["dataset"] = ds
    return ds


def state_digests(state_dict):
    """[key, dtype, shape, sha256 of the bytes] per state-dict entry: equal lists <=> bit-identical state dicts."""
    import hashlib
    out = []
    for k, v in state_dict.items():
        a = v.detach().cpu().contiguous().numpy()
        out.append([k, str(a.dtype), list(a.shape), hashlib.sha256(a.tobytes()).hexdigest()])
    return out


class Cfg(dict):
    """dict with attribute access — enough of a DictConfig for the reference."""

    def __getattr__(self, k):
        try:
            v = self[k]
        except KeyError as e:
            raise AttributeError(k) from e
        return Cfg(v) if isinstance(v, dict) else v


def make_cfg(model_name="resnet18", dataset="cifar10", mask_layer_type="ConvMask",
             precision="float32", prune_method="mag", **extra):
    cfg = {
        "model_params": {"model_name": model_name, "mask_layer_type": mask_layer_type, "use_compile": False},
        "dataset_params": {"dataset_name": dataset, "total_batch_size": 512},
        "experiment_params": {"distributed": False, "training_precision": precision, "seed": 0},
        "pruning_params": {"prune_method": prune_method, "prune_rate": 0.2, "target_sparsity": 0.8,
                           "training_type": "imp"},
        "optimizer_params": {"lr": 0.2, "momentum": 0.9, "weight_decay": 5e-4,
                             "scheduler_type": "TriangularSchedule", "warmup_fraction": 0.2},
    }
    for k, v in extra.items():
        cfg[k] = v
    return Cfg(cfg)


def make_harness(cfg, model, batch, tmp_dir=None):
    """A PruningHarness (the product's train-step surface, reference standard_pruning_harness.py:28-50) around a
    prebuilt wrapper model, with the optimizer of ``cfg.optimizer_params`` — what run_experiment.py builds per level."""
    import tempfile
    from turboprune_b200.harness_definitions.standard_pruning_harness import PruningHarness
    cfg["dataset_params"]["total_batch_size"] = batch
    cfg["dataset_params"]["synthetic_steps_per_epoch"] = 2
    h = PruningHarness(cfg=cfg, gpu_id=0, expt_dir=("test", tmp_dir or tempfile.gettempdir()), model=model)
    h._setup_optimizer()
    return h
