"""``PruningHarness`` — drop-in for the reference's ``harness_definitions/standard_pruning_harness.py``.

``PruningHarness(cfg, gpu_id, expt_dir, model=None)`` and ``.train_one_level(epochs_per_level, level)`` keep the
reference's behaviour (:28-50, :159-269): a fresh optimizer and LR schedule per level (momentum never carries
over), ``model_init.pt`` / ``optimizer_init.pt`` at level 0, ``model_rewind.pt`` at ``pruning_params.rewind_epoch``,
per-level CSV + summary CSV.  Optimizer = ``FusedSGD`` (same state-dict layout as torch.optim.SGD).  Loaders =
``utils.dataset.make_loaders``: the CIFAR data set under ``dataset_params.data_root_dir`` (``AirbenchLoaders``) when a
CIFAR config sets ``dataset_params.dataloader_type`` to anything but ``synthetic``, as the reference's configs do
(``torch``); otherwise, and for ImageNet, the synthetic on-device generator.
"""
import csv
import os
from typing import Optional

import torch
import torch.nn as nn

from ..optim import FusedSGD
from ..utils import schedulers
from ..utils.custom_models import CustomModel, TorchVisionModel
from ..utils.dataset import make_loaders
from ..utils.harness_utils import save_model
from .base_harness import BaseHarness


class PruningHarness(BaseHarness):
    def __init__(self, cfg, gpu_id: int, expt_dir, model: Optional[nn.Module] = None):
        self.gpu_id = gpu_id
        self.dataset_name = cfg.dataset_params.dataset_name.lower()
        self.use_compile = cfg.model_params.use_compile
        self.num_classes = 1000 if self.dataset_name.startswith("imagenet") else (100 if self.dataset_name.startswith("cifar100") else 10)
        local = int(os.environ.get("LOCAL_RANK", gpu_id))
        self.this_device = torch.device("cuda", local)
        self.prefix, self.expt_dir = expt_dir
        distributed = (cfg.experiment_params.distributed and torch.distributed.is_available()
                       and torch.distributed.is_initialized() and not self.dataset_name.startswith("cifar"))
        super().__init__(cfg=cfg, device=self.this_device, model=model, distributed=distributed)

    def _create_model(self):
        try:
            model = TorchVisionModel(cfg=self.cfg)
        except ValueError:
            model = CustomModel(cfg=self.cfg)            # the reference's fallback (broken upstream) for DeiT names
        return model

    def _setup_dataloaders(self):
        world = torch.distributed.get_world_size() if self.distributed else 1
        rank = torch.distributed.get_rank() if self.distributed else 0
        loaders = make_loaders(self.cfg, self.device, world, rank)
        return loaders.train_loader, loaders.test_loader

    def _setup_optimizer(self):
        o = self.cfg.optimizer_params
        if o.scheduler_type == "ScheduleFree":
            raise NotImplementedError("ScheduleFree optimizer (third-party package, off the benchmarked path)")
        # capturable: the learning rate is a device scalar refreshed by train_step (sync_lr), so the captured step
        # follows the per-iteration LR schedule without being re-recorded
        self.optimizer = FusedSGD(self.model.parameters(), lr=o.lr, momentum=o.momentum, weight_decay=o.weight_decay,
                                  capturable=True)

    def _setup_scheduler(self, epochs_per_level):
        kind = self.cfg.optimizer_params.scheduler_type
        if kind == "OneCycleLR":
            self.scheduler = torch.optim.lr_scheduler.OneCycleLR(self.optimizer, max_lr=self.cfg.optimizer_params.lr,
                                                                 epochs=epochs_per_level, steps_per_epoch=len(self.train_loader))
        elif kind == "TriangularSchedule":
            self.scheduler = schedulers.TriangularSchedule(self.cfg, self.optimizer, len(self.train_loader), epochs_per_level)
        else:
            raise NotImplementedError(f"scheduler {kind}: its reference call site passes arguments the class does not accept")

    def train_one_level(self, epochs_per_level: int, level: int) -> None:
        rows = []
        model = self.model
        self._setup_optimizer()
        self._setup_scheduler(epochs_per_level)
        ck = os.path.join(self.expt_dir, "checkpoints")
        art = os.path.join(self.expt_dir, "artifacts")
        if self.gpu_id == 0 and level == 0:
            save_model(self.model, os.path.join(ck, "model_init.pt"))
            torch.save(self.optimizer.state_dict(), os.path.join(art, "optimizer_init.pt"))
        rewind_epoch = getattr(self.cfg.pruning_params, "rewind_epoch", None)
        for epoch in range(epochs_per_level):
            self.epoch_counter += 1
            if self.gpu_id == 0:
                self.console.rule(f"Current Epoch: {epoch + 1}/{epochs_per_level}")
            metrics = {"epoch": int(self.epoch_counter), **self.train_epoch(), **self.test()}
            if self.gpu_id == 0 and rewind_epoch == epoch and level == 0:
                save_model(self.model, os.path.join(ck, "model_rewind.pt"))
                torch.save(self.optimizer.state_dict(), os.path.join(art, "optimizer_rewind.pt"))
            if self.gpu_id == 0:
                self.console.print({k: (round(v, 4) if isinstance(v, float) else v) for k, v in metrics.items()})
                rows.append({**metrics, "max_test_acc": max([r["test_acc"] for r in rows] + [metrics["test_acc"]]),
                             "sparsity": model.get_overall_sparsity()})
        if self.gpu_id == 0:
            path = os.path.join(self.expt_dir, "metrics", "level_wise_metrics", f"level_{level}_metrics.csv")
            with open(path, "w", newline="") as f:
                w = csv.DictWriter(f, fieldnames=list(rows[0].keys())); w.writeheader(); w.writerows(rows)
            summary = os.path.join(self.expt_dir, f"{self.prefix}_summary.csv")
            new = not os.path.exists(summary)
            with open(summary, "a", newline="") as f:
                w = csv.writer(f)
                if new:
                    w.writerow(["Level", "Sparsity", "Last_Test_Acc", "Max_Test_Acc"])
                w.writerow([level, model.get_overall_sparsity(), rows[-1]["test_acc"], max(r["test_acc"] for r in rows)])
