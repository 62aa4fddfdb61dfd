"""CPU arm of bench.py: one training step through the UNMODIFIED reference modules -- TEST / BASELINE
INFRASTRUCTURE ONLY (bench.py's `--impl reference` and `cpu_baseline` legs; nothing in the product path imports
this).

The reference is pure Python (no build step, not pip-installable: no setup.py), so its "install" is a copy of the
four files of the hot path -- agedb-dir/{resnet,fds,loss,utils}.py, identical to imdb-wiki-dir's -- into
oracle/_ref/agedb-dir/ (git-ignored), made by __graft_entry__.build() when a checkout of the reference is readable at
REFERENCE_ROOT (environment variable DIRB200_REFERENCE, else its default location); without one, build() goes on and
the CPU arm runs the port.  This module only adds the plumbing agedb-dir/train.py:246-262 has around them (train.py
itself cannot be imported: tensorboard_logger, argparse at import time):

    outputs, _ = model(inputs, targets, epoch); loss = weighted_l1_loss(outputs, targets, weights)
    optimizer.zero_grad(); loss.backward(); optimizer.step()

on the host CPU in fp32.  `.cuda()` is shimmed to the identity (fds.py:52 calls it unconditionally; this arm must
stay on the host cores even on a GPU box).  When oracle/_ref is absent, callers fall back to the port
(oracle/train_ref.py) and say so (`kind: "port"`).
"""
import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref", "agedb-dir")
REFERENCE_ROOT = os.environ.get("DIRB200_REFERENCE", "/root/reference")
FILES = ("resnet.py", "fds.py", "loss.py", "utils.py")


def available():
    return all(os.path.exists(os.path.join(REF_DIR, f)) for f in FILES)


def install(reference_root=REFERENCE_ROOT):
    """Copy the reference's hot-path modules into oracle/_ref (called by __graft_entry__.build()); False, and nothing
    copied, when no checkout of the reference is readable at `reference_root`."""
    import shutil
    src = os.path.join(reference_root, "agedb-dir")
    if not os.path.isdir(src):
        return False
    os.makedirs(REF_DIR, exist_ok=True)
    for f in FILES:
        shutil.copyfile(os.path.join(src, f), os.path.join(REF_DIR, f))
    return True


class ReferenceTrainer:
    """resnet50(fds=True, ...) + Adam of the reference, FDS brought to its epoch >= 2 state by the reference's own
    update_last_epoch_stats / update_running_stats on a synthetic epoch of features."""

    def __init__(self, bucket_num=100, bucket_start=0, lr=1e-3, seed=0, epoch_features=None, epoch_labels=None):
        if not available():
            raise RuntimeError("oracle/_ref is not populated (run __graft_entry__.build() with the reference readable)")
        saved_path, saved_mods = list(sys.path), {k: sys.modules.get(k) for k in ("resnet", "fds", "loss", "utils")}
        saved_cuda = (torch.Tensor.cuda, torch.nn.Module.cuda)
        torch.Tensor.cuda = lambda self, *a, **k: self
        torch.nn.Module.cuda = lambda self, *a, **k: self
        try:
            sys.path.insert(0, REF_DIR)
            for k in saved_mods:
                sys.modules.pop(k, None)
            resnet = importlib.import_module("resnet")
            loss = importlib.import_module("loss")
            torch.manual_seed(seed)
            self.model = resnet.resnet50(fds=True, bucket_num=bucket_num, bucket_start=bucket_start, start_update=0,
                                         start_smooth=1, kernel="gaussian", ks=5, sigma=2, momentum=0.9)
            self.loss_fn = loss.weighted_l1_loss
        finally:
            torch.Tensor.cuda, torch.nn.Module.cuda = saved_cuda
            sys.path[:] = saved_path
            for k, v in saved_mods.items():
                sys.modules.pop(k, None)
                if v is not None:
                    sys.modules[k] = v
        self.model.train()
        self.opt = torch.optim.Adam(self.model.parameters(), lr=lr)
        if epoch_features is not None:
            f, l = torch.as_tensor(epoch_features), torch.as_tensor(epoch_labels)
            for ep in (0, 1):
                self.model.FDS.update_last_epoch_stats(ep)
                self.model.FDS.update_running_stats(f, l, ep)
            self.model.FDS.update_last_epoch_stats(2)

    def step(self, x, targets, weights, epoch=2):
        outputs, _ = self.model(x, targets, epoch)
        loss = self.loss_fn(outputs, targets, weights)
        self.opt.zero_grad()
        loss.backward()
        self.opt.step()
        return float(loss.detach())

    def fds_timings(self, feats, labels):
        """ms of the reference's own FDS.update_running_stats (N x 2048) and FDS.smooth (first 256 rows)."""
        import time
        fds = self.model.FDS
        f, l = torch.as_tensor(feats), torch.as_tensor(labels)
        upd, smo = [], []
        for _ in range(3):
            t0 = time.perf_counter()
            fds.update_running_stats(f, l, int(fds.epoch.item()))
            upd.append(time.perf_counter() - t0)
        for _ in range(3):
            xb = f[:256].clone()
            t0 = time.perf_counter()
            fds.smooth(xb, l[:256].reshape(-1, 1), 3)
            smo.append(time.perf_counter() - t0)
        return {"update_running_stats_ms": round(1e3 * sorted(upd)[1], 2), "smooth_b256_ms": round(1e3 * sorted(smo)[1], 2),
                "rows": int(f.shape[0]), "impl": "reference fds.FDS (oracle/_ref)"}
