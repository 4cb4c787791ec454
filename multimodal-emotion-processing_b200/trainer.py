"""Epoch driver of the reference scripts (SURVEY.md §8f-4), restated once for all five of them and
fixed for current torch:  ``run()`` = Adam/AdamW + ``ReduceLROnPlateau(factor=0.1, patience=p)`` on
the validation loss + best-checkpoint saving + early stop after 4 epochs without a new best
(others/realformer.py:338-363, cmu-mosei/run.py:394-419, Ren-MME/run.py:370-401,
rencecps/run.py:198-223, robot_demo.py:498-523), and the contiguous k-fold split the scripts spell
out by hand (others/realformer.py:365-389).  The reference runs the folds one after the other;
``fit_folds`` trains them together, and ``fit`` is ``fit_folds`` with one fold.

Differences from the reference, all outside the hot path:
* ``ReduceLROnPlateau(verbose=True)`` raises ``TypeError`` on torch >= 2.7; the lr changes are
  reported through ``log`` instead.
* the model / batch / loss specifics live in two callables (``train_step``, ``valid_step``) so the
  same driver serves every script; with ``mmemo_b200.optim.AdamW(max_grad_norm=CLIP)`` the clip is
  part of ``optimizer.step()``.
* TensorBoard logging is optional (``writer`` may be any object with ``add_scalars``).

Host-side orchestration only: nothing here touches the GPU directly.
"""
from __future__ import annotations

import os
from typing import Callable, Dict, Iterable, List, Optional, Sequence, Tuple

import torch
from torch.optim.lr_scheduler import ReduceLROnPlateau

from . import optim


def kfold_splits(names: Sequence, k: int = 5) -> List[Tuple[list, list]]:
    """[(train_list, valid_list)] with validation fold i = ``names[int(n*i/k):int(n*(i+1)/k)]``
    — the slicing of others/realformer.py:366-389 (k = 5, 20 % folds; the last fold runs to the
    end of the list)."""
    n = len(names)
    names = list(names)
    out = []
    for i in range(k):
        lo = int(n * (i / k)) if i else 0
        hi = int(n * ((i + 1) / k)) if i + 1 < k else n
        out.append((names[:lo] + names[hi:], names[lo:hi]))
    return out


def checkpoint_name(name: str, valid_loss: float) -> str:
    """``model_1_1.31.pt``: first four characters of ``str(valid_loss)`` (others/realformer.py:359)."""
    return f"{name}_{str(valid_loss)[:4]}.pt"


class _Run:
    """The per-model bookkeeping of the reference's ``run()`` after each epoch: plateau schedule,
    log file, history, best checkpoint and early stop (``done``)."""

    def __init__(self, optimizer, name: str, log_dir: Optional[str], sched_patience: int,
                 sched_factor: float, stop_after: int, writer, log: Callable[[str], None]):
        self.optimizer, self.name, self.log_dir = optimizer, name, log_dir
        self.stop_after, self.writer, self.log = stop_after, writer, log
        self.scheduler = ReduceLROnPlateau(optimizer, factor=sched_factor, patience=sched_patience)
        self.log_file = None
        if log_dir is not None:
            os.makedirs(log_dir, exist_ok=True)
            self.log_file = os.path.join(log_dir, name + ".txt")
            with open(self.log_file, "w") as fh:
                fh.write("epoch, train_loss, valid_loss\n")
        self.hist = {"train": [], "valid": [], "best": None, "lrs": []}
        self.stop = 0
        self.done = False

    def end_epoch(self, model: torch.nn.Module, epoch: int, tr: float, va: float) -> None:
        name, hist = self.name, self.hist
        if self.writer is not None:
            self.writer.add_scalars(name, {"train_loss": tr, "valid_loss": va}, epoch)
        before = [g["lr"] for g in self.optimizer.param_groups]
        self.scheduler.step(va)
        after = [g["lr"] for g in self.optimizer.param_groups]
        if after != before:
            self.log(f"reducing learning rate: {before} -> {after}")
        hist["train"].append(tr)
        hist["valid"].append(va)
        hist["lrs"].append(after[0])
        if self.log_file is not None:
            with open(self.log_file, "a") as fh:
                fh.write("\n{epoch},{tr: 2.2f},{va: 2.2f}\n".format(epoch=epoch + 1, tr=tr, va=va))
        if va == min(hist["valid"]):
            self.stop = 0
            if self.log_dir is not None:
                hist["best"] = os.path.join(self.log_dir, checkpoint_name(name, va))
                torch.save(model.state_dict(), hist["best"])
        else:
            self.stop += 1
            self.done = self.stop >= self.stop_after


def fit(model: torch.nn.Module, optimizer: torch.optim.Optimizer,
        make_train_iter: Callable[[], Iterable], make_valid_iter: Callable[[], Iterable],
        train_step: Callable, valid_step: Optional[Callable] = None, *, epochs: int, name: str,
        log_dir: Optional[str] = None, clip: Optional[float] = 1.0, sched_patience: int = 2,
        sched_factor: float = 0.1, stop_after: int = 4, writer=None,
        log: Callable[[str], None] = print) -> dict:
    """The reference's ``run()``.  Returns ``{"train": [...], "valid": [...], "best": path | None,
    "lrs": [...]}``.  A new iterator is built every epoch (the reference reshuffles in
    ``data_loader``).  ``sched_patience`` is 2 in realformer and 1 in the other scripts."""
    valid_step = valid_step or train_step
    return fit_folds([model], [optimizer], [make_train_iter], [make_valid_iter],
                     lambda ms, bs: [train_step(ms[0], bs[0])],
                     lambda ms, bs: [valid_step(ms[0], bs[0])], epochs=epochs, names=[name],
                     log_dir=log_dir, clip=clip, sched_patience=sched_patience,
                     sched_factor=sched_factor, stop_after=stop_after, writer=writer, log=log)[0]


def _lockstep(iterables: Dict[int, Iterable]):
    """Yields ([fold], [batch]): the next batch of every fold whose iterator has not run out."""
    its = {k: iter(v) for k, v in iterables.items()}
    while its:
        ks, bs = [], []
        for k in list(its):
            try:
                bs.append(next(its[k]))
                ks.append(k)
            except StopIteration:
                del its[k]
        if ks:
            yield ks, bs


def _train_epoch_group(models, optimizers, iterables, train_step_group, clip) -> Dict[int, float]:
    for k in iterables:
        models[k].train()
    total = {k: 0.0 for k in iterables}
    count = {k: 0 for k in iterables}
    for ks, bs in _lockstep(iterables):
        opts = [optimizers[k] for k in ks]
        for o in opts:
            o.zero_grad()
        losses = list(train_step_group([models[k] for k in ks], bs))
        if len(losses) != len(ks):
            raise ValueError(f"train_step_group returned {len(losses)} losses for {len(ks)} folds")
        # the folds share no parameters: each receives exactly the gradients of its own loss
        total_loss = losses[0]
        for loss in losses[1:]:
            total_loss = total_loss + loss
        total_loss.backward()
        if clip is not None:
            for k in ks:
                torch.nn.utils.clip_grad_norm_(models[k].parameters(), clip)
        if all(isinstance(o, optim._FusedAdam) for o in opts):
            optim.step_group(opts)
        else:
            for o in opts:
                o.step()
        for k, loss in zip(ks, losses):
            total[k] += loss.item()
            count[k] += 1
    return {k: total[k] / max(count[k], 1) for k in iterables}


def _valid_epoch_group(models, iterables, valid_step_group) -> Dict[int, float]:
    for k in iterables:
        models[k].eval()
    total = {k: 0.0 for k in iterables}
    count = {k: 0 for k in iterables}
    with torch.no_grad():
        for ks, bs in _lockstep(iterables):
            for k, loss in zip(ks, valid_step_group([models[k] for k in ks], bs)):
                total[k] += float(loss)
                count[k] += 1
    return {k: total[k] / max(count[k], 1) for k in iterables}


def fit_folds(models: Sequence[torch.nn.Module], optimizers: Sequence[torch.optim.Optimizer],
              make_train_iters: Sequence[Callable[[], Iterable]],
              make_valid_iters: Sequence[Callable[[], Iterable]], train_step_group: Callable,
              valid_step_group: Optional[Callable] = None, *, epochs: int, names: Sequence[str],
              log_dir: Optional[str] = None, clip: Optional[float] = 1.0, sched_patience: int = 2,
              sched_factor: float = 0.1, stop_after: int = 4, writer=None,
              log: Callable[[str], None] = print) -> List[dict]:
    """``fit`` for the k folds of a cross-validation at once, in lockstep: every training step
    takes the next batch of each fold that still has one and calls
    ``train_step_group([model], [batch]) -> [loss]`` (one scalar loss per fold given), backpropagates
    the SUM of those losses once, clips each fold's gradients (``clip``) and steps all their
    optimizers together (``optim.step_group`` when they are all ``optim.Adam`` / ``AdamW``).
    Validation runs the same way through ``valid_step_group`` (default: ``train_step_group``).

    Each fold keeps its own scheduler, early stop, log file ``names[k].txt`` and best checkpoint
    ``checkpoint_name(names[k], valid_loss)``.  A fold whose epoch iterator runs out leaves the
    group for the rest of that epoch; one that stops early leaves it for good.  Returns one
    ``fit``-style history per fold, equal to what ``fit`` would return for that fold alone."""
    K = len(models)
    if not (len(optimizers) == len(make_train_iters) == len(make_valid_iters) == len(names) == K):
        raise ValueError("models, optimizers, iterator factories and names must have one entry "
                         "per fold")
    valid_step_group = valid_step_group or train_step_group
    runs = [_Run(optimizers[k], names[k], log_dir, sched_patience, sched_factor, stop_after, writer,
                 log) for k in range(K)]
    for epoch in range(epochs):
        live = [k for k in range(K) if not runs[k].done]
        if not live:
            break
        log(f"Epoch: {epoch + 1}")
        tr = _train_epoch_group(models, optimizers, {k: make_train_iters[k]() for k in live},
                                train_step_group, clip)
        va = _valid_epoch_group(models, {k: make_valid_iters[k]() for k in live}, valid_step_group)
        for k in live:
            runs[k].end_epoch(models[k], epoch, tr[k], va[k])
    return [r.hist for r in runs]
