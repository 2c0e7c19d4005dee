"""Data-parallel aware mirror of the reference ``engine.py`` (same class name, ctor arguments, method names and
loop shape: ``train`` / ``train_loop`` / ``evaluate`` / ``eval_loop`` / ``log`` / ``save`` / ``should_*``,
engine.py:14-208) - SURVEY 8f-4.  What changes, and only this:

* **one process per GPU** (torchrun): the constructor broadcasts rank 0's parameters and buffers; every rank iterates
  its own shard of the loaders, and the ranks' j-th batches together are the j-th batch of the single-process run.  Each
  loss term is scaled by local / global denominator before ``loss.backward()`` (engine.py:100): the denominator of a
  term is what its ``'mean'`` divides by (the targets that are not ``ignore_index``; the summed ``weight[target]`` of
  those when the criterion has class weights; 1 for ``reduction='sum'``, whose term is not scaled; the batch size for a
  criterion without ``reduction`` / ``ignore_index`` attributes), all-reduced in one small collective.  The gradients -
  views of ONE flat bucket, so there is nothing to pack - are then summed with a single all-reduce, which gives the
  gradient of the global-batch loss however the shards differ in size or in ignored pixels (engine.py has no such step:
  single device, engine.py:17,29-31).  Logged losses are global-batch values; progress bars, wandb and checkpoints are
  rank 0's business only.  Every rank must run the same number of training steps (checked when ``train`` starts);
  evaluation shards may differ, down to empty ones.
* **online evaluation**: the reference concatenates every batch's ``outputs`` on the CPU (``torch.concat`` inside the
  loop, O(n^2) copies, engine.py:162-163) and hands the tensor to ``compute_metrics``.  Here each batch goes through K3
  on the device (bicubic x4 + argmax + confusion matrix + per-image counts, metrics.py:84-101) and only integers
  accumulate; at the end of the pass ONE int64 all-reduce sums the confusion matrix over the ranks and the per-image
  statistics are all-gathered.  ``online_metrics=False`` keeps the reference behaviour (lists, one concat at the end,
  gathered from every rank) for a user-supplied ``compute_metrics(outputs=..., labels=...)``; it is the default when
  ``compute_metrics`` is given.
* **CUDA-graph step** (``cuda_graph=True``, static shapes): forward + criterion + backward of a training step are
  captured once after three eager warm-up steps and replayed from static input buffers; the bucket all-reduce and the
  optimizer step stay outside the graph, and the loss-term scales are static inputs of it.  A batch whose shapes differ
  from the first batch's (a short last batch) runs eagerly.

PyTorch is plumbing here (modules, autograd, optimizers, ``torch.distributed``); the head kernels are the mirrors in
``lc2is_b200.model`` / ``lc2is_b200.metrics`` that the model and the criteria are built from.
"""
from __future__ import annotations

from pathlib import Path
from typing import Callable, Optional

import numpy as np
import torch
import torch.distributed as dist
from torch import nn

from . import dp

_TERMS = ("loss", "aux_loss")          # the logged loss terms: criterion on "outputs", aux_criterion on "low_score_map"


def _local_denominator(crit, labels: torch.Tensor) -> torch.Tensor:
    """float64 scalar: what `crit`'s 'mean' divides the summed losses of this batch by (see the module docstring)."""
    reduction, ii = getattr(crit, "reduction", None), getattr(crit, "ignore_index", None)
    if reduction == "sum":
        return torch.ones((), dtype=torch.float64, device=labels.device)
    if reduction is None or ii is None:
        return torch.full((), float(labels.shape[0]), dtype=torch.float64, device=labels.device)
    counted = labels != ii
    weight = getattr(crit, "weight", None)
    if weight is None:
        return counted.sum().double()
    C = weight.numel()
    counted &= (labels >= 0) & (labels < C)
    w = weight.detach().double()[labels.clamp(0, C - 1)]
    return torch.where(counted, w, torch.zeros_like(w)).sum()


class _NoBar:
    def update(self, *a, **k): pass
    def set_postfix(self, *a, **k): pass
    def close(self): pass


def _bar(total, desc, enabled, **kw):
    if not enabled:
        return _NoBar()
    try:
        from tqdm import tqdm
        return tqdm(range(total), desc=desc, **kw)
    except Exception:  # noqa: BLE001
        return _NoBar()


class Engine:

    def __init__(self, name: str,
                 model: nn.Module, optimizer=None, criterion=None, lr_scheduler=None,
                 device="cuda", fp16: bool = False, aux_criterion=None,
                 train_loader=None, eval_loader=None, compute_metrics: Optional[Callable] = None,
                 max_epoch: int = 1, max_steps: Optional[int] = None, eval_step: Optional[int] = None,
                 log_step: Optional[int] = None, save_step: Optional[int] = None,
                 out_dir: str = "./", logger: Optional[str] = "wandb", logger_args: Optional[dict] = None,
                 *, online_metrics: Optional[bool] = None, n_cls: Optional[int] = None, ignore_index: Optional[int] = 0,
                 cuda_graph: bool = False) -> None:
        self.name = name
        self.model, self.optimizer, self.criterion, self.lr_scheduler = model, optimizer, criterion, lr_scheduler
        self.device, self.fp16 = device, fp16
        self.model.to(self.device)
        self.aux_criterion = aux_criterion
        self.train_loader, self.eval_loader, self.compute_metrics = train_loader, eval_loader, compute_metrics

        self.steps_in_epoch = len(train_loader) if train_loader is not None else 0
        self.train_steps = max(self.steps_in_epoch * max_epoch, max_steps) if max_steps is not None \
            else self.steps_in_epoch * max_epoch
        self.eval_step = self.steps_in_epoch * 10 if eval_step is None else eval_step
        self.log_step = self.steps_in_epoch if log_step is None else log_step
        self.save_step = self.steps_in_epoch * 10 if save_step is None else save_step
        self.out_dir = out_dir + name + "/"
        self.logger, self.logger_args = logger, logger_args

        # ---- data-parallel state -----------------------------------------------------------------------------
        self.distributed = dp.is_dist()
        self.rank = dist.get_rank() if self.distributed else 0
        self.world = dist.get_world_size() if self.distributed else 1
        self.is_main = self.rank == 0
        if self.distributed:
            for t in [*self.model.parameters(), *self.model.buffers()]:
                dist.broadcast(t.data, src=0)                       # replicas start from rank 0's state
        if online_metrics is None:
            online_metrics = compute_metrics is None                # a compute_metrics passed in is called
        self.online_metrics, self.n_cls, self.ignore_index = online_metrics, n_cls, ignore_index
        self.cuda_graph = cuda_graph
        self._graph = None
        self._bucket = None
        if self.distributed or cuda_graph:
            self._make_bucket()
        self.last_eval_stats = None

    # ---- gradients as views of one flat bucket ---------------------------------------------------------------
    def _make_bucket(self) -> None:
        params = [p for p in self.model.parameters() if p.requires_grad]
        if not params:
            return
        dev, dtype = params[0].device, params[0].dtype
        if dtype not in (torch.float32, torch.float64) or any(p.dtype != dtype for p in params):
            raise TypeError("the gradient bucket holds one dtype, fp32 or fp64: keep fp32 master parameters")
        self._bucket = dp.GradBucket([tuple(p.shape) for p in params], dev, dtype=dtype)
        for p, v in zip(params, self._bucket.views):
            p.grad = v                                              # autograd accumulates in place into the bucket

    def _zero_grad(self) -> None:
        if self._bucket is not None:
            self._bucket.zero_()                                    # one fill; p.grad stays a view of the bucket
        else:
            self.optimizer.zero_grad()

    def _allreduce_grads(self) -> None:
        if self.distributed and self._bucket is not None:
            self._bucket.allreduce_()                               # a plain sum: the terms carry their scales

    def _crit(self, key: str):
        return self.aux_criterion if key.endswith("aux_loss") else self.criterion

    def _summed(self, key: str) -> bool:
        return getattr(self._crit(key), "reduction", None) == "sum"

    def _local_denominators(self, keys, labels: torch.Tensor) -> torch.Tensor:
        return torch.stack([_local_denominator(self._crit(k), labels) for k in keys])

    def _denominators(self, keys, labels: torch.Tensor):
        """Distributed only: (float64 [n] this rank's denominator of each term, float64 [n] the scale local / global of
        each term's loss - 1 for a summed term).  The one collective of a step before backward."""
        den = self._local_denominators(keys, labels)
        tot = den.clone()
        dist.all_reduce(tot)
        scale = den / torch.where(tot > 0, tot, torch.ones_like(tot))
        summed = torch.tensor([self._summed(k) for k in keys], device=den.device)
        return den, torch.where(summed, torch.ones_like(scale), scale)

    @staticmethod
    def _total(losses: dict, scales: Optional[torch.Tensor]) -> torch.Tensor:
        terms = torch.stack([v for v in losses.values()])
        return (terms if scales is None else terms * scales.to(terms.dtype)).sum()

    # ---- one training step (engine.py:83-101) ----------------------------------------------------------------
    def _forward_losses(self, inputs: dict, labels: torch.Tensor) -> dict:
        outputs_dict = self.model(inputs)
        losses = dict(train_loss=self.criterion(outputs_dict["outputs"], labels))
        if "low_score_map" in outputs_dict.keys():
            losses.update(dict(train_aux_loss=self.aux_criterion(outputs_dict["low_score_map"], labels) * 0.4))
        return losses

    def _step_eager(self, inputs: dict, labels: torch.Tensor):
        """-> (losses, local denominators or None)"""
        self._zero_grad()
        den = scales = None
        if self.fp16:
            with torch.autocast(device_type=str(self.device).split(":")[0], dtype=torch.float16):
                losses = self._forward_losses(inputs, labels)
                if self.distributed:
                    den, scales = self._denominators(losses, labels)
                loss = self._total(losses, scales)
            self.scaler.scale(loss).backward()
            self._allreduce_grads()
            self.scaler.step(self.optimizer)
            self.scaler.update()
        else:
            losses = self._forward_losses(inputs, labels)
            if self.distributed:
                den, scales = self._denominators(losses, labels)
            self._total(losses, scales).backward()
            self._allreduce_grads()
            self.optimizer.step()
        return losses, den

    def _step_graphed(self, inputs: dict, labels: torch.Tensor):
        """Static-shape step: three eager steps, then forward + criteria + backward replayed from one CUDA graph.
        Batches whose shapes differ from the first batch's run eagerly."""
        g = self._graph
        shapes = (sorted((k, v.shape, v.dtype) for k, v in inputs.items()), labels.shape, labels.dtype)
        if g is None:
            # warm-up AND capture run on one side stream: autograd's AccumulateGrad nodes remember the stream they
            # were created on, and a node created on the default stream breaks the capture
            self._graph = g = dict(warm=0, stream=torch.cuda.Stream(), shapes=shapes)
        if self.fp16:
            return self._step_eager(inputs, labels)
        side, cur = g["stream"], torch.cuda.current_stream()
        if g["warm"] < 3 or shapes != g["shapes"]:
            g["warm"] += shapes == g["shapes"]
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                out = self._step_eager(inputs, labels)
            cur.wait_stream(side)
            g["keys"] = list(out[0])
            return out
        if "graph" not in g:
            g["inputs"] = {k: v.clone() for k, v in inputs.items()}
            g["labels"] = labels.clone()
            g["scales"] = torch.ones(len(g["keys"]), dtype=torch.float64, device=labels.device)
            side.wait_stream(cur)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.stream(side):
                with torch.cuda.graph(graph, stream=side, capture_error_mode="thread_local"):
                    self._bucket.zero_()
                    losses = self._forward_losses(g["inputs"], g["labels"])
                    self._total(losses, g["scales"]).backward()
            cur.wait_stream(side)
            g["graph"], g["losses"] = graph, losses
        den = None
        if self.distributed:
            den, scales = self._denominators(g["keys"], labels)
            g["scales"].copy_(scales)
        for k, v in inputs.items():
            g["inputs"][k].copy_(v, non_blocking=True)
        g["labels"].copy_(labels, non_blocking=True)
        g["graph"].replay()
        self._allreduce_grads()
        self.optimizer.step()
        return {k: v.detach().clone() for k, v in g["losses"].items()}, den

    # ---- reference loop shape ----------------------------------------------------------------------------------
    def train(self):
        self._wandb = None
        if self.logger == "wandb" and self.is_main:
            try:
                import wandb
                wandb.init(**(self.logger_args or {}))
                wandb.watch(self.model, log_freq=self.log_step)
                self._wandb = wandb
            except Exception:  # noqa: BLE001  (no wandb offline: keep training, log to the progress bar only)
                self._wandb = None
        if self.distributed:
            # every training step all-reduces: ranks that disagree on the step count would wait on each other forever
            n = torch.tensor([self.steps_in_epoch, self.train_steps], device=self._comm_device())
            ext = torch.cat([n, -n])
            dist.all_reduce(ext, op=dist.ReduceOp.MAX)
            hi, lo = ext[:2], -ext[2:]
            if not torch.equal(lo, hi):
                raise RuntimeError(f"rank {self.rank}: the ranks disagree on the number of training steps (batches per "
                                   f"epoch {int(-lo[0])}..{int(hi[0])}, steps {int(-lo[1])}..{int(hi[1])}); every rank "
                                   f"must get a train_loader of the same length")
        self.train_progress = _bar(self.train_steps, "Training", self.is_main)
        self.stop_train, self.train_step = False, 0
        self.train_metrics, self.eval_metrics = {}, {}
        self.all_train_metrics = []
        if self.fp16:
            self.scaler = torch.amp.GradScaler("cuda")
        metrics, save_path = {}, None
        while not self.stop_train:
            metrics, save_path = self.train_loop()
        if self._wandb is not None:
            self._wandb.finish()
        return metrics, save_path

    def train_loop(self):
        self.model.train()
        log_metrics, eval_metrics, save_path = {}, {}, None
        for data in self.train_loader:
            self.train_step += 1
            inputs, metas = data
            inputs = {k: v.to(self.device, non_blocking=True) for k, v in inputs.items()}
            labels = inputs.pop("label")
            losses_dict, den = (self._step_graphed if self.cuda_graph else self._step_eager)(inputs, labels)
            if self.lr_scheduler is not None:
                self.lr_scheduler.step()
            self.train_progress.update()
            # (device rows: converted to Python numbers when they are logged, not every step)
            self.all_train_metrics.append(self._loss_row("train_", losses_dict, den))
            eval_metrics = self.should_eval()
            log_metrics = self.should_log()
            save_path = self.should_save()
            if self.should_stop():
                self.stop_train = True
                break
        return {**log_metrics, **eval_metrics}, save_path

    def evaluate(self) -> dict:
        eval_metrics, eval_outputs = self.eval_loop()
        if self.online_metrics:
            return {**eval_metrics, **{"eval_" + k: v for k, v in self._metrics_from_stats(eval_outputs).items()}}
        if self.compute_metrics is not None:
            metrics = self.compute_metrics(**eval_outputs)
            eval_metrics = {**eval_metrics, **{"eval_" + k: v for k, v in metrics.items()}}
        return eval_metrics

    def eval_loop(self):
        from . import ops
        self.model.eval()
        eval_progress = _bar(len(self.eval_loader), "Evaluation", self.is_main, leave=False)
        self.all_eval_metrics = []
        outs, labs = [], []
        confmat, per_image = None, []
        for data in self.eval_loader:
            inputs, metas = data
            inputs = {k: v.to(self.device, non_blocking=True) for k, v in inputs.items()}
            labels = inputs.pop("label")
            with torch.no_grad():
                outputs_dict = self.model(inputs)
                losses_dict = dict(eval_loss=self.criterion(outputs_dict["outputs"], labels))
                if "low_score_map" in outputs_dict.keys():
                    losses_dict.update(dict(eval_aux_loss=self.aux_criterion(outputs_dict["low_score_map"], labels) * 0.4))
                den = self._local_denominators(losses_dict, labels) if self.distributed else None
            eval_progress.update()
            self.all_eval_metrics.append(self._loss_row("eval_", losses_dict, den))
            out = outputs_dict["outputs"]
            if self.online_metrics:
                # metrics.py:84-101 per batch on the device: only integers survive the batch
                h, w = out.shape[-2:]
                confmat, pi, _ = ops.argmax_confmat(out.float(), labels, confmat=confmat, per_image=True,
                                                    size=(4 * h, 4 * w), mode="bicubic")
                per_image.append(pi)
            else:
                outs.append(out.cpu())
                labs.append(labels.cpu())
        eval_progress.close()
        eval_metrics = self._global_losses("eval_", self.all_eval_metrics)
        # every rank enters every collective below, whatever its shard held (an empty shard included)
        if self.online_metrics:
            pi = torch.cat(per_image) if per_image else None
            if self.distributed:
                pi = dp.gather_ragged(pi, self._comm_device())
                if pi is not None:
                    if confmat is None:
                        C = pi.shape[-1]
                        confmat = torch.zeros(C, C, dtype=torch.int64, device=pi.device)
                    dp.allreduce_confmat_(confmat)                   # ONE int64 all-reduce for the pass
            eval_outputs = dict(confmat=confmat, per_image=pi)
        else:
            outputs = torch.cat(outs) if outs else None                # ONE concat, not one per batch
            labels = torch.cat(labs) if labs else None
            if self.distributed:
                outputs, labels = (dp.gather_ragged(t, self._comm_device()) for t in (outputs, labels))
                outputs, labels = (None if t is None else t.cpu() for t in (outputs, labels))
            eval_outputs = dict(outputs=outputs, labels=labels)
        return eval_metrics, eval_outputs

    def _comm_device(self) -> torch.device:
        return torch.device(self.device)

    def _loss_row(self, prefix: str, losses: dict, den: Optional[torch.Tensor]) -> torch.Tensor:
        """float64 [len(_TERMS), 3] of one batch: (numerator, denominator, present) of each term.  Single process:
        (loss, 1).  Distributed: (loss * local denominator, local denominator), so that the sums over the ranks give the
        global-batch value numerator / denominator; a summed term keeps (loss, 1) and its global value is the sum."""
        rows, dev = [], next(iter(losses.values())).device
        for name in _TERMS:
            key = prefix + name
            if key not in losses:
                rows.append(torch.zeros(3, dtype=torch.float64, device=dev))
                continue
            v = losses[key].detach().double().reshape(())
            d = torch.ones_like(v)
            if den is not None and not self._summed(key):
                d = den[list(losses).index(key)]
                v = torch.where(d > 0, v * d, torch.zeros_like(v))  # a shard with nothing counted adds 0, not NaN
            rows.append(torch.stack([v, d, torch.ones_like(v)]))
        return torch.stack(rows)

    def _global_losses(self, prefix: str, rows: list) -> dict:
        """Mean over batches of the global-batch value of each term (the ranks' j-th batches together are batch j of
        the single-process run).  Ranks may hold different numbers of batches, none included."""
        n = len(rows)
        t = torch.stack(rows) if rows else torch.zeros(0, len(_TERMS), 3, dtype=torch.float64,
                                                        device=self._comm_device())
        if self.distributed:
            m = torch.tensor([n], device=t.device)
            dist.all_reduce(m, op=dist.ReduceOp.MAX)
            t = torch.cat([t, t.new_zeros(int(m) - n, len(_TERMS), 3)])
            dist.all_reduce(t)
        out = {}
        for i, name in enumerate(_TERMS):
            num, den, present = t[:, i].unbind(-1)
            sel = present > 0
            if bool(sel.any()):
                key = prefix + name
                out[key] = float((num[sel] if self._summed(key) else num[sel] / den[sel]).mean())
        return out

    def _metrics_from_stats(self, stats: dict) -> dict:
        from . import metrics as M
        self.last_eval_stats = stats
        cm, pi = stats["confmat"], stats["per_image"]
        if cm is None:
            return {}
        return dict(mIOU_label=float(M._per_image_miou(pi, self.ignore_index).mean()),            # metrics.py:84-101
                    mIOU_global=float(M.miou_from_confmat(cm, self.ignore_index)),                # metrics.py:127-134
                    pixel_acc=float(M.pixel_accuracy_from_confmat(cm, self.ignore_index)))

    def log(self) -> dict:
        train_epoch = round(self.train_step / self.steps_in_epoch, 4) if self.steps_in_epoch else 0.0
        train_metrics = self._global_losses("train_", self.all_train_metrics)
        metrics = {**dict(train_step=self.train_step, train_epoch=train_epoch), **train_metrics, **self.eval_metrics}
        if self.is_main:
            self.train_progress.set_postfix(metrics)
            if getattr(self, "_wandb", None) is not None:
                self._wandb.log({"/".join(k.split("_")): v for k, v in metrics.items()})
        return metrics

    def save(self) -> Optional[str]:
        checkpoints_dir = self.out_dir + "checkpoints/"
        if self.is_main:
            Path(checkpoints_dir).mkdir(parents=True, exist_ok=True)
            torch.save(self.model.state_dict(), checkpoints_dir + "step-" + str(self.train_step) + ".pt")
        return checkpoints_dir

    def should_eval(self) -> dict:
        if self.eval_loader is not None and self.eval_step and (self.train_step % self.eval_step) == 0:
            self.eval_metrics = self.evaluate()
            self.model.train()
            return self.eval_metrics
        return {}

    def should_log(self) -> dict:
        if self.log_step and (self.train_step % self.log_step) == 0:
            metrics = self.log()
            self.all_train_metrics = []
            return metrics
        return {}

    def should_save(self) -> Optional[str]:
        if self.save_step and (self.train_step % self.save_step) == 0:
            return self.save()
        return None

    def should_stop(self) -> bool:
        return self.train_steps > 0 and (self.train_step % self.train_steps) == 0
