"""`Trainer` with the reference's constructor, attributes and methods (etpgt/train/trainer.py:17-251:
`train_epoch() -> float`, `evaluate() -> {"recall@k", "ndcg@k"}`, `save_checkpoint(is_best)`, `train() ->
history`, early stopping on recall@k_values[0], `checkpoint_latest.pt / checkpoint_best.pt / history.json`).

What differs is where the work runs:
  * a training step goes through the C++ step driver (`FusedTrainStep`) when the model / loss pair is one it
    covers, else through the per-operator autograd path — both give the same bits;
  * the loss is accumulated on the device and read once per epoch (the reference syncs twice per step,
    trainer.py:130-133);
  * evaluation keeps predictions on the device: fused scoring + top-k, hit / NDCG counters accumulated by
    `etpgt_topk_metrics`, one read-back per evaluation (the reference copies every batch's top-k to the host,
    trainer.py:158-159);
  * `process_group=` (not in the reference, which is single-GPU) makes this trainer one rank of a session-batch
    data-parallel job: loaders hand every rank its share of each global batch (`create_dataloader(..., rank,
    world_size)`), BatchNorm statistics / gradients / the item-table update are exchanged over peer memory
    (`exchange="peer"`, parallel.PeerDataParallel) or NCCL (`exchange="nccl"`), the loss is the global-batch mean,
    evaluation scores item shards (`parallel.sharded_predict`) and sums the counters over the ranks; rank 0 writes
    the checkpoints.
"""

from __future__ import annotations

import json
import logging
from pathlib import Path

import torch
import torch.distributed as dist

from .. import ops, parallel
from .losses import BPRLoss, DualLoss, ListwiseLoss
from .step import FusedTrainStep

logger = logging.getLogger(__name__)


def _driver_for(model, loss_fn):
    """FusedTrainStep for (model, loss_fn), or None when the pair needs the per-operator path."""
    if not FusedTrainStep.supported(model):
        return None
    if loss_fn is None or type(loss_fn) is BPRLoss:
        return FusedTrainStep(model, "bpr")
    if isinstance(loss_fn, ListwiseLoss):       # SampledSoftmaxLoss is the same arithmetic
        return FusedTrainStep(model, "listwise", temperature=loss_fn.temperature)
    if type(loss_fn) is DualLoss:
        return FusedTrainStep(model, "dual", alpha=loss_fn.alpha, temperature=loss_fn.listwise_loss.temperature)
    return None


class Trainer:
    def __init__(self, model, train_loader, val_loader, optimizer, device: str = "cuda",
                 output_dir: Path | str = "outputs", max_epochs: int = 100, patience: int = 10, eval_every: int = 1,
                 k_values: list[int] | None = None, loss_fn=None, process_group=None, exchange: str = "peer",
                 exclude_seen: bool = False):
        self.model = model.to(device)
        self.train_loader, self.val_loader, self.optimizer = train_loader, val_loader, optimizer
        self.device = device
        self.output_dir = Path(output_dir)
        self.max_epochs, self.patience, self.eval_every = max_epochs, patience, eval_every
        self.k_values = k_values if k_values is not None else [10, 20]
        self.loss_fn = loss_fn
        # evaluate() ranks without each session's own items and the padding id 0: the Recall / NDCG of what a
        # deployed recommender returns (the reference's serving filter, recommender.py:133-134)
        self.exclude_seen = exclude_seen
        self.output_dir.mkdir(parents=True, exist_ok=True)
        self.current_epoch = 0
        self.best_val_metric = 0.0
        self.patience_counter = 0
        self.history = {"train_loss": [], "val_metrics": []}
        # data parallelism: process_group=True (the default group) or a torch.distributed group
        self._group, self._world, self._rank, self._peer = None, 1, 0, None
        if process_group is not None and process_group is not False:
            if not (dist.is_available() and dist.is_initialized()):
                raise RuntimeError("Trainer(process_group=...) needs an initialised torch.distributed")
            self._group = None if process_group is True else process_group
            self._world, self._rank = dist.get_world_size(self._group), dist.get_rank(self._group)
        if self._world > 1:
            ours = hasattr(optimizer, "attach_peer")
            if exchange == "peer" and not ours:
                logger.warning("exchange='peer' needs an etpgt_b200.optim optimizer; using NCCL all-reduces")
                exchange = "nccl"
            elif exchange == "peer" and getattr(optimizer, "row_sparse", False):
                logger.warning("exchange='peer' has no row-sparse table update (lazy_rows=True / SparseAdam); "
                               "using NCCL all-reduces")
                exchange = "nccl"
            self._peer = parallel.enable_data_parallel(self.model, self._group, exchange)
            if self._peer is not None:
                optimizer.attach_peer(self._peer)      # the table moved into the peer region after the optimizer was built
        self._driver = _driver_for(self.model, loss_fn)

    # ------------------------------------------------------------------ one step
    def _total_sessions(self, batch, batch_size: int) -> int:
        """Sessions of the GLOBAL batch this rank's share belongs to (the loss is its mean)."""
        if self._world == 1:
            return batch_size
        total = getattr(batch, "total_sessions", None)
        if total is None:       # a loader that does not say: one collective + host read per step
            t = torch.tensor([batch_size], dtype=torch.int64, device=self.device)
            dist.all_reduce(t, group=self._group)
            total = int(t.item())
        return int(total)

    def _loss_and_backward(self, batch) -> torch.Tensor:
        """Backward of this rank's share of the global-batch loss; returns that share (its sum over the ranks is the
        global-batch mean loss).  Gradients are reduced here (NCCL exchange) or inside optimizer.step() (peer)."""
        batch_size = batch.target_item.shape[0]
        negatives = batch.negative_items.view(batch_size, -1)        # trainer.py:86-89
        total = self._total_sessions(batch, batch_size)
        if self._driver is not None and getattr(batch, "laplacian_pe", None) is None:
            loss = self._driver(batch, batch.target_item, negatives, total_sessions=total)[0]
            if self._world > 1 and self._peer is None:
                self._driver.allreduce_gradients(self._group)
            return loss
        sess = self.model(batch)
        if self.loss_fn is not None:
            out = self.loss_fn(sess, batch.target_item, negatives, self.model.item_embedding)
            loss = out[0] if isinstance(out, tuple) else out         # DualLoss returns (loss, parts)
        else:
            loss = self.model.compute_loss(sess, batch.target_item, negatives)
        if total != batch_size:
            loss = loss * (batch_size / total)       # mean over the local share -> share of the global mean
        loss.backward()
        if self._world > 1 and self._peer is None:
            parallel.allreduce_gradients(list(self.model.parameters()), self._group)
        return loss.detach()

    def train_epoch(self) -> float:
        self.model.train()
        total = torch.zeros((), dtype=torch.float64, device=self.device)
        steps = 0
        for batch in self.train_loader:
            batch = batch.to(self.device)
            self.optimizer.zero_grad()
            loss = self._loss_and_backward(batch)
            self.optimizer.step()
            prepared = getattr(batch, "prepared", None)
            if prepared is not None:
                prepared.release()        # the loader may refill that preparation slot once the step has run
            total += loss
            steps += 1
        if self._world > 1:
            dist.all_reduce(total, group=self._group)
        if self._peer is not None:
            self._peer.comm.check()
        ops.check_item_ids(self.device)       # IndexError if a batch held an id outside the table (one read per epoch)
        return float(total.item()) / max(steps, 1)

    # ------------------------------------------------------------------ evaluation
    @torch.no_grad()
    def evaluate(self) -> dict:
        self.model.eval()
        # k <= 64 and k > 64 are ranked by separate calls: "auto" may pick another scorer for k > 64 (the fp32 CUDA-core
        # scorer stops at 64), and a deep k must not change recall@20, the early-stopping metric, on any batch
        shallow = [k for k in self.k_values if k <= ops.SCORE_F32_MAX_K]
        deep = [k for k in self.k_values if k > ops.SCORE_F32_MAX_K]
        depths = [max(group) for group in (shallow, deep) if group]
        # [hits, ndcg] per k, then the session count: ONE tensor, so that data parallelism sums it in one collective
        acc = torch.zeros(2 * len(self.k_values) + 1, dtype=torch.float64, device=self.device)
        sessions = 0
        # exclusion rows of a fixed width when the loader says how long a session can be (no host read per batch,
        # and every rank of a data-parallel job agrees on it)
        max_len = getattr(self.val_loader, "max_session_length", None)
        width = max_len + 1 if max_len is not None else None
        for batch in self.val_loader:
            batch = batch.to(self.device)
            sess = self.model(batch)
            exclude = ops.seen_items(batch, num_sessions=sess.size(0), width=width) if self.exclude_seen else None
            if self._world > 1:
                # item-sharded scoring: every rank scores all sessions of the global batch against its id range
                counts = getattr(batch, "rank_sessions", None)
                if exclude is not None and width is None:
                    counts = None              # the ranks' list widths differ: exchanged with the counts
                hits = [parallel.sharded_predict(self.model, sess, k=d, group=self._group, counts=counts,
                                                 targets=batch.target_item, exclude=exclude, exclude_sorted=True)[1]
                        for d in depths]
                if getattr(batch, "replicated", False) and self._rank != 0:
                    continue                   # every rank holds the same sessions: counted once
                for j, k in enumerate(self.k_values):
                    ops.hit_metrics(hits[0 if k <= depths[0] else -1], k, acc[2 * j:2 * j + 2])
            else:
                # fused scoring + top-k; the target's position comes out of the scorer's select epilogue
                # (group=False: this Trainer is not data parallel, even if the process has a group initialised)
                hits = [parallel.sharded_predict(self.model, sess, k=d, group=False, targets=batch.target_item,
                                                 exclude=exclude, exclude_sorted=True)[1] for d in depths]
                for j, k in enumerate(self.k_values):
                    ops.hit_metrics(hits[0 if k <= depths[0] else -1], k, acc[2 * j:2 * j + 2])
            sessions += int(batch.target_item.shape[0])
        acc[-1] = sessions
        if self._world > 1:
            dist.all_reduce(acc, group=self._group)
        values = acc.tolist()
        sessions = values[-1]
        metrics = {}
        for j, k in enumerate(self.k_values):
            metrics[f"recall@{k}"] = values[2 * j] / sessions if sessions else 0.0
            metrics[f"ndcg@{k}"] = values[2 * j + 1] / sessions if sessions else 0.0
        return metrics

    # ------------------------------------------------------------------ checkpoints and the outer loop
    def save_checkpoint(self, is_best: bool = False) -> None:
        if self._peer is not None:      # every rank keeps only its own rows' moments current: collect them
            self._peer.gather_optimizer_state(self.optimizer)
        if self._rank != 0:
            return
        checkpoint = {"epoch": self.current_epoch, "model_state_dict": self.model.state_dict(),
                      "optimizer_state_dict": self.optimizer.state_dict(),
                      "best_val_metric": self.best_val_metric, "history": self.history}
        names = ["checkpoint_latest.pt"] + (["checkpoint_best.pt"] if is_best else [])
        for name in names:
            torch.save(checkpoint, self.output_dir / name)
            logger.info("Saved checkpoint to %s", self.output_dir / name)

    def train(self) -> dict:
        logger.info("Starting training for %d epochs on %s", self.max_epochs, self.device)
        for epoch in range(self.max_epochs):
            self.current_epoch = epoch
            train_loss = self.train_epoch()
            self.history["train_loss"].append(train_loss)
            logger.info("Epoch %d: train_loss=%.4f", epoch, train_loss)
            if (epoch + 1) % self.eval_every:
                continue
            metrics = self.evaluate()
            self.history["val_metrics"].append(metrics)
            logger.info("Epoch %d: %s", epoch, ", ".join(f"{k}={v:.4f}" for k, v in metrics.items()))
            watched = metrics[f"recall@{self.k_values[0]}"]
            is_best = watched > self.best_val_metric
            if is_best:
                self.best_val_metric, self.patience_counter = watched, 0
            else:
                self.patience_counter += 1
            self.save_checkpoint(is_best=is_best)
            if self.patience_counter >= self.patience:
                logger.info("Early stopping at epoch %d", epoch)
                break
        if self._rank == 0:
            with open(self.output_dir / "history.json", "w") as f:
                json.dump(self.history, f, indent=2)
        return self.history
