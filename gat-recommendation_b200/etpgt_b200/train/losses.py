"""BPR / listwise / dual / sampled-softmax / full-catalogue / shared-pool softmax losses with the reference's call signature
`loss(session_embeddings, target_items, negative_items, item_embeddings: nn.Embedding)`
(etpgt/train/losses.py), computed by the fused sampled-loss kernel (full_softmax: the tensor-core full-catalogue kernels;
shared_pool_softmax: the same kernels over one log-Q-corrected negative pool shared by the batch)."""

from __future__ import annotations

import torch
import torch.nn as nn

from .. import ops


class BPRLoss(nn.Module):
    def forward(self, session_embeddings, target_items, negative_items, item_embeddings) -> torch.Tensor:
        return ops.sampled_loss(session_embeddings, item_embeddings, target_items, negative_items, "bpr")[0]


class ListwiseLoss(nn.Module):
    def __init__(self, temperature: float = 1.0):
        super().__init__()
        self.temperature = temperature

    def forward(self, session_embeddings, target_items, negative_items, item_embeddings) -> torch.Tensor:
        return ops.sampled_loss(session_embeddings, item_embeddings, target_items, negative_items, "listwise",
                                temperature=self.temperature)[0]


class DualLoss(nn.Module):
    """alpha * listwise + (1 - alpha) * bpr; returns (loss, {"total","listwise","bpr"}) like the
    reference, with ONE device->host copy for the three floats instead of three syncs."""

    def __init__(self, alpha: float = 0.7, temperature: float = 1.0):
        super().__init__()
        self.alpha = alpha
        self.listwise_loss = ListwiseLoss(temperature=temperature)
        self.bpr_loss = BPRLoss()

    def forward(self, session_embeddings, target_items, negative_items, item_embeddings):
        losses = ops.sampled_loss(session_embeddings, item_embeddings, target_items, negative_items, "dual",
                                  alpha=self.alpha, temperature=self.listwise_loss.temperature)
        total, listwise, bpr = losses.detach().tolist()
        return losses[0], {"total": total, "listwise": listwise, "bpr": bpr}


class SampledSoftmaxLoss(ListwiseLoss):
    """Softmax over target + sampled negatives: identical to the listwise loss (losses.py:198-201)."""


class FullSoftmaxLoss(nn.Module):
    """Softmax cross-entropy over the whole catalogue (SR-GNN / GCE-GNN style) instead of the sampled negatives;
    `negative_items` is accepted for the common signature and not used.  Deliberately not a ListwiseLoss: the fused
    step driver has no full-catalogue mode, so the trainer takes the per-operator path for it.  `precision`:
    "bf16x3" (split-bf16, the default) or "bf16" (operands and softmax gradient rounded once to bf16), see
    ops.full_softmax_loss."""

    def __init__(self, temperature: float = 1.0, precision: str = "bf16x3"):
        super().__init__()
        ops._softmax_precision(precision)
        self.temperature = temperature
        self.precision = precision

    def forward(self, session_embeddings, target_items, negative_items, item_embeddings) -> torch.Tensor:
        return ops.full_softmax_loss(session_embeddings, item_embeddings, target_items, temperature=self.temperature,
                                     precision=self.precision)


class SharedPoolSoftmaxLoss(nn.Module):
    """Sampled softmax over one pool of `num_sampled` negatives shared by the whole batch, with the log-Q correction
    (ops.pool_softmax_loss).  The pool is drawn with replacement from item_counts ** sampling_power (uniform when
    item_counts is None; the padding row and zero-count items are never drawn), afresh on every call from
    (seed, this loss's own step counter), so every data-parallel rank draws the same pool.  `negative_items` is
    accepted for the common signature and not used.  Not a ListwiseLoss: the trainer takes the per-operator path.
    `precision` "bf16x3" (default) or "bf16", as FullSoftmaxLoss."""

    def __init__(self, num_sampled: int = 8192, item_counts=None, sampling_power: float = 0.75,
                 temperature: float = 1.0, seed: int = 0, precision: str = "bf16x3"):
        super().__init__()
        if int(num_sampled) < 1:
            raise ValueError(f"num_sampled must be >= 1; got {num_sampled}")
        ops._softmax_precision(precision)
        self.precision = precision
        self.num_sampled = int(num_sampled)
        self.item_counts = item_counts
        self.sampling_power = sampling_power
        self.temperature = temperature
        self.seed = int(seed)
        self.step = 0
        self._cum = None

    def forward(self, session_embeddings, target_items, negative_items, item_embeddings) -> torch.Tensor:
        weight, padding_idx = ops._weight_and_padding(item_embeddings)
        items = weight.size(0)
        if self._cum is None or self._cum.device != weight.device or self._cum.numel() != items + 1:
            self._cum = ops.item_sampling_table(self.item_counts, self.sampling_power,
                                                padding_idx=-1 if padding_idx is None else padding_idx,
                                                num_items=items, device=weight.device)
        pool, log_q = ops.sample_item_pool(self._cum, self.num_sampled, self.seed, self.step)
        self.step += 1
        return ops.PoolSoftmaxLoss.apply(session_embeddings, weight, target_items, pool, log_q, self.temperature,
                                         None, padding_idx, False, self.precision)[0]


def create_loss_function(loss_type: str = "dual", alpha: float = 0.7, temperature: float = 1.0, *,
                         num_sampled: int = 8192, item_counts=None, sampling_power: float = 0.75,
                         seed: int = 0, precision: str = "bf16x3") -> nn.Module:
    """The loss named `loss_type`.  num_sampled / item_counts / sampling_power / seed configure "shared_pool_softmax"
    and are ignored by the other types; precision ("bf16x3" or "bf16") configures "full_softmax" and
    "shared_pool_softmax" and is ignored by the other types."""
    if loss_type == "bpr":
        return BPRLoss()
    if loss_type == "listwise":
        return ListwiseLoss(temperature=temperature)
    if loss_type == "dual":
        return DualLoss(alpha=alpha, temperature=temperature)
    if loss_type == "sampled_softmax":
        return SampledSoftmaxLoss(temperature=temperature)
    if loss_type == "full_softmax":
        return FullSoftmaxLoss(temperature=temperature, precision=precision)
    if loss_type == "shared_pool_softmax":
        return SharedPoolSoftmaxLoss(num_sampled=num_sampled, item_counts=item_counts, sampling_power=sampling_power,
                                     temperature=temperature, seed=seed, precision=precision)
    raise ValueError(f"Unknown loss type: {loss_type}")
