"""BPR / listwise / dual / sampled-softmax / full-catalogue softmax losses with the reference's call signature
`loss(session_embeddings, target_items, negative_items, item_embeddings: nn.Embedding)`
(etpgt/train/losses.py), computed by the fused sampled-loss kernel (full_softmax: the tensor-core full-catalogue kernels)."""

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
    step driver has no full-catalogue mode, so the trainer takes the per-operator path for it."""

    def __init__(self, temperature: float = 1.0):
        super().__init__()
        self.temperature = temperature

    def forward(self, session_embeddings, target_items, negative_items, item_embeddings) -> torch.Tensor:
        return ops.full_softmax_loss(session_embeddings, item_embeddings, target_items, temperature=self.temperature)


def create_loss_function(loss_type: str = "dual", alpha: float = 0.7, temperature: float = 1.0) -> nn.Module:
    if loss_type == "bpr":
        return BPRLoss()
    if loss_type == "listwise":
        return ListwiseLoss(temperature=temperature)
    if loss_type == "dual":
        return DualLoss(alpha=alpha, temperature=temperature)
    if loss_type == "sampled_softmax":
        return SampledSoftmaxLoss(temperature=temperature)
    if loss_type == "full_softmax":
        return FullSoftmaxLoss(temperature=temperature)
    raise ValueError(f"Unknown loss type: {loss_type}")
