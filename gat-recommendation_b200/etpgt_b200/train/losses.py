"""BPR / listwise / dual / sampled-softmax / full-catalogue / shared-pool / in-batch softmax losses with the reference's
call signature `loss(session_embeddings, target_items, negative_items, item_embeddings: nn.Embedding)`
(etpgt/train/losses.py), computed by the fused sampled-loss kernel (full_softmax: the tensor-core full-catalogue kernels;
shared_pool_softmax: the same kernels over one log-Q-corrected negative pool shared by the batch; in_batch_softmax /
mixed_softmax: the same kernels over the batch's targets, plus such a pool for mixed_softmax)."""

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


class InBatchSoftmaxLoss(nn.Module):
    """Sampled softmax whose negatives are the batch's other targets (in-batch negatives), plus with num_sampled > 0
    a shared pool drawn exactly as SharedPoolSoftmaxLoss draws it ("mixed negative sampling", Yi et al., RecSys 2019;
    Yang et al., WWW 2020).  The columns are the B targets and the M pool entries:
        z_pos[b] = s_b . e_{t_b} / T,   z[b, c] = s_b . e_{col_c} / T - log_q[c]  (-inf where col_c is t_b or padding)
        loss = sum_b (logsumexp(z_pos[b], z[b, :]) - z_pos[b]) / B
    log_q[c] is the log of the expected copies of the item among its source's columns: log(B q_i) for an in-batch
    entry, log(M q(i)) for a pool entry.  An item in both sources appears twice, each copy corrected by its own source:
    the usual mixed-sampling approximation.  The positive is not corrected, as in pool_softmax_loss.

    q_i is a streaming estimate of item i's share of the batch's targets (ops.in_batch_columns): an exponential moving
    average over steps with weight freq_decay, updated lazily for the items of each step.  Yi et al. estimate the gap
    between sightings; this estimates the per-step share, so an item seen several times in one batch is counted by
    its copies.  Its prior is item_counts / sum (power 1; uniform without counts), 0 for the padding row.  item_counts
    ** sampling_power is the pool's proposal.  `freq`, `last` and `step` are buffers, so state_dict() /
    load_state_dict() resume the estimator and the pool sequence exactly.

    Data parallelism: each rank's columns are its own share's targets and each rank estimates their proposal from
    them, so no collective is needed; unlike the shared pool, the result depends on how the global batch is split.
    `negative_items` is accepted for the common signature and not used.  `precision` "bf16x3" (default) or "bf16",
    as FullSoftmaxLoss."""

    def __init__(self, num_sampled: int = 0, item_counts=None, sampling_power: float = 0.75,
                 temperature: float = 1.0, seed: int = 0, freq_decay: float = 0.01, precision: str = "bf16x3"):
        super().__init__()
        if int(num_sampled) < 0:
            raise ValueError(f"num_sampled must be >= 0; got {num_sampled}")
        if not 0.0 < float(freq_decay) <= 1.0:
            raise ValueError(f"freq_decay must be in (0, 1]; got {freq_decay}")
        ops._softmax_precision(precision)
        self.num_sampled = int(num_sampled)
        self.item_counts = item_counts
        self.sampling_power = sampling_power
        self.temperature = temperature
        self.seed = int(seed)
        self.freq_decay = float(freq_decay)
        self.precision = precision
        self.register_buffer("freq", torch.zeros(0, dtype=torch.float64))
        self.register_buffer("last", torch.zeros(0, dtype=torch.int64))
        self.register_buffer("step", torch.zeros((), dtype=torch.int64))
        self._step = 0                   # host copy of `step`: the forward reads no device value
        self._cum = None

    def _prior(self, items: int, padding_idx, device) -> torch.Tensor:
        if self.item_counts is None:
            q = torch.ones(items, dtype=torch.float64)
        else:
            q = torch.as_tensor(self.item_counts).detach().to("cpu", torch.float64).reshape(-1).clone()
            if q.numel() != items:
                raise ValueError(f"item_counts has {q.numel()} entries for {items} items")
            if bool((q < 0).any()) or not bool(torch.isfinite(q).all()):
                raise ValueError("item_counts must be finite and >= 0")
        if padding_idx is not None and 0 <= padding_idx < items:
            q[padding_idx] = 0.0
        if not float(q.sum()) > 0.0:
            raise ValueError("no item has a positive count")
        return (q / q.sum()).to(device)

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        for name in ("freq", "last"):    # the estimator is sized by the table at its first call
            src = state_dict.get(prefix + name)
            if src is not None and src.shape != self._buffers[name].shape:
                self._buffers[name] = torch.empty(src.shape, dtype=self._buffers[name].dtype,
                                                  device=self._buffers[name].device)
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)
        self._step = int(self.step)

    def forward(self, session_embeddings, target_items, negative_items, item_embeddings) -> torch.Tensor:
        weight, padding_idx = ops._weight_and_padding(item_embeddings)
        items, dev = weight.size(0), weight.device
        if self.freq.numel() != items:
            self.freq = self._prior(items, padding_idx, dev)
            self.last = torch.full((items,), -1, dtype=torch.int64, device=dev)
        elif self.freq.device != dev:
            self.freq, self.last = self.freq.to(dev), self.last.to(dev)
        pool = log_q = None
        if self.num_sampled > 0:
            if self._cum is None or self._cum.device != dev or self._cum.numel() != items + 1:
                self._cum = ops.item_sampling_table(self.item_counts, self.sampling_power,
                                                    padding_idx=-1 if padding_idx is None else padding_idx,
                                                    num_items=items, device=dev)
            pool, log_q = ops.sample_item_pool(self._cum, self.num_sampled, self.seed, self._step)
        columns, col_log_q = ops.in_batch_columns(target_items, self.freq, self.last, self._step, self.freq_decay,
                                                  padding_idx, pool, log_q)
        self._step += 1
        self.step.fill_(self._step)
        return ops.PoolSoftmaxLoss.apply(session_embeddings, weight, target_items, columns, col_log_q,
                                         self.temperature, None, padding_idx, False, self.precision)[0]


def create_loss_function(loss_type: str = "dual", alpha: float = 0.7, temperature: float = 1.0, *,
                         num_sampled: int = 8192, item_counts=None, sampling_power: float = 0.75,
                         seed: int = 0, precision: str = "bf16x3", freq_decay: float = 0.01) -> nn.Module:
    """The loss named `loss_type`.  num_sampled / item_counts / sampling_power / seed configure "shared_pool_softmax"
    and "mixed_softmax" (in-batch negatives plus a shared pool of num_sampled); "in_batch_softmax" (in-batch negatives
    only) ignores num_sampled; item_counts is also the prior of both in-batch losses' estimator, and freq_decay
    configures it (InBatchSoftmaxLoss).  The other
    types ignore them.  precision ("bf16x3" or "bf16") configures "full_softmax", "shared_pool_softmax" and both
    in-batch losses and is ignored by the other types."""
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
    if loss_type in ("in_batch_softmax", "mixed_softmax"):
        return InBatchSoftmaxLoss(num_sampled=num_sampled if loss_type == "mixed_softmax" else 0,
                                  item_counts=item_counts, sampling_power=sampling_power, temperature=temperature,
                                  seed=seed, freq_decay=freq_decay, precision=precision)
    raise ValueError(f"Unknown loss type: {loss_type}")
