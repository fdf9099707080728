"""Reference ranking with an exclusion list, the oracle of the filtered scorers (ops.score_topk(exclude=...)).

The serving filter of the reference's Recommender (recommender.py:133-134) sets the scores of the listed items to
-inf before `topk`; the ranking rule is the oracle's (score desc, ties to the lower id, model_ref.topk_lower_id).
Slots past a row's last eligible item are (-inf, INT64_MAX), as the library reports them."""

import torch

from oracle import model_ref

NO_ID = torch.iinfo(torch.int64).max


def predict_excluding(sess, table, k=20, exclude=None, bf16_inputs=False, id_base=0):
    """model_ref.predict with exclude [B, L] int64: ids outside [id_base, id_base + rows of table) are ignored.
    Returned ids are offset by id_base."""
    if bf16_inputs:
        sess = sess.to(torch.bfloat16).to(torch.float64)
        table = table.to(torch.bfloat16).to(torch.float64)
    scores = sess.double() @ table.double().t()
    b, n = scores.shape
    if exclude is None:
        exclude = torch.empty(b, 0, dtype=torch.int64)
    rel = torch.as_tensor(exclude, dtype=torch.int64).cpu() - id_base
    valid = (rel >= 0) & (rel < n)
    masked = torch.zeros(b, n + 1, dtype=torch.bool)
    masked.scatter_(1, torch.where(valid, rel, torch.full_like(rel, n)), True)   # column n collects ignored ids
    masked = masked[:, :n]
    val, idx = model_ref.topk_lower_id(scores.masked_fill(masked, float("-inf")), k)
    gone = masked.gather(1, idx)
    val = val.masked_fill(gone, float("-inf"))
    idx = torch.where(gone, torch.full_like(idx, NO_ID), idx + id_base)
    if idx.size(1) < k:   # fewer items than k
        val = torch.cat([val, torch.full((b, k - idx.size(1)), float("-inf"), dtype=val.dtype)], dim=1)
        idx = torch.cat([idx, torch.full((b, k - idx.size(1)), NO_ID)], dim=1)
    return val, idx


def hit_positions(idx, targets, k):
    """Position of each target among its row's first k ids, or -1 (etpgt/utils/metrics.py:49, first match)."""
    hit = idx[:, :k] == torch.as_tensor(targets).view(-1, 1)
    return torch.where(hit.any(dim=1), hit.int().argmax(dim=1), torch.full((idx.size(0),), -1)).int()
