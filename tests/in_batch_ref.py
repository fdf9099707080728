"""References for the in-batch and mixed-negative softmax (ops.in_batch_columns, train.losses.InBatchSoftmaxLoss): the
streaming estimate of each item's share of the batch's targets in fp64 numpy, its prior, and the merged column list."""

import numpy as np


def prior(num_items, padding_idx=0, counts=None):
    """freq at step 0: counts / sum (uniform without counts), 0 for the padding row."""
    q = np.ones(num_items) if counts is None else np.asarray(counts, dtype=np.float64).copy()
    if 0 <= padding_idx < num_items:
        q[padding_idx] = 0.0
    return q / q.sum()


def counted(t, num_items, padding_idx):
    return 0 <= t < num_items and t != padding_idx


def update(freq, last, targets, step, decay, padding_idx):
    """One lazy estimator step in place, as etpgt_in_batch_columns:
    freq[i] = freq[i] (1 - decay)^(step - last[i]) + decay n_i / B,  last[i] = step."""
    b = len(targets)
    ids, n = np.unique(np.asarray(targets, dtype=np.int64), return_counts=True)
    for i, c in zip(ids.tolist(), n.tolist()):
        if counted(i, freq.size, padding_idx):
            freq[i] = freq[i] * (1.0 - decay) ** (step - last[i]) + decay * c / b
            last[i] = step


def eager(q, targets, decay, padding_idx):
    """The eager EMA the lazy update equals: q <- (1 - decay) q + decay f over every item, f the step's shares."""
    f = np.zeros_like(q)
    for t in targets:
        if counted(int(t), q.size, padding_idx):
            f[int(t)] += 1.0 / len(targets)
    return (1.0 - decay) * q + decay * f


def columns(targets, freq, padding_idx, pool_ids=None, pool_log_q=None):
    """(columns int64, log_q float32) after the update: pool entries and in-batch entries by ascending id, pool entries
    first among equal ids, then in-batch entries in session order.  In-batch log_q = log(B freq[t]), +inf for the
    padding id and ids outside the table."""
    b = len(targets)
    entries = []
    if pool_ids is not None:
        entries += [(int(p), 0, j, float(lq)) for j, (p, lq) in enumerate(zip(pool_ids, pool_log_q))]
    for s, t in enumerate(np.asarray(targets, dtype=np.int64).tolist()):
        lq = float(np.float32(np.log(b * freq[t]))) if counted(t, freq.size, padding_idx) else np.inf
        entries.append((t, 1, s, lq))
    entries.sort(key=lambda e: e[:3])
    return (np.array([e[0] for e in entries], dtype=np.int64), np.array([e[3] for e in entries], dtype=np.float32))
