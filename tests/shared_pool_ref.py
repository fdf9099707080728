"""References for the shared-pool sampled softmax (ops.sample_item_pool, ops.pool_softmax_loss): the pool sampler
restated with Python integers on oracle/graph_ref's Philox, and the objective evaluated in fp64 with torch autograd."""

from bisect import bisect_right

import numpy as np
import torch

from oracle.graph_ref import philox4x32_10

_MASK = 0xFFFFFFFF
POOL_WORD = 0x504F4F4C   # "POOL": the second counter word, never a slot of sample_negatives (< 64)


def sample_item_pool(cum, num_sampled: int, seed: int, step: int):
    """(ids sorted ascending int64 [M], log_q float32 [M]) of etpgt_sample_item_pool.  Draw j: Philox4x32-10 with key
    (seed lo, seed hi) and counter (j >> 1, POOL_WORD, 0, step); u = c[2(j&1)] | c[2(j&1)+1] << 32; r = (u W) >> 64;
    the id i with cum[i] <= r < cum[i+1]; log_q = log(M w_i / W) in fp64."""
    cum = [int(c) for c in cum]
    total = cum[-1]
    key = (seed & _MASK, (seed >> 32) & _MASK)
    ids = []
    words = None
    for j in range(num_sampled):
        if j % 2 == 0:
            words = philox4x32_10((j >> 1, POOL_WORD, 0, step), key)
        h = 2 * (j & 1)
        u = words[h] | (words[h + 1] << 32)
        ids.append(bisect_right(cum, (u * total) >> 64) - 1)
    ids.sort()
    w = np.array([cum[i + 1] - cum[i] for i in ids], dtype=np.float64)
    log_q = np.log(float(num_sampled) * w / float(total)).astype(np.float32)
    return np.asarray(ids, dtype=np.int64), log_q


def pool_softmax_fp64(sess, table, targets, pool, log_q, temperature=1.0, total=None, padding_idx=0, d_loss=1.0):
    """fp64 (loss, lse [B], d_sess [B, D], d_table [I, D]) of
        z_pos[b] = s_b . e_{t_b} / T,  z[b, j] = s_b . e_{p_j} / T - log_q[j]  (-inf where p_j == t_b or padding)
        loss = sum_b (logsumexp(z_pos[b], z[b, :]) - z_pos[b]) / total."""
    s = sess.detach().double().requires_grad_(True)
    e = table.detach().double().requires_grad_(True)
    t, p = targets.long(), pool.long()
    b = s.shape[0]
    total = float(total) if total else float(b)
    z_pos = (s * e[t]).sum(1) / temperature
    z = s @ e[p].T / temperature - log_q.double()[None, :]
    mask = (p[None, :] == t[:, None]) | (p == padding_idx)[None, :]
    z = z.masked_fill(mask, -float("inf"))
    lse = torch.logsumexp(torch.cat([z_pos[:, None], z], dim=1), dim=1)
    loss = (lse - z_pos).sum() / total
    (loss * d_loss).backward()
    d_table = e.grad
    if padding_idx >= 0:
        d_table[padding_idx] = 0
    return loss.detach(), lse.detach(), s.grad, d_table
