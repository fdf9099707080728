"""Shared-pool sampled softmax (etpgt_sample_item_pool, etpgt_pool_softmax_*, ops.pool_softmax_loss,
train.losses.SharedPoolSoftmaxLoss) on the GPU: the sampler bit for bit against its CPU restatement, the loss against
the full-catalogue loss it reduces to and against the fp64 objective (tests/shared_pool_ref.py), the unbiasedness of
the log-Q correction, determinism, the model and Trainer levels and the host-side checks.  Errors are
max|got - want| / max|want| unless stated otherwise."""

import numpy as np
import pytest
import torch

from shared_pool_ref import pool_softmax_fp64, sample_item_pool
from softmax_loss_util import err, grads, model_and_batch

TOL = 1e-4


def _zipf_counts(num_items, a=1.5, seed=0):
    rng = np.random.default_rng(seed)
    return torch.from_numpy(np.bincount(rng.zipf(a, 4 * num_items) % num_items, minlength=num_items))


def _run(sess, table, targets, pool, log_q, temperature=1.0, total=None, padding_idx=0, d_table=None, d_loss=1.0):
    """One forward and one backward through the C ABI: (loss, lse, d_sess, d_table)."""
    from etpgt_b200 import _lib
    from etpgt_b200._lib import ptr

    b, dim = sess.shape
    items, m = table.shape[0], pool.numel()
    dev = sess.device
    lse = torch.empty(b, dtype=torch.float32, device=dev)
    z_pos = torch.empty(b, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    ws = _lib.workspace(_lib.size("etpgt_pool_softmax_workspace_bytes", b, m, dim), dev)
    tot = float(total) if total else 0.0
    _lib.call("etpgt_pool_softmax_fwd", ptr(sess), ptr(table), ptr(targets), ptr(pool), ptr(log_q), b, items, m, dim,
              float(temperature), tot, padding_idx, ptr(lse), ptr(z_pos), ptr(loss), ptr(ws), ws.numel(),
              _lib.stream())
    dl = torch.tensor([d_loss], dtype=torch.float32, device=dev)
    d_sess = torch.empty_like(sess)
    d_table = torch.zeros_like(table) if d_table is None else d_table
    _lib.call("etpgt_pool_softmax_bwd", ptr(sess), ptr(table), ptr(targets), ptr(pool), ptr(log_q), ptr(lse),
              ptr(z_pos), ptr(dl), b, items, m, dim, float(temperature), tot, padding_idx, ptr(d_sess), ptr(d_table),
              ptr(ws), ws.numel(), _lib.stream())
    torch.cuda.synchronize()
    return loss[0], lse, d_sess, d_table


def _inputs(b, items, dim, m, seed, scale=0.3):
    """Random operands and a sorted pool with duplicates in which row 0's target is the first pool entry and a few
    targets occur several times."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    sess = torch.randn(b, dim, device="cuda", generator=g) * scale
    table = torch.randn(items, dim, device="cuda", generator=g) * scale
    targets = torch.randint(1, items, (b,), device="cuda", generator=g)
    pool = torch.randint(1, items, (m,), device="cuda", generator=g)
    if m >= 8:
        pool[: m // 8] = targets[torch.arange(m // 8, device="cuda") % min(b, 3)]
    pool = torch.sort(pool).values
    targets[0] = pool[0]
    log_q = torch.rand(m, device="cuda", generator=g) * 4 - 2
    return sess, table, targets, pool, log_q


# ------------------------------------------------------------------------------ sampler


@pytest.mark.gpu
@pytest.mark.parametrize("items", [2, 82_174, 1_000_000])
@pytest.mark.parametrize("kind", ["uniform", "zipf"])
def test_sampler_is_bit_identical_to_the_restatement(items, kind):
    from etpgt_b200 import ops

    counts = None if kind == "uniform" else _zipf_counts(items)
    if counts is not None:
        counts[1] += 1                        # at least one drawable item when items == 2
    cum = ops.item_sampling_table(counts, 0.75, 0, num_items=items, device="cuda")
    cum_host = cum.cpu().numpy()
    for m in (1, 127, 128, 8_192):
        pool, log_q = ops.sample_item_pool(cum, m, seed=0x1234_5678_9ABC, step=7 + m)
        want_ids, _ = sample_item_pool(cum_host, m, 0x1234_5678_9ABC, 7 + m)
        got = pool.cpu().numpy()
        assert (got == want_ids).all(), (items, kind, m)
        assert (np.diff(got) >= 0).all()
        w = np.diff(cum_host)[got].astype(np.float64)
        want_lq = np.log(m * w / float(cum_host[-1]))
        ulp = np.spacing(np.abs(want_lq).astype(np.float32)).astype(np.float64)
        assert (np.abs(log_q.cpu().numpy().astype(np.float64) - want_lq) <= ulp).all()


# ------------------------------------------------------------------------------ the loss


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [64, 256])
@pytest.mark.parametrize("temperature", [1.0, 0.07])
def test_pool_of_every_item_reduces_to_the_full_loss(dim, temperature):
    from etpgt_b200 import _lib
    from etpgt_b200._lib import ptr

    b, items = 1_000, 5_000
    sess, table, targets, _, _ = _inputs(b, items, dim, 1, seed=dim)
    sess, table = sess * 0.5, table * 0.5
    pool = torch.arange(1, items, device="cuda")
    got = _run(sess, table, targets, pool, torch.zeros(items - 1, device="cuda"), temperature)
    lse = torch.empty(b, device="cuda")
    loss = torch.empty(1, device="cuda")
    ws = _lib.workspace(_lib.size("etpgt_full_softmax_workspace_bytes", b, items, dim), sess.device)
    _lib.call("etpgt_full_softmax_fwd", ptr(sess), ptr(table), ptr(targets), b, items, dim, temperature, 0.0, 0,
              ptr(lse), ptr(loss), ptr(ws), ws.numel(), _lib.stream())
    d_sess, d_table = torch.empty_like(sess), torch.zeros_like(table)
    dl = torch.ones(1, device="cuda")
    _lib.call("etpgt_full_softmax_bwd", ptr(sess), ptr(table), ptr(targets), ptr(lse), ptr(dl), b, items, dim,
              temperature, 0.0, 0, ptr(d_sess), ptr(d_table), ptr(ws), ws.numel(), _lib.stream())
    torch.cuda.synchronize()
    for name, g, w in zip(("loss", "lse", "d_sess", "d_table"), got, (loss[0], lse, d_sess, d_table)):
        assert err(g, w) <= 1e-5, (name, err(g, w))


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [64, 128, 192, 256])
@pytest.mark.parametrize("m", [1, 100, 128, 4_096, 8_192])
@pytest.mark.parametrize("batch", [1, 127, 128, 1_000, 32_768])
def test_matches_fp64_on_the_grid(batch, m, dim):
    items = 5_003
    sess, table, targets, pool, log_q = _inputs(batch, items, dim, m, seed=batch + m + dim)
    got = _run(sess, table, targets, pool, log_q, temperature=0.5)
    want = pool_softmax_fp64(sess, table, targets, pool, log_q, temperature=0.5)
    errs = {name: err(g, w) for name, g, w in zip(("loss", "lse", "d_sess", "d_table"), got, want)}
    assert all(v <= TOL for v in errs.values()), errs
    # row 0's target is pool[0]; with M = 1 its whole pool is its target: P = 1 exactly and its gradient is zero
    if m == 1:
        assert float(got[2][0].abs().max()) == 0.0


@pytest.mark.gpu
def test_pool_entirely_the_target_gives_zero_gradient_for_that_row():
    b, items, dim = 64, 300, 128
    sess, table, targets, _, _ = _inputs(b, items, dim, 1, seed=9)
    pool = torch.full((256,), int(targets[0]), device="cuda")
    targets[1:] = torch.where(targets[1:] == targets[0], targets[1:] % (items - 1) + 1, targets[1:])
    log_q = torch.zeros(256, device="cuda")
    got = _run(sess, table, targets, pool, log_q)
    want = pool_softmax_fp64(sess, table, targets, pool, log_q)
    assert float(got[2][0].abs().max()) == 0.0
    for name, g, w in zip(("loss", "lse", "d_sess", "d_table"), got, want):
        assert err(g, w) <= TOL, name


@pytest.mark.gpu
def test_accumulates_and_keeps_padding_and_untouched_rows():
    b, items, dim, m = 300, 2_000, 128, 700
    sess, table, targets, pool, log_q = _inputs(b, items, dim, m, seed=4)
    pool[:5] = 0                                           # padding entries in an explicit pool never count
    pool = torch.sort(pool).values
    targets[0] = pool[5]
    base = torch.randn(items, dim, device="cuda")
    got = _run(sess, table, targets, pool, log_q, d_table=base.clone())
    want = pool_softmax_fp64(sess, table, targets, pool, log_q)
    assert err(got[0], want[0]) <= TOL and err(got[2], want[2]) <= TOL
    assert err(got[3] - base, want[3]) <= TOL
    touched = torch.zeros(items, dtype=torch.bool, device="cuda")
    touched[pool] = True
    touched[targets] = True
    touched[0] = False
    assert torch.equal(got[3][~touched], base[~touched])   # padding row and untouched rows keep their bits


@pytest.mark.gpu
def test_log_q_correction_is_unbiased():
    from etpgt_b200 import _lib, ops
    from etpgt_b200._lib import ptr

    b, items, dim, m, pools = 16, 3_000, 64, 512, 64
    sess, table, targets, _, _ = _inputs(b, items, dim, 1, seed=21, scale=0.15)
    counts = _zipf_counts(items, seed=2) + 1
    cum = ops.item_sampling_table(counts, 0.75, 0, device="cuda")
    lse_full = torch.empty(b, device="cuda")
    loss = torch.empty(1, device="cuda")
    ws = _lib.workspace(_lib.size("etpgt_full_softmax_workspace_bytes", b, items, dim), sess.device)
    _lib.call("etpgt_full_softmax_fwd", ptr(sess), ptr(table), ptr(targets), b, items, dim, 1.0, 0.0, 0,
              ptr(lse_full), ptr(loss), ptr(ws), ws.numel(), _lib.stream())
    ratios = []
    for step in range(pools):
        pool, log_q = ops.sample_item_pool(cum, m, seed=77, step=step)
        lse = ops.PoolSoftmaxLoss.apply(sess, table, targets, pool, log_q, 1.0, None, 0, True)[1]
        ratios.append(torch.exp(lse.double() - lse_full.double()))
    r = torch.stack(ratios)                                  # E[exp(lse_pooled)] / exp(lse_full) = 1
    mean, se = r.mean(0), r.std(0) / pools ** 0.5
    assert bool(((mean - 1).abs() <= 5 * se).all()), ((mean - 1) / se).tolist()


@pytest.mark.gpu
def test_bit_reproducible_and_data_parallel_halves():
    b, items, dim, m = 2_048, 20_000, 256, 4_096
    sess, table, targets, pool, log_q = _inputs(b, items, dim, m, seed=13)
    a = _run(sess, table, targets, pool, log_q)
    c = _run(sess, table, targets, pool, log_q)
    for x, y in zip(a, c):
        assert torch.equal(x, y)
    # half the batch splits the pool's column ranges differently, so the sums round differently (measured ~1e-6)
    h = b // 2
    lo = _run(sess[:h].contiguous(), table, targets[:h].contiguous(), pool, log_q, total=b)
    hi = _run(sess[h:].contiguous(), table, targets[h:].contiguous(), pool, log_q, total=b)
    assert err(lo[0] + hi[0], a[0]) <= 1e-5
    assert err(torch.cat([lo[1], hi[1]]), a[1]) <= 1e-5
    assert err(torch.cat([lo[2], hi[2]]), a[2]) <= 1e-5
    assert err(lo[3] + hi[3], a[3]) <= 1e-5


# ------------------------------------------------------------------------------ host errors


@pytest.mark.gpu
def test_host_errors():
    from etpgt_b200 import ops

    sess, table, targets, pool, log_q = _inputs(8, 50, 64, 16, seed=1)
    with pytest.raises(RuntimeError, match="64, 128, 192, 256"):
        ops.pool_softmax_loss(torch.randn(8, 96, device="cuda"), torch.randn(50, 96, device="cuda"), targets, pool,
                              log_q)
    with pytest.raises(RuntimeError, match="num_sampled must be"):
        ops.sample_item_pool(ops.item_sampling_table(num_items=50, device="cuda"), 0, 0, 0)
    with pytest.raises(RuntimeError, match="pool_ids must be a non-empty"):
        ops.pool_softmax_loss(sess, table, targets, pool[:0], log_q[:0])
    bad = pool.clone()
    bad[-1] = 50
    with pytest.raises(RuntimeError, match="out of range"):
        ops.pool_softmax_loss(sess, table, targets, bad, log_q)
    bad[-1] = -1
    with pytest.raises(RuntimeError, match="out of range"):
        ops.pool_softmax_loss(sess, table, targets, bad, log_q)
    with pytest.raises(RuntimeError, match="log_q"):
        ops.pool_softmax_loss(sess, table, targets, pool, log_q[:-1])
    with pytest.raises(RuntimeError, match="target_items"):
        ops.pool_softmax_loss(sess, table, targets[:-1], pool, log_q)
    with pytest.raises(RuntimeError, match="sess"):
        ops.pool_softmax_loss(sess, table[:, :32].contiguous(), targets, pool, log_q)


@pytest.mark.gpu
def test_unsorted_pool_is_sorted_with_its_log_q():
    from etpgt_b200 import ops

    sess, table, targets, pool, log_q = _inputs(200, 400, 128, 300, seed=3)
    perm = torch.randperm(300, device="cuda")
    want = ops.pool_softmax_loss(sess, table, targets, pool, log_q)
    got = ops.pool_softmax_loss(sess, table, targets, pool[perm], log_q[perm])
    assert float(got) == float(want)


# ------------------------------------------------------------------------------ model and Trainer


@pytest.mark.gpu
def test_model_gradients_match_fp64_objective():
    from etpgt_b200 import ops

    temperature = 0.5
    model, batch, (d, _, _) = model_and_batch()
    model.train()
    cum = ops.item_sampling_table(num_items=d.num_items, device="cuda")
    pool, log_q = ops.sample_item_pool(cum, 300, seed=1, step=0)
    for p in model.parameters():
        p.grad = None
    loss = ops.pool_softmax_loss(model(batch), model.item_embedding, batch.target_item, pool, log_q,
                                 temperature=temperature)
    loss.backward()
    got, got_loss = grads(model), float(loss.detach())
    for p in model.parameters():
        p.grad = None
    sess = model(batch).double()
    e = model.item_embedding.weight.double()
    t = batch.target_item
    z_pos = (sess * e[t]).sum(1) / temperature
    z = sess @ e[pool].T / temperature - log_q.double()[None, :]
    z = z.masked_fill((pool[None, :] == t[:, None]) | (pool == 0)[None, :], -float("inf"))
    want_loss = (torch.logsumexp(torch.cat([z_pos[:, None], z], 1), 1) - z_pos).mean()
    want_loss.backward()
    want, want_loss = grads(model), float(want_loss.detach())
    assert abs(got_loss - want_loss) <= TOL * abs(want_loss)
    assert set(got) == set(want)
    scale = max(float(g.abs().max()) for g in want.values())
    for name in want:
        if float(want[name].abs().max()) <= 1e-6 * scale:
            assert float((got[name] - want[name]).abs().max()) <= 1e-6 * scale, name
            continue
        assert err(got[name], want[name]) <= TOL, (name, err(got[name], want[name]))


@pytest.mark.gpu
@pytest.mark.parametrize("opt_kind", ["lazy_adamw", "sparse_adam", "adamw"])
def test_trainer_learns_with_the_shared_pool(opt_kind, tmp_path):
    from etpgt_b200 import data, optim
    from etpgt_b200.train.losses import create_loss_function
    from etpgt_b200.train.trainer import Trainer

    model, _, (d, graph, store) = model_and_batch()

    def batches(lo, hi, step0):
        out = []
        for i, s in enumerate(range(lo, hi, 128)):
            ids = np.arange(s, min(hi, s + 128))
            bt = data.build_batch(graph, store, ids, 50, False, False)
            bt.negative_items = data.sample_negatives(store, ids, d.num_items, 5, seed=3, step=step0 + i).view(-1)
            out.append(bt)
        return out

    table = model.item_embedding.weight
    if opt_kind == "lazy_adamw":
        opt = optim.AdamW(model.parameters(), lr=3e-3, lazy_rows=True)
    elif opt_kind == "sparse_adam":
        rest = [p for p in model.parameters() if p is not table]
        opt = [optim.SparseAdam([table], lr=3e-3), optim.AdamW(rest, lr=3e-3)]
    else:
        opt = optim.AdamW(model.parameters(), lr=3e-3)
    counts = torch.bincount(torch.as_tensor(d.sess_items), minlength=d.num_items)
    loss_fn = create_loss_function("shared_pool_softmax", num_sampled=256, item_counts=counts, seed=3)
    if isinstance(opt, list):
        opt = _Chain(opt)
    trainer = Trainer(model, batches(0, 768, 0), batches(900, 1100, 100), opt, device="cuda", output_dir=tmp_path,
                      max_epochs=2, patience=5, k_values=[20], loss_fn=loss_fn)
    assert trainer._driver is None
    losses = trainer.train()["train_loss"]
    assert len(losses) == 2 and all(np.isfinite(losses)), losses
    assert losses[1] < losses[0], losses
    assert loss_fn.step == 12


class _Chain:
    """Two optimizers stepped together (the sparse table optimizer next to a dense one for the rest)."""

    def __init__(self, opts):
        self.opts = opts
        self.param_groups = [g for o in opts for g in o.param_groups]

    def zero_grad(self, set_to_none=True):
        for o in self.opts:
            o.zero_grad(set_to_none=set_to_none)

    def step(self):
        for o in self.opts:
            o.step()

    def state_dict(self):
        return [o.state_dict() for o in self.opts]
