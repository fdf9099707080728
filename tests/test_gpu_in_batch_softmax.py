"""In-batch and mixed-negative softmax (etpgt_in_batch_columns, ops.in_batch_columns,
train.losses.InBatchSoftmaxLoss) on the GPU: the column builder and its estimator against tests/in_batch_ref.py step
by step, the loss against the fp64 objective over the reference columns (tests/shared_pool_ref.py) and bit for bit
against ops.pool_softmax_loss, its properties, the model and Trainer levels and the argument checks.  Errors are
max|got - want| / max|want| unless stated otherwise."""

import numpy as np
import pytest
import torch

import in_batch_ref as ref
from shared_pool_ref import pool_softmax_fp64
from softmax_loss_util import err, grads, model_and_batch
from test_gpu_shared_pool_softmax import TOL
from test_gpu_softmax_bf16 import TOL_GRAD, TOL_VALUE, _pool_oracle

ITEMS = 5_003


def _targets(b, items, seed, a=1.3):
    """Zipf-distributed targets (duplicates; id 0, the padding row, now and then)."""
    rng = np.random.default_rng(seed)
    return torch.from_numpy(rng.zipf(a, b) % items).cuda()


def _state(items, pad=0, counts=None):
    freq = torch.from_numpy(ref.prior(items, pad, counts)).cuda()
    return freq, torch.full((items,), -1, dtype=torch.int64, device="cuda")


def _pool(items, m, step, seed=5):
    from etpgt_b200 import ops

    cum = ops.item_sampling_table(num_items=items, padding_idx=0, device="cuda")
    return ops.sample_item_pool(cum, m, seed, step)


# ------------------------------------------------------------------------------ the column builder


@pytest.mark.gpu
@pytest.mark.parametrize("m", [0, 4_096])
@pytest.mark.parametrize("batch", [1, 32_768, "all_equal"])
def test_builder_matches_the_reference_for_50_steps(batch, m):
    from etpgt_b200 import ops

    items, decay = ITEMS, 0.05
    freq, last = _state(items)
    freq_ref, last_ref = freq.cpu().numpy().copy(), last.cpu().numpy().copy()
    for step in range(50):
        if batch == "all_equal":
            t = torch.full((4_096,), 17 if step % 3 else 0, dtype=torch.int64, device="cuda")
        else:
            t = _targets(batch, items if step % 10 else 7, seed=step)      # every tenth step: only ids < 7
        pool, pool_lq = _pool(items, m, step) if m else (None, None)
        cols, lq = ops.in_batch_columns(t, freq, last, step, decay, 0, pool, pool_lq)
        t_host = t.cpu().numpy()
        ref.update(freq_ref, last_ref, t_host, step, decay, 0)
        want_cols, want_lq = ref.columns(t_host, freq_ref, 0, *(() if not m else (pool.cpu().numpy(),
                                                                                   pool_lq.cpu().numpy())))
        assert np.array_equal(cols.cpu().numpy(), want_cols), step
        np.testing.assert_allclose(lq.cpu().numpy(), want_lq, rtol=1e-6, atol=1e-6)
        np.testing.assert_array_equal(last.cpu().numpy(), last_ref)
        np.testing.assert_allclose(freq.cpu().numpy(), freq_ref, rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_builder_is_bitwise_deterministic_and_leaves_out_of_range_targets_alone():
    from etpgt_b200 import ops

    t = _targets(32_768, ITEMS, seed=3)
    t[:5] = torch.tensor([-4, ITEMS, ITEMS + 9, -1, 0], device="cuda")
    pool, pool_lq = _pool(ITEMS, 8_192, 0)
    outs = []
    for _ in range(2):
        freq, last = _state(ITEMS)
        outs.append((*ops.in_batch_columns(t, freq, last, 3, 0.01, 0, pool, pool_lq), freq, last))
    for x, y in zip(*outs):
        assert torch.equal(x, y)
    cols, lq, freq, last = outs[0]
    # the out-of-range ids sort to the ends with log_q = +inf, as the padding id does
    assert cols[:2].tolist() == [-4, -1] and sorted(cols[-2:].tolist()) == [ITEMS, ITEMS + 9]
    assert bool(torch.isinf(lq[:2]).all()) and bool(torch.isinf(lq[-2:]).all())
    assert bool((torch.diff(cols[2:-2]) >= 0).all())
    assert bool((lq[cols == 0] == float("inf")).all())
    assert float(freq[0]) == 0.0 and int(last[0]) == -1


@pytest.mark.gpu
def test_abi_workspace_and_argument_errors():
    from etpgt_b200 import _lib
    from etpgt_b200._lib import ptr

    t = torch.tensor([3, 1, 3], device="cuda")
    freq, last = _state(10)
    cols = torch.empty(3, dtype=torch.int64, device="cuda")
    lq = torch.empty(3, device="cuda")
    need = _lib.size("etpgt_in_batch_columns_workspace_bytes", 3, 0)
    ws = _lib.workspace(need, "cuda")
    args = [ptr(t), 3, None, None, 0, ptr(freq), ptr(last), 10, 0, 0, 0.01, ptr(cols), ptr(lq), ptr(ws), need,
            _lib.stream()]
    with pytest.raises(RuntimeError, match=r"\(-3\): in_batch_columns: workspace too small"):
        _lib.call("etpgt_in_batch_columns", *args[:-2], need - 1, args[-1])
    _lib.call("etpgt_in_batch_columns", *args)
    torch.cuda.synchronize()
    assert cols.tolist() == [1, 3, 3]


# ------------------------------------------------------------------------------ the loss


def _reference_columns(t, freq_before, last_before, step, decay, pool=None, pool_lq=None):
    f, l_ = freq_before.cpu().numpy().copy(), last_before.cpu().numpy().copy()
    ref.update(f, l_, t.cpu().numpy(), step, decay, 0)
    args = () if pool is None else (pool.cpu().numpy(), pool_lq.cpu().numpy())
    cols, lq = ref.columns(t.cpu().numpy(), f, 0, *args)
    return torch.from_numpy(cols).cuda(), torch.from_numpy(lq).cuda()


def _loss_inputs(b, dim, seed, scale=0.3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    sess = torch.randn(b, dim, device="cuda", generator=g) * scale
    table = torch.randn(ITEMS, dim, device="cuda", generator=g) * scale
    return sess, table, _targets(b, ITEMS, seed)


def _loss_and_grads(loss_fn, sess, table, t, d_table=None):
    s = sess.clone().requires_grad_(True)
    emb = torch.nn.Embedding.from_pretrained(table.clone(), freeze=False, padding_idx=0)
    loss = loss_fn(s, t, None, emb)
    loss.backward()
    return loss.detach(), s.grad, emb.weight.grad


@pytest.mark.gpu
@pytest.mark.parametrize("m", [0, 4_096])
@pytest.mark.parametrize("dim", [64, 128, 192, 256])
@pytest.mark.parametrize("batch", [1, 127, 128, 1_000, 32_768])
def test_matches_fp64_on_the_reference_columns(batch, dim, m):
    from etpgt_b200.train.losses import InBatchSoftmaxLoss

    sess, table, t = _loss_inputs(batch, dim, seed=batch + dim + m)
    loss_fn = InBatchSoftmaxLoss(num_sampled=m, temperature=0.5, seed=5)
    loss_fn(sess, t, None, torch.nn.Embedding(ITEMS, dim, padding_idx=0).cuda())   # step 0: a different batch
    freq, last = loss_fn.freq.clone(), loss_fn.last.clone()
    pool, pool_lq = _pool(ITEMS, m, 1) if m else (None, None)
    cols, lq = _reference_columns(t, freq, last, 1, 0.01, pool, pool_lq)
    loss, d_sess, d_table = _loss_and_grads(loss_fn, sess, table, t)
    assert int(loss_fn.last.max()) == 1
    _, lse = _lse(sess, table, t, cols, lq)
    want = pool_softmax_fp64(sess, table, t, cols, lq, temperature=0.5)
    errs = {"loss": err(loss, want[0]), "lse": err(lse, want[1]), "d_sess": err(d_sess, want[2]),
            "d_table": err(d_table, want[3])}
    assert all(v <= TOL for v in errs.values()), errs


def _lse(sess, table, t, cols, lq, precision="bf16x3"):
    from etpgt_b200 import ops

    return ops.PoolSoftmaxLoss.apply(sess, table, t, cols, lq, 0.5, None, 0, False, precision)


@pytest.mark.gpu
@pytest.mark.parametrize("m", [0, 4_096])
@pytest.mark.parametrize("batch", [127, 1_000])
def test_bf16_mode_matches_the_bf16_oracle(batch, m):
    from etpgt_b200.train.losses import InBatchSoftmaxLoss

    sess, table, t = _loss_inputs(batch, 256, seed=batch + m)
    loss_fn = InBatchSoftmaxLoss(num_sampled=m, temperature=0.5, seed=5, precision="bf16")
    freq, last = _state(ITEMS)
    pool, pool_lq = _pool(ITEMS, m, 0) if m else (None, None)
    cols, lq = _reference_columns(t, freq, last, 0, 0.01, pool, pool_lq)
    loss, d_sess, d_table = _loss_and_grads(loss_fn, sess, table, t)
    _, lse = _lse(sess, table, t, cols, lq, "bf16")
    want = _pool_oracle(sess, table, t, cols, lq, temperature=0.5)
    errs = {"loss": err(loss, want[0]), "lse": err(lse, want[1]), "d_sess": err(d_sess, want[3]),
            "d_table": err(d_table, want[4])}
    assert errs["loss"] <= TOL_VALUE and errs["lse"] <= TOL_VALUE, errs
    assert errs["d_sess"] <= TOL_GRAD and errs["d_table"] <= TOL_GRAD, errs


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
def test_bitwise_equal_to_pool_softmax_on_a_stably_sorted_concatenation(precision):
    from etpgt_b200 import ops
    from etpgt_b200.train.losses import InBatchSoftmaxLoss

    b, dim, m = 2_048, 128, 1_024
    sess, table, t = _loss_inputs(b, dim, seed=8)
    loss_fn = InBatchSoftmaxLoss(num_sampled=m, seed=5, freq_decay=0.2, precision=precision)
    got = _loss_and_grads(loss_fn, sess, table, t)
    pool, pool_lq = _pool(ITEMS, m, 0)
    freq = loss_fn.freq                                     # after the step's update
    in_lq = torch.where((t > 0) & (t < ITEMS), torch.log(b * freq[t.clamp(0, ITEMS - 1)]), float("inf")).float()
    cols, order = torch.sort(torch.cat([pool, t]), stable=True)
    lq = torch.cat([pool_lq, in_lq])[order]
    s = sess.clone().requires_grad_(True)
    e = torch.nn.Embedding.from_pretrained(table.clone(), freeze=False, padding_idx=0)
    want_loss = ops.pool_softmax_loss(s, e, t, cols, lq, precision=precision)
    want_loss.backward()
    for name, x, y in zip(("loss", "d_sess", "d_table"), got, (want_loss.detach(), s.grad, e.weight.grad)):
        assert torch.equal(x, y), name


# ------------------------------------------------------------------------------ properties


@pytest.mark.gpu
def test_all_targets_equal_leave_no_negative():
    from etpgt_b200.train.losses import InBatchSoftmaxLoss

    sess, table, _ = _loss_inputs(512, 128, seed=2)
    t = torch.full((512,), 42, dtype=torch.int64, device="cuda")
    loss, d_sess, d_table = _loss_and_grads(InBatchSoftmaxLoss(), sess, table, t)
    assert float(loss) == 0.0
    assert float(d_sess.abs().max()) == 0.0 and float(d_table.abs().max()) == 0.0


@pytest.mark.gpu
def test_padding_and_untouched_rows_keep_their_bits_in_the_optimizer_sink():
    from etpgt_b200 import optim
    from etpgt_b200.train.losses import InBatchSoftmaxLoss

    b, dim, m = 300, 128, 256
    sess, table, t = _loss_inputs(b, dim, seed=4)
    t[:7] = 0                                               # padding targets
    emb = torch.nn.Embedding.from_pretrained(table.clone(), freeze=False, padding_idx=0)
    opt = optim.AdamW(emb.parameters(), lr=1e-3, sink_bytes=table.numel() * 4)
    opt.zero_grad()
    sink = optim.grad_sink_for(emb.weight)
    base = torch.randn_like(table) * 1e-3
    sink.copy_(base)
    loss_fn = InBatchSoftmaxLoss(num_sampled=m, seed=5)
    loss_fn(sess, t, None, emb).backward()
    assert emb.weight.grad is sink
    pool, _ = _pool(ITEMS, m, 0)
    touched = torch.zeros(ITEMS, dtype=torch.bool, device="cuda")
    touched[pool] = True
    touched[t] = True
    touched[0] = False
    assert torch.equal(sink[~touched], base[~touched])
    ref_grad = _loss_and_grads(InBatchSoftmaxLoss(num_sampled=m, seed=5), sess, table, t)[2]
    assert err(sink - base, ref_grad) <= TOL


@pytest.mark.gpu
def test_estimate_converges_to_a_known_zipf_law():
    from etpgt_b200 import ops

    items, b, steps = 1_000, 4_096, 500
    w = np.zeros(items)
    w[1:] = 1.0 / np.arange(1, items) ** 1.1
    q = w / w.sum()
    rng = np.random.default_rng(0)
    freq, last = _state(items)
    for step in range(steps):
        t = torch.from_numpy(rng.choice(items, b, p=q)).cuda()
        ops.in_batch_columns(t, freq, last, step, 0.01, 0)
    f = freq.cpu().numpy() * (0.99 ** (steps - 1 - last.cpu().numpy()))      # brought up to date
    big = q > 1e-3
    rel = np.abs(f[big] - q[big]) / q[big]
    assert rel.max() <= 0.1, (rel.max(), int(big.sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("m", [0, 512])
def test_state_dict_round_trip_continues_bit_identically(m):
    from etpgt_b200.train.losses import InBatchSoftmaxLoss

    sess, table, _ = _loss_inputs(256, 64, seed=6)
    batches = [_targets(256, ITEMS, seed=100 + i) for i in range(5)]
    a = InBatchSoftmaxLoss(num_sampled=m, seed=9, freq_decay=0.3)
    for t in batches[:3]:
        _loss_and_grads(a, sess, table, t)
    state = {k: v.clone() for k, v in a.state_dict().items()}
    assert int(state["step"]) == 3 and state["freq"].numel() == ITEMS
    b = InBatchSoftmaxLoss(num_sampled=m, seed=9, freq_decay=0.3)
    b.load_state_dict(state)
    for t in batches[3:]:
        for x, y in zip(_loss_and_grads(a, sess, table, t), _loss_and_grads(b, sess, table, t)):
            assert torch.equal(x, y)
    for k, v in a.state_dict().items():
        assert torch.equal(v, b.state_dict()[k]), k


# ------------------------------------------------------------------------------ model and Trainer


@pytest.mark.gpu
def test_model_gradients_match_fp64_objective():
    from etpgt_b200.train.losses import create_loss_function

    temperature = 0.5
    model, batch, (d, _, _) = model_and_batch()
    model.train()
    t = batch.target_item
    loss_fn = create_loss_function("mixed_softmax", temperature=temperature, num_sampled=300, seed=1)
    freq, last = _state(d.num_items)
    pool, pool_lq = _pool(d.num_items, 300, 0, seed=1)
    f, l_ = freq.cpu().numpy(), last.cpu().numpy()
    ref.update(f, l_, t.cpu().numpy(), 0, 0.01, 0)
    cols, lq = (torch.from_numpy(x).cuda() for x in ref.columns(t.cpu().numpy(), f, 0, pool.cpu().numpy(),
                                                                 pool_lq.cpu().numpy()))
    for p in model.parameters():
        p.grad = None
    loss = loss_fn(model(batch), t, None, model.item_embedding)
    loss.backward()
    got, got_loss = grads(model), float(loss.detach())
    for p in model.parameters():
        p.grad = None
    sess = model(batch).double()
    e = model.item_embedding.weight.double()
    z_pos = (sess * e[t]).sum(1) / temperature
    z = sess @ e[cols].T / temperature - lq.double()[None, :]
    z = z.masked_fill((cols[None, :] == t[:, None]) | (cols == 0)[None, :], -float("inf"))
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
@pytest.mark.parametrize("kind", ["in_batch_softmax", "mixed_softmax"])
def test_trainer_learns_with_in_batch_negatives(kind, tmp_path):
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

    counts = torch.bincount(torch.as_tensor(d.sess_items), minlength=d.num_items)
    loss_fn = create_loss_function(kind, num_sampled=256, item_counts=counts, seed=3)
    trainer = Trainer(model, batches(0, 768, 0), batches(900, 1100, 100), optim.AdamW(model.parameters(), lr=3e-3),
                      device="cuda", output_dir=tmp_path, max_epochs=2, patience=5, k_values=[20], loss_fn=loss_fn)
    assert trainer._driver is None
    losses = trainer.train()["train_loss"]
    assert len(losses) == 2 and all(np.isfinite(losses)), losses
    assert losses[1] < losses[0], losses
    assert int(loss_fn.step) == 12 and loss_fn._step == 12


@pytest.mark.gpu
def test_host_errors():
    from etpgt_b200 import ops

    t = torch.tensor([1, 2], device="cuda")
    freq, last = _state(10)
    with pytest.raises(ValueError, match="decay"):
        ops.in_batch_columns(t, freq, last, 0, 0.0, 0)
    with pytest.raises(ValueError, match="step"):
        ops.in_batch_columns(t, freq, last, -1, 0.1, 0)
    with pytest.raises(ValueError, match="fp64"):
        ops.in_batch_columns(t, freq.float(), last, 0, 0.1, 0)
    with pytest.raises(ValueError, match="go together"):
        ops.in_batch_columns(t, freq, last, 0, 0.1, 0, pool_ids=t)
    with pytest.raises(ValueError, match="non-empty"):
        ops.in_batch_columns(t[:0], freq, last, 0, 0.1, 0)
