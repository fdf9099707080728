"""CPU checks of the in-batch estimator's reference (tests/in_batch_ref.py): the lazy update equals the eager moving
average over every item for many random steps, and the reference's column order; plus what needs no GPU: the loss's
prior against the reference, and the argument checks in Python and through the C ABI."""

import numpy as np
import pytest
import torch

import in_batch_ref as ref


@pytest.mark.parametrize("with_counts", [False, True])
@pytest.mark.parametrize("decay", [0.01, 0.3, 1.0])
def test_lazy_update_equals_the_eager_moving_average(with_counts, decay):
    rng = np.random.default_rng(int(decay * 100) + with_counts)
    items, pad = 200, 0
    counts = rng.integers(0, 50, items).astype(np.float64) if with_counts else None
    freq = ref.prior(items, pad, counts)
    assert freq[pad] == 0.0 and abs(freq.sum() - 1.0) < 1e-12
    if counts is not None:
        assert (freq[counts == 0] == 0.0).all()
    last = np.full(items, -1, dtype=np.int64)
    eager = freq.copy()
    for step in range(300):
        if step % 50 in range(20, 40):              # a long gap for the rare items: only a few ids for 20 steps
            targets = rng.integers(1, 6, rng.integers(1, 9))
        else:
            b = int(rng.choice([1, 2, 7, 64, 257]))  # changing B
            targets = rng.zipf(1.3, b) % items      # duplicates, and padding (id 0) targets
        if step % 7 == 0:
            targets = np.concatenate([targets, [pad, pad]])
        ref.update(freq, last, targets, step, decay, pad)
        eager = ref.eager(eager, targets, decay, pad)
        seen = np.unique(targets)
        seen = seen[seen != pad]
        np.testing.assert_allclose(freq[seen], eager[seen], rtol=1e-12, atol=1e-300)
        assert (last[seen] == step).all()
    # every item, brought up to date
    gap = (1.0 - decay) ** (299 - last)
    np.testing.assert_allclose(freq * gap, eager, rtol=1e-12, atol=1e-300)
    assert freq[pad] == 0.0 and last[pad] == -1


def test_out_of_range_and_padding_targets_are_not_counted():
    freq = ref.prior(10, 0)
    last = np.full(10, -1, dtype=np.int64)
    before = freq.copy()
    ref.update(freq, last, [-3, 10, 0, 12], 0, 0.5, 0)
    assert (freq == before).all() and (last == -1).all()


def test_column_order_puts_the_pool_first_then_sessions_in_order():
    freq = ref.prior(20, 0)
    targets = np.array([7, 3, 7, 0, 3, 7])
    last = np.full(20, -1, dtype=np.int64)
    ref.update(freq, last, targets, 0, 0.1, 0)
    pool = np.array([3, 7, 7, 15])
    pool_lq = np.array([0.5, 1.5, 2.5, 3.5], dtype=np.float32)
    cols, lq = ref.columns(targets, freq, 0, pool, pool_lq)
    assert cols.tolist() == [0, 3, 3, 3, 7, 7, 7, 7, 7, 15]
    # id 0: session 3 (padding: +inf).  id 3: the pool, then sessions 1 and 4.  id 7: the pool twice, then 0, 2, 5
    assert lq[0] == np.inf
    assert lq[1] == np.float32(0.5) and lq[4] == np.float32(1.5) and lq[5] == np.float32(2.5)
    assert lq[2] == lq[3] == np.float32(np.log(6 * freq[3]))
    assert lq[6] == lq[7] == lq[8] == np.float32(np.log(6 * freq[7]))
    assert lq[9] == np.float32(3.5)
    cols, lq = ref.columns(targets, freq, 0)
    assert cols.tolist() == [0, 3, 3, 7, 7, 7]


def test_loss_arguments_are_checked_in_python():
    from etpgt_b200 import ops
    from etpgt_b200.train.losses import InBatchSoftmaxLoss, create_loss_function

    with pytest.raises(ValueError, match="num_sampled"):
        InBatchSoftmaxLoss(num_sampled=-1)
    for bad in (0.0, -0.1, 1.5, float("nan")):
        with pytest.raises(ValueError, match="freq_decay"):
            InBatchSoftmaxLoss(freq_decay=bad)
    with pytest.raises(ValueError, match="precision"):
        InBatchSoftmaxLoss(precision="fp16")
    with pytest.raises(ValueError, match="freq_decay"):
        create_loss_function("mixed_softmax", freq_decay=2.0)
    loss = create_loss_function("in_batch_softmax", num_sampled=4096, freq_decay=0.05)
    assert isinstance(loss, InBatchSoftmaxLoss) and loss.num_sampled == 0 and loss.freq_decay == 0.05
    mixed = create_loss_function("mixed_softmax", num_sampled=4096, precision="bf16")
    assert mixed.num_sampled == 4096 and mixed.precision == "bf16" and mixed.freq_decay == 0.01
    assert set(mixed.state_dict()) == {"freq", "last", "step"}
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.in_batch_columns(torch.tensor([1, 2]), torch.zeros(5, dtype=torch.float64),
                             torch.zeros(5, dtype=torch.int64), 0, 0.01, 0)


@pytest.mark.parametrize("with_counts", [False, True])
def test_loss_prior_matches_the_reference(with_counts):
    from etpgt_b200.train.losses import InBatchSoftmaxLoss

    counts = np.arange(30, dtype=np.float64) % 4 if with_counts else None
    loss = InBatchSoftmaxLoss(item_counts=None if counts is None else torch.from_numpy(counts))
    got = loss._prior(30, 0, "cpu").numpy()
    np.testing.assert_allclose(got, ref.prior(30, 0, counts), rtol=1e-15, atol=0)


def test_abi_argument_errors_name_the_argument():
    from etpgt_b200 import _lib

    p = 16                   # never dereferenced: every call below fails its checks before any launch
    good = dict(targets=p, batch=4, pool_ids=None, pool_log_q=None, num_pool=0, freq=p, last=p, num_items=10,
                padding_idx=0, step=0, decay=0.01, columns=p, log_q=p, ws=p, ws_bytes=1 << 20, stream=None)
    cases = [(dict(batch=0), "batch must be"), (dict(num_pool=-1), "num_pool must be"),
             (dict(num_items=0), "num_items must be"), (dict(padding_idx=10), "padding_idx"),
             (dict(decay=0.0), "decay must be"), (dict(decay=1.5), "decay must be"),
             (dict(decay=float("nan")), "decay must be"), (dict(step=-1), "step must be"),
             (dict(freq=None), "targets, freq, last, columns and log_q are required"), (dict(columns=None), "targets, freq, last, columns and log_q are required"),
             (dict(num_pool=8), "pool_ids and pool_log_q are required")]
    for change, msg in cases:
        args = {**good, **change}
        with pytest.raises(RuntimeError, match=rf"\(-1\): in_batch_columns: {msg}"):
            _lib.call("etpgt_in_batch_columns", *args.values())
