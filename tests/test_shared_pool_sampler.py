"""The shared-pool sampler without a GPU: the proposal table of ops.item_sampling_table, the CPU restatement of
etpgt_sample_item_pool (tests/shared_pool_ref.py) against the proposal it draws from, and the boundary of the new
loss (C ABI declarations, create_loss_function)."""

import numpy as np
import pytest
import torch
from scipy import stats

from shared_pool_ref import sample_item_pool


def _table(counts=None, num_items=None, power=0.75, padding_idx=0):
    from etpgt_b200 import ops

    return ops.item_sampling_table(counts, power, padding_idx, num_items=num_items, device="cpu").numpy()


def _zipf_counts(num_items, a=1.5, seed=0):
    rng = np.random.default_rng(seed)
    c = np.bincount(rng.zipf(a, 200_000) % num_items, minlength=num_items).astype(np.int64)
    return torch.from_numpy(c)


def test_item_sampling_table_uniform_and_popularity():
    cum = _table(num_items=10)
    w = np.diff(cum)
    assert cum[0] == 0 and w[0] == 0 and (w[1:] == w[1]).all() and w[1] > 0
    assert 2 ** 60 <= cum[-1] < 2 ** 62
    counts = torch.tensor([7, 0, 1, 16, 81, 0])
    cum = _table(counts, power=0.75)
    w = np.diff(cum)
    assert w[0] == 0 and w[1] == 0 and w[5] == 0          # padding and zero counts are never drawn
    np.testing.assert_allclose(w[2:5] / w[2], [1.0, 8.0, 27.0], rtol=1e-12)
    assert cum[-1] < 2 ** 62
    with pytest.raises(ValueError, match="num_items"):
        _table()
    with pytest.raises(ValueError, match="positive weight"):
        _table(torch.tensor([5, 0, 0]))


def test_restatement_never_draws_padding_or_zero_weight():
    counts = _zipf_counts(300)
    counts[::7] = 0
    cum = _table(counts)
    w = np.diff(cum)
    for step in range(4):
        ids, log_q = sample_item_pool(cum, 2_000, seed=11, step=step)
        assert (np.diff(ids) >= 0).all()
        assert (w[ids] > 0).all() and not (ids == 0).any()
        np.testing.assert_allclose(log_q, np.log(2_000 * w[ids].astype(np.float64) / float(cum[-1])), rtol=1e-6)


@pytest.mark.parametrize("kind", ["uniform", "zipf"])
def test_restatement_draws_follow_the_proposal(kind):
    num_items = 200
    cum = _table(num_items=num_items) if kind == "uniform" else _table(_zipf_counts(num_items))
    w = np.diff(cum).astype(np.float64)
    draws = np.concatenate([sample_item_pool(cum, 50_000, seed=3, step=s)[0] for s in range(4)])
    observed = np.bincount(draws, minlength=num_items)
    expected = draws.size * w / w.sum()
    keep = expected > 0
    assert observed[~keep].sum() == 0
    # pool sparse cells so that every expected count is >= 5
    order = np.argsort(expected[keep])
    obs, exp = observed[keep][order], expected[keep][order]
    small = np.cumsum(exp) < 50
    obs = np.concatenate([[obs[small].sum()], obs[~small]]) if small.any() else obs
    exp = np.concatenate([[exp[small].sum()], exp[~small]]) if small.any() else exp
    _, p = stats.chisquare(obs, exp)
    assert p > 1e-4, p


def test_pool_depends_on_seed_and_step_only():
    cum = _table(num_items=1000)
    a = sample_item_pool(cum, 64, seed=5, step=9)[0]
    assert (a == sample_item_pool(cum, 64, seed=5, step=9)[0]).all()
    assert not (a == sample_item_pool(cum, 64, seed=5, step=10)[0]).all()
    assert not (a == sample_item_pool(cum, 64, seed=6, step=9)[0]).all()


def test_library_exports_and_header_declares_the_entry_points():
    from pathlib import Path

    from etpgt_b200 import _lib

    names = ("etpgt_sample_item_pool_workspace_bytes", "etpgt_sample_item_pool", "etpgt_pool_softmax_workspace_bytes",
             "etpgt_pool_softmax_fwd", "etpgt_pool_softmax_bwd")
    header = (Path(__file__).resolve().parents[1] / "include" / "etpgt_b200.h").read_text()
    for name in names:
        assert f"{name}(" in header
        assert name in _lib.exported_symbols()


def test_create_loss_function_shared_pool_softmax():
    from etpgt_b200.train.losses import ListwiseLoss, SharedPoolSoftmaxLoss, create_loss_function

    counts = torch.arange(10)
    loss = create_loss_function("shared_pool_softmax", temperature=0.2, num_sampled=64, item_counts=counts,
                                sampling_power=0.5, seed=4)
    assert isinstance(loss, SharedPoolSoftmaxLoss) and not isinstance(loss, ListwiseLoss)
    assert (loss.num_sampled, loss.temperature, loss.sampling_power, loss.seed) == (64, 0.2, 0.5, 4)
    assert loss.item_counts is counts
    default = create_loss_function("shared_pool_softmax")
    assert (default.num_sampled, default.item_counts, default.sampling_power, default.seed) == (8192, None, 0.75, 0)
    # the other types ignore the new keywords
    assert create_loss_function("full_softmax", num_sampled=3).temperature == 1.0
    with pytest.raises(ValueError, match="num_sampled"):
        SharedPoolSoftmaxLoss(num_sampled=0)


def test_cpu_tensors_are_rejected():
    from etpgt_b200 import ops

    with pytest.raises(RuntimeError, match="CUDA"):
        ops.pool_softmax_loss(torch.randn(4, 64), torch.randn(10, 64), torch.tensor([1, 2, 3, 4]),
                              torch.tensor([1, 2]), torch.zeros(2))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.sample_item_pool(torch.tensor([0, 1, 2]), 4, 0, 0)
