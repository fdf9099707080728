"""CPU tests of the exclusion reference (tests/exclude_ref.py) and of ops.seen_items, which is index plumbing and runs
on any device."""

import types

import pytest
import torch

from exclude_ref import NO_ID, predict_excluding


def _brute(scores, k, exclude):
    """Per row: drop the listed ids, sort the rest by (score desc, id asc), pad with sentinels."""
    vals, ids = [], []
    for b in range(scores.size(0)):
        banned = {int(e) for e in exclude[b]}
        cand = [(-float(scores[b, i]), i) for i in range(scores.size(1)) if i not in banned]
        cand.sort()
        cand = cand[:k] + [(float("inf"), NO_ID)] * max(0, k - len(cand))
        vals.append([-c[0] for c in cand])
        ids.append([c[1] for c in cand])
    return torch.tensor(vals, dtype=torch.float64), torch.tensor(ids, dtype=torch.int64)


@pytest.mark.parametrize("tied", [False, True])
def test_predict_excluding_matches_brute_force(tied):
    g = torch.Generator().manual_seed(5 + tied)
    b, n, d, k = 12, 40, 8, 10
    if tied:
        sess = torch.randint(-1, 2, (b, d), generator=g).double()
        table = torch.randint(-1, 2, (n, d), generator=g).double()
    else:
        sess, table = torch.randn(b, d, generator=g).double(), torch.randn(n, d, generator=g).double()
    width = 36
    exclude = torch.randint(-3, n + 5, (b, width), generator=g)     # padding and out-of-range ids too
    exclude[0] = -1                                                  # nothing excluded
    exclude[1, :35] = torch.arange(35)                               # 5 eligible items, k = 10
    exclude[2, :] = 7                                                # duplicates
    exclude[3, :width] = torch.arange(n - width, n)                  # the top of the id range
    want_v, want_i = _brute(sess @ table.t(), k, exclude)
    got_v, got_i = predict_excluding(sess, table, k, exclude)
    assert torch.equal(got_i, want_i)
    assert torch.equal(got_v, want_v)
    assert (got_i[1, 5:] == NO_ID).all() and torch.isinf(got_v[1, 5:]).all()
    # no exclusion: the oracle's own ranking
    from oracle import model_ref

    plain_v, plain_i = model_ref.predict(sess, table, k)
    none_v, none_i = predict_excluding(sess, table, k, None)
    assert torch.equal(none_i, plain_i) and torch.equal(none_v, plain_v)


def test_predict_excluding_shard_offsets():
    """A shard [lo, hi) with id_base = lo and the global list ranks its own ids exactly like the full table does."""
    g = torch.Generator().manual_seed(2)
    sess, table = torch.randn(6, 4, generator=g).double(), torch.randn(30, 4, generator=g).double()
    exclude = torch.randint(0, 30, (6, 9), generator=g)
    _, full_i = predict_excluding(sess, table, 30, exclude)
    lo, hi = 10, 22
    _, shard_i = predict_excluding(sess, table[lo:hi], 30, exclude, id_base=lo)
    for b in range(6):
        want = [int(i) for i in full_i[b] if lo <= int(i) < hi]
        got = [int(i) for i in shard_i[b] if int(i) != NO_ID]
        assert got == want


def test_seen_items_layout():
    import etpgt_b200.ops as ops

    x = torch.tensor([5, 3, 9, 4, 4, 8, 1, 2])
    bvec = torch.tensor([0, 0, 0, 1, 1, 2, 3, 3])
    ptr = torch.tensor([0, 3, 5, 6, 8], dtype=torch.int32)
    batch = types.SimpleNamespace(x=x, batch=bvec, ptr=ptr, num_graphs=4)
    want = torch.tensor([[0, 3, 5, 9], [-1, 0, 4, 4], [-1, -1, 0, 8], [-1, 0, 1, 2]])
    assert torch.equal(ops.seen_items(batch), want)
    assert torch.equal(ops.seen_items(batch, width=4), want)
    wide = ops.seen_items(batch, width=6)
    assert wide.shape == (4, 6) and torch.equal(wide[:, 2:], want)
    no_pad = ops.seen_items(batch, exclude_padding=False)
    assert torch.equal(no_pad, torch.tensor([[3, 5, 9], [-1, 4, 4], [-1, -1, 8], [-1, 1, 2]]))
    # without ptr: grouped by batch.batch; an empty session is all padding
    batch2 = types.SimpleNamespace(x=x, batch=bvec + (bvec >= 2).long(), num_graphs=5)
    got = ops.seen_items(batch2)
    assert torch.equal(got[2], torch.tensor([-1, -1, -1, 0]))
    assert torch.equal(got[[0, 1, 3, 4]], want)
