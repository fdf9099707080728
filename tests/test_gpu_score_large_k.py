"""GPU tests of top-k for 33 <= k <= 256 on the tcgen05 bf16 scorer (piece dump tracking the M-th largest score of a
piece, the one-CTA-per-row select, the exact CUDA-core fallback), the merges at k = 256, and the layers above them
(predict, sharded_predict, Trainer.evaluate).
Oracle: oracle/model_ref.predict(bf16_inputs=True) / topk_lower_id, and tests/exclude_ref.py for exclusion lists."""

import numpy as np
import pytest
import torch

from exclude_ref import NO_ID, hit_positions, predict_excluding
from oracle import model_ref

pytestmark = pytest.mark.gpu


def _exact_inputs(batch, items, dim, seed):
    """Small integers: exact in bf16 and in fp32 accumulation, with heavy ties (lower id wins)."""
    g = torch.Generator().manual_seed(seed)
    sess = torch.randint(-2, 3, (batch, dim), generator=g).float()
    table = torch.randint(-1, 2, (items, dim), generator=g).float()
    return sess, table


def _oracle(sess, table, k, exclude=None):
    return predict_excluding(sess, table, k, exclude, bf16_inputs=True)


# (k, dim, batch, items): every k class (33-64, 65-128, 129-256), every dim, batches across the 64-row and 256-row
# boundaries, item counts below, at and above k, and tables long enough for split ranges
CASES = [
    (33, 64, 63, 5000), (64, 128, 64, 3000), (65, 192, 257, 4096), (100, 256, 1000, 9001),
    (128, 64, 257, 128), (129, 128, 1, 20000), (200, 256, 63, 200), (200, 64, 257, 4999), (256, 64, 1000, 256),
    (256, 192, 300, 40000), (256, 256, 1000, 82174), (100, 64, 20000, 3000), (33, 256, 257, 33),
]


@pytest.mark.parametrize("k,dim,batch,items", CASES)
def test_exact_inputs_bit_for_bit(k, dim, batch, items):
    from etpgt_b200 import ops

    sess, table = _exact_inputs(batch, items, dim, seed=k + dim + items)
    want_v, want_i = model_ref.predict(sess, table, k, bf16_inputs=True)
    got_v, got_i = ops.score_topk(sess.cuda(), table.cuda(), k, precision="bf16")
    assert torch.equal(got_i.cpu(), want_i)
    assert torch.equal(got_v.cpu().double(), want_v)


@pytest.mark.parametrize("k", [33, 100, 256])
def test_random_inputs_within_ties(k):
    """Normal inputs against fp64 scores of the bf16-rounded operands: the values agree to fp32 rounding, and a
    position may hold another id only where the oracle's neighbouring scores are numerically tied."""
    from etpgt_b200 import ops

    g = torch.Generator().manual_seed(k)
    sess, table = torch.randn(700, 256, generator=g), torch.randn(30000, 256, generator=g)
    want_v, want_i = model_ref.predict(sess, table, k, bf16_inputs=True)
    got_v, got_i = ops.score_topk(sess.cuda(), table.cuda(), k, precision="bf16")
    got_v, got_i = got_v.cpu().double(), got_i.cpu()
    assert torch.allclose(got_v, want_v, rtol=0, atol=1e-3 * want_v.abs().max().item())
    differ = got_i != want_i
    tol = 2e-4 * want_v.abs().max().item()
    s_b = sess.to(torch.bfloat16).double()
    t_b = table.to(torch.bfloat16).double()
    exact = (s_b.unsqueeze(1) * t_b[got_i]).sum(-1)   # fp64 score of every returned id
    assert ((exact - want_v).abs()[differ] <= tol).all()
    assert (torch.sort(got_i, dim=1).values[:, 1:] != torch.sort(got_i, dim=1).values[:, :-1]).all()


@pytest.mark.parametrize("excl", [False, True])
@pytest.mark.parametrize("k", [33, 64, 65, 128, 129, 256])
def test_fallback_gives_the_same_bits(monkeypatch, k, excl):
    """ETPGT_SCORE_CAP = 1 overflows every row's slot buffer: every row takes the exact CUDA-core fallback."""
    from etpgt_b200 import ops

    sess, table = _exact_inputs(300, 7001, 128, seed=k)
    exclude = None
    if excl:
        exclude = torch.randint(-1, 7001, (300, 40), generator=torch.Generator().manual_seed(k))
        exclude[:, 0] = 0
    want_v, want_i = _oracle(sess, table, k, exclude)
    ex = exclude.cuda() if excl else None
    plain = ops.score_topk(sess.cuda(), table.cuda(), k, precision="bf16", exclude=ex)
    monkeypatch.setenv("ETPGT_SCORE_CAP", "1")
    forced = ops.score_topk(sess.cuda(), table.cuda(), k, precision="bf16", exclude=ex)
    for got_v, got_i in (plain, forced):
        assert torch.equal(got_i.cpu(), want_i)
        assert torch.equal(got_v.cpu().double(), want_v)


@pytest.mark.parametrize("cap", [None, "1"])
@pytest.mark.parametrize("k", [40, 100, 256])
def test_exclusion_and_sentinels(monkeypatch, cap, k):
    """Rows whose eligible items are fewer than k end in (-inf, INT64_MAX); an excluded target has hit_pos -1."""
    from etpgt_b200 import ops

    if cap is not None:
        monkeypatch.setenv("ETPGT_SCORE_CAP", cap)
    items = 300
    sess, table = _exact_inputs(200, items, 64, seed=k + 1)
    g = torch.Generator().manual_seed(k)
    exclude = torch.full((200, 290), -1, dtype=torch.int64)
    for r in range(200):
        n = [0, 10, items - k + 5, 290, 50][r % 5]
        exclude[r, :n] = torch.randperm(items, generator=g)[:n]
    _, plain = _oracle(sess, table, k)
    targets = plain[:, 3].clone()
    targets[::4] = exclude[::4, 0].clamp(min=0)
    want_v, want_i = _oracle(sess, table, k, exclude)
    got_v, got_i, hit = ops.score_topk(sess.cuda(), table.cuda(), k, precision="bf16", exclude=exclude.cuda(),
                                       targets=targets.cuda())
    assert torch.equal(got_i.cpu(), want_i)
    assert torch.equal(got_v.cpu().double(), want_v)   # sentinel slots included: -inf
    assert (want_i == NO_ID).any() and torch.isneginf(got_v[got_i == NO_ID]).all()
    assert torch.equal(hit.cpu(), hit_positions(want_i, targets, k))
    listed = (got_i.cpu().unsqueeze(2) == exclude.unsqueeze(1)).any(dim=2)
    assert not listed.any()


@pytest.mark.parametrize("cap", [None, "1"])
def test_target_positions(monkeypatch, cap):
    from etpgt_b200 import ops

    if cap is not None:
        monkeypatch.setenv("ETPGT_SCORE_CAP", cap)
    k, batch = 256, 350
    sess, table = _exact_inputs(batch, 12000, 256, seed=5)
    _, want_i = _oracle(sess, table, k)
    ranks = torch.tensor([0, 31, 32, 63, 64, 200, 255])
    targets = want_i[torch.arange(batch), ranks[torch.arange(batch) % 7]].clone()
    targets[::11] = 12005   # not an item: a miss
    _, got_i, hit = ops.score_topk(sess.cuda(), table.cuda(), k, precision="bf16", targets=targets.cuda())
    assert torch.equal(got_i.cpu(), want_i)
    want_pos = hit_positions(want_i, targets, k)
    assert torch.equal(hit.cpu(), want_pos)
    assert set(want_pos.tolist()) >= {-1, 0, 31, 32, 63, 64, 200, 255}


@pytest.mark.parametrize("shards", [2, 3, 8])
def test_item_shards_merge(shards):
    """Shards scored with id_base and merged with topk_merge_parts at k = 256 equal one unsharded call bit for bit
    (8 shards of 1,500 items: a shard smaller than k pads with sentinels, as sharded_predict does)."""
    from etpgt_b200 import ops

    items = 1500 if shards == 8 else 9000
    batch, k = 300, 256
    sess, table = _exact_inputs(batch, items, 64, seed=shards)
    sess, table = sess.cuda(), table.cuda()
    want_v, want_i = ops.score_topk(sess, table, k, precision="bf16")
    bounds = np.linspace(0, items, shards + 1).astype(int)
    val_bytes = (batch * k * 4 + 255) // 256 * 256
    stride = val_bytes + batch * k * 8
    parts = torch.empty(shards * stride, dtype=torch.uint8, device="cuda")
    for p in range(shards):
        lo, hi = int(bounds[p]), int(bounds[p + 1])
        block = parts[p * stride:(p + 1) * stride]
        val = block[:batch * k * 4].view(torch.float32).view(batch, k)
        idx = block[val_bytes:].view(torch.int64).view(batch, k)
        kk = min(k, hi - lo)
        val.fill_(float("-inf"))
        idx.fill_(NO_ID)
        v, i = ops.score_topk(sess, table[lo:hi], kk, id_base=lo, precision="bf16")
        val[:, :kk], idx[:, :kk] = v, i
    got_v, got_i, _ = ops.topk_merge_parts(parts, shards, stride, val_bytes, batch, k, 0, batch)
    assert torch.equal(got_i, want_i)
    assert torch.equal(got_v, want_v)
    cand_v = torch.stack([parts[p * stride:p * stride + batch * k * 4].view(torch.float32).view(batch, k)
                          for p in range(shards)], 1).reshape(batch, shards * k)
    cand_i = torch.stack([parts[p * stride + val_bytes:(p + 1) * stride].view(torch.int64).view(batch, k)
                          for p in range(shards)], 1).reshape(batch, shards * k)
    m_v, m_i = ops.topk_merge(cand_v, cand_i, k)
    assert torch.equal(m_i, want_i) and torch.equal(m_v, want_v)


@pytest.mark.parametrize("k,parts", [(65, 3), (100, 8), (256, 8), (256, 64)])
def test_merges_of_unsorted_candidates(k, parts):
    """topk_merge and topk_merge_parts at k > 64 on unsorted candidates with heavy score ties, exact duplicates and
    sentinels: the distinct (score, id) pairs by (score desc, id asc), padded with (-inf, INT64_MAX) — what the
    selection passes of the k <= 64 kernels give."""
    from etpgt_b200 import ops

    g = torch.Generator().manual_seed(k + parts)
    batch = 70
    val = torch.randint(-3, 4, (batch, parts * k), generator=g).float()
    idx = torch.randint(0, 5 * k, (batch, parts * k), generator=g)
    val[:, 1::7], idx[:, 1::7] = val[:, ::7][:, :val[:, 1::7].size(1)], idx[:, ::7][:, :idx[:, 1::7].size(1)]
    val[::3, k // 2:], idx[::3, k // 2:] = float("-inf"), NO_ID   # rows with fewer than k real candidates
    # the ::3 rows keep only k // 2 candidates: with duplicates they have fewer than k distinct ones
    want_v = torch.full((batch, k), float("-inf"))
    want_i = torch.full((batch, k), NO_ID)
    for r in range(batch):
        pairs = sorted(set(zip(val[r].tolist(), idx[r].tolist())), key=lambda p: (-p[0], p[1]))[:k]
        want_v[r, :len(pairs)] = torch.tensor([p[0] for p in pairs])
        want_i[r, :len(pairs)] = torch.tensor([p[1] for p in pairs])
    got_v, got_i = ops.topk_merge(val.cuda(), idx.cuda(), k)
    assert torch.equal(got_i.cpu(), want_i) and torch.equal(got_v.cpu(), want_v)
    val_bytes = (batch * k * 4 + 255) // 256 * 256
    stride = val_bytes + batch * k * 8
    buf = torch.empty(parts * stride, dtype=torch.uint8, device="cuda")
    for p in range(parts):
        buf[p * stride:p * stride + batch * k * 4].view(torch.float32).view(batch, k).copy_(val[:, p * k:(p + 1) * k])
        buf[p * stride + val_bytes:(p + 1) * stride].view(torch.int64).view(batch, k).copy_(idx[:, p * k:(p + 1) * k])
    targets = want_i[:, 5].clone()
    targets[::4] = 10 * k   # a miss
    got_v, got_i, hit = ops.topk_merge_parts(buf, parts, stride, val_bytes, batch, k, 0, batch, targets.cuda())
    assert torch.equal(got_i.cpu(), want_i) and torch.equal(got_v.cpu(), want_v)
    assert torch.equal(hit.cpu(), hit_positions(want_i, targets, k))


class _TableModel(torch.nn.Module):
    def __init__(self, table):
        super().__init__()
        self.table = table
        self.score_precision = "auto"

    def get_item_embeddings(self):
        return self.table


@pytest.mark.parametrize("k", [100, 256])
def test_predict_and_sharded_predict(k):
    """model.predict and parallel.sharded_predict (the Trainer's evaluation path) at k > 64 pick the tensor cores at
    every batch size, and give the oracle's ranking."""
    from etpgt_b200 import parallel
    from etpgt_b200.model.base import BaseRecommendationModel

    sess, table = _exact_inputs(90, 5000, 64, seed=k)
    model = _TableModel(table.cuda())
    for b in (1, 90):
        _, want_i = _oracle(sess[:b], table, k)
        got = BaseRecommendationModel.predict(model, sess[:b].cuda(), k)
        assert torch.equal(got.cpu(), want_i)
        targets = want_i[:, 7].clone()
        got2, hit = parallel.sharded_predict(model, sess[:b].cuda(), k=k, group=False, targets=targets.cuda())
        assert torch.equal(got2.cpu(), want_i)
        assert (hit.cpu() == 7).all()
    exclude = torch.randint(0, 5000, (90, 30), generator=torch.Generator().manual_seed(1))
    _, want_i = _oracle(sess, table, k, exclude)
    got = BaseRecommendationModel.predict(model, sess.cuda(), k, exclude_items=exclude.cuda())
    assert torch.equal(got.cpu(), want_i)


def test_explicit_precisions():
    from etpgt_b200 import ops

    sess, table = _exact_inputs(10, 3000, 64, seed=3)
    _, want_i = _oracle(sess, table, 50)
    got = ops.score_topk(sess.cuda(), table.cuda(), 50, precision="bf16")[1]   # 33 <= k <= 64 on the tensor cores
    assert torch.equal(got.cpu(), want_i)
    with pytest.raises(RuntimeError, match=r'64.*precision="bf16".*256'):
        ops.score_topk(sess.cuda(), table.cuda(), 65, precision="fp32")
    with pytest.raises(RuntimeError, match="256"):
        ops.score_topk(sess.cuda(), table.cuda(), 257, precision="bf16")


def test_evaluation_size():
    """23,861 x 82,174 x 256 at k = 256 (the oracle on the device in fp64, in row chunks)."""
    from etpgt_b200 import ops

    sess, table = _exact_inputs(23861, 82174, 256, seed=23)
    s_d, t_d = sess.cuda(), table.cuda()
    got_v, got_i = ops.score_topk(s_d, t_d, 256, precision="bf16")
    t64 = t_d.double()
    for r0 in range(0, sess.size(0), 2048):
        want_v, want_i = model_ref.topk_lower_id(s_d[r0:r0 + 2048].double() @ t64.t(), 256)
        assert torch.equal(got_i[r0:r0 + 2048], want_i)
        assert torch.equal(got_v[r0:r0 + 2048].double(), want_v)


def _synth_model_and_batches(sizes):
    from etpgt_b200 import data, synth
    from etpgt_b200.model import create_graph_transformer_optimized

    d = synth.generate(num_sessions=1200, graph_sessions=900, num_items=3000, clusters=16, seed=5)
    graph, store = data.ItemGraph(d.item_i, d.item_j, d.num_items), data.SessionStore(d.sess_ptr, d.sess_items)
    torch.manual_seed(1)
    model = create_graph_transformer_optimized(d.num_items, 64, 64, num_layers=2, num_heads=2, dropout=0.0,
                                               use_laplacian_pe=False).cuda().eval()
    batches, first = [], 900
    for n in sizes:
        batches.append(data.build_batch(graph, store, np.arange(first, first + n)))
        first += n
    return model, batches


def _near_tie_equal(got, sess, table, want_v, want_i):
    """Ids equal to the oracle's, or holding a score within fp32 rounding of the oracle's score at that position."""
    s_b, t_b = sess.to(torch.bfloat16).double(), table.to(torch.bfloat16).double()
    exact = (s_b @ t_b.t()).gather(1, got.clamp(0, table.size(0) - 1))
    return bool(((got == want_i) | ((exact - want_v).abs() < 1e-4)).all())


@pytest.mark.parametrize("k", [100, 256])
def test_recommend(k):
    """recommend(batch, k) = predict(forward, k, exclude_items=seen_items) on the tensor cores at every batch size,
    against the filtered oracle on the bf16-rounded operands."""
    from etpgt_b200 import ops

    model, batches = _synth_model_and_batches([100, 40])
    table = model.get_item_embeddings().detach().cpu()
    for batch in batches:
        batch = batch.to("cuda")
        with torch.no_grad():
            sess = model(batch)
        got = model.recommend(batch, k)
        seen = ops.seen_items(batch, num_sessions=sess.size(0))
        assert torch.equal(got, model.predict(sess, k, exclude_items=seen, exclude_sorted=True))
        want_v, want_i = predict_excluding(sess.cpu(), table, k, seen.cpu(), bf16_inputs=True)
        assert _near_tie_equal(got.cpu(), sess.cpu(), table, want_v, want_i)
        assert not (got.cpu().unsqueeze(2) == seen.cpu().unsqueeze(1)).any()
        assert torch.equal(model.recommend(batch, k, exclude_seen=False), model.predict(sess, k))


def test_trainer_evaluate_deep_k(tmp_path):
    """Trainer(k_values=[20, 100, 256]).evaluate() against the oracle's Recall / NDCG; its @20 metrics equal those of
    a k_values=[20] run bit for bit, also with a last batch of fewer than 64 sessions (where k = 20 is ranked by the
    fp32 scorer and k = 256 by the tensor cores)."""
    from etpgt_b200 import optim
    from etpgt_b200.train.trainer import Trainer

    model, val = _synth_model_and_batches([100, 100, 40])
    opt = optim.AdamW(model.parameters(), lr=1e-3)

    def metrics(ks, **kw):
        return Trainer(model, [], val, opt, output_dir=tmp_path, k_values=ks, **kw).evaluate()

    for kw in ({}, {"exclude_seen": True}):
        deep, shallow = metrics([20, 100, 256], **kw), metrics([20], **kw)
        assert deep["recall@20"] == shallow["recall@20"] and deep["ndcg@20"] == shallow["ndcg@20"]
        sums = {k: [0.0, 0.0] for k in (100, 256)}
        n = 0
        table = model.get_item_embeddings().detach().cpu()
        with torch.no_grad():
            for batch in val:
                batch = batch.to("cuda")
                sess = model(batch).cpu()
                seen = None
                if kw:
                    from etpgt_b200 import ops
                    seen = ops.seen_items(batch, num_sessions=sess.size(0)).cpu()
                _, ids = predict_excluding(sess, table, 256, seen, bf16_inputs=True)
                t = batch.target_item.cpu()
                for k in (100, 256):
                    sums[k][0] += model_ref.recall_at_k(ids, t, k) * len(t)
                    sums[k][1] += model_ref.ndcg_at_k(ids, t, k) * len(t)
                n += len(t)
        for k in (100, 256):   # a near-tie may move one target across the cut: within one session's worth
            assert abs(deep[f"recall@{k}"] - sums[k][0] / n) <= 1.5 / n
            assert abs(deep[f"ndcg@{k}"] - sums[k][1] / n) <= 1.5 / n
