"""GPU tests of the filtered scorers: ops.score_topk(exclude=...) on the tcgen05 bf16 scorer (piece-dump epilogue,
select kernel, CUDA-core fallback) and on the fp32 CUDA-core scorer, item shards, target positions, and the layers
above them (predict / recommend, sharded_predict, Trainer(exclude_seen=True)).
Oracle: tests/exclude_ref.py (the oracle's ranking with the listed ids at -inf; sentinels past the eligible items)."""

import os
import socket
from pathlib import Path

import numpy as np
import pytest
import torch

from exclude_ref import NO_ID, hit_positions, predict_excluding
from golden_util import Golden, rel_err

pytestmark = pytest.mark.gpu


def _exact_inputs(batch, items, dim, seed):
    """Small integers: exact in bf16 and in fp32 accumulation, with many ties (lower id wins)."""
    g = torch.Generator().manual_seed(seed)
    sess = torch.randint(-2, 3, (batch, dim), generator=g).float()
    table = torch.randint(-1, 2, (items, dim), generator=g).float()
    table[0] = 0
    return sess, table


def _exclusion_rows(sess, table, seed, width=48):
    """Unsorted rows of every kind: part of the row's own unfiltered top-20, its whole top-40, duplicates with -1
    padding and out-of-range ids, empty rows, ids in the table's last partial tile plus id 0, random ids."""
    b, items = sess.size(0), table.size(0)
    g = torch.Generator().manual_seed(seed)
    _, top40 = predict_excluding(sess, table, min(40, items), None, bf16_inputs=True)
    rows = torch.full((b, width), -1, dtype=torch.int64)
    for r in range(b):
        kind = r % 6
        if kind == 0:
            pick = torch.randperm(20, generator=g)[:5]
            rows[r, :5] = top40[r, pick]
        elif kind == 1:
            rows[r, :top40.size(1)] = top40[r]
        elif kind == 2:
            rows[r, :6] = top40[r, 0]
            rows[r, 6:9] = torch.tensor([items, items + 3, -7])
            rows[r, 9] = top40[r, 3]
        elif kind == 4:
            last = torch.arange(max(items - 9, 1), items)
            rows[r, :last.numel()] = last
            rows[r, last.numel()] = 0
        elif kind == 5:
            rows[r, :20] = torch.randint(0, items, (20,), generator=g)
        rows[r] = rows[r, torch.randperm(width, generator=g)]
    return rows


# (dim, batch, items, k): full-catalogue units (>= 74 CTA pairs of 256 rows), tail splits (items >= 128 tiles),
# small tables and the largest k
CASES = [(64, 19000, 3000, 20), (256, 300, 40000, 20), (256, 260, 7001, 32), (64, 200, 7001, 1), (64, 5, 300, 10)]


@pytest.mark.parametrize("cap", [None, "2"])
@pytest.mark.parametrize("dim,batch,items,k", CASES)
def test_bf16_exclusion_exact(monkeypatch, cap, dim, batch, items, k):
    """Bit for bit against the oracle; cap = 2 sends every row through the CUDA-core fallback kernel."""
    import etpgt_b200.ops as ops

    sess, table = _exact_inputs(batch, items, dim, seed=items + dim + k)
    exclude = _exclusion_rows(sess, table, seed=k)
    want_v, want_i = predict_excluding(sess, table, k, exclude, bf16_inputs=True)
    if cap is not None:
        monkeypatch.setenv("ETPGT_SCORE_CAP", cap)
    got_v, got_i = ops.score_topk(sess.cuda(), table.cuda(), k, precision="bf16", exclude=exclude.cuda())
    assert torch.equal(got_i.cpu(), want_i)
    assert torch.equal(got_v.cpu().double(), want_v)
    presorted = torch.sort(exclude, dim=1).values.cuda()
    again = ops.score_topk(sess.cuda(), table.cuda(), k, precision="bf16", exclude=presorted, exclude_sorted=True)[1]
    assert torch.equal(again.cpu(), want_i)
    listed = (got_i.cpu().unsqueeze(2) == exclude.unsqueeze(1)).any(dim=2)
    assert not listed.any()


@pytest.mark.parametrize("k", [1, 20, 40])
def test_fp32_exclusion_exact(k):
    import etpgt_b200.ops as ops

    sess, table = _exact_inputs(150, 5000, 128, seed=k)
    exclude = _exclusion_rows(sess, table, seed=k + 1)
    exclude[7, :45] = torch.arange(5000 - 45, 5000)
    want_v, want_i = predict_excluding(sess, table, k, exclude)
    got_v, got_i = ops.score_topk(sess.cuda(), table.cuda(), k, precision="fp32", exclude=exclude.cuda())
    assert torch.equal(got_i.cpu(), want_i)
    assert torch.equal(got_v.cpu().double(), want_v)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("shards", [2, 3, 8])
def test_item_shards_with_global_lists(precision, shards):
    """Scoring table[lo:hi] with id_base = lo and the unchanged global lists, then the exact merge of the shards'
    candidates, equals the single filtered pass bit for bit (8 shards of 150 items: fewer eligible items than k in
    a shard, whose missing slots are sentinels)."""
    import etpgt_b200.ops as ops

    items = 150 if shards == 8 else 6000
    batch, k = 300, 20
    sess, table = _exact_inputs(batch, items, 64, seed=shards)
    exclude = _exclusion_rows(sess, table, seed=shards).cuda()
    sess, table = sess.cuda(), table.cuda()
    want_v, want_i = ops.score_topk(sess, table, k, precision=precision, exclude=exclude)
    bounds = np.linspace(0, items, shards + 1).astype(int)
    val_bytes = (batch * k * 4 + 255) // 256 * 256
    stride = val_bytes + batch * k * 8
    parts = torch.empty(shards * stride, dtype=torch.uint8, device="cuda")
    for p in range(shards):
        lo, hi = int(bounds[p]), int(bounds[p + 1])
        block = parts[p * stride:(p + 1) * stride]
        val = block[:batch * k * 4].view(torch.float32).view(batch, k)
        idx = block[val_bytes:].view(torch.int64).view(batch, k)
        ops.score_topk(sess, table[lo:hi], k, id_base=lo, precision=precision, out=(val, idx), exclude=exclude)
    got_v, got_i, _ = ops.topk_merge_parts(parts, shards, stride, val_bytes, batch, k, 0, batch)
    assert torch.equal(got_i, want_i)
    assert torch.equal(got_v, want_v)


@pytest.mark.parametrize("cap", [None, "2"])
def test_target_positions_with_exclusion(monkeypatch, cap):
    """hit_pos: -1 for an excluded target; the others at their position in the filtered list."""
    import etpgt_b200.ops as ops

    if cap is not None:
        monkeypatch.setenv("ETPGT_SCORE_CAP", cap)
    batch, items, dim, k = 300, 4000, 256, 20
    sess, table = _exact_inputs(batch, items, dim, seed=9)
    exclude = _exclusion_rows(sess, table, seed=9)
    _, plain = predict_excluding(sess, table, k, None, bf16_inputs=True)
    targets = plain[torch.arange(batch), torch.arange(batch) % k].clone()   # in the unfiltered list
    targets[torch.arange(batch) % 5 == 0] = items + 5                       # a miss
    excluded_target = torch.arange(batch) % 7 == 0
    exclude[excluded_target, 0] = targets[excluded_target]
    _, want_i = predict_excluding(sess, table, k, exclude, bf16_inputs=True)
    want_pos = hit_positions(want_i, targets, k)
    assert (want_pos[excluded_target] == -1).all()
    _, idx, hit = ops.score_topk(sess.cuda(), table.cuda(), k, precision="bf16", targets=targets.cuda(),
                                 exclude=exclude.cuda())
    assert torch.equal(idx.cpu(), want_i)
    assert torch.equal(hit.cpu(), want_pos)
    # fp32 scorer: positions from its id matrix
    _, idx32, hit32 = ops.score_topk(sess.cuda(), table.cuda(), k, precision="fp32", targets=targets.cuda(),
                                     exclude=exclude.cuda())
    assert torch.equal(idx32.cpu(), want_i) and torch.equal(hit32.cpu(), want_pos)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_no_exclusion_changes_nothing(precision):
    """exclude=None, an all-padding list and a width-0 list give the unfiltered results bit for bit; a table of 300
    items with 295 excluded returns the 5 others and 5 sentinels."""
    import etpgt_b200.ops as ops

    g = torch.Generator().manual_seed(1)
    sess, table = torch.randn(300, 256, generator=g).cuda(), torch.randn(7001, 256, generator=g).cuda()
    ref_v, ref_i = ops.score_topk(sess, table, 20, precision=precision)
    for exclude in (None, torch.full((300, 17), -1, dtype=torch.int64), torch.empty(300, 0, dtype=torch.int64),
                    torch.full((300, 5), 7001, dtype=torch.int64)):
        v, i = ops.score_topk(sess, table, 20, precision=precision,
                              exclude=None if exclude is None else exclude.cuda())
        assert torch.equal(i, ref_i) and torch.equal(v, ref_v)
    small = table[:300]
    keep = torch.tensor([3, 77, 150, 298, 299])
    mask = torch.ones(300, dtype=torch.bool)
    mask[keep] = False
    exclude = torch.arange(300)[mask].repeat(300, 1).cuda()
    v, i = ops.score_topk(sess, small, 10, precision=precision, exclude=exclude)
    assert set(i[:, :5].flatten().tolist()) <= set(keep.tolist())
    assert torch.equal(torch.sort(i[:, :5], dim=1).values.cpu(), keep.repeat(300, 1))
    assert (i[:, 5:] == NO_ID).all() and torch.isinf(v[:, 5:]).all() and (v[:, 5:] < 0).all()
    want_v, want_i = predict_excluding(sess.cpu(), small.cpu(), 10, exclude.cpu(), bf16_inputs=precision == "bf16")
    assert torch.equal(i.cpu(), want_i)


def test_exclusion_argument_checks():
    import etpgt_b200.ops as ops

    sess, table = torch.randn(300, 64).cuda(), torch.randn(1000, 64).cuda()
    ex = torch.zeros(300, 1, dtype=torch.int64).cuda()
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.score_topk(sess, table, 10, precision="bf16", exclude=ex.cpu())
    with pytest.raises(RuntimeError, match="int64"):
        ops.score_topk(sess, table, 10, precision="bf16", exclude=ex.int())
    with pytest.raises(RuntimeError, match="B=300"):
        ops.score_topk(sess, table, 10, precision="bf16", exclude=ex[:5])


# ------------------------------------------------------------------------------ model level


class _GoldenBatch:
    def __init__(self, g):
        self.x = g.tensor("x").cuda()
        self.edge_index = g.tensor("edge_index").cuda()
        self.batch = g.tensor("batch").cuda()
        self.num_graphs = int(self.batch.max().item()) + 1


def test_predict_and_recommend_on_a_golden_model():
    """predict(exclude_items=seen_items(batch)) and recommend(batch) on the gt_opt_b32 fixture against the reference's
    eval forward plus the filtered ranking."""
    import etpgt_b200.ops as ops
    from etpgt_b200.model import create_graph_transformer_optimized

    g = Golden("gt_opt_b32")
    model = create_graph_transformer_optimized(**g.cfg())
    state = g.group("state")
    pe = state.pop("laplacian_pe._cached_pe", None)
    model.load_state_dict(state, strict=False)
    model = model.cuda().eval()
    if pe is not None:
        model.laplacian_pe._cached_pe = pe.cuda()
    batch = _GoldenBatch(g)
    with torch.no_grad():
        sess = model(batch)
    want_sess = torch.as_tensor(g.raw["eval_out_f64"])
    assert rel_err(sess, want_sess) < 1e-4
    seen = ops.seen_items(batch)
    x, bvec = batch.x.cpu(), batch.batch.cpu()
    for b in range(sess.size(0)):
        assert set(seen[b].tolist()) - {-1} == set(x[bvec == b].tolist()) | {0}
    table = model.get_item_embeddings().detach()
    k = 20
    top = model.predict(sess, k, exclude_items=seen)
    assert torch.equal(model.recommend(batch, k), top)
    assert torch.equal(model.predict(sess, k), model.recommend(batch, k, exclude_seen=False))
    want_v, want_i = predict_excluding(want_sess, table.cpu().double(), k, seen.cpu())
    exact = want_sess @ table.cpu().double().t()
    same = top.cpu() == want_i
    near_tie = (want_v - torch.gather(exact, 1, top.cpu().clamp(0, table.size(0) - 1))).abs() < 1e-3
    assert bool((same | near_tie).all()) and same.float().mean() > 0.99
    assert not (top.cpu().unsqueeze(2) == seen.cpu().unsqueeze(1)).any()


def _val_batches(d, graph, store, first, count, size):
    from etpgt_b200 import data

    return [data.build_batch(graph, store, np.arange(first + i * size, first + (i + 1) * size)) for i in range(count)]


def test_trainer_evaluate_exclude_seen(tmp_path):
    """Trainer(exclude_seen=True).evaluate() = the filtered oracle's Recall / NDCG@10/20 on the same batches;
    exclude_seen=False is today's evaluate bit for bit."""
    from etpgt_b200 import data, optim, synth
    from etpgt_b200.model import create_graph_transformer_optimized
    from etpgt_b200.train.trainer import Trainer
    from oracle import model_ref

    d = synth.generate(num_sessions=1200, graph_sessions=900, num_items=3000, clusters=16, seed=5)
    graph, store = data.ItemGraph(d.item_i, d.item_j, d.num_items), data.SessionStore(d.sess_ptr, d.sess_items)
    torch.manual_seed(1)
    model = create_graph_transformer_optimized(d.num_items, 64, 64, num_layers=2, num_heads=2, dropout=0.0,
                                               use_laplacian_pe=False).cuda()
    val = _val_batches(d, graph, store, 900, 3, 100)       # bf16 scorer (>= 64 sessions)
    val += _val_batches(d, graph, store, 1200 - 40, 1, 40)   # fp32 scorer
    opt = optim.AdamW(model.parameters(), lr=1e-3)

    def metrics(**kw):
        return Trainer(model, [], val, opt, output_dir=tmp_path, k_values=[10, 20], **kw).evaluate()

    plain = metrics()
    assert metrics(exclude_seen=False) == plain
    filtered = metrics(exclude_seen=True)
    assert set(filtered) == set(plain)
    hits = {k: [0.0, 0.0] for k in (10, 20)}
    n = 0
    model.eval()
    with torch.no_grad():
        for batch in val:
            sess = model(batch)
            seen = torch.stack(_seen_rows(batch))
            _, ids = predict_excluding(sess.cpu(), model.get_item_embeddings().cpu(), 20, seen,
                                       bf16_inputs=sess.size(0) >= 64)
            t = batch.target_item.cpu()
            for k in (10, 20):
                hits[k][0] += model_ref.recall_at_k(ids, t, k) * len(t)
                hits[k][1] += model_ref.ndcg_at_k(ids, t, k) * len(t)
            n += len(t)
    for k in (10, 20):   # a near-tie may move one target across the cut: within one session's worth
        assert abs(filtered[f"recall@{k}"] - hits[k][0] / n) <= 1.5 / n
        assert abs(filtered[f"ndcg@{k}"] - hits[k][1] / n) <= 1.5 / n


def _seen_rows(batch, width=None):
    """Host-built exclusion rows (the session's items plus 0, -1 padding) — independent of ops.seen_items."""
    x, ptr = batch.x.cpu(), batch.ptr.cpu().long()
    rows = [torch.cat([torch.zeros(1, dtype=torch.int64), x[ptr[b]:ptr[b + 1]]]) for b in range(len(ptr) - 1)]
    width = width or max(len(r) for r in rows)
    return [torch.cat([r, torch.full((width - len(r),), -1, dtype=torch.int64)]) for r in rows]


# ------------------------------------------------------------------------------ two GPUs


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _two_gpu_worker(rank, world, port, out):
    import faulthandler

    import torch.distributed as dist

    faulthandler.dump_traceback_later(300, exit=True)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from etpgt_b200 import ops, parallel

        class Model:
            def __init__(self, table):
                self.table = table

            def get_item_embeddings(self):
                return self.table

        g = torch.Generator().manual_seed(3)
        counts = (140, 160)
        sess_all = torch.randint(-2, 3, (sum(counts), 64), generator=g).float()
        table = torch.randint(-1, 2, (5001, 64), generator=g).float().cuda()
        exclude_all = torch.randint(-1, 5001, (sum(counts), 30), generator=g)
        lo = sum(counts[:rank])
        sess = sess_all[lo:lo + counts[rank]].cuda()
        ok, notes = True, []
        for precision in ("fp32", "bf16"):
            for known_counts, width in ((True, 30), (False, 12 + 9 * rank)):   # equal widths / widths exchanged
                exclude = exclude_all[lo:lo + counts[rank], :width].cuda()
                want = ops.score_topk(sess, table, 20, precision=precision, exclude=exclude)[1]
                got = parallel.sharded_predict(Model(table), sess, k=20, precision=precision, exclude=exclude,
                                               counts=counts if known_counts else None)
                same = bool(torch.equal(got, want))
                ok = ok and same
                notes.append(f"{precision} counts={known_counts}: {same}")
        out[rank] = (ok, notes)
    finally:
        faulthandler.cancel_dump_traceback_later()
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_two_gpus_sharded_predict_with_exclusion():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp

    manager = mp.get_context("spawn").Manager()
    out = manager.dict()
    mp.spawn(_two_gpu_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    for rank in (0, 1):
        ok, notes = out[rank]
        assert ok, (rank, notes)
