"""Generates tests/golden/*.npz by running the UNMODIFIED reference (/root/reference/etpgt)
on CPU, with `oracle/pyg_shim` standing in for the absent `torch_geometric`.

Run in the build container only (the GPU box has no /root/reference):
    python oracle/make_golden.py
The fixtures pin (a) the functional restatement in `oracle/model_ref.py` / `graph_ref.py`
against the reference's own classes and (b) the CUDA path against both.  Every case stores
inputs, the reference state_dict, fp32 outputs, and fp64 outputs + gradients (the model is
re-run with `.double()` for ground truth).
"""

from __future__ import annotations

import csv
import sys
import tempfile
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "oracle" / "pyg_shim"))
sys.path.insert(0, str(ROOT))
sys.path.insert(0, "/root/reference")

from torch_geometric.data import Batch, Data  # noqa: E402

sys.path.insert(0, str(ROOT / "tests"))
from golden_util import compact  # noqa: E402

from etpgt.model import (  # noqa: E402
    create_gat,
    create_graph_transformer,
    create_graph_transformer_optimized,
    create_graphsage,
)
from etpgt.model.base import SessionReadout  # noqa: E402
from etpgt.train.dataloader import SessionDataset, collate_fn  # noqa: E402
from etpgt.train.losses import create_loss_function  # noqa: E402
from etpgt.utils.metrics import compute_ndcg_at_k, compute_recall_at_k  # noqa: E402

OUT = ROOT / "tests" / "golden"


def npy(t):
    return t.detach().cpu().numpy()


def random_sessions_batch(rng, num_sessions, num_items, min_nodes=2, max_nodes=7, symmetric=True):
    """Block-diagonal batch of small session graphs with the shape statistics of
    docs/architecture/C4_CODE.md:46-67 (B=32 -> ~150 nodes, ~280 edges)."""
    graphs = []
    for _ in range(num_sessions):
        n = int(rng.integers(min_nodes, max_nodes + 1))
        ids = np.sort(rng.choice(np.arange(1, num_items), size=n, replace=False))
        pairs = [(a, b) for a in range(n) for b in range(a, n) if rng.random() < 0.45]
        src = [a for a, _ in pairs]
        dst = [b for _, b in pairs]
        if symmetric:
            src, dst = src + dst, dst + src
        ei = torch.tensor([src, dst], dtype=torch.long).reshape(2, -1)
        graphs.append(Data(x=torch.tensor(ids, dtype=torch.long), edge_index=ei))
    return Batch.from_data_list(graphs)


def run_model_case(name, factory, kwargs, batch, targets, negatives, loss_type, seed, pe=None, compact_pe_seed=None):
    """compact_pe_seed: `pe` is randn(num_items, k, seed compact_pe_seed).abs(); the fixture is written compact
    (tests/golden_util.py: the state as seeds + digest, large gradients sampled) to stay under 1 MB."""
    torch.manual_seed(seed)
    model = factory(**kwargs)
    if pe is not None:
        model.laplacian_pe._cached_pe = pe.clone()
    # make BN affine / running stats non-trivial so the fixture exercises them
    with torch.no_grad():
        for bn in model.batch_norms:
            bn.weight.uniform_(0.5, 1.5)
            bn.bias.uniform_(-0.2, 0.2)
            bn.running_mean.uniform_(-0.1, 0.1)
            bn.running_var.uniform_(0.5, 1.5)
    state0 = {k: v.clone() for k, v in model.state_dict().items()}
    out = {"cfg_" + k: np.asarray(v) for k, v in kwargs.items() if isinstance(v, (int, float, bool))}
    out.update({"x": npy(batch.x), "edge_index": npy(batch.edge_index), "batch": npy(batch.batch),
                "target": npy(targets), "negatives": npy(negatives)})
    for k, v in state0.items():
        out["state/" + k] = npy(v)
    loss_fn = create_loss_function(loss_type)

    for dtype, tag in ((torch.float32, "f32"), (torch.float64, "f64")):
        torch.set_default_dtype(dtype)  # base.py:140 allocates the readout in the default dtype
        model.load_state_dict(state0)
        model = model.to(dtype)
        if pe is not None:
            model.laplacian_pe._cached_pe = pe.clone().to(dtype)
        model.eval()
        with torch.no_grad():
            out[f"eval_out_{tag}"] = npy(model(batch))
        model.train()
        model.zero_grad()
        sess = model(batch)
        res = loss_fn(sess, targets, negatives, model.item_embedding)
        loss = res[0] if isinstance(res, tuple) else res
        loss.backward()
        out[f"train_out_{tag}"] = npy(sess)
        out[f"loss_{tag}"] = npy(loss)
        if tag == "f64":  # ground truth, stored rounded to fp32 to keep the fixtures small
            for pname, p in model.named_parameters():
                if p.grad is not None:
                    out["grad/" + pname] = npy(p.grad).astype(np.float32)
            for bname, b in model.named_buffers():
                if "running" in bname:
                    out["after/" + bname] = npy(b).astype(np.float32)
    torch.set_default_dtype(torch.float32)
    if compact_pe_seed is not None:
        out = compact(out, seed, compact_pe_seed)
    np.savez_compressed(OUT / f"{name}.npz", **out)
    print(f"wrote {name}.npz: N={batch.x.numel()} E={batch.edge_index.size(1)} loss={float(out['loss_f64']):.6f}")


def model_cases():
    rng = np.random.default_rng(20261018)
    # (1) the reference's own conftest fixture (tests/conftest.py:8-71)
    d1 = Data(x=torch.tensor([1, 2, 3]), edge_index=torch.tensor([[0, 1, 1, 2], [1, 0, 2, 1]]))
    d2 = Data(x=torch.tensor([4, 5, 6, 7]), edge_index=torch.tensor([[0, 1, 1, 2, 2, 3], [1, 0, 2, 1, 3, 2]]))
    dummy = Batch.from_data_list([d1, d2])
    tgt = torch.tensor([10, 20])
    neg = torch.tensor([[11, 12, 13, 14, 15], [21, 22, 23, 24, 25]])
    small = dict(num_items=100, embedding_dim=32, hidden_dim=32, num_layers=2, num_heads=2, dropout=0.0)
    pe_small = torch.randn(100, 16, generator=torch.Generator().manual_seed(7)).abs()
    run_model_case("gt_opt_dummy", create_graph_transformer_optimized, small, dummy, tgt, neg, "bpr", 1, pe_small)
    run_model_case("gt_opt_dummy_nope", create_graph_transformer_optimized,
                   {**small, "use_laplacian_pe": False}, dummy, tgt, neg, "listwise", 2)
    run_model_case("gt_ffn_dummy", create_graph_transformer, {**small, "use_laplacian_pe": False},
                   dummy, tgt, neg, "dual", 3)
    run_model_case("gat_dummy", create_gat, small, dummy, tgt, neg, "listwise", 4)
    sage_small = {k: v for k, v in small.items() if k != "num_heads"}
    run_model_case("sage_dummy", create_graphsage, sage_small, dummy, tgt, neg, "listwise", 5)

    # (2) C4 shape-trace batch: B=32, production widths (D=256, H=2, k_pe=16), small catalogue
    items = 400
    b32 = random_sessions_batch(rng, 32, items)
    tgt = torch.tensor(rng.integers(1, items, size=32))
    neg = torch.tensor(rng.integers(1, items, size=(32, 5)))
    prod = dict(num_items=items, embedding_dim=256, hidden_dim=256, num_layers=2, num_heads=2, dropout=0.0)
    pe = torch.randn(items, 16, generator=torch.Generator().manual_seed(7)).abs()
    run_model_case("gt_opt_b32", create_graph_transformer_optimized, prod, b32, tgt, neg, "bpr", 11, pe,
                   compact_pe_seed=7)
    mid_pe = dict(num_items=items, embedding_dim=64, hidden_dim=64, num_layers=2, num_heads=2, dropout=0.0)
    run_model_case("gt_opt_b32_dual", create_graph_transformer_optimized, mid_pe, b32, tgt, neg, "dual", 12, pe)

    # (3) directed low->high edges with self loops and edge-less sessions (train_baseline rule, N1)
    b_dir = random_sessions_batch(rng, 24, items, min_nodes=1, max_nodes=6, symmetric=False)
    tgt = torch.tensor(rng.integers(1, items, size=24))
    neg = torch.tensor(rng.integers(1, items, size=(24, 5)))
    mid = dict(num_items=items, embedding_dim=64, hidden_dim=64, num_layers=2, num_heads=2, dropout=0.0)
    run_model_case("gt_opt_directed", create_graph_transformer_optimized,
                   {**mid, "use_laplacian_pe": False}, b_dir, tgt, neg, "listwise", 13)
    run_model_case("gat_directed", create_gat, {**mid, "num_layers": 3, "num_heads": 4}, b_dir, tgt, neg, "bpr", 14)
    run_model_case("sage_directed", create_graphsage,
                   {k: v for k, v in {**mid, "num_layers": 3}.items() if k != "num_heads"},
                   b_dir, tgt, neg, "bpr", 15)
    for kind in ("max", "last", "attention"):
        run_model_case(f"gt_opt_readout_{kind}", create_graph_transformer_optimized,
                       {**mid, "use_laplacian_pe": False, "readout_type": kind}, b_dir, tgt, neg, "bpr", 16)


def loss_readout_metric_cases():
    torch.set_default_dtype(torch.float64)
    g = torch.Generator().manual_seed(99)
    sess = torch.randn(6, 32, generator=g, dtype=torch.float64)
    emb = torch.nn.Embedding(50, 32).double()
    tgt = torch.randint(1, 50, (6,), generator=g)
    neg = torch.randint(1, 50, (6, 5), generator=g)
    out = {"sess": npy(sess), "table": npy(emb.weight), "target": npy(tgt), "negatives": npy(neg)}
    for kind, kw in (("bpr", {}), ("listwise", {"temperature": 0.5}), ("dual", {"alpha": 0.7, "temperature": 2.0}),
                     ("sampled_softmax", {"temperature": 1.0})):
        s = sess.clone().requires_grad_(True)
        emb.zero_grad()
        res = create_loss_function(kind, **kw)(s, tgt, neg, emb)
        loss = res[0] if isinstance(res, tuple) else res
        loss.backward()
        out[f"{kind}/loss"], out[f"{kind}/dsess"], out[f"{kind}/dtable"] = npy(loss), npy(s.grad), npy(emb.weight.grad)
        if isinstance(res, tuple):
            out[f"{kind}/parts"] = np.asarray([res[1]["total"], res[1]["listwise"], res[1]["bpr"]])
    # readouts (etpgt/model/base.py:136-193)
    x = torch.randn(11, 32, generator=g, dtype=torch.float64)
    bvec = torch.tensor([0, 0, 0, 1, 2, 2, 2, 2, 3, 3, 3])
    out["ro/x"], out["ro/batch"] = npy(x), npy(bvec)
    for kind in ("mean", "max", "last", "attention"):
        ro = SessionReadout(32, kind).double()
        if kind == "attention":
            with torch.no_grad():
                ro.attention.bias.fill_(0.3)
            out["ro/att_w"], out["ro/att_b"] = npy(ro.attention.weight), npy(ro.attention.bias)
        out[f"ro/{kind}"] = npy(ro(x, bvec))
    # metrics known answers (tests/test_utils.py:62-93) + a random case
    preds = torch.tensor([[1, 2, 3, 4, 5], [6, 7, 8, 9, 10], [11, 12, 13, 14, 15]])
    tg = torch.tensor([1, 9, 99])
    out["met/preds"], out["met/targets"] = npy(preds), npy(tg)
    out["met/recall5"] = np.asarray(compute_recall_at_k(preds, tg, 5))
    out["met/recall2"] = np.asarray(compute_recall_at_k(preds, tg, 2))
    out["met/ndcg5"] = np.asarray(compute_ndcg_at_k(preds, tg, 5))
    torch.set_default_dtype(torch.float32)
    np.savez_compressed(OUT / "loss_readout_metrics.npz", **out)
    print("wrote loss_readout_metrics.npz")


def dataloader_case():
    """Drives the reference SessionDataset/collate_fn (etpgt/train/dataloader.py:12-202) over a
    small synthetic CSV pair so that the integer outputs of rows a1/a2 are pinned."""
    rng = np.random.default_rng(5)
    num_items, num_sessions = 60, 40
    sessions = []
    for s in range(num_sessions):
        length = int(rng.integers(3, 9)) if s != 7 else 58  # one session longer than max_session_length
        sessions.append(rng.integers(1, num_items, size=length))
    pairs = {}
    for items in sessions:  # window-5 co-occurrence, canonical i<=j (scripts/data/04_build_graph.py:57-71)
        for a in range(len(items)):
            for b in range(a + 1, min(a + 6, len(items))):
                i, j = sorted((int(items[a]), int(items[b])))
                pairs[(i, j)] = pairs.get((i, j), 0) + 1
    edges = sorted(pairs.items(), key=lambda kv: -kv[1])  # count-descending, like the stored CSV
    with tempfile.TemporaryDirectory() as tmp:
        sp, gp = Path(tmp) / "train.csv", Path(tmp) / "graph_edges.csv"
        with open(sp, "w", newline="") as f:
            w = csv.writer(f)
            w.writerow(["timestamp", "visitorid", "event", "itemid", "transactionid", "session_id"])
            for s, items in enumerate(sessions):
                for t, it in enumerate(items):
                    w.writerow([1000 * s + t, s, "view", int(it), "", s])
        with open(gp, "w", newline="") as f:
            w = csv.writer(f)
            w.writerow(["item_i", "item_j", "count", "last_ts", "event_pair_hist"])
            for (i, j), c in edges:
                w.writerow([i, j, c, 0, "{}"])
        ds = SessionDataset(sp, gp, num_negatives=5, max_session_length=50)
        torch.manual_seed(0)
        samples = [ds[i] for i in range(len(ds))]
        batch = collate_fn(samples)
    flat = np.concatenate(sessions)
    ptr = np.concatenate([[0], np.cumsum([len(s) for s in sessions])])
    np.savez_compressed(
        OUT / "dataloader.npz",
        item_i=np.asarray([e[0][0] for e in edges]), item_j=np.asarray([e[0][1] for e in edges]),
        sess_items=flat, sess_ptr=ptr, num_items=np.asarray(int(ds.num_items)),
        x=npy(batch.x), edge_index=npy(batch.edge_index), batch=npy(batch.batch),
        target=npy(batch.target_item), negatives=npy(batch.negative_items).reshape(len(samples), 5),
    )
    print(f"wrote dataloader.npz: N={batch.x.numel()} E={batch.edge_index.size(1)}")


def co_event_graph_case():
    """Runs the reference's own `build_co_event_graph` (scripts/data/04_build_graph.py:25-127, loaded by
    file path) on a small session frame with repeated items, equal items inside the window (self pairs),
    sessions shorter than the window and one long session; pins row f3."""
    import importlib.util

    import pandas as pd

    spec = importlib.util.spec_from_file_location("ref_build_graph", "/root/reference/scripts/data/04_build_graph.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    rng = np.random.default_rng(11)
    rows, ptr, items, stamps = [], [0], [], []
    for s in range(300):
        length = int(rng.integers(1, 12)) if s != 17 else 70
        its = rng.integers(1, 40, size=length)
        ts = np.sort(rng.integers(1_000, 2_000_000, size=length)) + s          # strictly per-session sorted
        ts = ts + np.arange(length)                                               # no equal timestamps
        for t, it in zip(ts, its):
            rows.append({"session_id": s, "timestamp": int(t), "itemid": int(it),
                         "event": ["view", "addtocart", "transaction"][int(rng.integers(0, 3))]})
        items += [int(i) for i in its]
        stamps += [int(t) for t in ts]
        ptr.append(len(items))
    df = pd.DataFrame(rows).sample(frac=1.0, random_state=3).reset_index(drop=True)   # shuffled rows
    edges_df, stats = mod.build_co_event_graph(df, window=5)
    np.savez_compressed(
        OUT / "co_event_graph.npz", sess_ptr=np.asarray(ptr), sess_items=np.asarray(items),
        timestamps=np.asarray(stamps), window=np.asarray(5),
        item_i=edges_df["item_i"].to_numpy(), item_j=edges_df["item_j"].to_numpy(),
        count=edges_df["count"].to_numpy(), last_ts=edges_df["last_ts"].to_numpy(),
        num_nodes=np.asarray(stats["num_nodes"]), num_edges=np.asarray(stats["num_edges"]))
    print(f"wrote co_event_graph.npz: {stats['num_edges']} edges, {stats['num_nodes']} nodes")


def trainer_case():
    """Drives the reference's own training loop — etpgt/train/trainer.py `Trainer.train()` (train_epoch, evaluate,
    checkpointing) with the reference model, `SessionDataset` + `collate_fn` batches and torch.optim.AdamW, as
    scripts/train/train_baseline.py:252-300 wires them — on CPU in fp32, for two loss settings.  The batches
    (negatives included) are materialised once and handed to the Trainer as lists, so that the B200 path can be fed
    the very same batches: the fixture pins epoch losses, Recall / NDCG per epoch and the final weights."""
    import logging

    from torch.utils.data import DataLoader

    from etpgt.train.trainer import Trainer

    logging.disable(logging.CRITICAL)
    rng = np.random.default_rng(21)
    num_items, n_train, n_val, dim, k_pe = 150, 96, 64, 32, 8
    sessions = [rng.integers(1, num_items, size=int(rng.integers(3, 10))) for _ in range(n_train + n_val)]
    pairs = {}
    for items in sessions[:n_train]:  # window-5 co-occurrence of the TRAIN sessions, canonical i<=j
        for a in range(len(items)):
            for b in range(a + 1, min(a + 6, len(items))):
                i, j = sorted((int(items[a]), int(items[b])))
                pairs[(i, j)] = pairs.get((i, j), 0) + 1
    edges = sorted(pairs.items(), key=lambda kv: -kv[1])

    def write_sessions(path, part, first_id):
        with open(path, "w", newline="") as f:
            w = csv.writer(f)
            w.writerow(["timestamp", "visitorid", "event", "itemid", "transactionid", "session_id"])
            for s, items in enumerate(part):
                for t, it in enumerate(items):
                    w.writerow([1000 * (first_id + s) + t, first_id + s, "view", int(it), "", first_id + s])

    out = {"cfg_num_items": np.asarray(num_items), "cfg_dim": np.asarray(dim), "cfg_k_pe": np.asarray(k_pe)}
    with tempfile.TemporaryDirectory() as tmp:
        tp, vp, gp = Path(tmp) / "train.csv", Path(tmp) / "val.csv", Path(tmp) / "graph_edges.csv"
        write_sessions(tp, sessions[:n_train], 0)
        write_sessions(vp, sessions[n_train:], n_train)
        with open(gp, "w", newline="") as f:
            w = csv.writer(f)
            w.writerow(["item_i", "item_j", "count", "last_ts", "event_pair_hist"])
            for (i, j), c in edges:
                w.writerow([i, j, c, 0, "{}"])
        torch.manual_seed(0)
        import random

        random.seed(0)
        np.random.seed(0)
        train_ds = SessionDataset(tp, gp, num_negatives=5, max_session_length=50)
        val_ds = SessionDataset(vp, gp, num_negatives=5, max_session_length=50)
        train_batches = list(DataLoader(train_ds, batch_size=32, shuffle=False, collate_fn=collate_fn))
        val_batches = list(DataLoader(val_ds, batch_size=32, shuffle=False, collate_fn=collate_fn))
        for split, batches in (("train", train_batches), ("val", val_batches)):
            out[f"n_{split}_batches"] = np.asarray(len(batches))
            for b, batch in enumerate(batches):
                out[f"{split}{b}/x"] = npy(batch.x)
                out[f"{split}{b}/edge_index"] = npy(batch.edge_index)
                out[f"{split}{b}/batch"] = npy(batch.batch)
                out[f"{split}{b}/target"] = npy(batch.target_item)
                out[f"{split}{b}/negatives"] = npy(batch.negative_items)      # flat [B * 5], as collate_fn leaves it
        pe = torch.randn(num_items, k_pe, generator=torch.Generator().manual_seed(7)).abs()
        out["pe"] = npy(pe)
        for tag, loss_type in (("bpr", None), ("dual", "dual")):
            torch.manual_seed(3)
            model = create_graph_transformer_optimized(num_items=num_items, embedding_dim=dim, hidden_dim=dim,
                                                       num_layers=2, num_heads=2, dropout=0.0, laplacian_k=k_pe)
            model.laplacian_pe._cached_pe = pe.clone()
            for k, v in model.state_dict().items():
                if "_cached_pe" not in k:
                    out[f"{tag}_init/{k}"] = npy(v).copy()      # a copy: the optimizer updates the parameters in place
            optimizer = torch.optim.AdamW(model.parameters(), lr=1e-3, weight_decay=1e-5)
            loss_fn = create_loss_function(loss_type) if loss_type else None
            trainer = Trainer(model, train_batches, val_batches, optimizer, device="cpu",
                              output_dir=Path(tmp) / f"out_{tag}", max_epochs=3, patience=5, k_values=[10, 20],
                              loss_fn=loss_fn)
            history = trainer.train()
            out[f"{tag}_train_loss"] = np.asarray(history["train_loss"], dtype=np.float64)
            for key in ("recall@10", "ndcg@10", "recall@20", "ndcg@20"):
                out[f"{tag}_{key}"] = np.asarray([m[key] for m in history["val_metrics"]], dtype=np.float64)
            out[f"{tag}_best_val_metric"] = np.asarray(trainer.best_val_metric)
            for k, v in model.state_dict().items():
                if "_cached_pe" not in k:
                    out[f"{tag}_final/{k}"] = npy(v)
            files = sorted(p.name for p in (Path(tmp) / f"out_{tag}").iterdir())
            out[f"{tag}_files"] = np.asarray(",".join(files))
            print(f"trainer[{tag}]: loss {history['train_loss']}, val {history['val_metrics'][-1]}, files {files}")
    logging.disable(logging.NOTSET)
    np.savez_compressed(OUT / "trainer_loop.npz", **out)
    print("wrote trainer_loop.npz")


def laplacian_pe_case():
    """Runs the reference's `compute_laplacian_pe` and `LaplacianPECached.precompute / forward / project`
    (etpgt/encodings/laplacian_pe.py:19-199) on (a) a directed edge list with item_i <= item_j — what
    scripts/train/train_baseline.py:234-243 passes — and (b) the same list symmetrised.  Pins the host path
    (`method="scipy"`) of etpgt_b200.encodings.laplacian_pe, which must reproduce what checkpoints store."""
    from etpgt.encodings.laplacian_pe import LaplacianPECached, compute_laplacian_pe

    rng = np.random.default_rng(13)
    n, k = 240, 8
    pairs = set()
    while len(pairs) < 900:
        a, b = (int(v) for v in rng.integers(1, n, size=2))
        pairs.add((min(a, b), max(a, b)))          # self pairs (a == b) are kept, as 04_build_graph.py keeps them
    directed = torch.tensor(sorted(pairs), dtype=torch.long).t().contiguous()
    symmetric = torch.cat([directed, directed.flip(0)], dim=1)
    out = {"num_nodes": np.asarray(n), "k": np.asarray(k), "directed": npy(directed), "symmetric": npy(symmetric)}
    for name, ei in (("directed", directed), ("symmetric", symmetric)):
        first = compute_laplacian_pe(ei, n, k=k)
        again = compute_laplacian_pe(ei, n, k=k)     # eigsh draws a new start vector on every call
        out[f"pe_{name}"] = npy(first)
        out[f"pe_{name}_again"] = npy(again)
        print(f"  {name}: two calls of the reference on the same input differ by {float((first - again).abs().max()):.3e}"
              f" (max entry {float(first.abs().max()):.3f})")

    class Graph:
        edge_index, num_nodes = directed, n

    torch.manual_seed(5)
    module = LaplacianPECached(k=k, embedding_dim=16)
    module.precompute(Graph)
    out["module_cached_pe"] = npy(module._cached_pe).copy()
    ids = torch.tensor([3, 7, 7, 100, 239])
    out["module_weight"] = npy(module.projection.weight).copy()
    out["module_bias"] = npy(module.projection.bias).copy()
    out["module_ids"] = npy(ids)
    out["module_forward"] = npy(module(ids))
    out["module_project"] = npy(module.project(module._cached_pe[ids]))
    np.savez_compressed(OUT / "laplacian_pe.npz", **out)
    print(f"wrote laplacian_pe.npz: directed {directed.size(1)} edges, pe max {float(out['pe_directed'].max()):.4f}")


if __name__ == "__main__":
    OUT.mkdir(parents=True, exist_ok=True)
    if "--only-laplacian" in sys.argv:
        laplacian_pe_case()
        raise SystemExit(0)
    if "--only-co-event" in sys.argv:
        co_event_graph_case()
        raise SystemExit(0)
    if "--only-trainer" in sys.argv:
        trainer_case()
        raise SystemExit(0)
    model_cases()
    loss_readout_metric_cases()
    dataloader_case()
    co_event_graph_case()
    trainer_case()
    laplacian_pe_case()
