"""Cost of the shared-pool sampled softmax (ops.pool_softmax_loss: csrc/softmax_tc.cu with POOL) next to the
full-catalogue loss at the same B x I, in the same process; with --quality, what the objectives give on synth data.

    python tools/bench_shared_pool_softmax.py [--reps 5] [--calls 5] [--shapes 1024x8192x82174,...] [--quality]
                                              [--precision bf16x3|bf16|both]

D = 256.  Forward + backward are timed through the C ABI with CUDA events around `calls` back-to-back pairs, median
over `reps` windows after a warm-up.  The backward adds into a d_table of the whole catalogue, as training does.
The pool is drawn once per shape by etpgt_sample_item_pool (popularity^0.75 of zipf counts); its own time is listed
apart.  Rates: executed MMA flops 15 * 2 * B * C * D (C = M for the pool, I for the full loss: three split-bf16 MMAs
for the forward logits, the two recomputed logits and the two gradient products) over the time.  Prints one JSON line.
--quality trains a 2-layer GraphTransformer (D = 64) for a few epochs on synth data with bpr, full_softmax and the
shared pool (uniform and popularity proposals) and reports Recall@20 / NDCG@20 on held-out sessions.

--precision bf16 or both (default bf16x3: the output above) times each precision on the same inputs, alternating window
by window: the pool's FWD, DS (the backward with d_sess only), DE (d_table only) and forward + backward, and the full
loss's forward + backward.  Executed MMA flops are 15 * 2 * B * C * D for bf16x3 and 5 * 2 * B * C * D for bf16.
With --quality, full_softmax and both shared-pool arms are trained in each precision from the same seeds.
"""

from __future__ import annotations

import argparse
import json
import sys
import tempfile
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "gat-recommendation_b200"))

from bench_full_softmax import MMAS_PER_PRODUCT, PRECISIONS, gpu_info, timed, timed_alternating  # noqa: E402

DIM = 256


def bench_shape(b: int, m: int, items: int, reps: int, calls: int) -> dict:
    from etpgt_b200 import _lib, ops
    from etpgt_b200._lib import ptr

    g = torch.Generator(device="cuda").manual_seed(b + m + items)
    sess = torch.randn(b, DIM, device="cuda", generator=g) * 0.3
    table = torch.randn(items, DIM, device="cuda", generator=g) * 0.3
    targets = torch.randint(1, items, (b,), device="cuda", generator=g)
    rng = np.random.default_rng(items)
    counts = torch.from_numpy(np.bincount(rng.zipf(1.5, 4 * items) % items, minlength=items) + 1)
    cum = ops.item_sampling_table(counts, 0.75, 0, device="cuda")
    pool, log_q = ops.sample_item_pool(cum, m, seed=1, step=0)
    sample_ms = timed(lambda: ops.sample_item_pool(cum, m, seed=1, step=0), reps, calls)
    lse = torch.empty(b, device="cuda")
    z_pos = torch.empty(b, device="cuda")
    loss = torch.empty(1, device="cuda")
    d_loss = torch.ones(1, device="cuda")
    d_sess = torch.empty_like(sess)
    d_table = torch.zeros_like(table)
    st = _lib.stream()
    ws = _lib.workspace(max(_lib.size("etpgt_pool_softmax_workspace_bytes", b, m, DIM),
                            _lib.size("etpgt_full_softmax_workspace_bytes", b, items, DIM)), "cuda")

    def pool_step():
        _lib.call("etpgt_pool_softmax_fwd", ptr(sess), ptr(table), ptr(targets), ptr(pool), ptr(log_q), b, items, m,
                  DIM, 1.0, 0.0, 0, ptr(lse), ptr(z_pos), ptr(loss), ptr(ws), ws.numel(), st)
        _lib.call("etpgt_pool_softmax_bwd", ptr(sess), ptr(table), ptr(targets), ptr(pool), ptr(log_q), ptr(lse),
                  ptr(z_pos), ptr(d_loss), b, items, m, DIM, 1.0, 0.0, 0, ptr(d_sess), ptr(d_table), ptr(ws),
                  ws.numel(), st)

    def full_step():
        _lib.call("etpgt_full_softmax_fwd", ptr(sess), ptr(table), ptr(targets), b, items, DIM, 1.0, 0.0, 0,
                  ptr(lse), ptr(loss), ptr(ws), ws.numel(), st)
        _lib.call("etpgt_full_softmax_bwd", ptr(sess), ptr(table), ptr(targets), ptr(lse), ptr(d_loss), b, items, DIM,
                  1.0, 0.0, 0, ptr(d_sess), ptr(d_table), ptr(ws), ws.numel(), st)

    pool_ms = timed(pool_step, reps, calls)
    full_ms = timed(full_step, reps, calls)
    pool_flops, full_flops = 15 * 2 * b * m * DIM, 15 * 2 * b * items * DIM
    out = {
        "batch": b, "num_sampled": m, "items": items, "dim": DIM,
        "pool_fwd_bwd_ms": round(pool_ms, 3), "sample_pool_ms": round(sample_ms, 3),
        "pool_executed_tflops": round(pool_flops / pool_ms / 1e9, 1),
        "full_fwd_bwd_ms": round(full_ms, 3),
        "full_executed_tflops": round(full_flops / full_ms / 1e9, 1),
        "full_ms_scaled_by_m_over_i": round(full_ms * m / items, 3),
        "pool_over_scaled_full": round(pool_ms / (full_ms * m / items), 2),
    }
    del ws, d_table
    torch.cuda.empty_cache()
    return out


def bench_precisions(b: int, m: int, items: int, reps: int, calls: int, precisions: list[str]) -> dict:
    """The pool's FWD, DS, DE and forward + backward and the full loss's forward + backward of each precision on the
    same inputs, alternating."""
    from etpgt_b200 import _lib, ops
    from etpgt_b200._lib import ptr

    g = torch.Generator(device="cuda").manual_seed(b + m + items)
    sess = torch.randn(b, DIM, device="cuda", generator=g) * 0.3
    table = torch.randn(items, DIM, device="cuda", generator=g) * 0.3
    targets = torch.randint(1, items, (b,), device="cuda", generator=g)
    rng = np.random.default_rng(items)
    counts = torch.from_numpy(np.bincount(rng.zipf(1.5, 4 * items) % items, minlength=items) + 1)
    cum = ops.item_sampling_table(counts, 0.75, 0, device="cuda")
    pool, log_q = ops.sample_item_pool(cum, m, seed=1, step=0)
    lse = torch.empty(b, device="cuda")
    z_pos = torch.empty(b, device="cuda")
    loss = torch.empty(1, device="cuda")
    d_loss = torch.ones(1, device="cuda")
    d_sess = torch.empty_like(sess)
    d_table = torch.zeros_like(table)
    st = _lib.stream()
    ws = _lib.workspace(max(_lib.size("etpgt_pool_softmax_workspace_bytes", b, m, DIM),
                            _lib.size("etpgt_full_softmax_workspace_bytes", b, items, DIM)), "cuda")

    def pool_fwd(p):
        _lib.call("etpgt_pool_softmax_fwd_ex", ptr(sess), ptr(table), ptr(targets), ptr(pool), ptr(log_q), b, items,
                  m, DIM, 1.0, 0.0, 0, ptr(lse), ptr(z_pos), ptr(loss), ptr(ws), ws.numel(), st, PRECISIONS[p])

    def pool_bwd(p, ds, dt):
        _lib.call("etpgt_pool_softmax_bwd_ex", ptr(sess), ptr(table), ptr(targets), ptr(pool), ptr(log_q), ptr(lse),
                  ptr(z_pos), ptr(d_loss), b, items, m, DIM, 1.0, 0.0, 0, ptr(ds), ptr(dt), ptr(ws), ws.numel(), st,
                  PRECISIONS[p])

    def full_step(p):
        _lib.call("etpgt_full_softmax_fwd_ex", ptr(sess), ptr(table), ptr(targets), b, items, DIM, 1.0, 0.0, 0,
                  ptr(lse), ptr(loss), ptr(ws), ws.numel(), st, PRECISIONS[p])
        _lib.call("etpgt_full_softmax_bwd_ex", ptr(sess), ptr(table), ptr(targets), ptr(lse), ptr(d_loss), b, items,
                  DIM, 1.0, 0.0, 0, ptr(d_sess), ptr(d_table), ptr(ws), ws.numel(), st, PRECISIONS[p])

    fns = {}
    for p in precisions:
        fns[(p, "fwd")] = lambda p=p: pool_fwd(p)
        fns[(p, "ds")] = lambda p=p: (pool_fwd(p), pool_bwd(p, d_sess, None))
        fns[(p, "de")] = lambda p=p: (pool_fwd(p), pool_bwd(p, None, d_table))
        fns[(p, "pair")] = lambda p=p: (pool_fwd(p), pool_bwd(p, d_sess, d_table))
        fns[(p, "full")] = lambda p=p: full_step(p)
    t = timed_alternating(fns, reps, calls)
    out = {"batch": b, "num_sampled": m, "items": items, "dim": DIM, "modes": {}}
    for p in precisions:
        k = 5 * MMAS_PER_PRODUCT[p]
        fwd = t[(p, "fwd")]
        out["modes"][p] = {
            "pool_fwd_ms": round(fwd, 3),
            "pool_ds_ms": round(t[(p, "ds")] - fwd, 3), "pool_de_ms": round(t[(p, "de")] - fwd, 3),
            "pool_fwd_bwd_ms": round(t[(p, "pair")], 3),
            "executed_flops": f"{k}*2*B*C*D",
            "pool_executed_tflops": round(k * 2 * b * m * DIM / t[(p, "pair")] / 1e9, 1),
            "full_fwd_bwd_ms": round(t[(p, "full")], 3),
            "full_executed_tflops": round(k * 2 * b * items * DIM / t[(p, "full")] / 1e9, 1),
        }
    if len(precisions) == 2:
        out["bf16x3_over_bf16_pool"] = round(t[("bf16x3", "pair")] / t[("bf16", "pair")], 2)
        out["bf16x3_over_bf16_full"] = round(t[("bf16x3", "full")] / t[("bf16", "full")], 2)
    del ws, d_table
    torch.cuda.empty_cache()
    return out


def quality(epochs: int, precisions: list[str] = ("bf16x3",)) -> list[dict]:
    from etpgt_b200 import data, optim, synth
    from etpgt_b200.model import create_graph_transformer_optimized
    from etpgt_b200.train.losses import create_loss_function
    from etpgt_b200.train.trainer import Trainer

    d = synth.generate(num_sessions=24_000, graph_sessions=18_000, num_items=5_000, clusters=64, seed=7)
    graph = data.ItemGraph(d.item_i, d.item_j, d.num_items)
    store = data.SessionStore(d.sess_ptr, d.sess_items)
    counts = torch.bincount(store.items, minlength=d.num_items)

    def batches(lo, hi, step0):
        out = []
        for i, s in enumerate(range(lo, hi, 512)):
            ids = np.arange(s, min(hi, s + 512))
            bt = data.build_batch(graph, store, ids, 50, False, False)
            bt.negative_items = data.sample_negatives(store, ids, d.num_items, 5, seed=3, step=step0 + i).view(-1)
            out.append(bt)
        return out

    train, val = batches(0, 18_000, 0), batches(18_000, 24_000, 10_000)
    arms = [("bpr", dict()), ("full_softmax", dict()),
            ("shared_pool_softmax_uniform", dict(num_sampled=1024)),
            ("shared_pool_softmax_popularity", dict(num_sampled=1024, item_counts=counts))]
    if list(precisions) != ["bf16x3"]:
        arms = [("bpr", dict())] + [(name, dict(kw, precision=p)) for name, kw in arms[1:] for p in precisions]
    results = []
    for name, kw in arms:
        torch.manual_seed(1)
        model = create_graph_transformer_optimized(d.num_items, 64, 64, num_layers=2, num_heads=2, dropout=0.0,
                                                   use_laplacian_pe=False).cuda()
        kind = "shared_pool_softmax" if name.startswith("shared_pool") else name
        loss_fn = create_loss_function(kind, **kw)
        with tempfile.TemporaryDirectory() as tmp:
            trainer = Trainer(model, train, val, optim.AdamW(model.parameters(), lr=3e-3), device="cuda",
                              output_dir=tmp, max_epochs=epochs, patience=epochs, k_values=[20], loss_fn=loss_fn)
            trainer.train()
            metrics = trainer.evaluate()
        row = {"loss": name, "recall@20": round(float(metrics["recall@20"]), 4),
               "ndcg@20": round(float(metrics["ndcg@20"]), 4)}
        if "precision" in kw:
            row = {"loss": name, "precision": kw["precision"], **{k: v for k, v in row.items() if k != "loss"}}
        results.append(row)
    return results


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--shapes", default="1024x8192x82174,32768x8192x82174,8192x8192x1000000,32768x16384x1000000")
    ap.add_argument("--quality", action="store_true")
    ap.add_argument("--epochs", type=int, default=5)
    ap.add_argument("--precision", choices=["bf16x3", "bf16", "both"], default="bf16x3")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_shared_pool_softmax needs a CUDA device")
    info = gpu_info()
    precisions = {"bf16x3": ["bf16x3"], "bf16": ["bf16"], "both": ["bf16x3", "bf16"]}[args.precision]
    results = []
    for shape in args.shapes.split(","):
        b, m, items = (int(v) for v in shape.split("x"))
        if args.precision == "bf16x3":
            results.append(bench_shape(b, m, items, args.reps, args.calls))
        else:
            results.append(bench_precisions(b, m, items, args.reps, args.calls, precisions))
    line = {"bench": "shared_pool_softmax", **info, "reps": args.reps, "calls": args.calls, "results": results}
    if args.precision != "bf16x3":
        line["precision"] = args.precision
    if args.quality:
        line["quality"] = quality(args.epochs, precisions)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
