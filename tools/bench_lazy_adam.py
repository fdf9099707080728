"""Row-sparse ("lazy") optimizer updates of the item table against the dense AdamW step.

    python tools/bench_lazy_adam.py [--part opt,step] [--quality] [--calls 30] [--steps 30]

(a) `opt`: the optimizer step alone on [I, 256] tables, I in {82,174, 466,865, 1,000,000}.  The touched rows come
    from synthetic batches of B in {32, 1,024, 32,768} sessions: the sessions' items, their targets and 5 uniform
    negatives per session, written into the gradient sink.  Timed: dense AdamW (`etpgt_adam_step`), lazy AdamW
    (`etpgt_adam_rows`), SparseAdam in scan mode over the same sink and in listed mode from the row list
    (`etpgt_sparse_adam`).  Every call clears the gradient (zero_grad), so before each timed call the sink's rows are
    written back and the L2 is overwritten with a 256 MB buffer, outside the timed window (CUDA events around the
    one call; the median is reported).  Bytes: dense 32 B per element; scan modes rows*dim*4 + touched*dim*28;
    listed mode touched*dim*(4 + 24) + touched*8.  Share of 6,452 GB/s (the copy rate this project measured on a
    B200 at a 1,000 W power limit).
(b) `step`: the whole training step (FusedTrainStep BPR forward + backward + optimizer.step) of the D = 256
    GraphTransformer at B in {1,024, 32,768} sessions and 82,174 (RR-synth) / 1,000,000 (scaled, graph from 2M
    sessions) items, dense against lazy AdamW; CUDA-event median of per-window means.
(c) `--quality`: a few Trainer epochs on RR-synth (batch 1,024) with dense and with lazy AdamW; Recall@10 / NDCG@10
    on the validation sessions.  Reported, not gated.

Prints one JSON line.
"""

from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "gat-recommendation_b200"))

PEAK_GBS = 6452.0
DIM = 256
NEG = 5


def gpu_info() -> dict:
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        power, clock = [v.strip() for v in out.strip().split(",")]
        info.update(power_limit_w=float(power), max_sm_clock_mhz=float(clock))
    except Exception as e:   # the numbers still stand, without the card's limits
        info["power_limit_w"] = f"unavailable ({type(e).__name__})"
    return info


def sessions_for(items: int, count: int):
    from etpgt_b200 import synth

    if items == 82_174:
        return synth.generate(num_sessions=count, graph_sessions=None, build_graph=False)
    if items == 1_000_000:
        return synth.generate_scaled(num_sessions=count, build_graph=False)
    return synth.generate(num_sessions=count, graph_sessions=None, num_items=items, clusters=items // 50,
                          build_graph=False)


def touched_rows(d, sessions: int, seed: int = 0) -> np.ndarray:
    """Distinct rows a batch of the first `sessions` sessions writes: its items (targets included) + negatives."""
    ids = d.sess_items[d.sess_ptr[0]:d.sess_ptr[sessions]]
    neg = np.random.default_rng(seed).integers(1, d.num_items, size=sessions * NEG)
    return np.unique(np.concatenate([ids, neg]))


def part_opt(args) -> dict:
    from etpgt_b200 import _lib, optim
    from etpgt_b200._lib import stream

    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")    # 256 MB > 126 MB of L2
    out = []
    for items in (82_174, 466_865, 1_000_000):
        d = sessions_for(items, 40_000)
        p = torch.randn(items, DIM, device="cuda") * 0.1
        m = torch.randn(items, DIM, device="cuda").abs() * 1e-3
        v = torch.randn(items, DIM, device="cuda").abs() * 1e-6
        sink = torch.zeros(items, DIM, device="cuda")
        for b in (32, 1024, 32_768):
            rows = torch.from_numpy(touched_rows(d, b)).cuda()
            vals = torch.randn(rows.numel(), DIM, device="cuda")
            touched = rows.numel()
            counter = torch.zeros(1, dtype=torch.int64, device="cuda")
            arr = (optim._AdamTensor * 1)(optim._AdamTensor(p.data_ptr(), sink.data_ptr(), m.data_ptr(),
                                                            v.data_ptr(), p.numel()))
            hp = (1e-3, 0.9, 0.999, 1e-8)
            paths = {
                "dense_adamw": (lambda: _lib.call("etpgt_adam_step", arr, 1, *hp, 1e-5, 1, 10, 1, stream()),
                                32.0 * items * DIM),
                "lazy_adamw": (lambda: _lib.call("etpgt_adam_rows", _lib.ptr(p), _lib.ptr(sink), _lib.ptr(m),
                                                 _lib.ptr(v), items, DIM, *hp, 1e-5, 1, 10, 1, None, stream()),
                               4.0 * items * DIM + 28.0 * touched * DIM),
                "sparse_adam_scan": (lambda: _lib.call("etpgt_sparse_adam", _lib.ptr(p), _lib.ptr(m), _lib.ptr(v),
                                                       items, DIM, _lib.ptr(sink), None, 0, *hp, 0, 10, 1, None,
                                                       stream()),
                                     4.0 * items * DIM + 28.0 * touched * DIM),
                "sparse_adam_listed": (lambda: _lib.call("etpgt_sparse_adam", _lib.ptr(p), _lib.ptr(m), _lib.ptr(v),
                                                         items, DIM, _lib.ptr(vals), _lib.ptr(rows), touched, *hp, 0,
                                                         10, 0, None, stream()),
                                       28.0 * touched * DIM + 8.0 * touched),
            }
            # the touched-row count as the kernels see it
            sink.index_copy_(0, rows, vals)
            _lib.call("etpgt_adam_rows", _lib.ptr(p), _lib.ptr(sink), _lib.ptr(m), _lib.ptr(v), items, DIM, *hp, 1e-5,
                      1, 10, 1, _lib.ptr(counter), stream())
            assert int(counter.item()) == touched and sink.abs().sum().item() == 0
            times = {name: [] for name in paths}
            for rep in range(args.calls + 3):
                for name, (fn, _) in paths.items():
                    sink.index_copy_(0, rows, vals)
                    flush.zero_()
                    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    start.record()
                    fn()
                    stop.record()
                    stop.synchronize()
                    if rep >= 3:
                        times[name].append(start.elapsed_time(stop))
            sink.zero_()
            entry = {"items": items, "sessions": b, "touched_rows": touched,
                     "touched_fraction": round(touched / items, 4)}
            for name, (_, nbytes) in paths.items():
                ms = float(np.median(times[name]))
                gbs = nbytes / (ms * 1e-3) / 1e9
                entry[name] = {"ms": round(ms, 4), "mb": round(nbytes / 1e6, 1), "gb_s": round(gbs, 0),
                               "of_peak": round(gbs / PEAK_GBS, 3)}
            entry["dense_over_lazy"] = round(entry["dense_adamw"]["ms"] / entry["lazy_adamw"]["ms"], 2)
            out.append(entry)
            print(json.dumps(entry), file=sys.stderr, flush=True)
        del p, m, v, sink
        torch.cuda.empty_cache()
    return {"optimizer_step": out}


def make_model(num_items):
    from etpgt_b200.model import create_graph_transformer_optimized

    torch.manual_seed(0)
    model = create_graph_transformer_optimized(num_items, DIM, DIM, 2, 2, dropout=0.1, laplacian_k=16).cuda()
    model.laplacian_pe._cached_pe = torch.randn(num_items, 16, generator=torch.Generator().manual_seed(7)).abs().cuda()
    return model.train()


def part_step(args) -> dict:
    from etpgt_b200 import data as ddata
    from etpgt_b200 import optim, synth
    from etpgt_b200.train.step import FusedTrainStep

    out = []
    for items in (82_174, 1_000_000):
        if items == 82_174:
            d = synth.generate(build_graph=True)
            store = ddata.SessionStore(d.sess_ptr, d.sess_items, "cuda")
            graph = ddata.ItemGraph(d.item_i, d.item_j, items, "cuda")
        else:
            d = synth.generate_scaled(num_sessions=2_000_000, build_graph=False)
            store = ddata.SessionStore(d.sess_ptr, d.sess_items, "cuda")
            gi, gj, _, _ = ddata.build_co_event_graph(d.sess_ptr, d.sess_items, None, 5, items, "cuda")
            graph = ddata.ItemGraph(gi, gj, items, "cuda")
        for b in (1024, 32_768):
            batches = []
            for i in range(2):
                ids = torch.from_numpy((i * b + np.arange(b)) % d.num_sessions).cuda()
                bt = ddata.build_batch(graph, store, ids, 50, False, False)
                bt.negative_items = ddata.sample_negatives(store, ids, items, NEG, seed=3, step=i).view(b, -1)
                batches.append(bt)
            entry = {"items": items, "sessions": b}
            runs = {}
            for lazy in (False, True):
                model = make_model(items)
                opt = optim.AdamW(model.parameters(), lr=1e-3, weight_decay=1e-5, lazy_rows=lazy)
                fused = FusedTrainStep(model, "bpr")

                def step(i, opt=opt, fused=fused):
                    bt = batches[i % 2]
                    opt.zero_grad()
                    fused(bt, bt.target_item, bt.negative_items)
                    opt.step()

                runs[lazy] = (step, model)
            for lazy in (False, True):
                for i in range(5):
                    runs[lazy][0](i)
            torch.cuda.synchronize()
            times = {False: [], True: []}
            for rep in range(args.reps):
                for lazy in (False, True):
                    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    start.record()
                    for i in range(args.steps):
                        runs[lazy][0](i)
                    stop.record()
                    stop.synchronize()
                    times[lazy].append(start.elapsed_time(stop) / args.steps)
            entry["dense_ms"] = round(float(np.median(times[False])), 4)
            entry["lazy_ms"] = round(float(np.median(times[True])), 4)
            entry["saved_ms"] = round(entry["dense_ms"] - entry["lazy_ms"], 4)
            out.append(entry)
            print(json.dumps(entry), file=sys.stderr, flush=True)
            del runs, batches
            torch.cuda.empty_cache()
    return {"training_step": out}


def part_quality(args) -> dict:
    import tempfile

    from etpgt_b200 import data as ddata
    from etpgt_b200 import optim, synth
    from etpgt_b200.train.trainer import Trainer

    d = synth.generate(build_graph=True)
    store = ddata.SessionStore(d.sess_ptr, d.sess_items, "cuda")
    graph = ddata.ItemGraph(d.item_i, d.item_j, d.num_items, "cuda")
    train_n, val_n, b = 120_436, 23_861, 1024

    def batches(lo, hi, step0):
        out = []
        for i, s in enumerate(range(lo, hi, b)):
            ids = torch.arange(s, min(hi, s + b), device="cuda")
            bt = ddata.build_batch(graph, store, ids, 50, False, False)
            bt.negative_items = ddata.sample_negatives(store, ids, d.num_items, NEG, seed=3, step=step0 + i)
            out.append(bt)
        return out

    train, val = batches(0, train_n, 0), batches(train_n, train_n + val_n, 10_000)
    out = {"epochs": args.epochs, "batch": b, "lr": 1e-3, "weight_decay": 1e-2}
    for lazy in (False, True):
        model = make_model(d.num_items)
        opt = optim.AdamW(model.parameters(), lr=1e-3, weight_decay=1e-2, lazy_rows=lazy)
        with tempfile.TemporaryDirectory() as tmp:
            trainer = Trainer(model, train, val, opt, device="cuda", output_dir=tmp, max_epochs=args.epochs,
                              patience=100, k_values=[10])
            history = trainer.train()
        last = history["val_metrics"][-1]
        out["lazy" if lazy else "dense"] = {"recall@10": round(last["recall@10"], 5), "ndcg@10": round(last["ndcg@10"], 5),
                                            "train_loss": [round(x, 5) for x in history["train_loss"]]}
    return {"quality": out}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--part", default="opt,step", help="comma list of: opt, step")
    ap.add_argument("--quality", action="store_true", help="also train a few epochs dense and lazy")
    ap.add_argument("--epochs", type=int, default=3)
    ap.add_argument("--calls", type=int, default=30, help="timed calls per path (optimizer step alone)")
    ap.add_argument("--steps", type=int, default=20, help="training steps per timed window")
    ap.add_argument("--reps", type=int, default=5, help="timed windows per path (training step)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lazy_adam.py: no CUDA device")
    result = {"tool": "bench_lazy_adam", **gpu_info(), "dim": DIM}
    parts = set(args.part.split(",")) if args.part else set()
    if "opt" in parts:
        result.update(part_opt(args))
    if "step" in parts:
        result.update(part_step(args))
    if args.quality:
        result.update(part_quality(args))
    print(json.dumps(result))


if __name__ == "__main__":
    main()
