"""Cost of the in-batch and mixed-negative softmax (train.losses.InBatchSoftmaxLoss): the column builder
(etpgt_in_batch_columns) and the loss's forward + backward over its columns, next to the shared-pool softmax over a
pool of the same total column count, in the same process.

    python tools/bench_in_batch_softmax.py [--reps 5] [--calls 5] [--batches 1024,8192,32768] [--pools 0,8192]
                                           [--precision bf16x3|bf16|both] [--items 82174]

D = 256.  Targets are zipf(1.3)-distributed ids, so the builder sees the duplicate runs of real traffic; the pool of
the mixed case is drawn by etpgt_sample_item_pool (popularity^0.75 of zipf counts), and its draw is not part of the
builder's time (the shared pool pays it too).  Each call of the builder advances the estimator's step.  Forward +
backward go through the C ABI (etpgt_pool_softmax_fwd_ex / _bwd_ex) over the C = num_sampled + B columns; the
backward adds into a d_table of the whole catalogue, as training does.  The shared-pool arm is a sampled pool of C
entries.  CUDA events around `calls` back-to-back calls, median over `reps` windows, all arms of a shape alternating
window by window after a warm-up.  Prints one JSON line with the card's name and power limit.
"""

from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "gat-recommendation_b200"))

from bench_full_softmax import PRECISIONS, gpu_info, timed_alternating  # noqa: E402

DIM = 256


def bench_shape(b: int, m: int, items: int, reps: int, calls: int, precisions: list[str]) -> dict:
    from etpgt_b200 import _lib, ops
    from etpgt_b200._lib import ptr

    g = torch.Generator(device="cuda").manual_seed(b + m + items)
    sess = torch.randn(b, DIM, device="cuda", generator=g) * 0.3
    table = torch.randn(items, DIM, device="cuda", generator=g) * 0.3
    rng = np.random.default_rng(b + m)
    targets = torch.from_numpy((rng.zipf(1.3, b) % (items - 1)) + 1).cuda()
    counts = torch.from_numpy(np.bincount(np.random.default_rng(items).zipf(1.5, 4 * items) % items,
                                          minlength=items) + 1)
    cum = ops.item_sampling_table(counts, 0.75, 0, device="cuda")
    c = m + b
    pool, pool_lq = ops.sample_item_pool(cum, m, seed=1, step=0) if m else (None, None)
    shared, shared_lq = ops.sample_item_pool(cum, c, seed=2, step=0)
    freq = torch.full((items,), 1.0 / (items - 1), dtype=torch.float64, device="cuda")
    freq[0] = 0.0
    last = torch.full((items,), -1, dtype=torch.int64, device="cuda")
    cols = torch.empty(c, dtype=torch.int64, device="cuda")
    lq = torch.empty(c, dtype=torch.float32, device="cuda")
    st = _lib.stream()
    bws = _lib.workspace(_lib.size("etpgt_in_batch_columns_workspace_bytes", b, m), "cuda")
    step = [0]

    def build():
        _lib.call("etpgt_in_batch_columns", ptr(targets), b, ptr(pool), ptr(pool_lq), m, ptr(freq), ptr(last), items,
                  0, step[0], 0.01, ptr(cols), ptr(lq), ptr(bws), bws.numel(), st)
        step[0] += 1

    build()
    lse = torch.empty(b, device="cuda")
    z_pos = torch.empty(b, device="cuda")
    loss = torch.empty(1, device="cuda")
    d_loss = torch.ones(1, device="cuda")
    d_sess = torch.empty_like(sess)
    d_table = torch.zeros_like(table)
    ws = _lib.workspace(_lib.size("etpgt_pool_softmax_workspace_bytes", b, c, DIM), "cuda")

    def fwd_bwd(ids, log_q, p):
        _lib.call("etpgt_pool_softmax_fwd_ex", ptr(sess), ptr(table), ptr(targets), ptr(ids), ptr(log_q), b, items,
                  c, DIM, 1.0, 0.0, 0, ptr(lse), ptr(z_pos), ptr(loss), ptr(ws), ws.numel(), st, PRECISIONS[p])
        _lib.call("etpgt_pool_softmax_bwd_ex", ptr(sess), ptr(table), ptr(targets), ptr(ids), ptr(log_q), ptr(lse),
                  ptr(z_pos), ptr(d_loss), b, items, c, DIM, 1.0, 0.0, 0, ptr(d_sess), ptr(d_table), ptr(ws),
                  ws.numel(), st, PRECISIONS[p])

    fns = {"build": build}
    for p in precisions:
        fns[(p, "in_batch")] = lambda p=p: fwd_bwd(cols, lq, p)
        fns[(p, "shared")] = lambda p=p: fwd_bwd(shared, shared_lq, p)
    t = timed_alternating(fns, reps, calls)
    out = {"batch": b, "num_sampled": m, "columns": c, "items": items, "dim": DIM,
           "builder_ms": round(t["build"], 4), "modes": {}}
    for p in precisions:
        fb = t[(p, "in_batch")]
        out["modes"][p] = {
            "in_batch_fwd_bwd_ms": round(fb, 3),
            "shared_pool_fwd_bwd_ms": round(t[(p, "shared")], 3),
            "in_batch_over_shared_pool": round(fb / t[(p, "shared")], 3),
            "builder_share_of_fwd_bwd": round(t["build"] / fb, 4),
        }
    del ws, d_table
    torch.cuda.empty_cache()
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--batches", default="1024,8192,32768")
    ap.add_argument("--pools", default="0,8192")
    ap.add_argument("--items", type=int, default=82_174)
    ap.add_argument("--precision", choices=["bf16x3", "bf16", "both"], default="both")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_in_batch_softmax needs a CUDA device")
    info = gpu_info()
    precisions = {"bf16x3": ["bf16x3"], "bf16": ["bf16"], "both": ["bf16x3", "bf16"]}[args.precision]
    results = [bench_shape(int(b), int(m), args.items, args.reps, args.calls, precisions)
               for b in args.batches.split(",") for m in args.pools.split(",")]
    print(json.dumps({"bench": "in_batch_softmax", **info, "reps": args.reps, "calls": args.calls,
                      "precision": args.precision, "results": results}))


if __name__ == "__main__":
    main()
