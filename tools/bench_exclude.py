"""Cost of the seen-item filter in full-catalogue scoring: the unfiltered tcgen05 bf16 scorer, the same scorer with
exclusion lists (ops.score_topk(exclude=...)), and the naive torch path a user would otherwise write (bf16 matmul into
the [B, I] score matrix, scatter_ of -inf, topk).

    python tools/bench_exclude.py [--reps 5] [--calls 10]

Shape: 23,861 RR-synth validation sessions x 82,174 items x 256, k = 20.  Exclusion rows are those sessions' context
items (their last max_len = 50 events before the target) plus the padding id 0, width 51.  Session vectors are the
mean of the context items' embeddings (random table), so the excluded items rank near the top, as they do for a
trained model.  The filtered scorer is timed with rows already ascending (as ops.seen_items returns them) and with
the row sort score_topk does otherwise.  The paths alternate in one process; times are CUDA-event medians over `reps`
windows of `calls` calls each.  Prints one JSON line.
"""

from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "gat-recommendation_b200"))


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


def validation_sessions(num_val=23_861, max_len=50):
    """RR-synth validation sessions (synth.generate's sessions after the 120,436 train ones): context item lists."""
    from etpgt_b200 import synth

    d = synth.generate(build_graph=False)
    first = 120_436
    ptr, items = d.sess_ptr, d.sess_items
    contexts = []
    for s in range(first, first + num_val):
        seq = items[ptr[s]:ptr[s + 1]]
        contexts.append(seq[:-1][-max_len:])   # the last event is the target
    return d.num_items, contexts


def score_stats(fn) -> dict:
    """One call with ETPGT_SCORE_STATS set: the library reports dump volume and fallback rows on stderr."""
    os.environ["ETPGT_SCORE_STATS"] = "1"
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as tmp:
        os.dup2(tmp.fileno(), 2)
        try:
            fn()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["ETPGT_SCORE_STATS"]
        tmp.seek(0)
        text = tmp.read()
    out = {}
    m = re.search(r"dump ([\d.]+) ms, select ([\d.]+) ms", text)
    if m:
        out.update(dump_ms=float(m.group(1)), select_ms=float(m.group(2)))
    m = re.search(r"([\d.]+) pieces per unit \(max (\d+)\), (\d+) rows recomputed", text)
    if m:
        out.update(pieces_per_row_range=float(m.group(1)), pieces_max=int(m.group(2)), fallback_rows=int(m.group(3)))
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--dim", type=int, default=256)
    ap.add_argument("--k", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_exclude.py measures on the GPU; no CUDA device found")
    import etpgt_b200.ops as ops

    dev = torch.device("cuda:0")
    num_items, contexts = validation_sessions()
    b, dim, k = len(contexts), args.dim, args.k
    width = 51
    ex = np.full((b, width), -1, dtype=np.int64)
    ex[:, 0] = 0
    for r, c in enumerate(contexts):
        ex[r, 1:1 + len(c)] = c
    exclude = torch.from_numpy(np.sort(ex, axis=1)).to(dev)
    g = torch.Generator(device=dev).manual_seed(0)
    table = (torch.randn(num_items, dim, device=dev, generator=g) / dim ** 0.5)
    table[0] = 0
    # session vectors: mean of the context embeddings (+ noise), so the seen items rank high
    flat = torch.from_numpy(np.concatenate(contexts)).to(dev)
    seg = torch.from_numpy(np.repeat(np.arange(b), [len(c) for c in contexts])).to(dev)
    sess = torch.zeros(b, dim, device=dev).index_add_(0, seg, table[flat])
    sess = sess / torch.bincount(seg, minlength=b).clamp(min=1).unsqueeze(1).float()
    sess = sess + 0.3 * torch.randn(b, dim, device=dev, generator=g) / dim ** 0.5
    sess_h, table_h = ops.to_bf16(sess), ops.to_bf16(table)
    naive_ex = torch.where(exclude < 0, torch.zeros_like(exclude), exclude)   # -1 padding -> id 0, excluded anyway

    def unfiltered():
        return ops.score_topk(sess_h, table_h, k, precision="bf16")

    def filtered():   # rows ascending, as ops.seen_items returns them
        return ops.score_topk(sess_h, table_h, k, precision="bf16", exclude=exclude, exclude_sorted=True)

    def filtered_sorting():   # unsorted rows: score_topk sorts them first
        return ops.score_topk(sess_h, table_h, k, precision="bf16", exclude=exclude)

    def naive():
        scores = sess_h @ table_h.t()
        scores.scatter_(1, naive_ex, float("-inf"))
        return torch.topk(scores, k, dim=1)

    paths = {"unfiltered_bf16": unfiltered, "filtered_bf16": filtered, "filtered_bf16_with_row_sort": filtered_sorting,
             "naive_torch": naive}
    # outputs: the filtered scorer against the naive path (same bf16 scores; ties may order differently there)
    fv, fi = filtered()
    nv, ni = naive()
    agree = float((fi == ni).float().mean().item())
    value_gap = float((fv - nv.float()).abs().max().item())
    leaked = int((fi.unsqueeze(2) == exclude.unsqueeze(1)).any(dim=2).sum().item())
    uv, ui = unfiltered()
    seen_in_unfiltered = float((ui.unsqueeze(2) == exclude.unsqueeze(1)).any(dim=2).float().sum(dim=1).mean().item())
    for fn in paths.values():   # warm-up
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {name: [] for name in paths}
    for _ in range(args.reps):
        for name, fn in paths.items():
            start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record()
            for _ in range(args.calls):
                fn()
            stop.record()
            stop.synchronize()
            times[name].append(start.elapsed_time(stop) / args.calls)
    flops = 2.0 * b * num_items * dim
    result = {"tool": "bench_exclude", **gpu_info(), "batch": b, "items": num_items, "dim": dim, "k": k,
              "exclude_width": width, "reps": args.reps, "calls_per_rep": args.calls}
    for name, ts in times.items():
        med = float(np.median(ts))
        result[name] = {"ms": round(med, 4), "ms_min": round(min(ts), 4), "ms_max": round(max(ts), 4),
                        "tflops": round(flops / (med * 1e-3) / 1e12, 1)}
    result["filtered_over_unfiltered"] = round(result["filtered_bf16"]["ms"] / result["unfiltered_bf16"]["ms"], 4)
    result["naive_over_filtered"] = round(result["naive_torch"]["ms"] / result["filtered_bf16"]["ms"], 2)
    result["stats_unfiltered"] = score_stats(unfiltered)
    result["stats_filtered"] = score_stats(filtered)
    result["check"] = {"filtered_vs_naive_id_agreement": round(agree, 5), "max_value_gap": value_gap,
                       "excluded_ids_returned": leaked, "seen_items_in_unfiltered_top_k": round(seen_in_unfiltered, 2)}
    print(json.dumps(result))


if __name__ == "__main__":
    main()
