#!/usr/bin/env python3
"""Times the tensor-core top-k scorer for k in {20, 64, 100, 128, 256}, unfiltered and with `seen_items`-style
exclusion lists, against torch bf16 matmul + topk and the fp32 CUDA-core scorer at k = 64.

    python tools/bench_score_large_k.py [--reps 10] [--out profiles/score_large_k.jsonl]

Shapes: 23,861 x 82,174 x 256 (the bf16 table, 42 MB, stays resident in L2 across calls) and 8,192 x 1,000,000 x 256.
Times are CUDA-event medians over `reps` calls after a warm-up.  The per-kernel split (dump / select / fallback),
dumped pieces per row and fallback rows come from a separate process: one warm-up call, then one call with
ETPGT_SCORE_STATS set (it synchronises, so it is not part of the medians).  Also times topk_merge_parts at k = 256
over 8 parts, the merge of sharded evaluation.  Prints the GPU name and power limit and appends one JSON line to --out.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "gat-recommendation_b200"))

from etpgt_b200 import _lib, ops  # noqa: E402

KS = [20, 64, 100, 128, 256]
SHAPES = [(23861, 82174, 256), (8192, 1000000, 256)]


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return sorted(times)[len(times) // 2]


def stats_of(sess_h, table_h, k, exclude):
    """One call with ETPGT_SCORE_STATS: the library's own report, parsed from stderr in a child process."""
    code = (
        "import sys, torch; sys.path.insert(0, %r); from etpgt_b200 import ops\n"
        "g = torch.Generator(device='cuda').manual_seed(0)\n"
        "b, n, d, k, ex = %d, %d, %d, %d, %d\n"
        "s = torch.randn(b, d, device='cuda', generator=g).bfloat16(); t = torch.randn(n, d, device='cuda', generator=g).bfloat16()\n"
        "e = torch.sort(torch.randint(0, n, (b, 20), device='cuda', generator=g), 1).values if ex else None\n"
        "ops.score_topk(s, t, k, precision='bf16', exclude=e, exclude_sorted=True); torch.cuda.synchronize()\n"
        "import os; os.environ['ETPGT_SCORE_STATS'] = '1'   # the warm-up call above is not reported\n"
        "ops.score_topk(s, t, k, precision='bf16', exclude=e, exclude_sorted=True); torch.cuda.synchronize()\n"
    ) % (str(ROOT / "gat-recommendation_b200"), sess_h.size(0), table_h.size(0), sess_h.size(1), k, int(exclude is not None))
    env = {key: v for key, v in os.environ.items() if key != "ETPGT_SCORE_STATS"}
    err = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=tempfile.gettempdir()).stderr
    out = {"dump_ms": 0.0, "select_ms": 0.0, "fallback_ms": 0.0, "pieces_per_unit": [], "redo_rows": 0, "calls": 0}
    for m in re.finditer(r"dump ([\d.]+) ms, select ([\d.]+) ms, fallback ([\d.]+) ms", err):
        out["dump_ms"] += float(m.group(1)); out["select_ms"] += float(m.group(2)); out["fallback_ms"] += float(m.group(3))
        out["calls"] += 1
    for m in re.finditer(r"cap (\d+), ([\d.]+) pieces per unit \(max (\d+)\), (\d+) rows recomputed", err):
        out["pieces_per_unit"].append(float(m.group(2)))
        out["redo_rows"] += int(m.group(4))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "score_large_k.jsonl"))
    ap.add_argument("--small", action="store_true", help="a tiny shape, for a dry run of the script")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_score_large_k: needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    gpu = q[0] if q else torch.cuda.get_device_name()
    print(f"GPU: {gpu}")
    shapes = [(1000, 20000, 256)] if args.small else SHAPES
    result = {"gpu": gpu, "reps": args.reps, "cases": []}
    for b, n, d in shapes:
        g = torch.Generator(device="cuda").manual_seed(0)
        sess_h = torch.randn(b, d, device="cuda", generator=g).bfloat16()
        table_h = torch.randn(n, d, device="cuda", generator=g).bfloat16()
        exclude = torch.sort(torch.randint(0, n, (b, 20), device="cuda", generator=g), 1).values
        for k in KS:
            row = {"batch": b, "items": n, "dim": d, "k": k,
                   "workspace_bytes": _lib.size("etpgt_score_topk_bf16_workspace_bytes", b, n, k)}
            row["ms"] = timed(lambda: ops.score_topk(sess_h, table_h, k, precision="bf16"), args.reps)
            row["ms_excl"] = timed(lambda: ops.score_topk(sess_h, table_h, k, precision="bf16", exclude=exclude,
                                                          exclude_sorted=True), args.reps)
            row["stats"] = stats_of(sess_h, table_h, k, None)
            row["stats_excl"] = stats_of(sess_h, table_h, k, exclude)
            chunk = max(1, (2 << 30) // (n * 2))   # torch: bf16 score rows in chunks of <= 2 GiB
            def torch_topk():
                for r0 in range(0, b, chunk):
                    torch.topk(sess_h[r0:r0 + chunk] @ table_h.t(), k, dim=1)
            row["torch_ms"] = timed(torch_topk, max(3, args.reps // 3))
            print(json.dumps(row), flush=True)
            result["cases"].append(row)
        # the sharded-evaluation merge at k = 256 over 8 parts (random candidates, each part sorted like a scorer's)
        k, parts = 256, 8
        val_bytes = (b * k * 4 + 255) // 256 * 256
        stride = val_bytes + b * k * 8
        buf = torch.empty(parts * stride, dtype=torch.uint8, device="cuda")
        for p in range(parts):
            blk = buf[p * stride:(p + 1) * stride]
            v = torch.sort(torch.randn(b, k, device="cuda", generator=g), dim=1, descending=True).values
            blk[:b * k * 4].view(torch.float32).view(b, k).copy_(v)
            blk[val_bytes:].view(torch.int64).view(b, k).copy_(torch.randint(0, n, (b, k), device="cuda", generator=g))
        targets = torch.randint(0, n, (b,), device="cuda", generator=g)
        ms = timed(lambda: ops.topk_merge_parts(buf, parts, stride, val_bytes, b, k, 0, b, targets), args.reps)
        result["cases"].append({"batch": b, "items": n, "k": k, "merge_parts": parts, "merge_ms": ms})
        print(f"topk_merge_parts {b} rows x {parts} parts, k={k}: {ms:.3f} ms", flush=True)
        del buf
        sess_f, table_f = sess_h.float(), table_h.float()
        ms = timed(lambda: ops.score_topk(sess_f, table_f, 64, precision="fp32"), 3)
        result["cases"].append({"batch": b, "items": n, "dim": d, "k": 64, "fp32_ms": ms})
        print(f"fp32 CUDA-core scorer {b}x{n}x{d} k=64: {ms:.3f} ms", flush=True)
        del sess_f, table_f
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    with open(args.out, "a") as f:
        f.write(json.dumps(result) + "\n")


if __name__ == "__main__":
    main()
