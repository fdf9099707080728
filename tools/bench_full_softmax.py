"""Cost of the full-catalogue softmax loss (ops.full_softmax_loss: csrc/softmax_tc.cu) against the same loss in torch
(fp32 matmul into the [B, I] logits, F.cross_entropy, backward).

    python tools/bench_full_softmax.py [--reps 5] [--calls 5] [--shapes 1024x82174,32768x82174,8192x1000000]
                                       [--precision bf16x3|bf16|both]

D = 256 throughout.  Forward and backward are timed separately through the C ABI (etpgt_full_softmax_fwd / _bwd),
with CUDA events around `calls` back-to-back launches, median over `reps` windows after a warm-up call.  The table of
every shape is larger than the 126 MB L2 once split into its bf16 pair.  Rates: executed MMA flops 15 * 2 * B * I * D
(three split-bf16 MMAs for the forward logits, the two recomputed logits and the two gradient products), algorithmic
flops 3 * 2 * B * I * D; both also as a share of the 1,673.7 TFLOP/s dense bf16 rate measured on this card.  Peak
memory is what a forward + backward allocates beyond its inputs.  The check compares the loss and a sample of rows of
both gradients of the timed inputs with torch's fp32 result (skipped where torch does not fit).  Prints one JSON line.

--precision bf16 or both (default bf16x3: the output above) times each precision's passes on the same inputs instead:
FWD, DS (the backward with d_sess only), DE (d_table only) and the pair (forward + full backward), the precisions
alternating window by window in one process.  Executed MMA flops are 15 * 2 * B * I * D for bf16x3 and 5 * 2 * B * I * D
for bf16 (one MMA per product); `both` also compares the bf16 loss and gradients with the bf16x3 ones.  No torch run.
"""

from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "gat-recommendation_b200"))

MEASURED_BF16_TFLOPS = 1673.7
DIM = 256


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


def timed(fn, reps: int, calls: int) -> float:
    """Median ms per call over `reps` windows of `calls` calls, after one warm-up call."""
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(calls):
            fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b) / calls)
    return sorted(times)[len(times) // 2]


PRECISIONS = {"bf16x3": 0, "bf16": 1}
MMAS_PER_PRODUCT = {"bf16x3": 3, "bf16": 1}


def timed_alternating(fns: dict, reps: int, calls: int) -> dict:
    """Median ms per call of each function, its windows of `calls` calls alternating with the others' (one warm-up
    call each)."""
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    times = {name: [] for name in fns}
    for _ in range(reps):
        for name, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(calls):
                fn()
            b.record()
            b.synchronize()
            times[name].append(a.elapsed_time(b) / calls)
    return {name: sorted(t)[len(t) // 2] for name, t in times.items()}


def bench_precisions(b: int, items: int, reps: int, calls: int, precisions: list[str]) -> dict:
    """FWD, DS, DE and forward + backward of each precision on the same inputs, alternating."""
    from etpgt_b200 import _lib
    from etpgt_b200._lib import ptr

    g = torch.Generator(device="cuda").manual_seed(b + items)
    sess = torch.randn(b, DIM, device="cuda", generator=g) * 0.3
    table = torch.randn(items, DIM, device="cuda", generator=g) * 0.3
    targets = torch.randint(1, items, (b,), device="cuda", generator=g)
    lse = {p: torch.empty(b, device="cuda") for p in precisions}
    loss = {p: torch.empty(1, device="cuda") for p in precisions}
    d_loss = torch.ones(1, device="cuda")
    d_sess = torch.empty_like(sess)
    d_table = torch.zeros_like(table)
    ws = _lib.workspace(_lib.size("etpgt_full_softmax_workspace_bytes", b, items, DIM), "cuda")
    st = _lib.stream()

    def fwd(p):
        _lib.call("etpgt_full_softmax_fwd_ex", ptr(sess), ptr(table), ptr(targets), b, items, DIM, 1.0, 0.0, 0,
                  ptr(lse[p]), ptr(loss[p]), ptr(ws), ws.numel(), st, PRECISIONS[p])

    def bwd(p, ds, dt):
        _lib.call("etpgt_full_softmax_bwd_ex", ptr(sess), ptr(table), ptr(targets), ptr(lse[p]), ptr(d_loss), b,
                  items, DIM, 1.0, 0.0, 0, ptr(ds), ptr(dt), ptr(ws), ws.numel(), st, PRECISIONS[p])

    fns = {}
    for p in precisions:
        fns[(p, "fwd")] = lambda p=p: fwd(p)
        fns[(p, "ds")] = lambda p=p: bwd(p, d_sess, None)
        fns[(p, "de")] = lambda p=p: bwd(p, None, d_table)
        fns[(p, "pair")] = lambda p=p: (fwd(p), bwd(p, d_sess, d_table))
    t = timed_alternating(fns, reps, calls)
    out = {"batch": b, "items": items, "dim": DIM, "modes": {}}
    for p in precisions:
        executed = 5 * MMAS_PER_PRODUCT[p] * 2 * b * items * DIM
        out["modes"][p] = {
            "fwd_ms": round(t[(p, "fwd")], 3), "ds_ms": round(t[(p, "ds")], 3), "de_ms": round(t[(p, "de")], 3),
            "fwd_bwd_ms": round(t[(p, "pair")], 3),
            "executed_flops": f"{5 * MMAS_PER_PRODUCT[p]}*2*B*I*D",
            "executed_tflops": round(executed / t[(p, "pair")] / 1e9, 1),
            "executed_share_of_measured_peak": round(executed / t[(p, "pair")] / 1e9 / MEASURED_BF16_TFLOPS, 3),
        }
    if len(precisions) == 2:
        out["bf16x3_over_bf16_fwd_bwd"] = round(t[("bf16x3", "pair")] / t[("bf16", "pair")], 2)
        res = {}
        for p in precisions:           # one clean forward + backward of each
            d_table.zero_()
            fwd(p)
            bwd(p, d_sess, d_table)
            torch.cuda.synchronize()
            res[p] = (loss[p].clone(), lse[p].clone(), d_sess.clone(), d_table.clone())

        def rel(a, w):
            return float((a - w).abs().max() / w.abs().max())

        out["bf16_vs_bf16x3"] = {name: rel(x, y) for name, x, y in
                                 zip(("loss", "lse", "d_sess", "d_table"), res["bf16"], res["bf16x3"])}
    del ws, d_sess, d_table
    torch.cuda.empty_cache()
    return out


def bench_shape(b: int, items: int, reps: int, calls: int) -> dict:
    from etpgt_b200 import _lib
    from etpgt_b200._lib import ptr

    g = torch.Generator(device="cuda").manual_seed(b + items)
    sess = torch.randn(b, DIM, device="cuda", generator=g) * 0.3
    table = torch.randn(items, DIM, device="cuda", generator=g) * 0.3
    targets = torch.randint(1, items, (b,), device="cuda", generator=g)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    lse = torch.empty(b, device="cuda")
    loss = torch.empty(1, device="cuda")
    d_loss = torch.ones(1, device="cuda")
    d_sess = torch.empty_like(sess)
    d_table = torch.zeros_like(table)
    ws = _lib.workspace(_lib.size("etpgt_full_softmax_workspace_bytes", b, items, DIM), "cuda")
    st = _lib.stream()

    def fwd():
        _lib.call("etpgt_full_softmax_fwd", ptr(sess), ptr(table), ptr(targets), b, items, DIM, 1.0, 0.0, 0,
                  ptr(lse), ptr(loss), ptr(ws), ws.numel(), st)

    def bwd():
        _lib.call("etpgt_full_softmax_bwd", ptr(sess), ptr(table), ptr(targets), ptr(lse), ptr(d_loss), b, items, DIM,
                  1.0, 0.0, 0, ptr(d_sess), ptr(d_table), ptr(ws), ws.numel(), st)

    fwd()
    torch.cuda.synchronize()
    fwd_ms = timed(fwd, reps, calls)
    bwd_ms = timed(bwd, reps, calls)
    peak = torch.cuda.max_memory_allocated() - base
    # the checked gradient: one clean backward
    d_table.zero_()
    fwd()
    bwd()
    torch.cuda.synchronize()
    ours = (float(loss), d_sess.clone(), d_table.clone())
    total_ms = fwd_ms + bwd_ms
    executed = 15 * 2 * b * items * DIM
    algorithmic = 3 * 2 * b * items * DIM
    out = {
        "batch": b, "items": items, "dim": DIM,
        "fwd_ms": round(fwd_ms, 3), "bwd_ms": round(bwd_ms, 3), "total_ms": round(total_ms, 3),
        "executed_tflops": round(executed / total_ms / 1e9, 1),
        "executed_share_of_measured_peak": round(executed / total_ms / 1e9 / MEASURED_BF16_TFLOPS, 3),
        "algorithmic_tflops": round(algorithmic / total_ms / 1e9, 1),
        "algorithmic_share_of_measured_peak": round(algorithmic / total_ms / 1e9 / MEASURED_BF16_TFLOPS, 3),
        "peak_mem_beyond_inputs_mb": round(peak / 2**20, 1),
    }
    del ws, d_sess, d_table
    torch.cuda.empty_cache()
    # torch: fp32 logits [B, I] + cross_entropy + backward (padding column 0 left out as a -inf mask)
    need = 4 * b * items * 3
    free, _ = torch.cuda.mem_get_info()
    if need > 0.8 * free:
        out["torch"] = f"not run: needs ~{need / 2**30:.0f} GB of logits and gradients"
        return out
    s = sess.clone().requires_grad_(True)
    e = table.clone().requires_grad_(True)
    mask = torch.zeros(items, device="cuda")
    mask[0] = -float("inf")
    prev_tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False

    def torch_step():
        s.grad = e.grad = None
        z = s @ e.T + mask
        torch.nn.functional.cross_entropy(z, targets).backward()

    torch_step()
    torch.cuda.synchronize()
    base_t = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    torch_ms = timed(torch_step, reps, max(1, calls // 2))
    out["torch_fp32_ms"] = round(torch_ms, 3)
    out["torch_peak_mem_beyond_inputs_mb"] = round((torch.cuda.max_memory_allocated() - base_t) / 2**20, 1)
    out["speedup_vs_torch"] = round(torch_ms / total_ms, 2)
    torch_step()
    torch.backends.cuda.matmul.allow_tf32 = prev_tf32
    rows = torch.randperm(b, device="cuda")[:256]
    item_rows = torch.randperm(items, device="cuda")[:1024]

    def rel(a, w):
        return float((a - w).abs().max() / w.abs().max())

    with torch.no_grad():
        z = s @ e.T + mask
        want_loss = float(torch.nn.functional.cross_entropy(z, targets))
    out["check"] = {"loss_rel_err": abs(ours[0] - want_loss) / abs(want_loss),
                    "d_sess_rows_rel_err": rel(ours[1][rows], s.grad[rows]),
                    "d_table_rows_rel_err": rel(ours[2][item_rows], e.grad[item_rows])}
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--shapes", default="1024x82174,32768x82174,8192x1000000")
    ap.add_argument("--precision", choices=["bf16x3", "bf16", "both"], default="bf16x3")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_full_softmax needs a CUDA device")
    info = gpu_info()
    results = []
    for shape in args.shapes.split(","):
        b, items = (int(v) for v in shape.split("x"))
        if args.precision == "bf16x3":
            results.append(bench_shape(b, items, args.reps, args.calls))
        else:
            precisions = ["bf16x3", "bf16"] if args.precision == "both" else ["bf16"]
            results.append(bench_precisions(b, items, args.reps, args.calls, precisions))
    line = {"bench": "full_softmax", **info, "reps": args.reps, "calls": args.calls, "results": results}
    if args.precision != "bf16x3":
        line["precision"] = args.precision
    print(json.dumps(line))


if __name__ == "__main__":
    main()
