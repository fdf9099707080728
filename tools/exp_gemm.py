"""Timing of the three GEMMs of one TransformerConv layer at the bench batch (N = 99,132 nodes, D = 256): forward
projection [N,256]x[1024,256]^T, dX [N,1024]x[1024,256] (+ TMA reduce-add), dW [1024,N]x[N,256] (split-K).
Prints ms per GEMM and the worst error vs fp64."""
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "gat-recommendation_b200"))
from etpgt_b200 import ops  # noqa: E402

torch.manual_seed(0)
n, d, w4 = 99_132, 256, 1024
dev = "cuda"
x = torch.randn(n, d, device=dev)
w = torch.randn(w4, d, device=dev) / 16
b = torch.randn(w4, device=dev)
dy = torch.randn(n, w4, device=dev)
x_hi, x_lo, *_ = ops._split(x, True, False)
w_hi, w_lo, *_ = ops._split(w, True, False)
g_hi, g_lo, *_ = ops._split(dy, True, False)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def timed(fn, reps=20):
    for _ in range(3):
        fn()
    tot = 0.0
    for _ in range(reps):
        flush.zero_()
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        tot += a.elapsed_time(e)
    return tot / reps


fwd = lambda: ops._gemm_x3(x_hi, x_lo, w_hi, w_lo, n, w4, d, d, d, b)                       # noqa: E731
res = torch.zeros(n, d, device=dev)
dx = lambda: ops._gemm_x3(g_hi, g_lo, w_hi, w_lo, n, d, w4, w4, d, None, b_mn=True, accumulate_into=res)   # noqa: E731
dw = lambda: ops._gemm_x3(g_hi, g_lo, x_hi, x_lo, w4, d, n, w4, d, None, split_k=0, a_mn=True, b_mn=True)  # noqa: E731
y = fwd()
err_f = ((y.double() - (x.double() @ w.double().t() + b.double())).abs().max() / y.double().abs().max()).item()
res.zero_()
gx = dx()
err_x = ((gx.double() - dy.double() @ w.double()).abs().max() / gx.double().abs().max()).item()
gw = dw()
ref_w = dy.double().t() @ x.double()
err_w = ((gw.double() - ref_w).abs().max() / ref_w.abs().max()).item()
print(f"errors fwd {err_f:.2e} dX {err_x:.2e} dW {err_w:.2e}")
print(f"fwd {timed(fwd):.4f} ms, dX {timed(dx):.4f} ms, dW {timed(dw):.4f} ms")
