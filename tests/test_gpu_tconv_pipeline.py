"""The TransformerConv row kernels walk each warp's nodes one ahead and hold a row's edge metadata in lanes, one chunk
of lanes-per-node edges at a time (csrc/tconv.cuh, csrc/tconv.cu).  These graphs put the chunk and prefetch edges in
front of all four row kernels: destinations and sources of 0, 1, 31, 32, 33, 64, 256 and 257 edges (the 257-edge rows
go to the hub kernels when the hub plan is used, and through nine chunks of the row kernels when it is not), at the
last node of the grid, with enough nodes that the persistent grids stride more than once and warps find their next
node past the end.  Checked against the fp64 oracle at the bounds of test_gpu_kernels.py, with and without the
attention mask and w_beta, fp32 and split-bf16 gradients, the fused BatchNorm sums, and run-to-run bits."""

import math

import numpy as np
import pytest
import torch

from golden_util import rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-4
DEGS = [0, 1, 31, 32, 33, 64, 256, 257]


@pytest.fixture(scope="module")
def ops():
    from etpgt_b200 import ops as _ops

    return _ops


def pipeline_graph(rng, n):
    """The last len(DEGS) nodes are destinations of exactly DEGS in-edges, the first len(DEGS) sources of exactly DEGS
    out-edges; every other node has 0-5 in-edges from the other nodes."""
    k = len(DEGS)
    mid = np.arange(k, n - k)
    src, dst = [], []
    for i, d in enumerate(DEGS):
        src.append(rng.choice(mid, size=d))
        dst.append(np.full(d, n - k + i))
        src.append(np.full(d, i))
        dst.append(rng.choice(mid, size=d))
    fill = rng.integers(0, 6, size=n - 2 * k)
    dst.append(np.repeat(mid, fill))
    src.append(rng.choice(mid, size=int(fill.sum())))
    ei = np.stack([np.concatenate(src), np.concatenate(dst)]).astype(np.int64)
    return ei[:, rng.permutation(ei.shape[1])]


def oracle(qkvs, ei, heads, amask, wb):
    from oracle.conv_ref import _scatter_rows, segment_softmax

    n, dim = qkvs.size(0), qkvs.size(1) // 4
    q, k, v, s = qkvs.split(dim, dim=1)
    c = dim // heads
    src, dst = ei[0], ei[1]
    logits = (q.view(n, heads, c)[dst] * k.view(n, heads, c)[src]).sum(-1) / math.sqrt(c)
    alpha = segment_softmax(logits, dst, n)
    if amask is not None:
        alpha = alpha * amask
    agg = _scatter_rows(v.view(n, heads, c)[src] * alpha.unsqueeze(-1), dst, n).reshape(n, dim)
    if wb is None:
        return agg + s
    bta = torch.sigmoid(torch.cat([agg, s, agg - s], dim=-1) @ wb.t())
    return bta * s + (1 - bta) * agg


@pytest.mark.parametrize("dim,heads,n,mask,beta,hub", [
    (256, 2, 12_000, True, True, False),
    (256, 2, 12_000, True, True, True),
    (256, 8, 10_001, False, False, False),
    (128, 1, 10_001, True, True, False),
    (64, 2, 20_003, True, False, True),
    (32, 4, 40_001, False, True, False),
])
def test_tconv_pipeline_edges(ops, dim, heads, n, mask, beta, hub):
    rng = np.random.default_rng(dim * 7 + heads + n)
    g = torch.Generator().manual_seed(dim + heads + n)
    ei = torch.from_numpy(pipeline_graph(rng, n))
    e = ei.size(1)
    qkvs64 = torch.randn(n, 4 * dim, generator=g, dtype=torch.float64).requires_grad_(True)
    wb64 = (torch.randn(1, 3 * dim, generator=g, dtype=torch.float64) * 0.2).requires_grad_(True) if beta else None
    amask = (torch.rand(e, heads, generator=g) > 0.1).double() / 0.9 if mask else None
    d_out = torch.randn(n, dim, generator=g, dtype=torch.float64)
    ref = oracle(qkvs64, ei, heads, amask, wb64)
    ref.backward(d_out)

    index = ops.GraphIndex(ei.cuda(), n)
    if not hub:
        index._hub = False          # the 257-edge rows stay with the row kernels
    assert (index.hub_plan() is not None) == hub

    f32 = dict(dtype=torch.float32, device="cuda")
    qkvs = qkvs64.detach().float().cuda()
    wb = wb64.detach().float().cuda().reshape(-1) if beta else None
    am = amask.float().cuda() if mask else None
    dout = d_out.float().cuda()

    def forward(bn_sums=None):
        out, agg = torch.empty(n, dim, **f32), torch.empty(n, dim, **f32)
        bt, m, inv_l = torch.empty(n, **f32), torch.empty(n, heads, **f32), torch.empty(n, heads, **f32)
        ops._tconv_fwd(qkvs, n, dim, heads, index, wb, am, out, agg, bt, m, inv_l, bn_sums)
        return out, agg, bt, m, inv_l

    def backward(saved, split):
        _, agg, bt, m, inv_l = saved
        d_wb = torch.empty(3 * dim, **f32) if beta else None
        if split:
            hi = torch.empty(n, 4 * dim, dtype=torch.bfloat16, device="cuda")
            lo, colsum = torch.empty_like(hi), torch.empty(4 * dim, **f32)
            ops._tconv_bwd(qkvs, dout, n, dim, heads, index, wb, am, agg, bt, m, inv_l, None, hi, lo, colsum, d_wb)
            return hi, lo, colsum, d_wb
        d_qkvs = torch.empty(n, 4 * dim, **f32)
        ops._tconv_bwd(qkvs, dout, n, dim, heads, index, wb, am, agg, bt, m, inv_l, d_qkvs, None, None, None, d_wb)
        return d_qkvs, d_wb

    saved = forward()
    assert rel_err(saved[0], ref) < TOL, "forward"
    d_qkvs, d_wb = backward(saved, split=False)
    assert rel_err(d_qkvs, qkvs64.grad) < TOL, "d_qkvs"
    if beta:
        assert rel_err(d_wb, wb64.grad.reshape(-1)) < TOL, "d_w_beta"

    # training forward (persistent, BatchNorm sums): the same rows as the eval forward, and the column sums of out
    bn = torch.empty(2 * dim, dtype=torch.float64, device="cuda")
    saved_bn = forward(bn)
    for a, b in zip(saved, saved_bn):
        assert torch.equal(a, b)
    o = saved[0].double()
    assert rel_err(bn, torch.cat([o.sum(0), (o * o).sum(0)])) < 1e-9

    # split-bf16 gradients: the bf16 pair of the fp32 gradient, plus the bias column sums
    hi, lo, colsum, d_wb2 = backward(saved, split=True)
    want_hi = d_qkvs.to(torch.bfloat16)
    assert torch.equal(hi, want_hi)
    assert torch.equal(lo, (d_qkvs - want_hi.float()).to(torch.bfloat16))
    assert rel_err(colsum, d_qkvs.double().sum(0)) < 1e-5
    if beta:
        assert torch.equal(d_wb, d_wb2)

    # run to run: the same bits
    again = forward(torch.empty_like(bn))
    for a, b in zip(saved, again):
        assert torch.equal(a, b)
    d_qkvs2, d_wb3 = backward(again, split=False)
    assert torch.equal(d_qkvs, d_qkvs2)
    hi2, lo2, colsum2, _ = backward(again, split=True)
    assert torch.equal(hi, hi2) and torch.equal(lo, lo2) and torch.equal(colsum, colsum2)
    if beta:
        assert torch.equal(d_wb, d_wb3)
