"""GPU parity tests of the reference's two baselines, GraphSAGE and GAT, at the widths and batch sizes the reference
trains them at, against the fp64 oracle (oracle/conv_ref.py, oracle/model_ref.py) run on the device.

  A. the SAGE mean kernels (etpgt_sage_mean_fwd / _fwd_split / _bwd / _bwd_ld) bit for bit, on inputs for which every
     sum, every 1/deg and every fma of the kernels is exact in fp32;
  B. SAGEConv, fused (ops.SageLayerFn: one split-bf16 GEMM over [mean | x]) and fallback (ops.SageMeanFn + linear), up
     to ~100k nodes, where the weight gradient runs split-K;
  C. GATConv with concat=True (ops.GatAggregateFn, the d_agg branch of the edge backward) and concat=False
     (ops.GatLayerFn, ops.GatConvFn) on graphs with a hub of > 5,000 in-edges;
  D. create_graphsage / create_gat (with and without concatenated heads) on a ~4,096-session batch: session
     embeddings, loss, every parameter gradient, BatchNorm running statistics, eval forward;
  E. widths outside the supported set fail with an error that names the set.

Errors are `golden_util.rel_err` (max |diff| over max |ref| of the whole tensor).  A whole-tensor bound hides a wrong
small row (a hub row's mean is ~1/sqrt(deg) the size of an ordinary row), so B and C also bound the hub, isolated and
degree-1 rows against their own row's size."""

import numpy as np
import pytest
import torch

from golden_util import rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-4
DIMS = (32, 64, 128, 256)


# ------------------------------------------------------------------------------ graphs


def _graph(n, seed, *, hub_deg=0, fan_out=0, pow2=False, loops=0.03, dups=0.3):
    """A destination-ordered-at-random edge list [2, E] (CPU int64) with the rows kernels get wrong:
      * in-degrees 1..5 (pow2: 1, 2, 4, ..., 64), ~15% of the nodes with in-degree 0;
      * a hub `n // 2` with `hub_deg` in-edges whose sources are zipf-like over the other nodes, including 8 self loops
        and many duplicates;
      * a source `n - 1` with `fan_out` out-edges (kept off the hub);
      * self loops (fraction `loops`) and duplicated edges (a row repeats its previous source with probability `dups`).
    Self loops and duplicates count towards the in-degree (PyG's mean counts them).  Returns (edge_index, rows) with
    rows = {"hub", "fan", "isolated", "deg1"} (degrees without self loops, as GAT sees them)."""
    g = torch.Generator().manual_seed(seed)
    deg = (2 ** torch.randint(0, 7, (n,), generator=g)) if pow2 else torch.randint(1, 6, (n,), generator=g)
    deg[torch.rand(n, generator=g) < 0.15] = 0
    hub, fan = n // 2, n - 1
    if n == 1:
        deg[0] = 4 if pow2 else 3
    if hub_deg:
        assert n >= 3
        deg[hub] = hub_deg
    dst = torch.repeat_interleave(torch.arange(n), deg)
    src = torch.randint(0, n, (dst.numel(),), generator=g)
    same = torch.zeros_like(dst, dtype=torch.bool)
    same[1:] = (dst[1:] == dst[:-1]) & (torch.rand(dst.numel() - 1, generator=g) < dups)
    for k in torch.nonzero(same).flatten().tolist():      # chains of repeated (src, dst) pairs
        src[k] = src[k - 1]
    src[torch.rand(dst.numel(), generator=g) < loops] = -1
    src = torch.where(src < 0, dst, src)
    if fan_out:
        cand = torch.nonzero(dst != hub).flatten()
        assert cand.numel() >= fan_out
        src[cand[torch.randperm(cand.numel(), generator=g)[:fan_out]]] = fan
    if hub_deg:
        at = torch.nonzero(dst == hub).flatten()
        u = torch.rand(at.numel(), generator=g)
        src[at] = ((n - 1) * u * u).long()                # zipf-like over 0..n-2: never the fan-out source
        src[at[:8]] = hub                                 # self loops on the hub
    if n == 1:
        src.zero_()
    perm = torch.randperm(dst.numel(), generator=g)
    ei = torch.stack([src, dst])[:, perm]
    real = ei[:, ei[0] != ei[1]]
    indeg = torch.bincount(real[1], minlength=n)
    rows = {"hub": hub if hub_deg else None, "fan": fan if fan_out else None,
            "isolated": torch.nonzero(indeg == 0).flatten(), "deg1": torch.nonzero(indeg == 1).flatten()[:64]}
    return ei, rows


def _row_err(got, want, rows):
    """max over `rows` of (max |diff| in the row) / (max |ref| in the row).  A row whose reference is below 1e-3 of the
    tensor's largest entry (an exactly-zero row, e.g. a node whose only edge is masked) is measured on that 1e-3."""
    rows = torch.as_tensor(rows, dtype=torch.long).reshape(-1)
    if rows.numel() == 0:
        return 0.0
    floor = 1e-3 * float(want.detach().abs().max())
    got = got.detach().double()[rows.to(got.device)]
    want = want.detach().double()[rows.to(want.device)].to(got.device)
    return ((got - want).abs().amax(1) / want.abs().amax(1).clamp_min(floor)).max().item()


def _check_rows(got, want, rows, keys, tol):
    for key in keys:
        r = rows[key]
        if r is None:
            continue
        err = _row_err(got, want, r)
        assert err < tol, f"{key} rows: {err}"


# ------------------------------------------------------------------------------ A. SAGE mean kernels, exact


def _exact_case(n, case, dim, seed):
    """Inputs of the exact SAGE tests: every in-degree 0 or a power of two, features on a 1/512 grid in (-2, 2) (more
    significant bits than bf16 holds, so the split's lo half is not trivially zero), integer gradients in [-2, 2]."""
    if case == "empty":
        ei = torch.empty(2, 0, dtype=torch.long)
    else:
        ei, _ = _graph(n, seed, hub_deg=4096 if case == "hub" else 0, fan_out=3000 if n > 1000 else 0, pow2=True)
    src, dst = ei
    g = torch.Generator().manual_seed(seed + dim)
    x = torch.randint(-1023, 1024, (n, dim), generator=g, dtype=torch.float64) / 512
    d_mean = torch.randint(-2, 3, (n, dim), generator=g, dtype=torch.float64)
    d_root = torch.randint(-2, 3, (n, dim), generator=g, dtype=torch.float64)
    deg = torch.bincount(dst, minlength=n)
    assert bool(((deg == 0) | ((deg & (deg - 1)) == 0)).all()), "an in-degree is not a power of two"
    # exactness in fp32 (24-bit significand): forward partial sums are multiples of 2^-9 below deg * 2; backward
    # partial sums at a source j are multiples of 1 / (largest degree among j's destinations) below 2 * outdeg(j) + 2
    assert int(deg.max()) * 2 * 512 < 2 ** 24
    if ei.numel():
        outdeg = torch.bincount(src, minlength=n)
        finest = torch.zeros(n, dtype=torch.long).scatter_reduce(0, src, deg[dst], "amax")
        assert int(((2 * outdeg + 2) * finest).max()) < 2 ** 24, "a backward partial sum would round in fp32"
        if case == "hub":
            assert int(deg.max()) == 4096 and (n < 1000 or int(outdeg.max()) >= 1000)
            assert bool((src == dst).any()) and ei.unique(dim=1).size(1) < ei.size(1)
    return ei, x, d_mean, d_root


def _sage_mean_oracle(x64, ei, d_mean, d_root):
    """The SAGE aggregation through the oracle: conv_ref.sage_conv with lin_l = identity, lin_r = 0 (both products
    exact in fp64) is the neighbour mean; its gradient with respect to x is the scatter of d_mean_i / deg_i."""
    from oracle import conv_ref

    dim = x64.size(1)
    x64 = x64.clone().requires_grad_(True)
    eye = torch.eye(dim, dtype=torch.float64, device=x64.device)
    mean = conv_ref.sage_conv(x64, ei, eye, None, torch.zeros_like(eye))
    mean.backward(d_mean)
    return mean.detach(), x64.grad, x64.grad + d_root


def _split_ref(t):
    hi = t.to(torch.bfloat16)
    return hi, (t - hi.float()).to(torch.bfloat16)


@pytest.mark.parametrize("dim", DIMS)
@pytest.mark.parametrize("n,case", [(1, "empty"), (1, "loops"), (45, "empty"), (37, "hub"), (3001, "hub")])
def test_sage_mean_kernels_are_exact(dim, n, case):
    """Node counts are not multiples of the nodes per CTA (32 / 16 / 8 / 8 at D = 32 / 64 / 128 / 256).  A lost,
    repeated or misrouted edge, a wrong degree or a wrong pitch changes at least one value."""
    from etpgt_b200 import ops
    from etpgt_b200._lib import call, ptr, stream

    ei, x64, d_mean64, d_root64 = _exact_case(n, case, dim, seed=n + dim)
    dev = torch.device("cuda")
    eic = ei.to(dev)
    want_mean, want_dx, want_dx_root = _sage_mean_oracle(x64.to(dev), eic, d_mean64.to(dev), d_root64.to(dev))
    for t in (want_mean, want_dx, want_dx_root):
        assert torch.equal(t.float().double(), t), "the reference is not exact in fp32"
    x, d_mean, d_root = x64.float().to(dev), d_mean64.float().to(dev), d_root64.float().to(dev)
    index = ops.GraphIndex(eic, n)
    isolated = torch.bincount(ei[1], minlength=n) == 0

    mean = torch.full((n, dim), float("nan"), device=dev)
    call("etpgt_sage_mean_fwd", ptr(x), n, dim, ptr(index.rowptr), ptr(index.col), ptr(mean), stream())
    assert torch.equal(mean, want_mean.float())
    assert bool((mean[isolated.to(dev)] == 0).all())

    # the fused layer's operand: mean split into the left half of a [n, 2*dim] bf16 pair, x into the right half
    sentinel = float("nan")
    a_hi = torch.full((n, 2 * dim), sentinel, dtype=torch.bfloat16, device=dev)
    a_lo = torch.full((n, 2 * dim), sentinel, dtype=torch.bfloat16, device=dev)
    call("etpgt_sage_mean_fwd_split", ptr(x), n, dim, ptr(index.rowptr), ptr(index.col), None, ptr(a_hi), ptr(a_lo),
         2 * dim, stream())
    ops._split_into(x, a_hi, a_lo, dim)
    m_hi, m_lo = _split_ref(want_mean.float())
    x_hi, x_lo = _split_ref(x)
    assert torch.equal(a_hi[:, :dim], m_hi) and torch.equal(a_lo[:, :dim], m_lo)
    assert torch.equal(a_hi[:, dim:], x_hi) and torch.equal(a_lo[:, dim:], x_lo)
    if case == "hub":
        assert bool((m_lo != 0).any()) and bool((x_lo != 0).any())   # the lo halves carry information

    d_x = torch.full((n, dim), float("nan"), device=dev)
    call("etpgt_sage_mean_bwd", ptr(d_mean), n, dim, ptr(index.rowptr), ptr(index.colptr), ptr(index.row), ptr(d_x),
         stream())
    assert torch.equal(d_x, want_dx.float())

    # the fused layer's backward: [d_mean | d_root] as the two column halves of one GEMM output
    d_a = torch.cat([d_mean, d_root], dim=1).contiguous()
    d_x.fill_(float("nan"))
    call("etpgt_sage_mean_bwd_ld", ptr(d_a), 2 * dim, ptr(d_a.view(-1)[dim:]), n, dim, ptr(index.rowptr),
         ptr(index.colptr), ptr(index.row), ptr(d_x), stream())
    assert torch.equal(d_x, want_dx_root.float())


# ------------------------------------------------------------------------------ B. SAGEConv vs fp64

_GRAPHS = {}


def _layer_graph(n, seed):
    """The graph of the layer tests at n nodes: a hub of 4,096 (n < 1,000) or 5,200 in-edges, a fan-out source of
    3,000 edges from 1,000 nodes on, isolated nodes, self loops and duplicates; cached across parameter sets."""
    key = (n, seed)
    if key not in _GRAPHS:
        hub = 0 if n < 3 else (4096 if n < 1000 else 5200)
        _GRAPHS[key] = _graph(n, seed, hub_deg=hub, fan_out=3000 if n >= 1000 else 0)
    return _GRAPHS[key]


def _sage_inputs(in_dim, out_dim, n, seed):
    from etpgt_b200.nn import SAGEConv

    ei, rows = _layer_graph(n, seed)
    torch.manual_seed(seed + in_dim + out_dim)
    conv = SAGEConv(in_dim, out_dim)
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(n, in_dim, generator=g)
    d_y = torch.randn(n, out_dim, generator=g)
    return conv, ei, rows, x, d_y


def _sage_oracle(conv, ei, x, d_y):
    from oracle import conv_ref

    dev = torch.device("cuda")
    params = [p.detach().double().to(dev).requires_grad_(True)
              for p in (conv.lin_l.weight, conv.lin_l.bias, conv.lin_r.weight)]
    x64 = x.double().to(dev).requires_grad_(True)
    want = conv_ref.sage_conv(x64, ei.to(dev), params[0], params[1], params[2])
    want.backward(d_y.double().to(dev))
    return want.detach(), [x64.grad] + [p.grad for p in params]


def _sage_run(conv, ei, x, d_y):
    conv = conv.cuda()
    for p in conv.parameters():
        p.grad = None
    xc = x.cuda().requires_grad_(True)
    out = conv(xc, ei.cuda())
    out.backward(d_y.cuda())
    torch.cuda.synchronize()
    return out.detach(), [xc.grad, conv.lin_l.weight.grad, conv.lin_l.bias.grad, conv.lin_r.weight.grad]


def _check_sage(out, grads, want, want_grads, rows):
    assert rel_err(out, want) < TOL, "forward"
    for name, got, ref in zip(("x", "lin_l.weight", "lin_l.bias", "lin_r.weight"), grads, want_grads):
        assert rel_err(got, ref) < TOL, name
    _check_rows(out, want, rows, ("hub", "isolated", "deg1"), TOL)
    _check_rows(grads[0], want_grads[0], rows, ("hub", "fan", "isolated", "deg1"), TOL)


_SAGE_FUSED = [(i, o, n) for n in (1, 300, 5003) for i in DIMS for o in sorted({i, 256, 40})] + \
    [(256, 256, 99_133), (32, 40, 99_133), (128, 256, 99_133)]


@pytest.mark.parametrize("in_dim,out_dim,n", _SAGE_FUSED)
def test_sage_conv_fused_layer_matches_fp64(in_dim, out_dim, n):
    """ops.SageLayerFn: etpgt_sage_mean_fwd_split + _split_into build [mean | x] as one bf16 operand pair, one GEMM
    against [W_l | W_r], etpgt_sage_mean_bwd_ld and a split-K [dW_l | dW_r] (K = n; at 99,133 nodes the last split ends
    in a partial k-block).  out = 40 leaves a partial N tile.  A dropped lo term costs ~4e-3 and fails the bound; the
    split-bf16 products themselves are good to ~1e-5.  The backward is deterministic: no atomics, fixed split-K."""
    from etpgt_b200 import ops

    conv, ei, rows, x, d_y = _sage_inputs(in_dim, out_dim, n, seed=7)
    assert ops.sage_layer_supported(x.cuda(), in_dim, out_dim)
    want, want_grads = _sage_oracle(conv, ei, x, d_y)
    out, grads = _sage_run(conv, ei, x, d_y)
    _check_sage(out, grads, want, want_grads, rows)
    out2, grads2 = _sage_run(conv, ei, x, d_y)
    assert torch.equal(out, out2)
    for a, b in zip(grads, grads2):
        assert torch.equal(a, b), "two backward passes differ"


@pytest.mark.parametrize("in_dim,out_dim,n", [(32, 32, 1), (64, 40, 300), (128, 256, 5003), (256, 256, 5003),
                                              (256, 256, 99_133)])
def test_sage_conv_fallback_matches_fp64_and_fused(in_dim, out_dim, n, monkeypatch):
    """ops.SageMeanFn (etpgt_sage_mean_fwd / etpgt_sage_mean_bwd) + ops.linear, the route SAGEConv takes when the fused
    layer is not available; checked against fp64 and against the fused layer on the same inputs."""
    from etpgt_b200 import ops

    conv, ei, rows, x, d_y = _sage_inputs(in_dim, out_dim, n, seed=7)
    want, want_grads = _sage_oracle(conv, ei, x, d_y)
    fused, fused_grads = _sage_run(conv, ei, x, d_y)
    monkeypatch.setattr(ops, "PROJECTION_BACKEND", "library")
    assert not ops.sage_layer_supported(x.cuda(), in_dim, out_dim)
    calls = []
    real = ops.SageMeanFn.apply
    monkeypatch.setattr(ops.SageMeanFn, "apply", lambda *a: calls.append(1) or real(*a))
    out, grads = _sage_run(conv, ei, x, d_y)
    assert calls, "the fallback did not run the mean kernels"
    _check_sage(out, grads, want, want_grads, rows)
    assert rel_err(out, fused) < 2 * TOL
    for a, b in zip(grads, fused_grads):
        assert rel_err(a, b) < 2 * TOL
    out2, grads2 = _sage_run(conv, ei, x, d_y)
    for a, b in zip(grads, grads2):
        assert torch.equal(a, b), "two backward passes differ"


# ------------------------------------------------------------------------------ C. GATConv vs fp64


def _gat_case(in_dim, c, heads, concat, n, e_kind, seed):
    from etpgt_b200.nn import GATConv

    if e_kind == "empty":
        ei, rows = torch.empty(2, 0, dtype=torch.long), {"hub": None, "fan": None, "isolated": torch.arange(n),
                                                          "deg1": torch.empty(0, dtype=torch.long)}
    else:
        ei, rows = _layer_graph(n, seed)
    e = ei.size(1)
    torch.manual_seed(seed + in_dim + c)
    conv = GATConv(in_dim, c, heads=heads, concat=concat, dropout=0.0)
    g = torch.Generator().manual_seed(seed + 3)
    with torch.no_grad():
        conv.bias.copy_(torch.randn(conv.bias.shape, generator=g) * 0.1)
    x = torch.randn(n, in_dim, generator=g)
    mask_edges = (torch.rand(e, heads, generator=g) > 0.2).float() / 0.8
    mask_self = (torch.rand(n, heads, generator=g) > 0.2).float() / 0.8
    d_out = torch.randn(n, heads * c if concat else c, generator=g)
    return conv, ei, rows, x, mask_edges, mask_self, d_out


def _gat_oracle(conv, ei, x, mask_edges, mask_self, d_out):
    """oracle/conv_ref.gat_conv in fp64 on the device; its edge order is the kept edges, then one self loop per node."""
    from oracle import conv_ref

    dev = torch.device("cuda")
    keep = ei[0] != ei[1]
    oracle_mask = torch.cat([mask_edges[keep], mask_self]).double().to(dev)
    params = [p.detach().double().to(dev).requires_grad_(True)
              for p in (conv.lin.weight, conv.att_src, conv.att_dst, conv.bias)]
    x64 = x.double().to(dev).requires_grad_(True)
    want = conv_ref.gat_conv(x64, ei.to(dev), params[0], params[1], params[2], params[3], conv.heads, conv.concat, 0.2,
                             oracle_mask)
    want.backward(d_out.double().to(dev))
    return want.detach(), [x64.grad] + [p.grad for p in params]


def _gat_run(conv, ei, x, mask_edges, mask_self, d_out):
    conv = conv.cuda()
    for p in conv.parameters():
        p.grad = None
    xc = x.cuda().requires_grad_(True)
    out = conv(xc, ei.cuda(), mask_edges=mask_edges.cuda(), mask_self=mask_self.cuda())
    out.backward(d_out.cuda())
    torch.cuda.synchronize()
    return out.detach(), [xc.grad] + [p.grad for p in (conv.lin.weight, conv.att_src, conv.att_dst, conv.bias)]


def _check_gat(case, route, monkeypatch):
    conv, ei, rows, x, mask_edges, mask_self, d_out = case
    want, want_grads = _gat_oracle(conv, ei, x, mask_edges, mask_self, d_out)
    calls = []
    real = route.apply
    monkeypatch.setattr(route, "apply", lambda *a: calls.append(1) or real(*a))
    out, grads = _gat_run(conv, ei, x, mask_edges, mask_self, d_out)
    assert calls, f"{route.__name__} was not reached"
    assert out.shape == want.shape
    assert rel_err(out, want) < TOL, "forward"
    # analytically zero gradients (the attention vectors of an edgeless graph: a softmax over the one self loop) are
    # compared on the scale of the layer's largest parameter gradient, as test_gpu_models.check_case does
    scale = max(float(g.abs().max()) for g in want_grads[1:])
    assert rel_err(grads[0], want_grads[0], floor=1e-2 * float(want_grads[0].abs().max())) < 5 * TOL, "x"
    for name, got, ref in zip(("lin.weight", "att_src", "att_dst", "bias"), grads[1:], want_grads[1:]):
        assert rel_err(got, ref, floor=1e-2 * scale) < 5 * TOL, name
    _check_rows(out, want, rows, ("hub", "isolated", "deg1"), TOL)
    _check_rows(grads[0], want_grads[0], rows, ("hub", "fan", "isolated"), 5 * TOL)
    out2, grads2 = _gat_run(conv, ei, x, mask_edges, mask_self, d_out)
    assert torch.equal(out, out2)
    for a, b in zip(grads, grads2):
        assert torch.equal(a, b), "two backward passes differ"


@pytest.mark.parametrize("in_dim,c,heads", [(32, 32, 1), (64, 64, 4), (256, 256, 4), (1024, 128, 8)])
@pytest.mark.parametrize("n,e_kind", [(3001, "graph"), (77, "empty")])
def test_gat_conv_concat_matches_fp64(in_dim, c, heads, n, e_kind, monkeypatch):
    """GATConv(concat=True): linear + attention scalars, then ops.GatAggregateFn (etpgt_gat_fwd, and etpgt_gat_bwd with
    the [N, heads*C] d_agg), W = heads*C from 32 to 1,024 — the widths of create_gat(concat_heads=True).  The hub
    destination has 5,200 in-edges; the projection's weight gradient (K = 3,001 nodes) runs split-K."""
    from etpgt_b200 import ops

    _check_gat(_gat_case(in_dim, c, heads, True, n, e_kind, seed=11), ops.GatAggregateFn, monkeypatch)


@pytest.mark.parametrize("in_dim,c,heads,route", [(256, 256, 4, "GatLayerFn"), (64, 128, 8, "GatLayerFn"),
                                                  (64, 64, 4, "GatConvFn")])
@pytest.mark.parametrize("n,e_kind", [(20_011, "graph"), (77, "empty")])
def test_gat_conv_mean_at_batch_scale_matches_fp64(in_dim, c, heads, route, n, e_kind, monkeypatch):
    """GATConv(concat=False) through ops.GatLayerFn (scores from the input through the folded attention vectors, head
    mean in the edge kernel's epilogue) and ops.GatConvFn (separate head-mean pass, C = 64) at ~20k nodes with a hub of
    5,200 in-edges: the projection-gradient GEMM runs split-K together with the fold terms att (x) d_u."""
    from etpgt_b200 import ops

    _check_gat(_gat_case(in_dim, c, heads, False, n, e_kind, seed=13), getattr(ops, route), monkeypatch)


def test_gat_concat_unsupported_width_names_the_supported_widths():
    """heads*C = 2,048 is past the edge kernels' widths: the projection runs, then etpgt_gat_fwd refuses."""
    from etpgt_b200.nn import GATConv

    conv = GATConv(64, 256, heads=8, concat=True).cuda()
    x = torch.randn(10, 64, device="cuda")
    ei = torch.tensor([[0, 1, 2], [1, 2, 3]], device="cuda")
    with pytest.raises(RuntimeError, match=r"heads\*channels=2048.*32\.\.1024"):
        conv(x, ei)


# ------------------------------------------------------------------------------ D. whole models vs fp64


@pytest.fixture(scope="module")
def session_batch():
    """~4,096 sessions of a synthetic catalogue of 3,000 items built the way the training loop builds them: ~12k nodes,
    so every layer's weight gradient runs split-K."""
    from etpgt_b200 import data, synth

    d = synth.generate(num_sessions=6000, graph_sessions=5000, num_items=3000, clusters=60, seed=17)
    graph = data.ItemGraph(d.item_i, d.item_j, d.num_items)
    store = data.SessionStore(d.sess_ptr, d.sess_items)
    ids = np.arange(4096)
    batch = data.build_batch(graph, store, ids)
    negatives = data.sample_negatives(store, ids, d.num_items, 5, seed=2, step=0)
    assert batch.x.numel() > 1000 and batch.num_graphs == 4096
    return d.num_items, batch, negatives


def _randomize(model):
    g = torch.Generator().manual_seed(23)
    with torch.no_grad():
        for bn in model.batch_norms:
            for t, lo, hi in ((bn.weight, 0.5, 1.5), (bn.bias, -0.2, 0.2), (bn.running_mean, -0.1, 0.1),
                              (bn.running_var, 0.5, 1.5)):
                t.copy_(torch.rand(t.shape, generator=g) * (hi - lo) + lo)
        for conv in model.convs:
            if hasattr(conv, "bias") and conv.bias is not None:
                conv.bias.copy_(torch.randn(conv.bias.shape, generator=g) * 0.1)


KINK = 1e-5     # relative distance from a ReLU / leaky_relu kink within which fp32 and fp64 may take different branches


@pytest.mark.parametrize("kind", ["graphsage", "gat", "gat_concat"])
def test_baseline_model_at_batch_scale_matches_fp64(kind, session_batch, monkeypatch):
    """create_graphsage(I, 256, 256, 3) / create_gat(I, 256, 256, 3, 4) (/ concat_heads=True: widths 1,024 and a
    1,024-wide BatchNorm) in training mode against model_ref in fp64 on the model's own state.

    ReLU's derivative jumps at 0.  Over the ~3M activations of a layer a few lie within fp32 rounding of 0 (|y| ~ 1e-6
    of the largest), and fp32 and fp64 put them on different sides.  Each such element moves a weight gradient by one
    whole term of its sum over ~12k rows, ~1e-2 relative, while changing no output by more than its own |y|.  So the
    oracle takes the product's ReLU gates (the zero pattern of the product's layer outputs), and the test asserts that
    every element where they differ from the oracle's own is within KINK of 0.  GAT's leaky_relu has the same kink at
    logit 0, and there one flip moves the analytically small attention-vector gradients by several percent: the oracle
    takes the slope of the fp32 logit a_src[j] + a_dst[i] the edge kernels compare with 0 (their attention scalars,
    read from the autograd nodes), under the same assertion."""
    import torch.nn.functional as F

    import etpgt_b200.model.gat as gat_module
    import etpgt_b200.model.graphsage as sage_module
    from etpgt_b200 import ops
    from etpgt_b200.model import create_gat, create_graphsage
    from oracle import model_ref

    num_items, batch, negatives = session_batch
    torch.manual_seed(5)
    if kind == "graphsage":
        model = create_graphsage(num_items, 256, 256, 3, dropout=0.0)
    else:
        model = create_gat(num_items, 256, 256, 3, 4, dropout=0.0, concat_heads=kind == "gat_concat")
    _randomize(model)
    model = model.cuda().train()
    state = {k: v.detach().double().clone().requires_grad_(v.is_floating_point() and "running" not in k)
             if v.is_floating_point() else v.clone() for k, v in model.state_dict().items()}

    module = sage_module if kind == "graphsage" else gat_module
    relu_out = []
    real_bn_rows = module.batch_norm_rows

    def recording_bn_rows(*a, **k):
        y = real_bn_rows(*a, **k)
        if k.get("relu"):
            relu_out.append(y.detach())
        return y

    scalars = []     # (a_src, a_dst) [N, heads] of each GAT layer, in layer order

    def recording_layer(*a):
        out = real_layer(*a)
        scalars.append(tuple(t.detach() for t in out.grad_fn.saved_tensors[10:12]))   # GatLayerFn's a_src, a_dst
        return out

    def recording_aggregate(*a):
        scalars.append((a[1].detach(), a[2].detach()))
        return real_aggregate(*a)

    real_layer, real_aggregate = ops.GatLayerFn.apply, ops.GatAggregateFn.apply
    with monkeypatch.context() as m:
        m.setattr(module, "batch_norm_rows", recording_bn_rows)
        m.setattr(ops.GatLayerFn, "apply", recording_layer)
        m.setattr(ops.GatAggregateFn, "apply", recording_aggregate)
        sess = model(batch)
    loss = model.compute_loss(sess, batch.target_item, negatives)
    loss.backward()
    torch.cuda.synchronize()

    ei, n = batch.edge_index, batch.x.numel()
    keep, loops = ei[0] != ei[1], torch.arange(n, device=ei.device)
    src, dst = torch.cat([ei[0][keep], loops]), torch.cat([ei[1][keep], loops])   # the oracle's edge order
    real_bn, real_leaky = model_ref.batch_norm_rows, F.leaky_relu
    fwd = model_ref.graphsage_forward if kind == "graphsage" else model_ref.gat_forward
    kw = {"num_layers": 3} if kind == "graphsage" else {"num_convs": 3, "num_heads": 4,
                                                         "concat_heads": kind == "gat_concat"}

    def oracle(state, stats):
        """model_ref forward + BPR loss + backward on `state`, on the product's ReLU gates and logit branches."""
        gates, layer_scalars = iter(relu_out), iter(scalars)

        def product_gated_relu(y):
            gate = next(gates) > 0
            differ = (y > 0) != gate
            if bool(differ.any()):
                assert float(y.detach()[differ].abs().max()) <= KINK * float(y.detach().abs().max()), "ReLU gates"
            return y * gate.to(y.dtype)

        def product_branch_leaky(z, slope):
            a_src, a_dst = next(layer_scalars)
            positive = (a_src[src] + a_dst[dst]) > 0
            differ = (z > 0) != positive
            if bool(differ.any()):
                assert float(z.detach()[differ].abs().max()) <= KINK * float(z.detach().abs().max()), "logit branches"
            return torch.where(positive, z, slope * z)

        with monkeypatch.context() as m:
            m.setattr(model_ref, "batch_norm_rows", lambda *a, **k: stats.append(real_bn(*a, **k)) or stats[-1])
            m.setattr(torch, "relu", product_gated_relu)
            m.setattr(F, "leaky_relu", product_branch_leaky)
            want = fwd(state, batch.x, batch.edge_index, batch.batch, training=True, **kw)
        assert next(gates, None) is None and len(relu_out) == (3 if kind == "graphsage" else 2)
        assert next(layer_scalars, None) is None and len(scalars) == (0 if kind == "graphsage" else 3)
        want_loss = model_ref.bpr_loss(want, state["item_embedding.weight"], batch.target_item, negatives)
        want_loss.backward()
        return want, want_loss

    stats = []
    want, want_loss = oracle(state, stats)
    assert rel_err(sess, want) < TOL, "session embeddings"
    assert abs(loss.item() - want_loss.item()) < TOL * abs(want_loss.item()), (loss.item(), want_loss.item())

    grads = {k: v.grad for k, v in state.items() if v.is_floating_point() and v.grad is not None}
    named = dict(model.named_parameters())
    assert set(grads) == set(named)
    # a conv bias in front of BatchNorm has an analytically zero gradient: compared on the scale of the model's
    # largest gradient entry, as test_gpu_models.check_case does.  What remains of it is the rounding of a column sum
    # over all ~12k rows of BatchNorm's input gradient, which grows with the batch: at this size it can exceed that
    # floor, so these biases may also be as close to fp64 as the same oracle evaluated in fp32 (twice its error).
    scale = max(float(g.abs().max()) for g in grads.values())
    state32 = {k: v.detach().float().requires_grad_(v.requires_grad) if v.is_floating_point() else v
               for k, v in state.items()}
    oracle(state32, [])
    for name, ref in grads.items():
        assert named[name].grad is not None, name
        bound = 5 * TOL
        if name.startswith("convs.") and name.endswith("bias"):
            bound = max(bound, 2 * rel_err(state32[name].grad, ref, floor=1e-2 * scale))
        assert rel_err(named[name].grad, ref, floor=1e-2 * scale) < bound, name

    assert len(stats) == 3
    new_stats = {}
    for layer, (bn, ref) in enumerate(zip(model.batch_norms, stats)):
        assert rel_err(bn.running_mean, ref.running_mean) < TOL, f"running_mean {layer}"
        assert rel_err(bn.running_var, ref.running_var) < TOL, f"running_var {layer}"
        new_stats[f"batch_norms.{layer}.running_mean"] = ref.running_mean.detach()
        new_stats[f"batch_norms.{layer}.running_var"] = ref.running_var.detach()

    model.eval()
    with torch.no_grad():
        got_eval = model(batch)
        want_eval = fwd({**{k: v.detach() for k, v in state.items()}, **new_stats}, batch.x, batch.edge_index,
                        batch.batch, training=False, **kw)
    assert rel_err(got_eval, want_eval) < TOL, "eval forward"


# ------------------------------------------------------------------------------ E. supported widths


def test_sage_conv_unsupported_width_names_the_supported_set():
    from etpgt_b200.nn import SAGEConv

    conv = SAGEConv(72, 64).cuda()
    x = torch.randn(10, 72, device="cuda")
    ei = torch.tensor([[0, 1, 2], [1, 2, 3]], device="cuda")
    with pytest.raises(RuntimeError, match="32, 64, 128, 256"):
        conv(x, ei)


def test_graphsage_unsupported_hidden_width_names_the_supported_set():
    from etpgt_b200.model import create_graphsage

    model = create_graphsage(50, hidden_dim=100, dropout=0.0).cuda()

    class Batch:
        x = torch.tensor([3, 4, 5, 6], device="cuda")
        edge_index = torch.tensor([[0, 1, 2], [1, 2, 3]], device="cuda")
        batch = torch.tensor([0, 0, 1, 1], device="cuda")
        num_graphs = 2

    with pytest.raises(RuntimeError, match="32, 64, 128, 256"):
        model(Batch())
