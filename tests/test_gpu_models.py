"""GPU parity tests at the model boundary: the etpgt_b200 modules, loaded with the reference's
state dict, against the golden vectors produced by the unmodified reference classes
(tests/golden, oracle/make_golden.py): eval output, training output, loss, every parameter
gradient and the BatchNorm running statistics."""

import pytest
import torch

from golden_util import Golden, pick, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-4


class Batch:
    def __init__(self, g, with_graphs=True):
        self.x = g.tensor("x").cuda()
        self.edge_index = g.tensor("edge_index").cuda()
        self.batch = g.tensor("batch").cuda()
        if with_graphs:
            self.num_graphs = int(self.batch.max().item()) + 1


def build(g, factory, **extra):
    cfg = {**g.cfg(), **extra}
    model = factory(**cfg)
    state = g.group("state")
    pe = state.pop("laplacian_pe._cached_pe", None)
    model.load_state_dict(state, strict=False)
    model = model.cuda()
    if pe is not None:
        model.laplacian_pe._cached_pe = pe.cuda()
    return model


def oracle_gradients(g, loss_kind):
    """fp64 parameter gradients of the oracle (oracle/model_ref.py) on the fixture's state and batch.  A compact
    fixture keeps a sample of the reference's large gradients; the oracle, pinned to that sample and to the
    reference's outputs and loss in tests/test_oracle.py, stands in for the other entries."""
    from oracle import model_ref

    assert loss_kind == "bpr", loss_kind
    state = {k: (v.double().requires_grad_(True) if v.is_floating_point() else v) for k, v in g.group("state").items()}
    cfg = g.cfg()
    sess = model_ref.graph_transformer_forward(state, g.tensor("x"), g.tensor("edge_index"), g.tensor("batch"),
                                               num_layers=cfg["num_layers"], num_heads=cfg["num_heads"], training=True)
    model_ref.bpr_loss(sess, state["item_embedding.weight"], g.tensor("target"), g.tensor("negatives")).backward()
    return {k: v.grad for k, v in state.items() if v.is_floating_point() and v.grad is not None}


def check_case(name, factory, loss_kind, **extra):
    from etpgt_b200.train.losses import create_loss_function

    g = Golden(name)
    model = build(g, factory, **extra)
    batch = Batch(g)
    model.eval()
    with torch.no_grad():
        assert rel_err(model(batch), g.raw["eval_out_f64"]) < TOL, "eval forward"
    model.train()
    sess = model(batch)
    assert rel_err(sess, g.raw["train_out_f64"]) < TOL, "train forward"
    res = create_loss_function(loss_kind)(sess, g.tensor("target").cuda(), g.tensor("negatives").cuda(),
                                          model.item_embedding)
    loss = res[0] if isinstance(res, tuple) else res
    want = g.raw["loss_f64"].item()
    assert abs(loss.item() - want) < TOL * abs(want), "loss"
    loss.backward()
    grads = g.gradients()
    full = oracle_gradients(g, loss_kind) if any(index is not None for _, index in grads.values()) else {}
    checked = 0
    # Some gradients are analytically zero (a bias in front of BatchNorm, the key bias under the
    # per-destination softmax): they are compared on the scale of the model's largest gradient
    # entry instead of their own rounding noise.
    scale = max(want.abs().max().item() for want, _ in grads.values())
    for pname, p in model.named_parameters():
        if pname in grads:
            want, index = grads[pname]
            assert p.grad is not None, pname
            assert rel_err(pick(p.grad, index), want, floor=1e-2 * scale) < 5 * TOL, pname
            if index is not None:
                assert rel_err(p.grad, full[pname], floor=1e-2 * scale) < 5 * TOL, pname
            checked += 1
    assert checked == len(grads)
    for bname, want_b in g.group("after").items():
        got = dict(model.named_buffers())[bname]
        assert rel_err(got, want_b) < TOL, bname
    return model, batch


@pytest.mark.parametrize("name,loss", [("gt_opt_dummy", "bpr"), ("gt_opt_dummy_nope", "listwise"),
                                       ("gt_opt_b32", "bpr"), ("gt_opt_b32_dual", "dual"),
                                       ("gt_opt_directed", "listwise"), ("gt_ffn_dummy", "dual")])
def test_graph_transformer_matches_reference(name, loss):
    from etpgt_b200.model import create_graph_transformer, create_graph_transformer_optimized

    factory = create_graph_transformer if "ffn" in name else create_graph_transformer_optimized
    check_case(name, factory, loss)


@pytest.mark.parametrize("kind", ["max", "last", "attention"])
def test_graph_transformer_readout_variants(kind):
    from etpgt_b200.model import create_graph_transformer_optimized

    check_case(f"gt_opt_readout_{kind}", create_graph_transformer_optimized, "bpr", readout_type=kind)


@pytest.mark.parametrize("name,loss", [("gat_dummy", "listwise"), ("gat_directed", "bpr")])
def test_gat_matches_reference(name, loss):
    from etpgt_b200.model import create_gat

    check_case(name, create_gat, loss)


@pytest.mark.parametrize("name,loss", [("sage_dummy", "listwise"), ("sage_directed", "bpr")])
def test_graphsage_matches_reference(name, loss):
    from etpgt_b200.model import create_graphsage

    check_case(name, create_graphsage, loss)


def test_reference_api_contract_on_gpu():
    """The reference's own acceptance tests (tests/test_models.py:46-57,221-226), on the B200 path."""
    from etpgt_b200.model import create_graph_transformer_optimized

    g = Golden("gt_opt_dummy")
    model = build(g, create_graph_transformer_optimized)
    batch = Batch(g, with_graphs=False)   # bare Data-like object: num_sessions comes from batch.max()
    out = model(batch)
    assert out.shape == (2, 32) and torch.isfinite(out).all()
    out.sum().backward()
    assert model.item_embedding.weight.grad is not None and torch.isfinite(model.item_embedding.weight.grad).all()
    top = model.predict(out.detach(), k=10)
    assert top.shape == (2, 10) and top.dtype == torch.long
    # explicit per-node PE overrides the cached table (graph_transformer.py:144-150)
    batch.laplacian_pe = model.laplacian_pe._cached_pe[batch.x]
    assert rel_err(model(batch), out.detach()) < 1e-6
    # predict() agrees with the fp32 reference formula
    scores = out.detach() @ model.item_embedding.weight.detach().t()
    assert torch.equal(top, torch.sort(scores, dim=1, descending=True, stable=True).indices[:, :10])


def test_training_dropout_is_applied_and_finite():
    from etpgt_b200.model import create_graph_transformer_optimized

    g = Golden("gt_opt_b32")
    model = build(g, create_graph_transformer_optimized, dropout=0.1)
    batch = Batch(g)
    model.train()
    torch.manual_seed(0)
    a = model(batch)
    b = model(batch)
    assert torch.isfinite(a).all() and not torch.equal(a, b)   # masks differ between calls
    loss = model.compute_loss(a, g.tensor("target").cuda(), g.tensor("negatives").cuda())
    loss.backward()
    assert all(torch.isfinite(p.grad).all() for p in model.parameters() if p.grad is not None)


def test_fused_layer_equals_unfused_layer_bit_for_bit():
    """ops.TransformerLayer (conv + BN + residual + dropout in one autograd node, split hand-over between
    layers, residual gradient accumulated by the GEMM's TMA reduce-add) against the same kernels driven
    as separate autograd nodes: identical outputs, gradients and running statistics (p = 0)."""
    import numpy as np

    import etpgt_b200.ops as ops
    from etpgt_b200 import data, synth
    from etpgt_b200.model import create_graph_transformer_optimized

    d = synth.generate(num_sessions=900, graph_sessions=700, num_items=500, clusters=16, seed=5)
    graph = data.ItemGraph(d.item_i, d.item_j, d.num_items)
    store = data.SessionStore(d.sess_ptr, d.sess_items)
    ids = np.arange(300)
    results = []
    for fused in (True, False):
        ops.FUSED_LAYER = fused
        try:
            torch.manual_seed(3)
            model = create_graph_transformer_optimized(d.num_items, 256, 256, dropout=0.0).cuda()
            model.laplacian_pe._cached_pe = torch.randn(d.num_items, 16, generator=torch.Generator().manual_seed(7)).abs().cuda()
            model.train()
            batch = data.build_batch(graph, store, ids, 50, True, True)
            neg = data.sample_negatives(store, ids, d.num_items, 5, seed=3, step=0)
            out = model(batch)
            model.compute_loss(out, batch.target_item, neg).backward()
            results.append((out.detach().clone(), {k: p.grad.clone() for k, p in model.named_parameters()},
                            {k: v.clone() for k, v in model.state_dict().items() if "running" in k}))
        finally:
            ops.FUSED_LAYER = True
    (o1, g1, r1), (o2, g2, r2) = results
    assert torch.equal(o1, o2)
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k
    for k in r1:
        assert torch.equal(r1[k], r2[k]), k


def test_fused_layer_training_mode_dropout_statistics():
    """With dropout 0.5 the fused layer zeroes about half of every layer's outputs, is reproducible under
    torch.manual_seed, and still back-propagates finite gradients to every parameter."""
    import numpy as np

    from etpgt_b200 import data, synth
    from etpgt_b200.model import create_graph_transformer_optimized

    d = synth.generate(num_sessions=900, graph_sessions=700, num_items=500, clusters=16, seed=5)
    graph = data.ItemGraph(d.item_i, d.item_j, d.num_items)
    store = data.SessionStore(d.sess_ptr, d.sess_items)
    batch = data.build_batch(graph, store, np.arange(400), 50, True, True)
    torch.manual_seed(3)
    model = create_graph_transformer_optimized(d.num_items, 256, 256, dropout=0.5, readout_type="last").cuda()
    model.laplacian_pe._cached_pe = torch.randn(d.num_items, 16).abs().cuda()
    model.train()
    torch.manual_seed(11)
    a = model(batch)
    torch.manual_seed(11)
    b = model(batch)
    assert torch.equal(a, b)
    zero_frac = (a == 0).float().mean().item()          # "last" readout = rows of the last layer's output
    assert 0.45 < zero_frac < 0.55
    a.square().mean().backward()
    for name, p in model.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), name
    model.eval()
    assert (model(batch) == 0).float().mean().item() < 0.01


@pytest.mark.parametrize("n,e,in_dim,c,heads", [(300, 1500, 64, 128, 4), (257, 900, 256, 256, 4), (64, 0, 32, 128, 2),
                                                (200, 800, 64, 64, 4)])
def test_gat_conv_layer_with_wide_heads_matches_fp64(n, e, in_dim, c, heads):
    """GATConv(concat=False) as one layer at the reference's width (heads*C up to 1024): for C a multiple of 128 the
    head mean + bias come out of the edge kernel's epilogue (etpgt_gat_fwd_mean) and the backward kernels expand
    d_out / heads in registers (etpgt_gat_bwd_mean); the last case takes the separate head-mean pass in forward.
    Oracle: oracle/conv_ref.gat_conv in fp64 (output and every gradient), with an injected attention-dropout mask."""
    from etpgt_b200.nn import GATConv
    from oracle import conv_ref

    g = torch.Generator().manual_seed(n + c)
    x = torch.randn(n, in_dim, generator=g, dtype=torch.float64)
    src = torch.randint(0, n, (e,), generator=g)
    dst = torch.randint(0, n, (e,), generator=g)
    if e > 10:
        dst[:5] = src[:5]                      # existing self loops are dropped, one per node is appended
    ei = torch.stack([src, dst])
    conv = GATConv(in_dim, c, heads=heads, concat=False, dropout=0.0)
    with torch.no_grad():
        conv.bias.copy_(torch.randn(c, generator=g) * 0.1)
    keep = src != dst
    n_kept = int(keep.sum())
    mask_edges = (torch.rand(e, heads, generator=g) > 0.2).double() / 0.8
    mask_self = (torch.rand(n, heads, generator=g) > 0.2).double() / 0.8
    # the oracle's edge order: kept edges, then the appended self loops
    oracle_mask = torch.cat([mask_edges[keep], mask_self])
    assert oracle_mask.size(0) == n_kept + n
    params64 = [p.detach().double().clone().requires_grad_(True) for p in (conv.lin.weight, conv.att_src, conv.att_dst,
                                                                          conv.bias)]
    x64 = x.clone().requires_grad_(True)
    want = conv_ref.gat_conv(x64, ei, params64[0], params64[1], params64[2], params64[3], heads, False, 0.2, oracle_mask)
    d_out = torch.randn(n, c, generator=g, dtype=torch.float64)
    want.backward(d_out)
    conv = conv.cuda()
    xc = x.float().cuda().requires_grad_(True)
    got = conv(xc, ei.cuda(), mask_edges=mask_edges.float().cuda(), mask_self=mask_self.float().cuda())
    got.backward(d_out.float().cuda())
    torch.cuda.synchronize()
    assert got.shape == (n, c)
    assert rel_err(got, want) < TOL
    # analytically zero gradients (the attention vectors of an edgeless graph: a softmax over the one self loop)
    # are compared on the scale of the layer's largest gradient, as in check_case
    scale = max(float(q.grad.abs().max()) for q in params64)
    assert rel_err(xc.grad, x64.grad, floor=1e-2 * float(x64.grad.abs().max())) < 5 * TOL
    for p, q in zip((conv.lin.weight, conv.att_src, conv.att_dst, conv.bias), params64):
        assert rel_err(p.grad, q.grad, floor=1e-2 * scale) < 5 * TOL
