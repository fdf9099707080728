"""CPU tests: the oracle restatement (oracle/model_ref.py, graph_ref.py, conv_ref.py) against the
golden vectors that oracle/make_golden.py produced from the unmodified reference classes, and
against the reference's own known-answer tests (tests/test_utils.py:62-93) and published
parameter counts (docs/EXPERIMENTS.md:85-88)."""

import numpy as np
import pytest
import torch

from golden_util import GOLDEN as GOLDEN_DIR, Golden, pick, rel_err
from oracle import graph_ref, model_ref

GT_CASES = ["gt_opt_dummy", "gt_opt_dummy_nope", "gt_opt_b32", "gt_opt_b32_dual", "gt_opt_directed",
            "gt_opt_readout_max", "gt_opt_readout_last", "gt_opt_readout_attention", "gt_ffn_dummy"]


def _gt_forward(g, dtype, training):
    state = g.group("state", None)
    state = {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in state.items()}
    cfg = g.cfg()
    return model_ref.graph_transformer_forward(
        state, g.tensor("x"), g.tensor("edge_index"), g.tensor("batch"),
        num_layers=cfg["num_layers"], num_heads=cfg["num_heads"],
        readout=str(g.raw.get("cfg_readout_type", "mean")), training=training,
        use_ffn="ffns.0.0.weight" in state)


@pytest.mark.parametrize("name", GT_CASES)
def test_graph_transformer_restatement_matches_reference(name):
    g = Golden(name)
    if "readout" in name:
        g.raw["cfg_readout_type"] = name.rsplit("_", 1)[1]
    assert rel_err(_gt_forward(g, torch.float64, False), g.raw["eval_out_f64"]) < 1e-10
    assert rel_err(_gt_forward(g, torch.float64, True), g.raw["train_out_f64"]) < 1e-10
    assert rel_err(_gt_forward(g, torch.float32, True), g.raw["train_out_f32"]) < 1e-4


@pytest.mark.parametrize("name,layers,heads", [("gat_dummy", 2, 2), ("gat_directed", 3, 4)])
def test_gat_restatement_matches_reference(name, layers, heads):
    g = Golden(name)
    state = g.group("state", torch.float64)
    convs = 1 + max(layers - 2, 0) + (1 if layers > 1 else 0)  # etpgt/model/gat.py:45-111
    for training, key in ((False, "eval_out_f64"), (True, "train_out_f64")):
        out = model_ref.gat_forward(state, g.tensor("x"), g.tensor("edge_index"), g.tensor("batch"),
                                    num_convs=convs, num_heads=heads, training=training)
        assert rel_err(out, g.raw[key]) < 1e-10


@pytest.mark.parametrize("name,layers", [("sage_dummy", 2), ("sage_directed", 3)])
def test_graphsage_restatement_matches_reference(name, layers):
    g = Golden(name)
    state = g.group("state", torch.float64)
    for training, key in ((False, "eval_out_f64"), (True, "train_out_f64")):
        out = model_ref.graphsage_forward(state, g.tensor("x"), g.tensor("edge_index"), g.tensor("batch"),
                                          num_layers=layers, training=training)
        assert rel_err(out, g.raw[key]) < 1e-10


def test_training_gradients_and_running_stats_match_reference():
    g = Golden("gt_opt_b32")
    state = {k: (v.double().requires_grad_(True) if v.is_floating_point() else v)
             for k, v in g.group("state").items()}
    cfg = g.cfg()
    sess, _, stats = model_ref.graph_transformer_forward(
        state, g.tensor("x"), g.tensor("edge_index"), g.tensor("batch"), num_layers=cfg["num_layers"],
        num_heads=cfg["num_heads"], training=True, return_nodes=True)
    loss = model_ref.bpr_loss(sess, state["item_embedding.weight"], g.tensor("target"), g.tensor("negatives"))
    assert abs(loss.item() - g.raw["loss_f64"].item()) < 1e-12
    loss.backward()
    for name, (want, index) in g.gradients().items():
        assert rel_err(pick(state[name].grad, index), want) < 1e-6, name
    for name, want in g.group("after").items():
        if name in stats:
            assert rel_err(stats[name], want) < 1e-6, name


def test_losses_match_reference():
    g = Golden("loss_readout_metrics")
    sess0, table0 = g.tensor("sess"), g.tensor("table")
    tgt, neg = g.tensor("target"), g.tensor("negatives")
    cases = {
        "bpr": lambda s, t: model_ref.bpr_loss(s, t, tgt, neg),
        "listwise": lambda s, t: model_ref.listwise_loss(s, t, tgt, neg, 0.5),
        "dual": lambda s, t: model_ref.dual_loss(s, t, tgt, neg, 0.7, 2.0)[0],
        "sampled_softmax": lambda s, t: model_ref.listwise_loss(s, t, tgt, neg, 1.0),
    }
    for kind, fn in cases.items():
        s, t = sess0.clone().requires_grad_(True), table0.clone().requires_grad_(True)
        loss = fn(s, t)
        loss.backward()
        assert abs(loss.item() - g.raw[f"{kind}/loss"].item()) < 1e-12, kind
        assert rel_err(s.grad, g.raw[f"{kind}/dsess"]) < 1e-10, kind
        assert rel_err(t.grad, g.raw[f"{kind}/dtable"]) < 1e-10, kind
    total, lw, bp = model_ref.dual_loss(sess0, table0, tgt, neg, 0.7, 2.0)
    assert np.allclose([total.item(), lw.item(), bp.item()], g.raw["dual/parts"], atol=1e-12)


def test_readouts_match_reference():
    g = Golden("loss_readout_metrics")
    x, bvec = g.tensor("ro/x"), g.tensor("ro/batch")
    for kind in ("mean", "max", "last", "attention"):
        out = model_ref.session_readout(x, bvec, 4, kind, g.tensor("ro/att_w"), g.tensor("ro/att_b"))
        assert rel_err(out, g.raw[f"ro/{kind}"]) < 1e-12, kind
    with pytest.raises(ValueError, match="Unknown readout type"):
        model_ref.session_readout(x, bvec, 4, "median")


def test_metrics_known_answers():
    # the reference's only known-answer tests: tests/test_utils.py:62-93
    g = Golden("loss_readout_metrics")
    preds, tg = g.tensor("met/preds"), g.tensor("met/targets")
    assert model_ref.recall_at_k(preds, tg, 5) == pytest.approx(2 / 3)
    assert model_ref.recall_at_k(preds, tg, 2) == pytest.approx(1 / 3)
    assert 0.4 < model_ref.ndcg_at_k(preds, tg, 5) < 0.5
    assert model_ref.recall_at_k(preds, tg, 5) == pytest.approx(g.raw["met/recall5"].item())
    assert model_ref.ndcg_at_k(preds, tg, 5) == pytest.approx(g.raw["met/ndcg5"].item(), abs=1e-7)


def test_published_parameter_counts():
    """docs/EXPERIMENTS.md:85-88 — 188 items, D=64, L=2, H=2: the structural pin of the PyG
    stand-in (4 biased Linears + bias-free beta; one bias-free GAT lin; SAGE lin_l/lin_r)."""
    from oracle import conv_ref  # noqa: F401  (puts the stand-in on sys.path)
    from torch_geometric.nn import GATConv, SAGEConv, TransformerConv

    count = lambda m: sum(p.numel() for p in m.parameters())  # noqa: E731
    emb, bn = 188 * 64, 2 * 64
    tconv = count(TransformerConv(64, 32, heads=2, beta=True))
    assert emb + 2 * (tconv + bn) == 45952
    ffn = 64 * 256 + 256 + 256 * 64 + 64
    assert emb + 2 * (tconv + bn + ffn) == 112128
    assert emb + 2 * (count(GATConv(64, 64, heads=2, concat=False)) + bn) == 29312
    assert emb + 2 * (count(SAGEConv(64, 64)) + bn) == 28800


def test_topk_ties_go_to_lower_id():
    scores = torch.tensor([[1.0, 3.0, 3.0, 2.0, 3.0], [0.0, 0.0, 0.0, 0.0, 0.0]])
    _, idx = model_ref.topk_lower_id(scores, 3)
    assert idx.tolist() == [[1, 2, 4], [0, 1, 2]]


# ------------------------------------------------------------------ integer oracle


def test_dataloader_restatement_is_bit_exact():
    g = Golden("dataloader")
    ptr = g.raw["sess_ptr"]
    sessions = [g.raw["sess_items"][ptr[i]:ptr[i + 1]] for i in range(len(ptr) - 1)]
    out = graph_ref.collate_sessions(sessions, g.raw["item_i"], g.raw["item_j"])
    assert np.array_equal(out["x"], g.raw["x"])
    assert np.array_equal(np.stack([out["edge_src"], out["edge_dst"]]), g.raw["edge_index"])
    assert np.array_equal(out["batch"], g.raw["batch"])
    assert np.array_equal(out["target"], g.raw["target"])
    # the reference's negatives obey the acceptance rule our sampler restates
    for s, items in enumerate(sessions):
        assert not set(g.raw["negatives"][s]) & set(items[-50:])
        assert g.raw["negatives"][s].min() >= 1


def test_philox_known_answers():
    # Random123 kat_vectors, philox4x32 10 rounds
    assert graph_ref.philox4x32_10((0, 0, 0, 0), (0, 0)) == (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)
    assert graph_ref.philox4x32_10((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2) == (
        0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)
    assert graph_ref.philox4x32_10((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0)) == (
        0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)


def test_negative_sampler_rule():
    items = np.arange(1, 40)
    neg = graph_ref.sample_negatives(seed=42, step=3, session_index=17, session_items=items, num_items=50, num_neg=64)
    assert neg.min() >= 40 and neg.max() < 50  # never a session item, never padding id 0
    again = graph_ref.sample_negatives(42, 3, 17, items, 50, 64)
    assert np.array_equal(neg, again)
    assert not np.array_equal(neg, graph_ref.sample_negatives(42, 4, 17, items, 50, 64))


def test_csr_from_coo_is_stable():
    src = np.array([2, 0, 1, 2, 0, 2, 1])
    dst = np.array([1, 1, 0, 1, 2, 0, 1])
    c = graph_ref.csr_from_coo(src, dst, 4)
    assert c["rowptr"].tolist() == [0, 2, 6, 7, 7]
    assert c["eperm"].tolist() == [2, 5, 0, 1, 3, 6, 4]
    assert c["col"].tolist() == [1, 2, 2, 0, 2, 1, 0]
    assert c["colptr"].tolist() == [0, 2, 4, 7, 7]
    assert c["cpos"].tolist() == [3, 6, 0, 5, 1, 2, 4]
    assert c["row"].tolist() == [1, 2, 0, 1, 0, 1, 1]


def test_co_event_graph_restatement_matches_reference_function():
    """oracle/graph_ref.co_event_graph vs the reference's build_co_event_graph
    (scripts/data/04_build_graph.py:25-127) run by oracle/make_golden.py: same edge set, counts and
    last timestamps; both count-descending (the reference's order inside equal counts is pandas'
    unstable quicksort, so ties are compared as sets)."""
    g = dict(np.load(GOLDEN_DIR / "co_event_graph.npz"))
    i, j, c, t = graph_ref.co_event_graph(g["sess_ptr"], g["sess_items"], g["timestamps"], int(g["window"]))
    assert len(i) == int(g["num_edges"]) == len(g["item_i"])
    want = {(int(a), int(b)): (int(cc), int(tt)) for a, b, cc, tt in zip(g["item_i"], g["item_j"], g["count"], g["last_ts"])}
    got = {(int(a), int(b)): (int(cc), int(tt)) for a, b, cc, tt in zip(i, j, c, t)}
    assert got == want
    assert (np.diff(c) <= 0).all() and (np.diff(g["count"]) <= 0).all()
    assert np.array_equal(c, g["count"])                       # the count column itself is identical
    assert len(set(i) | set(j)) == int(g["num_nodes"])
    # without timestamps the structure is unchanged
    i2, j2, c2, _ = graph_ref.co_event_graph(g["sess_ptr"], g["sess_items"], None, int(g["window"]))
    assert np.array_equal(i, i2) and np.array_equal(j, j2) and np.array_equal(c, c2)


def test_oracle_training_loop_matches_the_reference_trainer():
    """The CPU arm of bench.py (oracle/model_ref.py forward + BPR + torch.optim.AdamW, bench.py::oracle_training_steps)
    restates the reference's training loop: on the batches of tests/golden/trainer_loop.npz — produced by the
    reference's own `Trainer.train()` (oracle/make_golden.py::trainer_case) — the same three epochs give the
    reference's epoch losses, Recall@k / NDCG@k and final weights."""
    from golden_util import Golden, rel_err
    from oracle import model_ref

    g = Golden("trainer_loop")
    state = {k: v.clone() for k, v in g.group("bpr_init").items()}
    state["laplacian_pe._cached_pe"] = g.tensor("pe")
    params = [k for k, v in state.items() if v.is_floating_point() and "running" not in k and "_cached_pe" not in k]
    for k in params:
        state[k].requires_grad_(True)
    opt = torch.optim.AdamW([state[k] for k in params], lr=1e-3, weight_decay=1e-5)

    def batch(prefix):
        return {name: g.tensor(f"{prefix}/{name}") for name in ("x", "edge_index", "batch", "target", "negatives")}

    train = [batch(f"train{b}") for b in range(int(g.raw["n_train_batches"]))]
    val = [batch(f"val{b}") for b in range(int(g.raw["n_val_batches"]))]
    for epoch in range(3):
        total = 0.0
        for b in train:
            sess, _, stats = model_ref.graph_transformer_forward(state, b["x"], b["edge_index"], b["batch"], num_layers=2,
                                                                 num_heads=2, training=True, return_nodes=True)
            loss = model_ref.bpr_loss(sess, state["item_embedding.weight"], b["target"],
                                      b["negatives"].view(b["target"].numel(), -1))
            opt.zero_grad()
            loss.backward()
            opt.step()
            total += loss.item()
            state.update({k: v.detach() for k, v in stats.items()})      # BatchNorm running statistics
        assert abs(total / len(train) - g.raw["bpr_train_loss"][epoch]) <= 1e-5 * abs(g.raw["bpr_train_loss"][epoch])
        with torch.no_grad():
            tops, targets = [], []
            for b in val:
                sess = model_ref.graph_transformer_forward(state, b["x"], b["edge_index"], b["batch"], num_layers=2,
                                                           num_heads=2, training=False)
                tops.append(model_ref.predict(sess, state["item_embedding.weight"], 20)[1])
                targets.append(b["target"])
            top, tgt = torch.cat(tops), torch.cat(targets)
            for k in (10, 20):
                assert abs(model_ref.recall_at_k(top[:, :k], tgt, k) - g.raw[f"bpr_recall@{k}"][epoch]) < 1e-9
                assert abs(model_ref.ndcg_at_k(top[:, :k], tgt, k) - g.raw[f"bpr_ndcg@{k}"][epoch]) < 1e-6
    # Parameters whose gradient is analytically zero (the key bias cancels in the per-destination softmax, the value /
    # skip biases in the BatchNorm that follows) receive rounding noise as gradient, which Adam turns into steps of
    # +-lr: they drift differently in any two implementations and are left out of the weight comparison.
    noise_driven = ("lin_key.bias", "lin_value.bias", "lin_skip.bias")
    for k, want in g.group("bpr_final").items():
        if want.is_floating_point() and not k.endswith(noise_driven):
            assert rel_err(state[k].detach(), want, floor=1e-6) < 1e-4, k


def test_laplacian_pe_host_path_against_the_reference_function():
    """tests/golden/laplacian_pe.npz holds outputs of the reference's `compute_laplacian_pe` /
    `LaplacianPECached` (etpgt/encodings/laplacian_pe.py:19-199; oracle/make_golden.py::laplacian_pe_case).
    On a SYMMETRIC edge list the result is well defined and the package's host path (`method="scipy"`) reproduces
    it to the solver's tolerance (two calls of the reference itself agree to ~1e-5).  On the directed list that
    scripts/train/train_baseline.py:234-243 passes (item_i <= item_j) the reference does not reproduce ITSELF: its
    two recorded calls on the same input differ by the size of the entries — there is nothing to pin, only the
    call sequence is kept.  The cached-table module (gather + projection) is pinned exactly."""
    from golden_util import Golden

    from etpgt_b200.encodings.laplacian_pe import LaplacianPECached, compute_laplacian_pe

    g = Golden("laplacian_pe")
    n, k = int(g.raw["num_nodes"]), int(g.raw["k"])
    ref, ref_again = g.tensor("pe_symmetric"), g.tensor("pe_symmetric_again")
    self_agreement = float((ref - ref_again).abs().max())
    assert self_agreement < 1e-3
    got = compute_laplacian_pe(g.tensor("symmetric"), n, k=k)
    assert got.shape == (n, k) and got.dtype == torch.float32 and bool((got >= 0).all())
    assert float((got - ref).abs().max()) < max(10 * self_agreement, 2e-4)
    # the reference's own run-to-run spread on its directed input is of the order of the values themselves
    d0, d1 = g.tensor("pe_directed"), g.tensor("pe_directed_again")
    assert float((d0 - d1).abs().max()) > 0.1 * float(d0.abs().max())
    ours = compute_laplacian_pe(g.tensor("directed"), n, k=k)        # same call sequence: runs, same shape / sign rule
    assert ours.shape == (n, k) and bool((ours >= 0).all())
    # LaplacianPECached.forward / project on the reference's cached table and projection weights
    module = LaplacianPECached(k=k, embedding_dim=16)
    module._cached_pe = g.tensor("module_cached_pe")
    with torch.no_grad():
        module.projection.weight.copy_(g.tensor("module_weight"))
        module.projection.bias.copy_(g.tensor("module_bias"))
    ids = g.tensor("module_ids")
    assert torch.allclose(module(ids), g.tensor("module_forward"), atol=1e-6)
    assert torch.allclose(module.project(module._cached_pe[ids]), g.tensor("module_project"), atol=1e-6)
