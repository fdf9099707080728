"""Full-catalogue softmax cross-entropy (csrc/softmax_tc.cu, ops.full_softmax_loss, train.losses.FullSoftmaxLoss):
the kernels against an fp64 torch recomputation chunked over rows, the autograd op inside a model against
F.cross_entropy in fp64, the Trainer on the per-operator path, and the host-side checks.  Errors are
max|got - want| / max|want| unless stated otherwise."""

import numpy as np
import pytest
import torch

from softmax_loss_util import err, grads, model_and_batch

TOL = 1e-4


# ------------------------------------------------------------------------------ CPU: the boundary


def test_library_exports_and_header_declares_the_entry_points():
    import ctypes
    from pathlib import Path

    from etpgt_b200 import _lib

    names = ("etpgt_full_softmax_workspace_bytes", "etpgt_full_softmax_fwd", "etpgt_full_softmax_bwd")
    header = (Path(__file__).resolve().parents[1] / "include" / "etpgt_b200.h").read_text()
    for name in names:
        assert f"{name}(" in header
        assert name in _lib.exported_symbols()
    if _lib.lib_path().exists():
        handle = ctypes.CDLL(str(_lib.lib_path()))
        for name in names:
            assert hasattr(handle, name)


def test_create_loss_function_full_softmax():
    from etpgt_b200.train.losses import FullSoftmaxLoss, ListwiseLoss, create_loss_function

    loss = create_loss_function("full_softmax", temperature=0.5)
    assert isinstance(loss, FullSoftmaxLoss)
    assert loss.temperature == 0.5
    assert create_loss_function("full_softmax").temperature == 1.0
    # the step driver's listwise mode is chosen by isinstance(ListwiseLoss)
    assert not isinstance(loss, ListwiseLoss)


def test_cpu_tensors_are_rejected():
    from etpgt_b200 import ops

    with pytest.raises(RuntimeError, match="CUDA"):
        ops.full_softmax_loss(torch.randn(4, 64), torch.randn(10, 64), torch.tensor([1, 2, 3, 4]))


# ------------------------------------------------------------------------------ GPU helpers


def _run(sess, table, targets, temperature=1.0, total=None, padding_idx=0, d_table=None, d_loss=1.0):
    """One forward and one backward through the C ABI: (loss, lse, d_sess, d_table)."""
    from etpgt_b200 import _lib
    from etpgt_b200._lib import ptr

    b, dim = sess.shape
    items = table.shape[0]
    dev = sess.device
    lse = torch.empty(b, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    ws = _lib.workspace(_lib.size("etpgt_full_softmax_workspace_bytes", b, items, dim), dev)
    tot = float(total) if total else 0.0
    _lib.call("etpgt_full_softmax_fwd", ptr(sess), ptr(table), ptr(targets), b, items, dim, float(temperature), tot,
              padding_idx, ptr(lse), ptr(loss), ptr(ws), ws.numel(), _lib.stream())
    dl = torch.tensor([d_loss], dtype=torch.float32, device=dev)
    d_sess = torch.empty_like(sess)
    d_table = torch.zeros_like(table) if d_table is None else d_table
    _lib.call("etpgt_full_softmax_bwd", ptr(sess), ptr(table), ptr(targets), ptr(lse), ptr(dl), b, items, dim,
              float(temperature), tot, padding_idx, ptr(d_sess), ptr(d_table), ptr(ws), ws.numel(), _lib.stream())
    torch.cuda.synchronize()
    return loss[0], lse, d_sess, d_table


def _reference(sess, table, targets, temperature=1.0, total=None, padding_idx=0, d_loss=1.0, rows_only=None):
    """fp64: (loss, lse [B], d_sess [B, D], d_table [I, D]), chunked over rows (at most ~2 GB of logits at once).
    rows_only: compute d_sess for these rows only (d_table and lse still need every row)."""
    s, e = sess.double(), table.double()
    t = targets.long()
    b, items = s.shape[0], e.shape[0]
    total = float(total) if total else float(b)
    scale = d_loss / (temperature * total)
    chunk = max(1, min(b, (2 << 30) // (8 * items * 2)))
    lse = torch.empty(b, dtype=torch.float64, device=s.device)
    d_sess = torch.zeros_like(s)
    d_table = torch.zeros_like(e)
    loss = 0.0
    for r0 in range(0, b, chunk):
        r1 = min(b, r0 + chunk)
        z = s[r0:r1] @ e.T / temperature
        if padding_idx >= 0:
            z[:, padding_idx] = -float("inf")
        l = torch.logsumexp(z, dim=1)
        lse[r0:r1] = l
        ar = torch.arange(r1 - r0, device=s.device)
        loss += float((l - z[ar, t[r0:r1]]).sum())
        g = torch.exp(z - l[:, None])
        g[ar, t[r0:r1]] -= 1.0
        g *= scale
        d_table += g.T @ s[r0:r1]
        if rows_only is None:
            d_sess[r0:r1] = g @ e
        else:
            sel = rows_only[(rows_only >= r0) & (rows_only < r1)]
            if sel.numel():
                d_sess[sel] = g[sel - r0] @ e
        del z, g
    if padding_idx >= 0:
        d_table[padding_idx] = 0
    return loss * d_loss / total, lse, d_sess, d_table


def _inputs(b, items, dim, seed, scale=0.3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    sess = torch.randn(b, dim, device="cuda", generator=g) * scale
    table = torch.randn(items, dim, device="cuda", generator=g) * scale
    targets = torch.randint(1, items, (b,), device="cuda", generator=g)
    return sess, table, targets


def _check(sess, table, targets, temperature=1.0, total=None, padding_idx=0, tol=TOL):
    got = _run(sess, table, targets, temperature, total, padding_idx)
    want = _reference(sess, table, targets, temperature, total, padding_idx)
    errs = {name: err(g, w) for name, g, w in zip(("loss", "lse", "d_sess", "d_table"), got, want)}
    assert all(v <= tol for v in errs.values()), errs
    return got


# ------------------------------------------------------------------------------ GPU: kernels against fp64


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [64, 256])
@pytest.mark.parametrize("items", [2, 1000, 82174])
@pytest.mark.parametrize("batch", [1, 37, 128, 1000, 4096])
def test_matches_fp64_on_the_grid(batch, items, dim):
    sess, table, targets = _inputs(batch, items, dim, seed=batch * 7 + items + dim)
    if items == 2:
        targets.fill_(1)             # id 0 is the padding column: with two items the target is id 1
    for temperature in (1.0, 0.5):
        for total in (None, 3 * batch + 5):
            _check(sess, table, targets, temperature, total)


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [128, 192])
def test_other_supported_dims(dim):
    sess, table, targets = _inputs(300, 5000, dim, seed=dim)
    _check(sess, table, targets, 0.7, None)


@pytest.mark.gpu
def test_large_logits_exercise_the_online_max():
    # logits of magnitude ~80: exp overflows fp32 without the running max
    g = torch.Generator(device="cuda").manual_seed(11)
    sess = torch.randn(777, 256, device="cuda", generator=g)
    table = torch.randn(20000, 256, device="cuda", generator=g)
    table *= 80.0 / float((sess[:64] @ table.T).abs().max())
    targets = torch.randint(1, 20000, (777,), device="cuda", generator=g)
    loss, lse, d_sess, d_table = _check(sess, table, targets)
    assert float(lse.abs().max()) > 60
    # the same with the sign flipped: the maxima now sit at the other end
    _check(-sess, table, targets)


@pytest.mark.gpu
def test_all_equal_logits():
    b, items, dim = 300, 3000, 64
    sess = torch.full((b, dim), 0.25, device="cuda")
    table = torch.full((items, dim), 0.5, device="cuda")
    targets = torch.randint(1, items, (b,), device="cuda")
    loss, lse, d_sess, d_table = _run(sess, table, targets)
    w_loss, w_lse, _, w_dt = _reference(sess, table, targets)
    assert err(loss, w_loss) <= TOL and err(lse, w_lse) <= TOL and err(d_table, w_dt) <= TOL
    want = np.log(items - 1) + 0.0                     # every logit equal: lse - z_t = log(I - 1)
    assert abs(float(loss) - want) <= 1e-5 * want
    # dS = mean_j E_j - E_t = 0 exactly when every row of E is the same: there is no scale to be relative to, so
    # the rounding left over is measured against one term of the sum, |E| / B
    assert float(d_sess.abs().max()) <= TOL * 0.5 / b


@pytest.mark.gpu
def test_targets_at_edges_tile_boundaries_and_duplicates():
    items = 1000
    edge = [1, items - 1, 127, 128, 129, 255, 256, 511, 512, 767, 768, 895, 896, 999]
    sess, table, _ = _inputs(2 * len(edge) + 100, items, 256, seed=3)
    targets = torch.tensor(edge + edge + [5] * 100, device="cuda")     # duplicates across rows
    _check(sess, table, targets, 0.5, None)


@pytest.mark.gpu
def test_padding_column_and_row():
    sess, table, targets = _inputs(500, 1000, 64, seed=4)
    _, _, _, d_table = _check(sess, table, targets, padding_idx=0)
    assert torch.count_nonzero(d_table[0]) == 0
    # a padding id inside the table (not row 0) is left out the same way (a target must not be the padding id)
    targets[targets == 700] = 701
    _, _, _, d_table = _check(sess, table, targets, padding_idx=700)
    assert torch.count_nonzero(d_table[700]) == 0
    # no padding: column 0 takes part, row 0 receives gradient, targets may be 0
    targets[:50] = 0
    _, _, _, d_table = _check(sess, table, targets, padding_idx=-1)
    assert torch.count_nonzero(d_table[0]) == table.shape[1]


@pytest.mark.gpu
def test_d_table_accumulates_onto_existing_values():
    sess, table, targets = _inputs(1000, 82174, 256, seed=5)
    base = torch.randn_like(table) * 1e-3
    base[0] = 7.0
    _, _, _, d_table = _run(sess, table, targets, d_table=base.clone())
    want = _reference(sess, table, targets)[3] + base.double()
    assert err(d_table - base, want - base.double()) <= TOL
    assert torch.all(d_table[0] == 7.0)                 # the padding row is left untouched


@pytest.mark.gpu
def test_upstream_gradient_scales_the_backward():
    sess, table, targets = _inputs(200, 3000, 64, seed=6)
    got = _run(sess, table, targets, d_loss=-2.5)
    want = _reference(sess, table, targets, d_loss=-2.5)
    assert err(got[2], want[2]) <= TOL and err(got[3], want[3]) <= TOL


@pytest.mark.gpu
@pytest.mark.parametrize("batch,items", [(4096, 82174), (1000, 1000)])
def test_bit_reproducible(batch, items):
    sess, table, targets = _inputs(batch, items, 256, seed=8)
    a = _run(sess, table, targets)
    b = _run(sess, table, targets)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_full_size():
    """B = 32,768 sessions x I = 82,174 items x D = 256: the loss and lse, and sampled rows of both gradients."""
    b, items, dim = 32768, 82174, 256
    sess, table, targets = _inputs(b, items, dim, seed=9)
    loss, lse, d_sess, d_table = _run(sess, table, targets)
    rows = torch.randperm(b, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))[:512]
    w_loss, w_lse, w_ds, w_dt = _reference(sess, table, targets, rows_only=rows)
    assert err(loss, torch.tensor(w_loss)) <= TOL
    assert err(lse, w_lse) <= TOL
    assert err(d_sess[rows], w_ds[rows]) <= TOL
    item_rows = torch.randperm(items, device="cuda")[:2048]
    assert err(d_table[item_rows], w_dt[item_rows]) <= TOL


@pytest.mark.gpu
def test_unsupported_dim_names_the_supported_set():
    from etpgt_b200 import ops

    sess = torch.randn(8, 96, device="cuda")
    table = torch.randn(50, 96, device="cuda")
    with pytest.raises(RuntimeError, match="64, 128, 192, 256"):
        ops.full_softmax_loss(sess, table, torch.ones(8, dtype=torch.long, device="cuda"))


@pytest.mark.gpu
def test_bad_targets_shape_is_rejected():
    from etpgt_b200 import ops

    sess, table, _ = _inputs(8, 50, 64, seed=1)
    with pytest.raises(RuntimeError, match="target_items"):
        ops.full_softmax_loss(sess, table, torch.ones(7, dtype=torch.long, device="cuda"))


# ------------------------------------------------------------------------------ GPU: autograd and model level


@pytest.mark.gpu
@pytest.mark.parametrize("opt_kind", ["torch", "etpgt"])
def test_model_gradients_match_fp64_cross_entropy(opt_kind):
    import torch.nn.functional as F

    from etpgt_b200 import ops, optim

    temperature = 0.5
    model, batch, _ = model_and_batch()
    model.train()
    table = model.item_embedding.weight
    if opt_kind == "torch":
        opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    else:
        opt = optim.AdamW(model.parameters(), lr=1e-3, sink_bytes=table.numel() * 4)
    # ours
    opt.zero_grad()
    loss = ops.full_softmax_loss(model(batch), model.item_embedding, batch.target_item, temperature=temperature)
    loss.backward()
    if opt_kind == "etpgt":
        assert optim.grad_sink_for(table) is table.grad        # the table gradient went into the sink
    got = grads(model)
    got_loss = float(loss.detach())
    # the same forward, then the fp64 torch loss over the table without its padding column
    for p in model.parameters():
        p.grad = None
    sess = model(batch)
    logits = sess.double() @ table.double()[1:].T / temperature
    want_loss = F.cross_entropy(logits, batch.target_item - 1)
    want_loss.backward()
    want = grads(model)
    want_loss = float(want_loss.detach())
    assert abs(got_loss - want_loss) <= TOL * abs(want_loss)
    assert set(got) == set(want)
    # parameters with an analytically zero gradient (the key bias under the attention softmax) get rounding noise
    # (~1e-10) on both paths: relative error is meaningless there, the noise is compared with the largest gradient
    scale = max(float(g.abs().max()) for g in want.values())
    for name in want:
        if float(want[name].abs().max()) <= 1e-6 * scale:
            assert float((got[name] - want[name]).abs().max()) <= 1e-6 * scale, name
            continue
        assert err(got[name], want[name]) <= TOL, (name, err(got[name], want[name]))
    # one optimizer step runs on either gradient path
    opt.step()


@pytest.mark.gpu
def test_trainer_takes_the_per_operator_path_and_learns(tmp_path):
    from etpgt_b200 import data, optim
    from etpgt_b200.train.losses import create_loss_function
    from etpgt_b200.train.trainer import Trainer

    model, _, (d, graph, store) = model_and_batch()

    def batches(lo, hi, step0):
        out = []
        for i, s in enumerate(range(lo, hi, 128)):
            ids = np.arange(s, min(hi, s + 128))
            bt = data.build_batch(graph, store, ids, 50, False, False)
            bt.negative_items = data.sample_negatives(store, ids, d.num_items, 5, seed=3, step=step0 + i).view(-1)
            out.append(bt)
        return out

    trainer = Trainer(model, batches(0, 768, 0), batches(900, 1100, 100), optim.AdamW(model.parameters(), lr=3e-3),
                      device="cuda", output_dir=tmp_path, max_epochs=2, patience=5, k_values=[10, 20],
                      loss_fn=create_loss_function("full_softmax"))
    assert trainer._driver is None
    history = trainer.train()
    losses = history["train_loss"]
    assert len(losses) == 2 and all(np.isfinite(losses)), losses
    assert losses[1] < losses[0], losses
    metrics = trainer.evaluate()
    for key in ("recall@10", "ndcg@10", "recall@20", "ndcg@20"):
        assert key in metrics and np.isfinite(metrics[key])
