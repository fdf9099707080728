"""GPU tests of the row-sparse optimizer updates of etpgt_b200.optim: `SparseAdam` (etpgt_sparse_adam) against
torch.optim.SparseAdam, `AdamW / Adam(lazy_rows=True)` (etpgt_adam_rows) against the dense step on gathered rows
and the fp64 oracle (tests/lazy_adam_ref.py), training with both, the argument checks and data parallelism."""

import copy
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 2e-6   # fp32: relative to the largest parameter magnitude (as tests/test_gpu_optim.py)


def _bits(t):
    return t.detach().contiguous().view(torch.int32).cpu()


def _same(a, b):
    return torch.equal(_bits(a), _bits(b))


# ---------------------------------------------------------------------------------------------- SparseAdam
def _sparse_grads(rows, dim, steps, seed, zero_row_step=None):
    """Per step: (ascending row ids, values) with magnitudes 1e-3 .. 1e2; the row sets change between steps, rows
    skipped for a few steps come back.  At `zero_row_step` one listed row is all zero."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for s in range(steps):
        if rows == 1:
            ids = torch.tensor([0] if s % 3 != 1 else [], dtype=torch.int64)
        else:
            keep = torch.rand(rows, generator=g) < (0.15 if s % 2 else 0.4)
            ids = torch.nonzero(keep).view(-1)
        scale = 10.0 ** (torch.rand(ids.numel(), 1, generator=g) * 5 - 3)
        vals = torch.randn(ids.numel(), dim, generator=g) * scale
        if s == zero_row_step and ids.numel():
            vals[ids.numel() // 2] = 0
        out.append((ids, vals))
    return out


def _sparse(ids, vals, rows, dim, device):
    return torch.sparse_coo_tensor(ids.view(1, -1), vals, (rows, dim)).coalesce().to(device)


HYPER = [dict(), dict(lr=3e-2, betas=(0.8, 0.95), eps=1e-4, maximize=True)]


@pytest.mark.parametrize("hyper", range(len(HYPER)))
@pytest.mark.parametrize("rows", [1, 1003])
@pytest.mark.parametrize("dim", [4, 32, 100, 256])
@pytest.mark.parametrize("mode", ["listed", "scan"])
def test_sparse_adam_is_bit_identical_to_torch(mode, dim, rows, hyper):
    from etpgt_b200 import optim

    kw = HYPER[hyper]
    init = torch.randn(rows, dim, generator=torch.Generator().manual_seed(dim + rows))
    mine = torch.nn.Parameter(init.clone().cuda())
    ref = torch.nn.Parameter(init.clone().cuda())
    cpu = torch.nn.Parameter(init.clone())
    # scan mode through a gradient sink (every 2-D parameter gets one at sink_bytes=0)
    opt_m = optim.SparseAdam([mine], **kw, sink_bytes=0 if mode == "scan" else 4 << 20)
    opt_t = torch.optim.SparseAdam([ref], **kw)
    opt_c = torch.optim.SparseAdam([cpu], **kw)
    assert (len(opt_m._sinks) == 1) == (mode == "scan")
    for ids, vals in _sparse_grads(rows, dim, 6, seed=dim * rows, zero_row_step=3 if mode == "listed" else None):
        before = mine.detach().clone()
        sp = _sparse(ids, vals, rows, dim, "cuda")
        if mode == "listed":
            mine.grad = sp.clone()
        else:
            mine.grad.copy_(sp.to_dense())
        ref.grad = sp.clone()
        cpu.grad = sp.cpu()
        opt_m.step()
        opt_t.step()
        opt_c.step()
        for name in ("exp_avg", "exp_avg_sq"):
            assert _same(opt_m.state[mine][name], opt_t.state[ref][name]), name
            assert _same(opt_m.state[mine][name], opt_c.state[cpu][name]), name
        assert _same(mine, ref)
        # torch's CPU kernels round some parameters differently from its CUDA ones (the moments agree bit for bit)
        assert (mine.detach().cpu() - cpu.detach()).abs().max().item() <= TOL * cpu.detach().abs().max().item()
        untouched = torch.ones(rows, dtype=torch.bool)
        untouched[ids] = False
        assert _same(mine[untouched.cuda()], before[untouched.cuda()])
        if mode == "scan":
            assert mine.grad.abs().sum().item() == 0      # the sink is cleared by the step
    assert opt_m.state[mine]["step"] == opt_t.state[ref]["step"] == 6


def test_listed_zero_row_is_updated_and_scan_zero_row_is_not():
    from etpgt_b200 import optim

    rows, dim = 64, 32
    init = torch.randn(rows, dim).cuda()
    listed = torch.nn.Parameter(init.clone())
    scan = torch.nn.Parameter(init.clone())
    ref = torch.nn.Parameter(init.clone())
    opt_l, opt_s, opt_t = optim.SparseAdam([listed]), optim.SparseAdam([scan]), torch.optim.SparseAdam([ref])
    # warm the moments of row 5 so that a zero gradient still moves it
    for step, zero in ((0, False), (1, True)):
        ids = torch.tensor([3, 5, 9])
        vals = torch.randn(3, dim)
        if zero:
            vals[1] = 0
        sp = _sparse(ids, vals, rows, dim, "cuda")
        before, before_l = scan.detach().clone(), listed.detach().clone()
        listed.grad, ref.grad, scan.grad = sp.clone(), sp.clone(), sp.to_dense()
        opt_l.step()
        opt_t.step()
        opt_s.step()
        assert _same(listed, ref)
    assert not _same(listed[5], before_l[5])        # listed: torch's index-set semantics
    assert _same(scan[5], before[5])                # scan: an all-zero row is not touched
    assert not _same(scan[3], before[3])


def test_sparse_adam_state_dicts_round_trip_with_torch():
    from etpgt_b200 import optim

    rows, dim = 1003, 100
    grads = _sparse_grads(rows, dim, 6, seed=11)
    init = torch.randn(rows, dim).cuda()
    mine = torch.nn.Parameter(init.clone())
    ref = torch.nn.Parameter(init.clone())
    opt_m, opt_t = optim.SparseAdam([mine], betas=(0.85, 0.99)), torch.optim.SparseAdam([ref], betas=(0.85, 0.99))
    for ids, vals in grads[:3]:
        mine.grad = ref.grad = _sparse(ids, vals, rows, dim, "cuda")
        opt_m.step()
        opt_t.step()
    # swap: torch continues from our state and we continue from torch's
    mine2 = torch.nn.Parameter(ref.detach().clone())
    ref2 = torch.nn.Parameter(mine.detach().clone())
    opt_m2, opt_t2 = optim.SparseAdam([mine2], betas=(0.85, 0.99)), torch.optim.SparseAdam([ref2], betas=(0.85, 0.99))
    # (load_state_dict keeps tensors already on the right device: copies, so that no two optimizers share moments)
    opt_m2.load_state_dict(copy.deepcopy(opt_t.state_dict()))
    opt_t2.load_state_dict(copy.deepcopy(opt_m.state_dict()))
    assert isinstance(opt_t2.state[ref2]["step"], int) and opt_t2.state[ref2]["step"] == 3
    for ids, vals in grads[3:]:
        sp = _sparse(ids, vals, rows, dim, "cuda")
        for p in (mine, ref, mine2, ref2):
            p.grad = sp.clone()
        for o in (opt_m, opt_t, opt_m2, opt_t2):
            o.step()
    for p in (ref, mine2, ref2):
        assert _same(mine, p)


def test_sparse_adam_constructor_checks_match_torch():
    from etpgt_b200 import optim

    p = [torch.nn.Parameter(torch.zeros(4, 4, device="cuda"))]
    for kw, msg in ((dict(lr=0.0), "Invalid learning rate"), (dict(eps=0.0), "Invalid epsilon"),
                    (dict(betas=(1.0, 0.9)), "index 0"), (dict(betas=(0.9, -0.1)), "index 1")):
        with pytest.raises(ValueError, match=msg):
            torch.optim.SparseAdam(p, **kw)
        with pytest.raises(ValueError, match=msg):
            optim.SparseAdam(p, **kw)
    with pytest.raises(ValueError, match="complex"):
        optim.SparseAdam([torch.nn.Parameter(torch.zeros(3, dtype=torch.complex64, device="cuda"))])


# ---------------------------------------------------------------------------------------------- lazy AdamW / Adam
def _adam_rows_on_gathered(p, g, m, v, hit, step, lr, wd, decoupled):
    """etpgt_adam_step (the dense kernel) over a gathered copy of the touched rows."""
    from etpgt_b200 import _lib, optim
    from etpgt_b200._lib import stream

    P, G, M, V = (t[hit].contiguous() for t in (p, g, m, v))
    arr = (optim._AdamTensor * 1)(optim._AdamTensor(P.data_ptr(), G.data_ptr(), M.data_ptr(), V.data_ptr(), P.numel()))
    _lib.call("etpgt_adam_step", arr, 1, lr, 0.9, 0.999, 1e-8, wd, int(decoupled), step, 0, stream())
    return P, M, V


@pytest.mark.parametrize("kind", ["adamw", "adam"])
@pytest.mark.parametrize("wd", [0.0, 1e-5, 1e-2])
@pytest.mark.parametrize("dim", [256, 64, 100])
def test_lazy_rows_match_dense_step_on_gathered_rows_and_oracle(kind, wd, dim):
    from etpgt_b200 import optim
    from lazy_adam_ref import lazy_adam_step

    rows, lr = (4 << 20) // (4 * dim) + 17, 1e-3           # just above the sink threshold
    gen = torch.Generator().manual_seed(dim)
    table = torch.nn.Parameter(torch.randn(rows, dim, generator=gen).cuda())
    bias = torch.nn.Parameter(torch.randn(300, generator=gen).cuda())
    twin_bias = torch.nn.Parameter(bias.detach().clone())
    cls = optim.AdamW if kind == "adamw" else optim.Adam
    opt = cls([table, bias], lr=lr, weight_decay=wd, lazy_rows=True)
    dense = cls([twin_bias], lr=lr, weight_decay=wd)
    assert opt._sinks == [table] and opt.lazy_rows
    ref = (table.detach().double().cpu().numpy(), np.zeros((rows, dim)), np.zeros((rows, dim)))
    for step in range(1, 5):
        keep = torch.rand(rows, generator=gen) < (0.05 if step % 2 else 0.3)
        g = torch.randn(rows, dim, generator=gen) * keep[:, None] * 10.0 ** (step - 3)
        g[torch.nonzero(keep)[0, 0], : dim // 2] = 0         # a touched row with zeros in it
        g[torch.nonzero(~keep)[0, 0], 0] = -0.0              # -0 does not touch a row
        table.grad.copy_(g)
        bias.grad = twin_bias.grad = torch.randn(300, generator=gen).cuda()
        st = opt.state.get(table, {})
        m0 = st["exp_avg"].clone() if st else torch.zeros_like(table)
        v0 = st["exp_avg_sq"].clone() if st else torch.zeros_like(table)
        p0 = table.detach().clone()
        hit = keep.cuda()
        want_p, want_m, want_v = _adam_rows_on_gathered(p0, table.grad.clone(), m0, v0, hit, step, lr, wd,
                                                        kind == "adamw")
        opt.step()
        dense.step()
        st = opt.state[table]
        assert _same(table[hit], want_p) and _same(st["exp_avg"][hit], want_m) and _same(st["exp_avg_sq"][hit], want_v)
        assert _same(table[~hit], p0[~hit]) and _same(st["exp_avg"][~hit], m0[~hit])
        assert _same(st["exp_avg_sq"][~hit], v0[~hit])
        assert table.grad.abs().sum().item() == 0 and opt._is_sink(table)
        assert _same(bias, twin_bias)                     # parameters without a sink take the dense step
        rp, rm, rv, rhit = lazy_adam_step(ref[0], g.double().numpy(), ref[1], ref[2], step, lr=lr, weight_decay=wd,
                                          decoupled=kind == "adamw")
        assert np.array_equal(rhit, keep.numpy())
        ref = (rp, rm, rv)
        scale = np.abs(rp).max()
        assert np.abs(table.detach().double().cpu().numpy() - rp).max() <= TOL * scale, step
        assert np.abs(st["exp_avg"].double().cpu().numpy() - rm).max() <= TOL * max(np.abs(rm).max(), 1e-30)
        assert np.abs(st["exp_avg_sq"].double().cpu().numpy() - rv).max() <= TOL * max(np.abs(rv).max(), 1e-30)
    assert int(opt.state[table]["step"].item()) == 4
    torch.optim.AdamW([table.detach().clone(), bias.detach().clone()]).load_state_dict(opt.state_dict())


@pytest.mark.parametrize("kind", ["adamw", "adam"])
def test_lazy_rows_with_every_row_touched_equal_the_dense_step(kind):
    from etpgt_b200 import optim

    cls = optim.AdamW if kind == "adamw" else optim.Adam
    init = torch.randn(8192, 128).cuda()
    a, b = torch.nn.Parameter(init.clone()), torch.nn.Parameter(init.clone())
    opt_a, opt_b = cls([a], weight_decay=1e-2, lazy_rows=True), cls([b], weight_decay=1e-2)
    for step in range(3):
        g = torch.randn(8192, 128).cuda() + 3.0          # no all-zero row
        a.grad.copy_(g)
        b.grad.copy_(g)
        opt_a.step()
        opt_b.step()
        assert _same(a, b) and _same(opt_a.state[a]["exp_avg_sq"], opt_b.state[b]["exp_avg_sq"])


def test_nan_gradient_row_counts_as_touched():
    from etpgt_b200 import _lib, optim

    table = torch.nn.Parameter(torch.randn(8192, 256).cuda())
    before = table.detach().clone()
    opt = optim.AdamW([table], lazy_rows=True)
    table.grad[7, 3] = float("nan")
    table.grad[9, 0] = 1.0
    opt.step()
    assert torch.isnan(table[7, 3]) and torch.isnan(opt.state[table]["exp_avg"][7, 3])
    # the rest of row 7 was updated (decayed) like row 9's zero elements: the row counts as touched
    others = torch.arange(256, device="cuda") != 3
    assert torch.isfinite(table[7, others]).all() and not _same(table[7, others], before[7, others])
    assert not _same(table[9], before[9]) and table.grad.abs().sum().item() == 0
    rest = (torch.arange(8192, device="cuda") != 7) & (torch.arange(8192, device="cuda") != 9)
    assert _same(table[rest], before[rest])
    # the touched-row counter of the C entry points
    counter = torch.full((1,), -5, dtype=torch.int64, device="cuda")
    p, g, m, v = (torch.zeros(1000, 100, device="cuda") for _ in range(4))
    g[[0, 10, 999]] = 1.0
    _lib.call("etpgt_adam_rows", _lib.ptr(p), _lib.ptr(g), _lib.ptr(m), _lib.ptr(v), 1000, 100, 1e-3, 0.9, 0.999,
              1e-8, 0.0, 1, 1, 1, _lib.ptr(counter), _lib.stream())
    assert counter.item() == 3 and g.abs().sum().item() == 0
    idx = torch.tensor([-1, 2, 5, 1000], device="cuda")
    vals = torch.zeros(4, 100, device="cuda")
    _lib.call("etpgt_sparse_adam", _lib.ptr(p), _lib.ptr(m), _lib.ptr(v), 1000, 100, _lib.ptr(vals), _lib.ptr(idx),
              4, 1e-3, 0.9, 0.999, 1e-8, 0, 1, 0, _lib.ptr(counter), _lib.stream())
    assert counter.item() == 2                          # out-of-range listed rows are skipped


# ---------------------------------------------------------------------------------------------- training
def _setup(num_items=20000, dim=64, seed=5):
    from etpgt_b200 import data, synth

    d = synth.generate(num_sessions=1200, graph_sessions=900, num_items=num_items, clusters=16, seed=seed)
    return d, data.ItemGraph(d.item_i, d.item_j, d.num_items), data.SessionStore(d.sess_ptr, d.sess_items)


def _model(d, dim=64):
    from etpgt_b200.model import create_graph_transformer_optimized

    torch.manual_seed(1)
    return create_graph_transformer_optimized(d.num_items, dim, dim, dropout=0.0, use_laplacian_pe=False).cuda().train()


def _batch(d, graph, store, step, sessions=256):
    from etpgt_b200 import data

    ids = np.arange(step * sessions, (step + 1) * sessions) % d.num_sessions
    batch = data.build_batch(graph, store, ids, 50, False, False)
    batch.negative_items = data.sample_negatives(store, ids, d.num_items, 5, seed=3, step=step)
    return batch


def test_fused_step_lazy_and_dense_adamw_agree_on_touched_rows():
    from etpgt_b200 import optim
    from etpgt_b200.train.step import FusedTrainStep

    d, graph, store = _setup()
    lr, wd = 1e-3, 1e-2
    out = {}
    for lazy in (False, True):
        model = _model(d)
        init = model.item_embedding.weight.detach().clone()
        opt = optim.AdamW(model.parameters(), lr=lr, weight_decay=wd, lazy_rows=lazy)
        fused = FusedTrainStep(model, "bpr")
        opt.zero_grad()
        batch = _batch(d, graph, store, 0)
        fused(batch, batch.target_item, batch.negative_items.view(batch.target_item.shape[0], -1))
        hit = (model.item_embedding.weight.grad != 0).any(1)
        opt.step()
        out[lazy] = ({n: p.detach().clone() for n, p in model.named_parameters()}, hit, init)
    (dense, hit_d, init), (lazy, hit_l, _) = out[False], out[True]
    assert torch.equal(hit_d, hit_l) and 0 < hit_l.sum().item() < d.num_items // 2
    for name in dense:
        if name != "item_embedding.weight":
            assert _same(dense[name], lazy[name]), name
    td, tl = dense["item_embedding.weight"], lazy["item_embedding.weight"]
    assert _same(td[hit_l], tl[hit_l])
    assert _same(tl[~hit_l], init[~hit_l])
    decay = torch.tensor(1.0 - lr * wd, dtype=torch.float32, device="cuda")
    assert _same(td[~hit_l], init[~hit_l] * decay)


def test_per_operator_listwise_steps_match_a_replay_through_the_oracle():
    from etpgt_b200 import optim
    from etpgt_b200.train.losses import create_loss_function
    from lazy_adam_ref import lazy_adam_step
    from oracle import optim_ref

    d, graph, store = _setup()
    model = _model(d)
    loss_fn = create_loss_function("listwise")
    lr, wd = 2e-3, 1e-5
    opt = optim.AdamW(model.parameters(), lr=lr, weight_decay=wd, lazy_rows=True)
    ref = {n: (p.detach().double().cpu().numpy(), 0.0, 0.0) for n, p in model.named_parameters()}
    for step in range(1, 4):
        batch = _batch(d, graph, store, step)
        opt.zero_grad()
        sess = model(batch)
        loss = loss_fn(sess, batch.target_item, batch.negative_items.view(sess.shape[0], -1), model.item_embedding)
        loss.backward()
        grads = {n: p.grad.detach().double().cpu().numpy() for n, p in model.named_parameters() if p.grad is not None}
        opt.step()
        for n in grads:
            p, m, v = ref[n]
            m = np.zeros_like(p) if np.isscalar(m) else m
            v = np.zeros_like(p) if np.isscalar(v) else v
            if n == "item_embedding.weight":
                p, m, v, _ = lazy_adam_step(p, grads[n], m, v, step, lr=lr, weight_decay=wd)
            else:
                p, m, v = optim_ref.adam_step(p, grads[n], m, v, step, lr=lr, weight_decay=wd)
            ref[n] = (p, m, v)
    for n, p in model.named_parameters():
        want = ref[n][0]
        assert np.abs(p.detach().double().cpu().numpy() - want).max() <= TOL * max(np.abs(want).max(), 1e-30), n


def test_full_softmax_lazy_equals_dense_except_the_padding_row():
    from etpgt_b200 import optim
    from etpgt_b200.train.losses import create_loss_function

    d, graph, store = _setup()
    loss_fn = create_loss_function("full_softmax")
    out = {}
    for lazy in (False, True):
        model = _model(d)
        opt = optim.AdamW(model.parameters(), lr=1e-3, weight_decay=1e-2, lazy_rows=lazy)
        for step in range(2):
            batch = _batch(d, graph, store, step)
            opt.zero_grad()
            sess = model(batch)
            loss_fn(sess, batch.target_item, batch.negative_items.view(sess.shape[0], -1), model.item_embedding).backward()
            opt.step()
        out[lazy] = {n: p.detach().clone() for n, p in model.named_parameters()}
    for name in out[False]:
        a, b = out[False][name], out[True][name]
        if name == "item_embedding.weight":
            # the padding row has no gradient: lazy leaves it alone, dense decays it (it is zero, and stays so)
            assert _same(a[1:], b[1:]) and (a[0] == 0).all() and (b[0] == 0).all()
        else:
            assert _same(a, b), name


def test_trainer_checkpoints_of_a_lazy_run_load_into_torch_adamw(tmp_path):
    from etpgt_b200 import optim
    from etpgt_b200.train.trainer import Trainer

    d, graph, store = _setup()
    model = _model(d)
    train = [_batch(d, graph, store, s, 128) for s in range(6)]
    val = [_batch(d, graph, store, 8 + s, 128) for s in range(2)]
    opt = optim.AdamW(model.parameters(), lr=3e-3, lazy_rows=True)
    trainer = Trainer(model, train, val, opt, device="cuda", output_dir=tmp_path, max_epochs=2, patience=5,
                      k_values=[10])
    history = trainer.train()
    assert len(history["train_loss"]) == 2 and all(np.isfinite(history["train_loss"]))
    ckpt = torch.load(tmp_path / "checkpoint_latest.pt", weights_only=False)
    twin = _model(d)
    twin.load_state_dict(ckpt["model_state_dict"])
    ref = torch.optim.AdamW(twin.parameters(), lr=3e-3)
    ref.load_state_dict(ckpt["optimizer_state_dict"])
    table_state = ref.state[twin.item_embedding.weight]
    assert float(table_state["step"]) == 12 and table_state["exp_avg"].shape == twin.item_embedding.weight.shape
    dense_again = optim.AdamW(twin.parameters(), lr=3e-3)
    dense_again.load_state_dict(ckpt["optimizer_state_dict"])


# ---------------------------------------------------------------------------------------------- errors, data parallelism
def test_argument_checks():
    from etpgt_b200 import _lib, optim

    s = _lib.stream()
    p, g, m, v = (torch.zeros(10, 32, device="cuda") for _ in range(4))
    P = [_lib.ptr(t) for t in (p, g, m, v)]
    good = (1e-3, 0.9, 0.999, 1e-8)
    with pytest.raises(RuntimeError, match="NULL pointer"):
        _lib.call("etpgt_adam_rows", P[0], None, P[2], P[3], 10, 32, *good, 0.0, 1, 1, 1, None, s)
    with pytest.raises(RuntimeError, match="step must be >= 1"):
        _lib.call("etpgt_adam_rows", *P, 10, 32, *good, 0.0, 1, 0, 1, None, s)
    with pytest.raises(RuntimeError, match="hyper-parameters out of range"):
        _lib.call("etpgt_adam_rows", *P, 10, 32, 1e-3, 1.0, 0.999, 1e-8, 0.0, 1, 1, 1, None, s)
    with pytest.raises(RuntimeError, match="bad shape"):
        _lib.call("etpgt_adam_rows", *P, 10, 0, *good, 0.0, 1, 1, 1, None, s)
    flat, flat_g = torch.zeros(400, device="cuda"), torch.zeros(400, device="cuda")
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        _lib.call("etpgt_adam_rows", flat.data_ptr() + 4, *P[1:], 10, 32, *good, 0.0, 1, 1, 1, None, s)
    flat_g[1:34] = 1.0
    _lib.call("etpgt_adam_rows", flat.data_ptr() + 4, flat_g.data_ptr() + 4, *P[2:], 3, 33, *good, 0.0, 1, 1, 1,
              None, s)                                   # scalar path: no alignment needed
    assert (flat[1:34] < 0).all() and (flat[34:] == 0).all() and flat_g.abs().sum().item() == 0
    flat.zero_()
    with pytest.raises(RuntimeError, match="NULL pointer"):
        _lib.call("etpgt_sparse_adam", P[0], None, P[3], 10, 32, P[1], None, 0, *good, 0, 1, 1, None, s)
    with pytest.raises(RuntimeError, match="step must be >= 1"):
        _lib.call("etpgt_sparse_adam", P[0], P[2], P[3], 10, 32, P[1], None, 0, *good, 0, 0, 1, None, s)
    with pytest.raises(RuntimeError, match="hyper-parameters out of range"):
        _lib.call("etpgt_sparse_adam", P[0], P[2], P[3], 10, 32, P[1], None, 0, 1e-3, 0.9, 0.999, -1.0, 0, 1, 1,
                  None, s)
    idx = torch.arange(3, device="cuda")
    with pytest.raises(RuntimeError, match="zero_grad"):
        _lib.call("etpgt_sparse_adam", P[0], P[2], P[3], 10, 32, P[1], _lib.ptr(idx), 3, *good, 0, 1, 1, None, s)
    with pytest.raises(RuntimeError, match="listed rows"):
        _lib.call("etpgt_sparse_adam", P[0], P[2], P[3], 10, 32, P[1], _lib.ptr(idx), -1, *good, 0, 1, 0, None, s)
    torch.cuda.synchronize()
    assert p.abs().sum().item() == 0                    # nothing was launched by a rejected call
    table = [torch.nn.Parameter(torch.zeros(8192, 256, device="cuda"))]
    with pytest.raises(ValueError, match="grad_sinks"):
        optim.AdamW(table, lazy_rows=True, grad_sinks=False)
    with pytest.raises(ValueError, match="grad_sinks"):
        optim.Adam(table, lazy_rows=True, grad_sinks=False)
    with pytest.raises(RuntimeError, match="dense fp32"):
        opt = optim.AdamW([torch.nn.Parameter(torch.zeros(4, 4, device="cuda"))], lazy_rows=True)
        opt.param_groups[0]["params"][0].grad = torch.zeros(4, 4, device="cuda").to_sparse()
        opt.step()


def test_row_sparse_tables_in_a_peer_region_are_refused():
    from etpgt_b200 import _lib, optim, parallel
    from etpgt_b200.model import create_graph_transformer_optimized

    def model():
        torch.manual_seed(0)
        return create_graph_transformer_optimized(500, 64, 64, dropout=0.0, use_laplacian_pe=False).cuda()

    m = model()
    dense = sum(p.numel() for p in m.parameters()) - m.item_embedding.weight.numel()
    need = int(_lib.size("etpgt_comm_control_bytes")) + 4 * dense + 8 * m.item_embedding.weight.numel() + 4096
    (comm,) = parallel.PeerComm.local_group(1, need)
    peer = parallel.PeerDataParallel(m, comm=comm)
    for make in (lambda ps: optim.AdamW(ps, lazy_rows=True), lambda ps: optim.Adam(ps, lazy_rows=True),
                 lambda ps: optim.SparseAdam(ps)):
        with pytest.raises(NotImplementedError, match='exchange="nccl"'):
            make(list(m.parameters()))
    # created before the peer region (Trainer's order): attach_peer refuses
    m2 = model()
    opt = optim.AdamW(m2.parameters(), lazy_rows=True, sink_bytes=0)
    (comm2,) = parallel.PeerComm.local_group(1, need)
    peer2 = parallel.PeerDataParallel(m2, comm=comm2)
    with pytest.raises(NotImplementedError, match='exchange="nccl"'):
        opt.attach_peer(peer2)
    del peer, peer2


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, out):
    import faulthandler

    import torch.distributed as dist

    faulthandler.dump_traceback_later(300, exit=True)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from etpgt_b200 import optim
        from etpgt_b200.train.step import FusedTrainStep
        from etpgt_b200.train.trainer import Trainer

        d, graph, store = _setup()
        model = _model(d)
        opt = optim.AdamW(model.parameters(), lr=1e-3, weight_decay=1e-2, lazy_rows=True)
        trainer = Trainer(model, [], [], opt, device="cuda", output_dir=f"/tmp/etpgt_lazy_{port}", process_group=True,
                          exchange="peer")
        peer_is_none = trainer._peer is None           # warned and fell back to NCCL
        fused = FusedTrainStep(model, "bpr")
        for step in range(3):
            batch = _batch(d, graph, store, 2 * step + rank, 128)
            opt.zero_grad()
            fused(batch, batch.target_item, batch.negative_items.view(128, -1), total_sessions=256)
            fused.allreduce_gradients()
            opt.step()
        torch.cuda.synchronize()
        flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
        gathered = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(gathered, flat)
        out[rank] = (peer_is_none, all(torch.equal(gathered[0], g) for g in gathered))
    finally:
        dist.destroy_process_group()


def test_two_gpus_nccl_lazy_replicas_stay_identical():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp

    manager = mp.get_context("spawn").Manager()
    out = manager.dict()
    mp.spawn(_nccl_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    for rank in (0, 1):
        assert out[rank] == (True, True), (rank, out[rank])
