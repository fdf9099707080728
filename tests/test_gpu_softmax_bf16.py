"""The plain-bf16 mode of the full-catalogue and shared-pool softmax losses (precision="bf16",
ETPGT_SOFTMAX_BF16): the kernels against an fp64 oracle of the bf16 arithmetic, against the default split-bf16 path,
its properties (determinism, exact zero gradient, padding row, accumulation), the pool's reduction to the full loss,
the model and Trainer levels and the argument checks.  Errors are max|got - want| / max|want|.

The oracle: S and E rounded to bf16, logits, lse and the loss in fp64; G = (P - onehot) / (T B_total) from the
oracle's own lse in fp64, then rounded to bf16 before the gradient products (in fp64).  For the pool the positive is
z_pos = bf16(s_b) . bf16(e_t) / T and its entry of G is rounded like the rest.  lse, the loss and z_pos are held to
1e-4; the gradients to 1e-3 of max|ref|, which leaves room for an element of G that rounds to the other bf16
neighbour where the kernel's fp32 value and the oracle's fp64 value lie on either side of a rounding boundary."""

import numpy as np
import pytest
import torch

from softmax_loss_util import err, model_and_batch

TOL_VALUE = 1e-4        # lse, loss, z_pos against the oracle
TOL_GRAD = 1e-3         # d_sess, d_table against the oracle, of max|ref|
TOL_SPLIT_LOSS = 1e-3   # against the split-bf16 path, for a loss that is a mean over SPLIT_LOSS_ROWS rows or more
TOL_SPLIT_GRAD = 1e-2
# With a handful of rows the loss is a few single logits, and rounding S and E to bf16 moves one dot product of
# D = 256 terms by up to ~1e-2 relative (measured: z_pos of one row, 1.2e-2): that compares the two inputs, not the
# kernels, so below this many rows only the oracle bounds apply to the loss.
SPLIT_LOSS_ROWS = 128
BF16X3, BF16 = 0, 1
NUM_SMS, DRAIN_TILES = 148, 8


# ------------------------------------------------------------------------------ CPU: the boundary


def test_bad_precision_is_rejected_in_python():
    from etpgt_b200 import ops
    from etpgt_b200.train.losses import FullSoftmaxLoss, SharedPoolSoftmaxLoss, create_loss_function

    for bad in ("fp32", "BF16", "", None, 1):
        with pytest.raises(ValueError, match='"bf16x3" or "bf16"'):
            ops._softmax_precision(bad)
        with pytest.raises(ValueError, match='"bf16x3" or "bf16"'):
            FullSoftmaxLoss(precision=bad)
        with pytest.raises(ValueError, match='"bf16x3" or "bf16"'):
            SharedPoolSoftmaxLoss(precision=bad)
    with pytest.raises(ValueError, match='"bf16x3" or "bf16"'):
        create_loss_function("full_softmax", precision="fp16")
    # the Python check comes before anything touches a tensor
    with pytest.raises(ValueError, match='"bf16x3" or "bf16"'):
        ops.full_softmax_loss(torch.randn(4, 64), torch.randn(10, 64), torch.tensor([1, 2, 3, 4]), precision="fp8")
    with pytest.raises(ValueError, match='"bf16x3" or "bf16"'):
        ops.pool_softmax_loss(torch.randn(4, 64), torch.randn(10, 64), torch.tensor([1, 2, 3, 4]),
                              torch.tensor([1, 2]), torch.zeros(2), precision="fp8")


def test_bad_precision_is_rejected_by_the_abi():
    """Any precision other than 0 or 1 returns ETPGT_EINVAL (-1) and names both, before any argument is read."""
    from etpgt_b200 import _lib

    lib = _lib.load()
    z = None
    calls = {
        "etpgt_full_softmax_fwd_ex": (z, z, z, 4, 10, 64, 1.0, 0.0, 0, z, z, z, 0, z),
        "etpgt_full_softmax_bwd_ex": (z, z, z, z, z, 4, 10, 64, 1.0, 0.0, 0, z, z, z, 0, z),
        "etpgt_pool_softmax_fwd_ex": (z, z, z, z, z, 4, 10, 2, 64, 1.0, 0.0, 0, z, z, z, z, 0, z),
        "etpgt_pool_softmax_bwd_ex": (z, z, z, z, z, z, z, z, 4, 10, 2, 64, 1.0, 0.0, 0, z, z, z, 0, z),
    }
    for name, args in calls.items():
        for bad in (-1, 2, 3):
            assert getattr(lib, name)(*args, bad) == -1, name
            msg = _lib.last_error()
            assert "ETPGT_SOFTMAX_BF16X3" in msg and "ETPGT_SOFTMAX_BF16 " in msg, msg
        # a valid precision gets as far as the argument checks (null pointers)
        assert getattr(lib, name)(*args, BF16) == -1
        assert "null argument" in _lib.last_error()


def test_create_loss_function_stores_the_precision():
    from etpgt_b200.train.losses import (BPRLoss, FullSoftmaxLoss, SharedPoolSoftmaxLoss, create_loss_function)

    assert create_loss_function("full_softmax").precision == "bf16x3"
    assert create_loss_function("shared_pool_softmax").precision == "bf16x3"
    full = create_loss_function("full_softmax", temperature=0.5, precision="bf16")
    assert isinstance(full, FullSoftmaxLoss) and full.precision == "bf16" and full.temperature == 0.5
    pool = create_loss_function("shared_pool_softmax", num_sampled=64, precision="bf16")
    assert isinstance(pool, SharedPoolSoftmaxLoss) and pool.precision == "bf16" and pool.num_sampled == 64
    # the other loss types ignore it, as they ignore num_sampled
    assert isinstance(create_loss_function("bpr", precision="bf16"), BPRLoss)
    with pytest.raises(TypeError):
        create_loss_function("full_softmax", 0.7, 1.0, 8192, None, 0.75, 0, "bf16")   # keyword-only


# ------------------------------------------------------------------------------ helpers


def _plan_ranges(rows, cols, max_ranges):
    """softmax_tc.cu's plan_ranges: (tiles_per_range, ranges, grid)."""
    row_tiles, col_tiles = -(-rows // 128), -(-cols // 128)
    best = None
    for want in range(1, min(col_tiles, max_ranges) + 1):
        tpr = -(-col_tiles // want)
        r = -(-col_tiles // tpr)
        cost = -(-(row_tiles * r) // NUM_SMS) * tpr
        if best is None or cost < best[0]:
            best = (cost, tpr, r, row_tiles * r)
    return best[1:]


def _plans(batch, items):
    """The column-range plans of FWD, DS and DE (plan_fwd, plan_grad(B, I), plan_grad(I, B))."""
    def grad(rows, cols):
        row_tiles = -(-rows // 128)
        return _plan_ranges(rows, cols, max(1, (4 * NUM_SMS + row_tiles - 1) // row_tiles))
    return {"fwd": _plan_ranges(batch, items, 1 << 20), "ds": grad(batch, items), "de": grad(items, batch)}


def _bf16(x):
    """fp32 -> bf16 (round to nearest even) -> fp64."""
    return x.float().to(torch.bfloat16).double()


def _full_oracle(sess, table, targets, temperature=1.0, total=None, padding_idx=0, d_loss=1.0):
    """fp64 (loss, lse, d_sess, d_table) of the bf16 full loss, chunked over rows."""
    s, e = _bf16(sess), _bf16(table)
    t = targets.long()
    b, items = s.shape[0], e.shape[0]
    total = float(total) if total else float(b)
    scale = d_loss / (temperature * total)
    chunk = max(1, min(b, (1 << 30) // (8 * items * 2)))
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
        g = _bf16(g * scale)
        d_table += g.T @ s[r0:r1]
        d_sess[r0:r1] = g @ e
        del z, g
    if padding_idx >= 0:
        d_table[padding_idx] = 0
    return torch.tensor(loss * d_loss / total, dtype=torch.float64), lse, d_sess, d_table


def _pool_oracle(sess, table, targets, pool, log_q, temperature=1.0, total=None, padding_idx=0, d_loss=1.0):
    """fp64 (loss, lse, z_pos, d_sess, d_table) of the bf16 shared-pool loss."""
    s, e = _bf16(sess), _bf16(table)
    t, p = targets.long(), pool.long()
    b = s.shape[0]
    total = float(total) if total else float(b)
    scale = d_loss / (temperature * total)
    z_pos = (s * e[t]).sum(1) / temperature
    z = s @ e[p].T / temperature - log_q.double()[None, :]
    z = z.masked_fill((p[None, :] == t[:, None]) | (p == padding_idx)[None, :], -float("inf"))
    lse = torch.logsumexp(torch.cat([z_pos[:, None], z], dim=1), dim=1)
    loss = (lse - z_pos).sum() / total * d_loss
    g = _bf16(torch.exp(z - lse[:, None]) * scale)
    c = _bf16((torch.exp(z_pos - lse) - 1.0) * scale)
    d_sess = g @ e[p] + c[:, None] * e[t]
    d_table = torch.zeros_like(e)
    d_table.index_add_(0, p, g.T @ s)
    d_table.index_add_(0, t, c[:, None] * s)
    if padding_idx >= 0:
        d_table[padding_idx] = 0
    return loss, lse, z_pos, d_sess, d_table


def _run_full(sess, table, targets, temperature=1.0, total=None, padding_idx=0, d_table=None, d_loss=1.0,
              precision=BF16):
    """One forward and one backward through the _ex ABI: (loss, lse, d_sess, d_table)."""
    from etpgt_b200 import _lib
    from etpgt_b200._lib import ptr

    b, dim = sess.shape
    items = table.shape[0]
    dev = sess.device
    lse = torch.empty(b, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    ws = _lib.workspace(_lib.size("etpgt_full_softmax_workspace_bytes", b, items, dim), dev)
    tot = float(total) if total else 0.0
    _lib.call("etpgt_full_softmax_fwd_ex", ptr(sess), ptr(table), ptr(targets), b, items, dim, float(temperature),
              tot, padding_idx, ptr(lse), ptr(loss), ptr(ws), ws.numel(), _lib.stream(), precision)
    dl = torch.tensor([d_loss], dtype=torch.float32, device=dev)
    d_sess = torch.empty_like(sess)
    d_table = torch.zeros_like(table) if d_table is None else d_table
    _lib.call("etpgt_full_softmax_bwd_ex", ptr(sess), ptr(table), ptr(targets), ptr(lse), ptr(dl), b, items, dim,
              float(temperature), tot, padding_idx, ptr(d_sess), ptr(d_table), ptr(ws), ws.numel(), _lib.stream(),
              precision)
    torch.cuda.synchronize()
    return loss[0], lse, d_sess, d_table


def _run_pool(sess, table, targets, pool, log_q, temperature=1.0, total=None, padding_idx=0, d_table=None,
              d_loss=1.0, precision=BF16):
    """One forward and one backward through the _ex ABI: (loss, lse, z_pos, d_sess, d_table)."""
    from etpgt_b200 import _lib
    from etpgt_b200._lib import ptr

    b, dim = sess.shape
    items, m = table.shape[0], pool.numel()
    dev = sess.device
    lse = torch.empty(b, dtype=torch.float32, device=dev)
    z_pos = torch.empty(b, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    ws = _lib.workspace(_lib.size("etpgt_pool_softmax_workspace_bytes", b, m, dim), dev)
    tot = float(total) if total else 0.0
    _lib.call("etpgt_pool_softmax_fwd_ex", ptr(sess), ptr(table), ptr(targets), ptr(pool), ptr(log_q), b, items, m,
              dim, float(temperature), tot, padding_idx, ptr(lse), ptr(z_pos), ptr(loss), ptr(ws), ws.numel(),
              _lib.stream(), precision)
    dl = torch.tensor([d_loss], dtype=torch.float32, device=dev)
    d_sess = torch.empty_like(sess)
    d_table = torch.zeros_like(table) if d_table is None else d_table
    _lib.call("etpgt_pool_softmax_bwd_ex", ptr(sess), ptr(table), ptr(targets), ptr(pool), ptr(log_q), ptr(lse),
              ptr(z_pos), ptr(dl), b, items, m, dim, float(temperature), tot, padding_idx, ptr(d_sess), ptr(d_table),
              ptr(ws), ws.numel(), _lib.stream(), precision)
    torch.cuda.synchronize()
    return loss[0], lse, z_pos, d_sess, d_table


def _inputs(b, items, dim, seed, scale=0.3, padding_idx=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    sess = torch.randn(b, dim, device="cuda", generator=g) * scale
    table = torch.randn(items, dim, device="cuda", generator=g) * scale
    targets = torch.randint(1 if padding_idx == 0 else 0, items, (b,), device="cuda", generator=g)
    return sess, table, targets


def _pool_inputs(b, items, dim, m, seed, scale=0.3):
    """A sorted pool with duplicates, entries equal to rows' targets (row 0's target is the first entry) and five
    padding entries (id 0)."""
    sess, table, targets = _inputs(b, items, dim, seed, scale)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    pool = torch.randint(1, items, (m,), device="cuda", generator=g)
    if m >= 16:
        pool[: m // 8] = targets[torch.arange(m // 8, device="cuda") % min(b, 3)]
        pool[m // 8: m // 8 + 5] = 0
    pool = torch.sort(pool).values
    targets[0] = pool[-1]
    log_q = torch.rand(m, device="cuda", generator=g) * 4 - 2
    return sess, table, targets, pool, log_q


def _fmt(errs):
    return "{" + ", ".join(f"{n} {v:.2e}" for n, v in errs.items()) + "}"


def _check_full(sess, table, targets, temperature=1.0, total=None, padding_idx=0, label=""):
    got = _run_full(sess, table, targets, temperature, total, padding_idx)
    want = _full_oracle(sess, table, targets, temperature, total, padding_idx)
    split = _run_full(sess, table, targets, temperature, total, padding_idx, precision=BF16X3)
    names = ("loss", "lse", "d_sess", "d_table")
    errs = {n: err(g, w) for n, g, w in zip(names, got, want)}
    vs_split = {n: err(g, w) for n, g, w in zip(names, got, split)}
    print(f"full bf16 {label} B={sess.shape[0]} I={table.shape[0]} D={sess.shape[1]}: vs oracle {_fmt(errs)}, "
          f"vs split {_fmt(vs_split)}")
    assert errs["loss"] <= TOL_VALUE and errs["lse"] <= TOL_VALUE, errs
    assert errs["d_sess"] <= TOL_GRAD and errs["d_table"] <= TOL_GRAD, errs
    assert sess.shape[0] < SPLIT_LOSS_ROWS or vs_split["loss"] <= TOL_SPLIT_LOSS, vs_split
    assert vs_split["d_sess"] <= TOL_SPLIT_GRAD and vs_split["d_table"] <= TOL_SPLIT_GRAD, vs_split
    return got


def _check_pool(sess, table, targets, pool, log_q, temperature=1.0, total=None, padding_idx=0, label=""):
    got = _run_pool(sess, table, targets, pool, log_q, temperature, total, padding_idx)
    want = _pool_oracle(sess, table, targets, pool, log_q, temperature, total, padding_idx)
    split = _run_pool(sess, table, targets, pool, log_q, temperature, total, padding_idx, precision=BF16X3)
    names = ("loss", "lse", "z_pos", "d_sess", "d_table")
    errs = {n: err(g, w) for n, g, w in zip(names, got, want)}
    vs_split = {n: err(g, w) for n, g, w in zip(names, got, split)}
    print(f"pool bf16 {label} B={sess.shape[0]} M={pool.numel()} D={sess.shape[1]}: vs oracle {_fmt(errs)}, "
          f"vs split {_fmt(vs_split)}")
    assert errs["loss"] <= TOL_VALUE and errs["lse"] <= TOL_VALUE and errs["z_pos"] <= TOL_VALUE, errs
    assert errs["d_sess"] <= TOL_GRAD and errs["d_table"] <= TOL_GRAD, errs
    assert sess.shape[0] < SPLIT_LOSS_ROWS or vs_split["loss"] <= TOL_SPLIT_LOSS, vs_split
    assert vs_split["d_sess"] <= TOL_SPLIT_GRAD and vs_split["d_table"] <= TOL_SPLIT_GRAD, vs_split
    return got


# ------------------------------------------------------------------------------ GPU: full loss


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [64, 128, 192, 256])
@pytest.mark.parametrize("batch,items", [(1, 2), (1, 3001), (300, 5003), (129, 2)])
def test_full_matches_the_bf16_oracle(batch, items, dim):
    sess, table, targets = _inputs(batch, items, dim, seed=batch + items + dim)
    if items == 2:
        targets.fill_(1)             # id 0 is the padding column
    _check_full(sess, table, targets, 0.5, None, label="T=0.5")
    _check_full(sess, table, targets, 1.0, 3 * batch + 5, label="total")


@pytest.mark.gpu
@pytest.mark.parametrize("padding_idx", [0, -1])
def test_full_padding(padding_idx):
    sess, table, targets = _inputs(500, 1000, 128, seed=4, padding_idx=padding_idx)
    if padding_idx == -1:
        targets[:50] = 0
    _, _, _, d_table = _check_full(sess, table, targets, padding_idx=padding_idx, label=f"pad={padding_idx}")
    if padding_idx == 0:
        assert torch.count_nonzero(d_table[0]) == 0
    else:
        assert torch.count_nonzero(d_table[0]) == table.shape[1]


@pytest.mark.gpu
def test_full_several_column_ranges_of_many_drain_groups():
    """B = 4,100, I = 50,011: 33 row tiles x 391 column tiles.  The forward and dS are split into column ranges, and
    both gradient passes (the ones that drain the accumulator) have well over kDrainTiles tiles per range."""
    b, items, dim = 4100, 50011, 256
    plans = _plans(b, items)
    print("ranges plan (tiles_per_range, ranges, grid):", plans)
    assert plans["fwd"][1] > 1 and plans["ds"][1] > 1
    for name in ("ds", "de"):
        assert plans[name][0] > 2 * DRAIN_TILES, (name, plans[name])
    sess, table, targets = _inputs(b, items, dim, seed=41)
    _check_full(sess, table, targets, 0.5, None, label="multi-range")


@pytest.mark.gpu
def test_full_properties():
    sess, table, targets = _inputs(1000, 20000, 256, seed=8)
    a = _run_full(sess, table, targets)
    b = _run_full(sess, table, targets)
    for x, y in zip(a, b):
        assert torch.equal(x, y)                         # bit-reproducible
    # explicit bf16x3 through the _ex call gives the default call's bits
    from etpgt_b200 import _lib
    from etpgt_b200._lib import ptr

    default = _run_full(sess, table, targets, precision=BF16X3)
    lse = torch.empty(1000, device="cuda")
    loss = torch.empty(1, device="cuda")
    ws = _lib.workspace(_lib.size("etpgt_full_softmax_workspace_bytes", 1000, 20000, 256), sess.device)
    _lib.call("etpgt_full_softmax_fwd", ptr(sess), ptr(table), ptr(targets), 1000, 20000, 256, 1.0, 0.0, 0, ptr(lse),
              ptr(loss), ptr(ws), ws.numel(), _lib.stream())
    torch.cuda.synchronize()
    assert torch.equal(default[0], loss[0]) and torch.equal(default[1], lse)
    # d_table is added to, and its padding row keeps its bits
    base = torch.randn_like(table) * 1e-3
    base[0] = 7.0
    got = _run_full(sess, table, targets, d_table=base.clone())
    assert err(got[3] - base, a[3]) <= 1e-6
    assert torch.all(got[3][0] == 7.0)


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [64, 256])
def test_full_exact_softmax_gives_an_exactly_zero_gradient(dim):
    # two items, id 0 the padding column: one eligible column, P = 1 exactly
    sess, table, _ = _inputs(300, 2, dim, seed=dim)
    targets = torch.ones(300, dtype=torch.long, device="cuda")
    loss, lse, d_sess, d_table = _run_full(sess, table, targets)
    assert float(loss) == 0.0
    assert float(d_sess.abs().max()) == 0.0 and float(d_table.abs().max()) == 0.0


# ------------------------------------------------------------------------------ GPU: shared pool


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [64, 128, 192, 256])
@pytest.mark.parametrize("batch,m", [(1, 1), (1, 129), (300, 1000), (1000, 8192)])
def test_pool_matches_the_bf16_oracle(batch, m, dim):
    sess, table, targets, pool, log_q = _pool_inputs(batch, 5003, dim, m, seed=batch + m + dim)
    got = _check_pool(sess, table, targets, pool, log_q, temperature=0.5)
    if m == 1:   # row 0's whole pool is its target: P = 1 exactly and its gradient is zero
        assert float(got[3][0].abs().max()) == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [64, 256])
@pytest.mark.parametrize("temperature", [1.0, 0.07])
def test_pool_of_every_item_is_the_bf16_full_loss(dim, temperature):
    b, items = 1000, 5000
    sess, table, targets = _inputs(b, items, dim, seed=dim)
    sess, table = sess * 0.5, table * 0.5
    pool = torch.arange(1, items, device="cuda")
    got = _run_pool(sess, table, targets, pool, torch.zeros(items - 1, device="cuda"), temperature)
    want = _run_full(sess, table, targets, temperature)
    errs = {n: err(g, w) for n, g, w in zip(("loss", "lse", "d_sess", "d_table"),
                                            (got[0], got[1], got[3], got[4]), want)}
    print(f"pool of every item vs full, bf16, D={dim} T={temperature}: {_fmt(errs)}")
    assert all(v <= 1e-5 for v in errs.values()), errs


@pytest.mark.gpu
def test_pool_properties():
    b, items, dim, m = 2048, 20000, 256, 4096
    sess, table, targets, pool, log_q = _pool_inputs(b, items, dim, m, seed=13)
    a = _run_pool(sess, table, targets, pool, log_q)
    c = _run_pool(sess, table, targets, pool, log_q)
    for x, y in zip(a, c):
        assert torch.equal(x, y)
    base = torch.randn(items, dim, device="cuda") * 1e-3
    got = _run_pool(sess, table, targets, pool, log_q, d_table=base.clone())
    assert err(got[4] - base, a[4]) <= 1e-5                # fp32 rounding of the additions onto base
    touched = torch.zeros(items, dtype=torch.bool, device="cuda")
    touched[pool] = True
    touched[targets] = True
    touched[0] = False
    assert torch.equal(got[4][~touched], base[~touched])   # padding row and untouched rows keep their bits
    # the pool entirely one row's target: that row's gradient is exactly zero
    pool1 = torch.full((256,), int(targets[0]), device="cuda")
    t = targets.clone()
    t[1:] = torch.where(t[1:] == t[0], t[1:] % (items - 1) + 1, t[1:])
    got = _run_pool(sess, table, t, pool1, torch.zeros(256, device="cuda"))
    assert float(got[3][0].abs().max()) == 0.0


# ------------------------------------------------------------------------------ GPU: through the layers


def _model_grads(loss_fn, batch, model, opt=None):
    from softmax_loss_util import grads

    for p in model.parameters():
        p.grad = None
    if opt is not None:
        opt.zero_grad()
    loss = loss_fn(model(batch), batch.target_item, None, model.item_embedding)
    loss.backward()
    return float(loss.detach()), grads(model)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["full_softmax", "shared_pool_softmax"])
def test_model_gradients_match_the_split_path(kind):
    from etpgt_b200 import optim
    from etpgt_b200.train.losses import create_loss_function

    model, batch, _ = model_and_batch()
    model.train()
    kw = {"num_sampled": 300, "seed": 1} if kind == "shared_pool_softmax" else {}
    split_loss, split = _model_grads(create_loss_function(kind, temperature=0.5, **kw), batch, model)
    bf16_loss, got = _model_grads(create_loss_function(kind, temperature=0.5, precision="bf16", **kw), batch, model)
    assert abs(bf16_loss - split_loss) <= TOL_SPLIT_LOSS * abs(split_loss), (bf16_loss, split_loss)
    assert set(got) == set(split)
    scale = max(float(g.abs().max()) for g in split.values())
    errs = {}
    for name in split:
        if float(split[name].abs().max()) <= 1e-6 * scale:   # analytically zero: rounding noise on both paths
            assert float((got[name] - split[name]).abs().max()) <= 1e-4 * scale, name
            continue
        errs[name] = err(got[name], split[name])
    print(f"{kind}: loss bf16 {bf16_loss:.6f} split {split_loss:.6f}; max gradient error vs split "
          f"{max(errs.values()):.2e}")
    assert all(v <= TOL_SPLIT_GRAD for v in errs.values()), errs
    # the table gradient lands in the optimizer's sink when one is registered
    table = model.item_embedding.weight
    opt = optim.AdamW(model.parameters(), lr=1e-3, sink_bytes=table.numel() * 4)
    _, sunk = _model_grads(create_loss_function(kind, temperature=0.5, precision="bf16", **kw), batch, model, opt)
    assert optim.grad_sink_for(table) is table.grad
    assert err(sunk["item_embedding.weight"], got["item_embedding.weight"]) <= 1e-6
    opt.step()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["full_softmax", "shared_pool_softmax"])
def test_trainer_runs_an_epoch_in_bf16(kind, tmp_path):
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

    kw = {"num_sampled": 256, "seed": 3} if kind == "shared_pool_softmax" else {}
    loss_fn = create_loss_function(kind, precision="bf16", **kw)
    trainer = Trainer(model, batches(0, 768, 0), batches(900, 1100, 100), optim.AdamW(model.parameters(), lr=3e-3),
                      device="cuda", output_dir=tmp_path, max_epochs=1, patience=5, k_values=[20], loss_fn=loss_fn)
    assert trainer._driver is None
    losses = trainer.train()["train_loss"]
    assert len(losses) == 1 and np.isfinite(losses[0]), losses
    metrics = trainer.evaluate()
    assert np.isfinite(metrics["recall@20"]) and np.isfinite(metrics["ndcg@20"])
