"""Optimizer step of the training loop on the device (SURVEY.md §8 a11 / f1).

`AdamW` / `Adam` are drop-ins for the `torch.optim.AdamW(model.parameters(), lr, weight_decay)` the
reference builds at scripts/train/train_baseline.py:252-256 and the `torch.optim.Adam(lr=1e-3)` of
scripts/pipeline/run_full_pipeline.py:210: same constructor arguments, `step() / zero_grad() /
state_dict() / load_state_dict()`, same per-parameter state keys (`step`, `exp_avg`, `exp_avg_sq`),
so `Trainer` (etpgt/train/trainer.py:125-127) and its checkpoints work unchanged.  The arithmetic of
torch's dense single-tensor update runs as ONE launch of `etpgt_adam_step` over every parameter.

Persistent gradient buffers ("grad sinks"): for large tables (>= `sink_bytes`, i.e. the item embedding)
the optimizer owns a zero-initialised gradient buffer that the path's backward kernels ACCUMULATE rows
into directly (ops.EmbedPE / ops.SampledLoss look the buffer up by the table's storage address), and
the step kernel clears it while it updates the parameter.  That removes, per step, two 84 MB memsets,
the 3 x 84 MB add that autograd needs to sum the two table gradients, and a separate zero_grad pass.

Data parallelism over peer memory (`parallel.PeerDataParallel`, created BEFORE the optimizer): the sink is the
gradient buffer inside this rank's peer region, and `step()` runs the whole gradient exchange itself —
barrier, dense-gradient sum over the peers, the table's reduce-scatter + AdamW + all-gather as one kernel
(`etpgt_dp_adam_table`), barrier — so no `allreduce_gradients` call and no NCCL collective is on the step.

Row-sparse ("lazy") updates of the sink tables, for large catalogues and small batches where a step touches a few
percent of the item rows: `AdamW(..., lazy_rows=True)` / `Adam(..., lazy_rows=True)` step each sink table with
`etpgt_adam_rows` (rows whose gradient row is all zero keep their value and moments: no weight decay, no moment
decay — NOT the reference's dense semantics), and `SparseAdam` is torch.optim.SparseAdam on `etpgt_sparse_adam`.
Both read the whole gradient but move p / m / v only for touched rows.  Under data parallelism they need the NCCL
exchange (every rank sees the same summed sink, so all make the same row decisions); a row-sparse table inside a
peer region raises NotImplementedError.
"""

from __future__ import annotations

import ctypes
import weakref

import torch

from . import _lib
from ._lib import stream


class _AdamTensor(ctypes.Structure):
    _fields_ = [("param", ctypes.c_void_p), ("grad", ctypes.c_void_p), ("exp_avg", ctypes.c_void_p),
                ("exp_avg_sq", ctypes.c_void_p), ("numel", ctypes.c_int64)]


# table storage address -> (weakref to the parameter, gradient buffer, owner optimizer)
_GRAD_SINKS: dict[int, tuple] = {}


def grad_sink_for(table: torch.Tensor):
    """The persistent gradient buffer registered for `table` (a parameter or its data), or None."""
    entry = _GRAD_SINKS.get(table.data_ptr())
    if entry is None:
        return None
    ref, buf, owner = entry
    param = ref()
    if param is None or param.data_ptr() != table.data_ptr() or buf.shape != table.shape:
        _GRAD_SINKS.pop(table.data_ptr(), None)
        return None
    owner_opt = owner()
    if param.grad is None:
        # `model.zero_grad()` / `table.grad = None` detached the buffer: its contents were "cleared" by that call,
        # and the next backward must find it attached again or the table would silently stop training
        if owner_opt is None or owner_opt._dirty:
            buf.zero_()
        param.grad = buf
    elif param.grad is not buf:
        # somebody installed a gradient of their own: accumulate there through autograd, not into the sink
        _GRAD_SINKS.pop(table.data_ptr(), None)
        return None
    if owner_opt is not None:
        owner_opt._dirty = True
    return buf


class _SinkOptimizer(torch.optim.Optimizer):
    """Gradient-sink bookkeeping shared by the device optimizers (see the module docstring)."""

    # row-sparse update of the sink tables (lazy AdamW / Adam, SparseAdam): they keep no exchange over peer memory
    row_sparse = False

    def _install_sinks(self, grad_sinks: bool, sink_bytes: int) -> None:
        self._dirty = False
        self._sinks: list[torch.nn.Parameter] = []
        self._plan_key = None
        self._plan = None
        self._peer = None          # parallel.PeerDataParallel owning the item table, if any
        from .parallel import peer_for

        for group in self.param_groups:
            for p in group["params"]:
                if not (p.is_cuda and p.dtype == torch.float32 and p.dim() == 2 and p.is_contiguous()):
                    continue
                # a table that lives in a peer region (data parallelism) always uses the region's gradient buffer
                if peer_for(p) is not None or (grad_sinks and p.numel() * 4 >= sink_bytes):
                    self._install_sink(p)

    # ------------------------------------------------------------------ gradient sinks
    def _install_sink(self, p):
        from .parallel import peer_for

        peer = peer_for(p)
        if peer is not None and self.row_sparse:
            self._refuse_peer()
        if peer is not None:       # the gradient buffer inside the peer region: the other ranks read it
            buf, self._peer = peer.table_grad, peer
        else:
            buf = torch.zeros_like(p)
        p.grad = buf
        _GRAD_SINKS[p.data_ptr()] = (weakref.ref(p), buf, weakref.ref(self))
        self._sinks.append(p)

    def attach_peer(self, peer) -> None:
        """Moves the item table's gradient sink into the peer region of `peer` (parallel.PeerDataParallel created
        AFTER this optimizer, e.g. by Trainer(process_group=...)): the table's storage address changed when it was
        re-homed, so the old registration is dropped and the region's gradient buffer takes over."""
        if self.row_sparse:
            self._refuse_peer()
        for group in self.param_groups:
            for p in group["params"]:
                if p.data_ptr() != peer.table.data_ptr():
                    continue
                for key, entry in list(_GRAD_SINKS.items()):
                    if entry[0]() is p:
                        _GRAD_SINKS.pop(key, None)
                self._sinks = [q for q in self._sinks if q is not p]
                self._install_sink(p)
        self._plan_key = None

    def _refuse_peer(self):
        raise NotImplementedError(
            f"{type(self).__name__}: a row-sparse table update over peer memory is not implemented; "
            'use data parallelism with exchange="nccl" (Trainer(..., exchange="nccl") or '
            'parallel.enable_data_parallel(model, group, exchange="nccl"))')

    def _is_sink(self, p) -> bool:
        entry = _GRAD_SINKS.get(p.data_ptr())
        return entry is not None and entry[0]() is p and p.grad is entry[1]

    def zero_grad(self, set_to_none: bool = True):
        """torch semantics, except that sink gradients stay allocated (they are already zero after a
        step; they are cleared here only if a backward ran since)."""
        for group in self.param_groups:
            for p in group["params"]:
                if self._is_sink(p):
                    if self._dirty:
                        p.grad.zero_()
                elif p.grad is not None:
                    if set_to_none:
                        p.grad = None
                    else:
                        p.grad.detach_()
                        p.grad.zero_()
        self._dirty = False


class _DeviceAdam(_SinkOptimizer):
    _decoupled = True

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, amsgrad=False,
                 grad_sinks=True, sink_bytes=4 << 20, lazy_rows=False):
        if amsgrad:
            raise NotImplementedError("etpgt_b200 optimizers implement amsgrad=False (the reference's setting)")
        if lr < 0.0 or eps < 0.0 or weight_decay < 0.0 or not 0.0 <= betas[0] < 1.0 or not 0.0 <= betas[1] < 1.0:
            raise ValueError("Invalid optimizer hyper-parameter")
        if lazy_rows and not grad_sinks:
            raise ValueError("lazy_rows=True updates the tables that have a gradient sink: it needs grad_sinks=True")
        defaults = dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay, amsgrad=False)
        super().__init__(params, defaults)
        self.lazy_rows = self.row_sparse = bool(lazy_rows)
        self._install_sinks(grad_sinks, sink_bytes)

    # ------------------------------------------------------------------ the step
    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        for group in self.param_groups:
            todo: dict[int, list] = {}
            bumped: dict[int, int] = {}       # id(step tensor) -> its new value: one increment per distinct tensor
            for p in group["params"]:
                if p.grad is None:
                    continue
                state = self.state[p]
                if len(state) == 0:
                    if not p.is_cuda:
                        raise RuntimeError("etpgt_b200 optimizers run on CUDA parameters only (no CPU fallback)")
                    if p.grad.is_sparse or p.dtype != torch.float32:
                        raise RuntimeError("etpgt_b200 optimizers need dense fp32 parameters and gradients")
                    # the parameters of a group step together: they share ONE step counter tensor (a host scalar,
                    # as in torch), so a step costs one host increment instead of one per parameter
                    shared = group.get("_shared_step")
                    state["step"] = shared if shared is not None else torch.tensor(0.0)
                    if shared is None and not bumped:
                        group["_shared_step"] = state["step"]
                    state["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    state["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                counter = state["step"]
                step_no = bumped.get(id(counter))
                if step_no is None:
                    counter += 1
                    step_no = bumped[id(counter)] = int(counter.item())
                todo.setdefault(step_no, []).append(p)
            for step_no, plist in todo.items():
                self._launch(group, step_no, plist)
        self._dirty = False
        return loss

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        self._plan_key = None      # the moment tensors were replaced: the cached launch plan holds freed pointers
        for group in self.param_groups:     # loaded counters are per parameter again: share equal ones
            group.pop("_shared_step", None)
            by_value: dict[float, torch.Tensor] = {}
            for p in group["params"]:
                state = self.state.get(p)
                if state and "step" in state:
                    value = float(state["step"])
                    state["step"] = by_value.setdefault(value, torch.as_tensor(state["step"], dtype=torch.float32).cpu())

    def state_dict(self):
        """torch's format; every parameter gets its own copy of the (shared) step counter."""
        out = super().state_dict()
        # (the packed per-parameter dicts are the live ones: copy before un-sharing the counter)
        out["state"] = {k: ({**st, "step": st["step"].clone()} if "step" in st else dict(st))
                        for k, st in out["state"].items()}
        for group in out["param_groups"]:
            group.pop("_shared_step", None)
        return out

    def add_param_group(self, param_group):
        super().add_param_group(param_group)
        self._plan_key = None

    def _launch(self, group, step_no, plist):
        beta1, beta2 = group["betas"]
        peer = self._peer
        if peer is not None and peer.world > 1:
            # data parallelism over peer memory: the gradient exchange is part of the step
            reduced = peer.exchange_dense()
            rest = []
            for p in plist:
                if p.data_ptr() == peer.table.data_ptr():
                    st = self.state[p]
                    peer.update_table(st["exp_avg"], st["exp_avg_sq"], group["lr"], beta1, beta2, group["eps"],
                                      group["weight_decay"], self._decoupled, step_no)
                else:
                    rest.append(p)
            peer.end_exchange()
            plist = rest
            if not plist:
                return
            if not reduced:    # gradients from the per-operator autograd path: not in the peer region
                from .parallel import allreduce_gradients

                allreduce_gradients(plist, group=peer.group)
        grads = [p.grad if p.grad.is_contiguous() else p.grad.contiguous() for p in plist]
        # the plan holds raw pointers of the moments too: load_state_dict / restore-best replace those tensors
        key = tuple((p.data_ptr(), g.data_ptr(), self.state[p]["exp_avg"].data_ptr(),
                     self.state[p]["exp_avg_sq"].data_ptr()) for p, g in zip(plist, grads))
        if key != self._plan_key:
            plain, sinks, lazy = [], [], []
            for p, g in zip(plist, grads):
                if not p.is_contiguous():
                    raise RuntimeError("etpgt_b200 optimizers need contiguous parameters")
                st = self.state[p]
                entry = _AdamTensor(p.data_ptr(), g.data_ptr(), st["exp_avg"].data_ptr(),
                                    st["exp_avg_sq"].data_ptr(), p.numel())
                if not self._is_sink(p):
                    plain.append(entry)
                elif self.lazy_rows:      # one row-sparse launch per table
                    lazy.append((entry.param, entry.grad, entry.exp_avg, entry.exp_avg_sq, p.size(0), p.size(1)))
                else:
                    sinks.append(entry)
            self._plan_key = key
            self._plan = ((_AdamTensor * max(len(plain), 1))(*plain), len(plain),
                          (_AdamTensor * max(len(sinks), 1))(*sinks), len(sinks), lazy)
        arr_plain, n_plain, arr_sink, n_sink, lazy = self._plan
        common = (float(group["lr"]), float(beta1), float(beta2), float(group["eps"]), float(group["weight_decay"]),
                  int(self._decoupled), int(step_no))
        # the sink gradients are cleared by the kernel (zero_grad flag); the others are released by
        # zero_grad(set_to_none=True) as usual
        if n_plain:
            _lib.call("etpgt_adam_step", arr_plain, n_plain, *common, 0, stream())
        if n_sink:
            _lib.call("etpgt_adam_step", arr_sink, n_sink, *common, 1, stream())
        for table in lazy:
            _lib.call("etpgt_adam_rows", *table, *common, 1, None, stream())


class AdamW(_DeviceAdam):
    """torch.optim.AdamW semantics (decoupled weight decay, default 1e-2) on `etpgt_adam_step`."""

    _decoupled = True

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, amsgrad=False, **kw):
        super().__init__(params, lr, betas, eps, weight_decay, amsgrad, **kw)


class Adam(_DeviceAdam):
    """torch.optim.Adam semantics (L2 weight decay added to the gradient, default 0)."""

    _decoupled = False

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, amsgrad=False, **kw):
        super().__init__(params, lr, betas, eps, weight_decay, amsgrad, **kw)


class SparseAdam(_SinkOptimizer):
    """torch.optim.SparseAdam on `etpgt_sparse_adam`: the same constructor checks, the same state (integer `step`,
    `exp_avg`, `exp_avg_sq`; state dicts load both ways with torch's class) and the same fp32 arithmetic, one
    rounding per torch operation.  Only the rows present in a step's gradient move: their moments and values are
    updated, every other row keeps its bits.

    * A sparse COO gradient (`nn.Embedding(sparse=True)`) is coalesced and every listed row is updated, all-zero
      rows included, as in torch.
    * Unlike torch, a dense gradient is accepted too: its rows with a nonzero element (or a NaN) are updated.  This
      is how the item table is trained here: 2-D fp32 CUDA parameters of at least `sink_bytes` get a persistent
      gradient buffer (a sink, as for `AdamW`) that the backward kernels accumulate rows into and the step clears.
    """

    row_sparse = True

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, maximize=False, *, grad_sinks=True,
                 sink_bytes=4 << 20):
        if isinstance(lr, torch.Tensor) and lr.numel() != 1:
            raise ValueError("Tensor lr must be 1-element")
        if not 0.0 < lr:
            raise ValueError(f"Invalid learning rate: {lr}")
        if not 0.0 < eps:
            raise ValueError(f"Invalid epsilon value: {eps}")
        if not 0.0 <= betas[0] < 1.0:
            raise ValueError(f"Invalid beta parameter at index 0: {betas[0]}")
        if not 0.0 <= betas[1] < 1.0:
            raise ValueError(f"Invalid beta parameter at index 1: {betas[1]}")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, maximize=maximize))
        for index, group in enumerate(self.param_groups):
            for d_index, p in enumerate(group["params"]):
                if p.is_sparse:
                    raise ValueError(f"Sparse params at indices {[[index, d_index]]}: SparseAdam requires dense "
                                     "parameter tensors")
                if p.is_complex():
                    raise ValueError(f"Complex params at indices {[[index, d_index]]}: SparseAdam does not support "
                                     "complex parameters")
        self._install_sinks(grad_sinks, sink_bytes)

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        for group in self.param_groups:
            beta1, beta2 = group["betas"]
            lr = float(group["lr"])
            for p in group["params"]:
                if p.grad is None:
                    continue
                if not (p.is_cuda and p.dtype == torch.float32 and p.is_contiguous()):
                    raise RuntimeError("etpgt_b200 SparseAdam needs contiguous fp32 CUDA parameters (no CPU fallback)")
                state = self.state[p]
                if len(state) == 0:
                    state["step"] = 0
                    state["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    state["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                state["step"] += 1
                rows = p.size(0) if p.dim() else 1
                dim = p.numel() // rows if rows else 1
                grad = p.grad
                if grad.is_sparse:
                    grad = grad.coalesce()
                    if grad.sparse_dim() != 1 or grad.dtype != torch.float32:
                        raise RuntimeError("SparseAdam: sparse gradients must be fp32 with one sparse dimension "
                                           "(rows, as nn.Embedding(sparse=True) produces)")
                    index = grad._indices()[0].contiguous()
                    values = grad._values().contiguous()
                    if values.numel() == 0:      # torch skips an empty gradient (the step still counts)
                        continue
                    g_ptr, i_ptr, nnz, zero = _lib.ptr(values), _lib.ptr(index), index.numel(), 0
                else:
                    if grad.dtype != torch.float32 or not grad.is_contiguous():
                        raise RuntimeError("SparseAdam: dense gradients must be contiguous fp32")
                    g_ptr, i_ptr, nnz, zero = _lib.ptr(grad), None, 0, int(self._is_sink(p))
                _lib.call("etpgt_sparse_adam", _lib.ptr(p), _lib.ptr(state["exp_avg"]),
                          _lib.ptr(state["exp_avg_sq"]), rows, dim, g_ptr, i_ptr, nnz, lr, float(beta1),
                          float(beta2), float(group["eps"]), int(bool(group["maximize"])), int(state["step"]), zero,
                          None, stream())
        self._dirty = False
        return loss
