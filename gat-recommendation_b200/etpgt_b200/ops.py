"""Host side of the hot path: graph index construction and the autograd Functions that hand
raw device pointers + the current stream to the C-ABI kernels (include/etpgt_b200.h).

PyTorch is plumbing here (device memory, streams, autograd bookkeeping); all arithmetic on the
path runs in libetpgt_b200.so — the dense node projections included (etpgt_gemm_bf16x3: tcgen05 split-bf16 GEMMs
on CTA pairs).  What stays in torch is element-wise work on parameter-sized tensors (the GAT score folds, weight
concatenations) and `torch.nn.functional.linear` for layer widths that are not multiples of 8 (no configuration of
the reference has one; `linear` warns once when it takes that route).
"""

from __future__ import annotations

import weakref

import torch
import torch.distributed as dist

from . import _lib
from ._lib import call, ptr, size, stream, workspace

READOUT_MODES = {"mean": 0, "max": 1, "last": 2, "attention": 3}
LOSS_MODES = {"bpr": 0, "listwise": 1, "dual": 2}


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"etpgt_b200: {what} must be a CUDA tensor (the B200 path has no CPU fallback)")


def _f32(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous() if t.dtype == torch.float32 else t.float().contiguous()


def _grad_sink(table: torch.Tensor):
    """Persistent gradient buffer of `table` if an etpgt_b200.optim optimizer registered one."""
    from .optim import grad_sink_for

    return grad_sink_for(table) if table.dtype == torch.float32 and table.is_contiguous() else None


def _table_grad(ctx, shape, device):
    """(buffer the library ADDS the table gradient into, what backward returns for the table, input 1): the optim
    gradient sink and None when one is registered, else a dense fp32 zero tensor twice; (None, None) if not needed."""
    if not ctx.needs_input_grad[1]:
        return None, None
    sink = _grad_sink(ctx.table_ref)
    d_table = sink if sink is not None else torch.zeros(shape, dtype=torch.float32, device=device)
    return d_table, (None if sink is not None else d_table)


def _weight_and_padding(item_embeddings):
    return getattr(item_embeddings, "weight", item_embeddings), getattr(item_embeddings, "padding_idx", None)


def _i64(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous() if t.dtype == torch.int64 else t.long().contiguous()


# ------------------------------------------------------------------------------ graph index


class GraphIndex:
    """Destination-sorted CSR + source-sorted CSC of one batched graph, built once per batch on
    the device and shared by every conv layer (forward and backward)."""

    __slots__ = ("num_nodes", "num_edges", "rowptr", "col", "eperm", "colptr", "row", "cpos", "slot", "generation",
                 "_hub")

    HUB_THRESHOLD = 256      # kHubThreshold of csrc/tconv.cuh

    def __init__(self, edge_index: torch.Tensor, num_nodes: int, out: torch.Tensor | None = None,
                 ws: torch.Tensor | None = None, build: bool = True):
        """`out` (optional): an int32 buffer of at least `GraphIndex.out_elems(num_nodes, num_edges)` elements the
        six arrays are carved from; `ws`: a byte workspace of at least etpgt_csr_workspace_bytes; build=False
        only carves the arrays (the caller fills them, see prepare_batch)."""
        _require_cuda(edge_index, "edge_index")
        edge_index = _i64(edge_index)
        dev = edge_index.device
        e = int(edge_index.size(1))
        num_nodes = int(num_nodes)
        self.num_nodes, self.num_edges = num_nodes, e
        self.slot, self.generation = None, 0      # set by prepare_batch when the arrays live in a BatchPreparer slot
        self._hub = None
        if out is None:
            out = torch.empty(self.out_elems(num_nodes, e), dtype=torch.int32, device=dev)
        o1 = _pad64(num_nodes + 1)
        o2, oe = 2 * o1, _pad64(e)
        self.rowptr, self.colptr = out[:num_nodes + 1], out[o1:o1 + num_nodes + 1]
        self.col, self.eperm = out[o2:o2 + e], out[o2 + oe:o2 + oe + e]
        self.row, self.cpos = out[o2 + 2 * oe:o2 + 2 * oe + e], out[o2 + 3 * oe:o2 + 3 * oe + e]
        if not build:
            return
        if ws is None:
            ws = workspace(size("etpgt_csr_workspace_bytes", e, num_nodes), dev)
        call("etpgt_csr_from_coo", ptr(edge_index[0]), ptr(edge_index[1]), e, num_nodes,
             ptr(self.rowptr), ptr(self.col), ptr(self.eperm), ptr(self.colptr), ptr(self.row), ptr(self.cpos),
             ptr(ws), ws.numel(), stream())

    @staticmethod
    def out_elems(num_nodes: int, num_edges: int) -> int:
        return 2 * _pad64(num_nodes + 1) + 4 * _pad64(num_edges)

    def hub_plan(self) -> torch.Tensor | None:
        """The hub-row plan of this graph (etpgt_hub_plan: destinations / sources with more than 256 edges cut into
        chunks) or None when it has no such row.  Built at first use and kept with the index; costs one host read
        of the four counts (session batches, whose rows have at most 51 edges, answer None every time)."""
        if self._hub is None:
            self._hub = False
            if self.num_edges > self.HUB_THRESHOLD:
                dev = self.rowptr.device
                plan = torch.empty(size("etpgt_hub_plan_bytes", self.num_edges), dtype=torch.uint8, device=dev)
                ws = workspace(size("etpgt_hub_plan_workspace_bytes", self.num_nodes), dev)
                call("etpgt_hub_plan", ptr(self.rowptr), ptr(self.colptr), self.num_nodes, self.num_edges, ptr(plan),
                     ptr(ws), ws.numel(), stream())
                counts = plan[:16].view(torch.int32).tolist()
                if counts[0] or counts[2]:
                    self._hub = plan
        return self._hub if self._hub is not False else None


def _pad64(n: int) -> int:
    """int32 element counts rounded to 256 bytes, so that every array carved from one buffer stays aligned."""
    return (int(n) + 63) // 64 * 64


def graph_index_of(batch, edge_index: torch.Tensor, num_nodes: int) -> GraphIndex:
    """Cached on the batch object so that L layers and the backward pass share one build."""
    cached = getattr(batch, "_etpgt_index", None)
    if cached is not None and cached[0] is edge_index and cached[1].num_nodes == num_nodes and _slot_valid(cached[1]):
        return cached[1]
    index = GraphIndex(edge_index, num_nodes)
    try:
        object.__setattr__(batch, "_etpgt_index", (edge_index, index))
    except Exception:  # exotic batch containers: just rebuild next time
        pass
    return index


def _slot_valid(obj) -> bool:
    """An index / plan carved from a BatchPreparer slot is valid until that slot is refilled."""
    return obj.slot is None or obj.slot.generation == obj.generation


def segment_ptr(batch_vec: torch.Tensor, num_sessions: int) -> torch.Tensor:
    _require_cuda(batch_vec, "batch")
    batch_vec = _i64(batch_vec)
    out = torch.empty(num_sessions + 1, dtype=torch.int32, device=batch_vec.device)
    call("etpgt_segment_ptr", ptr(batch_vec), batch_vec.numel(), num_sessions, ptr(out), stream())
    return out


# ------------------------------------------------------------------------------ scatter plans


class ScatterPlan:
    """Stable sort of the keys of one row scatter (`etpgt_scatter_plan`): `sorted_key [m]`, `perm [m]`.
    The keys of both table-gradient scatters of a step — the batch's node ids (embedding backward) and
    [target | negatives] per session (loss backward) — are inputs of the batch, so their sorts are batch
    preparation (the device-side counterpart of the reference's collate, dataloader.py:157-202), not part
    of the step's dependent chain."""

    __slots__ = ("m", "sorted_key", "perm", "slot", "generation")

    def __init__(self, keys: torch.Tensor, num_rows: int, negatives: torch.Tensor | None = None,
                 out: torch.Tensor | None = None, ws: torch.Tensor | None = None, build: bool = True):
        """keys [m] — or, with `negatives` [B, num_neg], keys = targets [B] and the plan covers the loss layout
        [b][0] = target, [b][1 + c] = negative c.  `out`: int32 buffer of >= 2 * _pad64(m) elements; build=False
        only carves the two arrays (the caller fills them, see prepare_batch)."""
        _require_cuda(keys, "scatter keys")
        keys = _i64(keys).reshape(-1)
        dev = keys.device
        self.slot, self.generation = None, 0
        if negatives is not None:
            negatives = _i64(negatives)
            b = int(keys.numel())
            num_neg = negatives.numel() // max(b, 1)
            self.m = b * (num_neg + 1)
        else:
            self.m = int(keys.numel())
        if out is None:
            out = torch.empty(2 * _pad64(self.m), dtype=torch.int32, device=dev)
        self.sorted_key, self.perm = out[:self.m], out[_pad64(self.m):_pad64(self.m) + self.m]
        if not build:
            return
        if ws is None:
            ws = workspace(size("etpgt_scatter_plan_workspace_bytes", self.m), dev)
        if negatives is not None:
            call("etpgt_scatter_plan_loss", ptr(keys), ptr(negatives), b, num_neg, int(num_rows),
                 ptr(self.sorted_key), ptr(self.perm), ptr(ws), ws.numel(), stream())
        else:
            call("etpgt_scatter_plan", ptr(keys), self.m, int(num_rows), ptr(self.sorted_key), ptr(self.perm),
                 ptr(ws), ws.numel(), stream())


# Plans are found again by the identity of the key tensors' memory: (data_ptr, numel) of the tensors the plan
# was made from, valid while those tensors are alive and unmodified (weak references + version counters).
_PLANS: dict = {}


def _plan_key(*tensors):
    return tuple((t.data_ptr(), t.numel()) for t in tensors)


def _register_plan(plan: ScatterPlan, *tensors) -> None:
    key = _plan_key(*tensors)

    def drop(_ref, key=key):
        _PLANS.pop(key, None)

    _PLANS[key] = (plan, tuple(weakref.ref(t, drop) for t in tensors), tuple(t._version for t in tensors))


def _find_plan(*tensors):
    if not _PLANS:
        return None
    entry = _PLANS.get(_plan_key(*tensors))
    if entry is None:
        return None
    plan, refs, versions = entry
    for t, ref, version in zip(tensors, refs, versions):
        base = ref()
        # a view of the planned tensor (e.g. the trainer's negative_items.view(B, -1), trainer.py:87-89)
        # shares its version counter
        if base is None or base.device != t.device or t._version != version:
            return None
    return plan if _slot_valid(plan) else None


class PreparedBatch:
    """What `prepare_batch` built: the graph index and the two scatter plans, all carved from ONE int32 buffer
    (`tensors()` lists what a caller must `record_stream` when preparation runs on a side stream)."""

    __slots__ = ("index", "plan_nodes", "plan_loss", "buffer", "scratch", "slot")

    def tensors(self):
        return [self.buffer, self.scratch]

    def release(self) -> None:
        """Call on the stream that consumed the batch, after its last kernel is queued: the pool slot behind this
        preparation may then be refilled once that stream gets here (no-op without a pool)."""
        if getattr(self, "slot", None) is not None:
            self.slot.free.record()
            self.slot.busy = False


class _PrepareSlot:
    __slots__ = ("buffer", "scratch", "free", "busy", "generation")


class BatchPreparer:
    """Ring of reusable preparation buffers for a loader that prepares batches ahead of the training step on a side
    stream: `prepare_batch(batch, num_items, pool=...)` fills the next slot instead of allocating, after making
    its stream wait (on the device, no host sync) for the step that last consumed that slot —
    `prepared.release()`, called by the consumer.  A slot that was never released is left alone and replaced by a
    fresh one; slots grow (with head-room) when a larger batch arrives, so a steady loop allocates nothing."""

    def __init__(self, depth: int = 4):
        self.depth, self.slots, self.next = int(depth), [], 0

    def acquire(self, elems: int, scratch_bytes: int, device) -> _PrepareSlot:
        if len(self.slots) < self.depth:
            self.slots.append(None)
        i = self.next % self.depth
        self.next += 1
        slot = self.slots[i]
        if slot is not None and (slot.busy or slot.buffer.numel() < elems or slot.scratch.numel() < scratch_bytes
                                 or slot.buffer.device != torch.device(device)):
            if slot.busy:      # its consumer never released it: it may still be in use
                slot = None
            else:              # too small: the consumer is done with it once `free` has passed
                torch.cuda.current_stream().wait_event(slot.free)
                slot = None
        if slot is None:
            slot = _PrepareSlot()
            slot.buffer = torch.empty(elems + elems // 8, dtype=torch.int32, device=device)
            slot.scratch = workspace(scratch_bytes + scratch_bytes // 8, device)
            slot.free = torch.cuda.Event()
            slot.generation = 0
            self.slots[i] = slot
        else:
            torch.cuda.current_stream().wait_event(slot.free)
        slot.busy = True
        slot.generation += 1      # indexes / plans carved from the previous filling are no longer valid
        return slot


def prepare_batch(batch, num_items: int | None = None, pool: "BatchPreparer | None" = None) -> PreparedBatch:
    """Integer preparation of one batch on the current stream: CSR / CSC index of `batch.edge_index` and, when
    the table size is given, the scatter plans of `batch.x` and of `batch.target_item | batch.negative_items`.
    Everything here depends on the batch's inputs only, so a loader (or a side stream one step ahead) runs
    it off the training step's critical path; the model and the loss find the results again through the
    batch object / the key tensors.  Without this call the step builds the same things inline.
    Host cost: two allocations (none with a `pool`) and one library call."""
    prepared = PreparedBatch()
    edge_index, ids = batch.edge_index, batch.x
    _require_cuda(ids, "batch.x")
    n, e = int(ids.numel()), int(edge_index.size(1))
    dev = ids.device
    prepared.plan_nodes = prepared.plan_loss = None
    prepared.slot = None

    def buffers(elems: int, scratch_bytes: int):
        if pool is None:
            return torch.empty(elems, dtype=torch.int32, device=dev), workspace(scratch_bytes, dev)
        prepared.slot = pool.acquire(elems, scratch_bytes, dev)
        return prepared.slot.buffer[:elems], prepared.slot.scratch

    if num_items is None or n == 0:      # the index alone
        prepared.buffer, prepared.scratch = buffers(GraphIndex.out_elems(n, e), size("etpgt_csr_workspace_bytes", e, n))
        prepared.index = GraphIndex(edge_index, n, out=prepared.buffer, ws=prepared.scratch)
    else:
        # index + both scatter plans from ONE library call (etpgt_batch_prepare: the destination sort and the two
        # plan sorts are a single segmented radix sort), outputs carved from one buffer
        edge_index, ids = _i64(edge_index), _i64(ids)
        targets, negatives = getattr(batch, "target_item", None), getattr(batch, "negative_items", None)
        plan_loss = targets is not None and negatives is not None and targets.numel() > 0
        b = int(targets.numel()) if plan_loss else 0
        num_neg = int(negatives.numel()) // b if plan_loss else 0
        m_loss = b * (num_neg + 1)
        if plan_loss:
            targets, negatives = _i64(targets), _i64(negatives)
        elems_index, elems_nodes = GraphIndex.out_elems(n, e), 2 * _pad64(n)
        prepared.buffer, prepared.scratch = buffers(elems_index + elems_nodes + 2 * _pad64(m_loss),
                                                    size("etpgt_batch_prepare_workspace_bytes", e, n, m_loss))
        index = prepared.index = GraphIndex(edge_index, n, out=prepared.buffer, build=False)
        nodes = prepared.plan_nodes = ScatterPlan(ids, num_items, out=prepared.buffer[elems_index:], build=False)
        loss = None
        if plan_loss:
            loss = prepared.plan_loss = ScatterPlan(targets, num_items, negatives=negatives,
                                                    out=prepared.buffer[elems_index + elems_nodes:], build=False)
        call("etpgt_batch_prepare", ptr(edge_index[0]), ptr(edge_index[1]), e, n, ptr(ids),
             ptr(targets) if plan_loss else None, ptr(negatives) if plan_loss else None, b, num_neg, int(num_items),
             ptr(index.rowptr), ptr(index.col), ptr(index.eperm), ptr(index.colptr), ptr(index.row), ptr(index.cpos),
             ptr(nodes.sorted_key), ptr(nodes.perm), ptr(loss.sorted_key) if loss else None,
             ptr(loss.perm) if loss else None, ptr(prepared.scratch), prepared.scratch.numel(), stream())
        _register_plan(nodes, batch.x)
        if loss is not None:
            _register_plan(loss, batch.target_item, batch.negative_items)
        # ids index the table (and its gradient buffer) raw: flag anything outside [0, num_items)
        call("etpgt_ids_check", ptr(ids), n, ptr(targets) if plan_loss else None, b,
             ptr(negatives) if plan_loss else None, b * num_neg, int(num_items), ptr(_bad_ids_flag(dev)), stream())
    if prepared.slot is not None:
        for obj in (prepared.index, prepared.plan_nodes, prepared.plan_loss):
            if obj is not None:
                obj.slot, obj.generation = prepared.slot, prepared.slot.generation
    try:
        object.__setattr__(batch, "_etpgt_index", (batch.edge_index, prepared.index))
        object.__setattr__(batch, "_etpgt_prepared", prepared)   # keeps the plans alive with the batch
    except Exception:
        pass
    return prepared


_BAD_IDS: dict = {}


def _bad_ids_flag(device) -> torch.Tensor:
    """Sticky device flag (int32[1]) set by etpgt_ids_check when a prepared batch held an item id outside the
    table."""
    key = torch.device(device).index or 0
    flag = _BAD_IDS.get(key)
    if flag is None:
        flag = _BAD_IDS[key] = torch.zeros(1, dtype=torch.int32, device=device)
    return flag


def check_item_ids(device="cuda") -> None:
    """Raises IndexError (what the reference's nn.Embedding raises, etpgt/model/base.py:36) if any batch prepared
    on `device` since the last call held an item id outside [0, num_items).  One host read; trainers call it once
    per epoch, loaders validate their CSV ids up front."""
    flag = _BAD_IDS.get(torch.device(device).index or 0)
    if flag is not None and int(flag.item()):
        flag.zero_()
        raise IndexError("index out of range in self: a batch holds item ids outside [0, num_items) "
                         "(e.g. a validation file with items the model was not sized for)")


# ------------------------------------------------------------------------------ embedding + PE


class EmbedPE(torch.autograd.Function):
    """x0 = table[ids] (+ pe @ w_pe^T + b_pe)   — etpgt/model/graph_transformer.py:140-152."""

    @staticmethod
    def forward(ctx, ids, table, pe, pe_per_node, w_pe, b_pe, padding_idx, want_split=False):
        """want_split: also return the bf16 hi/lo split of x0 (non-differentiable), the operand format of the
        first layer's tensor-core projection — (x0, hi, lo) instead of x0."""
        _require_cuda(table, "item_embedding.weight")
        ids = _i64(ids)
        table_c = _f32(table)
        n, dim = ids.numel(), table_c.size(1)
        out = torch.empty(n, dim, dtype=torch.float32, device=table_c.device)
        k_pe = 0
        if pe is not None:
            pe, w_pe_c, b_pe_c = _f32(pe), _f32(w_pe), _f32(b_pe)
            k_pe = pe.size(1)
        else:
            w_pe_c = b_pe_c = None
        hi = lo = None
        if want_split:
            hi = torch.empty(n, dim, dtype=torch.bfloat16, device=table_c.device)
            lo = torch.empty(n, dim, dtype=torch.bfloat16, device=table_c.device)
        call("etpgt_embed_pe_fwd_split", ptr(ids), n, ptr(table_c), table_c.size(0), ptr(pe), int(bool(pe_per_node)),
             ptr(w_pe_c), ptr(b_pe_c), k_pe, dim, ptr(out), ptr(hi), ptr(lo), stream())
        ctx.save_for_backward(ids, pe)
        ctx.table_ref = table
        ctx.plan = _find_plan(ids)          # per-batch sort of the node ids, if prepare_batch made one
        ctx.meta = (table_c.size(0), dim, k_pe, int(bool(pe_per_node)), -1 if padding_idx is None else int(padding_idx))
        if want_split:
            ctx.set_materialize_grads(False)
            ctx.mark_non_differentiable(hi, lo)
            return out, hi, lo
        return out

    @staticmethod
    def backward(ctx, d_out, *_unused):
        ids, pe = ctx.saved_tensors
        num_items, dim, k_pe, per_node, padding_idx = ctx.meta
        d_out = _f32(d_out)
        dev = d_out.device
        n = ids.numel()
        d_table, table_grad = _table_grad(ctx, (num_items, dim), dev)
        d_w = d_b = None
        if pe is not None:
            d_w = torch.empty(dim, k_pe, dtype=torch.float32, device=dev)
            d_b = torch.empty(dim, dtype=torch.float32, device=dev)
        ws = workspace(size("etpgt_embed_pe_bwd_workspace_bytes", n, dim, max(k_pe, 1)), dev)
        plan = ctx.plan if d_table is not None and ctx.plan is not None and ctx.plan.m == n else None
        call("etpgt_embed_pe_bwd_planned", ptr(ids), n, ptr(d_out), num_items, ptr(pe), per_node, k_pe, dim,
             padding_idx, ptr(plan.sorted_key) if plan else None, ptr(plan.perm) if plan else None,
             ptr(d_table), ptr(d_w), ptr(d_b), ptr(ws), ws.numel(), stream())
        return None, table_grad, None, None, d_w, d_b, None, None


# ------------------------------------------------------------------------------ TransformerConv


def _tconv_fwd(qkvs, n, dim, heads, index: GraphIndex, w_beta, mask, out, agg, beta, m, inv_l, bn_sums=None) -> None:
    """etpgt_tconv_fwd, with the hub-row kernels when the graph has rows of more than 256 edges; bn_sums (double
    [>= 2*dim]): the BatchNorm statistics of `out` are taken by the same kernel (etpgt_tconv_fwd_bn)."""
    hub = index.hub_plan()
    hub_ws = workspace(size("etpgt_tconv_hub_workspace_bytes", index.num_edges, dim), qkvs.device) if hub is not None else None
    hub_bytes = hub_ws.numel() if hub_ws is not None else 0
    if bn_sums is None:
        call("etpgt_tconv_fwd_hub", ptr(qkvs), n, dim, heads, ptr(index.rowptr), ptr(index.col), ptr(index.eperm),
             index.num_edges, ptr(w_beta), ptr(mask), ptr(out), ptr(agg), ptr(beta), ptr(m), ptr(inv_l), ptr(hub),
             ptr(hub_ws), hub_bytes, stream())
        return
    ws = workspace(size("etpgt_tconv_fwd_bn_workspace_bytes", dim), qkvs.device)
    call("etpgt_tconv_fwd_bn", ptr(qkvs), n, dim, heads, ptr(index.rowptr), ptr(index.col), ptr(index.eperm),
         index.num_edges, ptr(w_beta), ptr(mask), ptr(out), ptr(agg), ptr(beta), ptr(m), ptr(inv_l), ptr(hub),
         ptr(hub_ws), hub_bytes, ptr(bn_sums), ptr(ws), ws.numel(), stream())


def _tconv_bwd(qkvs, d_out, n, dim, heads, index: GraphIndex, w_beta, mask, agg, beta, m, inv_l, d_qkvs, g_hi, g_lo,
               d_bias, d_w_beta) -> None:
    """etpgt_tconv_bwd_split (fp32 d_qkvs, or the bf16 hi / lo operand pair + bias column sums), hub rows included."""
    dev = qkvs.device
    ws = workspace(size("etpgt_tconv_bwd_workspace_bytes", n, index.num_edges, dim, heads), dev)
    hub = index.hub_plan()
    hub_ws = workspace(size("etpgt_tconv_hub_workspace_bytes", index.num_edges, dim), dev) if hub is not None else None
    call("etpgt_tconv_bwd_split_hub", ptr(qkvs), ptr(d_out), n, dim, heads, ptr(index.rowptr), ptr(index.col),
         ptr(index.eperm), ptr(index.colptr), ptr(index.row), ptr(index.cpos), index.num_edges, ptr(w_beta), ptr(mask),
         ptr(agg), ptr(beta), ptr(m), ptr(inv_l), ptr(d_qkvs), ptr(g_hi), ptr(g_lo), ptr(d_bias), ptr(d_w_beta), ptr(ws),
         ws.numel(), ptr(hub), ptr(hub_ws), hub_ws.numel() if hub_ws is not None else 0, stream())


class TransformerConvFn(torch.autograd.Function):
    """Fused attention + aggregation + gate over the CSR (etpgt_tconv_fwd / _bwd)."""

    @staticmethod
    def forward(ctx, qkvs, w_beta, alpha_mask, index: GraphIndex, heads: int):
        _require_cuda(qkvs, "node features")
        qkvs = _f32(qkvs)
        n, dim = qkvs.size(0), qkvs.size(1) // 4
        dev = qkvs.device
        w_beta_c = _f32(w_beta).reshape(-1) if w_beta is not None else None
        mask_c = _f32(alpha_mask) if alpha_mask is not None else None
        f32 = dict(dtype=torch.float32, device=dev)
        out = torch.empty(n, dim, **f32)
        agg = torch.empty(n, dim, **f32)
        beta = torch.empty(n, **f32)
        m = torch.empty(n, heads, **f32)
        inv_l = torch.empty(n, heads, **f32)
        _tconv_fwd(qkvs, n, dim, heads, index, w_beta_c, mask_c, out, agg, beta, m, inv_l)
        ctx.save_for_backward(qkvs, w_beta_c, mask_c, agg, beta, m, inv_l)
        ctx.index, ctx.heads = index, heads
        ctx.w_beta_shape = None if w_beta is None else tuple(w_beta.shape)
        return out

    @staticmethod
    def backward(ctx, d_out):
        qkvs, w_beta, mask, agg, beta, m, inv_l = ctx.saved_tensors
        index, heads = ctx.index, ctx.heads
        d_out = _f32(d_out)
        n, dim = qkvs.size(0), qkvs.size(1) // 4
        dev = qkvs.device
        d_qkvs = torch.empty_like(qkvs)
        d_w_beta = torch.empty(3 * dim, dtype=torch.float32, device=dev) if w_beta is not None else None
        _tconv_bwd(qkvs, d_out, n, dim, heads, index, w_beta, mask, agg, beta, m, inv_l, d_qkvs, None, None, None,
                   d_w_beta)
        if d_w_beta is not None:
            d_w_beta = d_w_beta.view(ctx.w_beta_shape)
        return d_qkvs, d_w_beta, None, None, None


# ------------------------------------------------------------------------------ dense projections


def _split(src: torch.Tensor, rowmajor: bool, transposed: bool, colsum: bool = False):
    """fp32 [R, C] -> bf16 hi/lo parts (x = hi + lo), row-major and/or transposed, + column sums."""
    r, c = src.shape
    dev = src.device
    bf = dict(dtype=torch.bfloat16, device=dev)
    hi = lo = hi_t = lo_t = sums = None
    ld_t = (r + 7) // 8 * 8
    if rowmajor:
        hi, lo = torch.empty(r, c, **bf), torch.empty(r, c, **bf)
    if transposed:
        hi_t, lo_t = torch.empty(c, ld_t, **bf), torch.empty(c, ld_t, **bf)
    if colsum:
        sums = torch.empty(c, dtype=torch.float32, device=dev)
    ws = workspace(size("etpgt_split_bf16_workspace_bytes", r, c) if colsum else 256, dev)
    call("etpgt_split_bf16", ptr(src), r, c, c, ptr(hi), ptr(lo), c, ptr(hi_t), ptr(lo_t), ld_t, ptr(sums), ptr(ws),
         ws.numel(), stream())
    return hi, lo, hi_t, lo_t, ld_t, sums


def _gemm_x3(a_hi, a_lo, b_hi, b_lo, m, n, k, lda, ldb, bias, split_k=1, a_mn=False, b_mn=False,
             accumulate_into=None) -> torch.Tensor:
    """C[m,n] = A B^T (+bias).  a_mn / b_mn: that operand is stored as its transpose ([k, m] / [k, n]
    row-major) and read MN-major by the tensor cores — no transposed copy is made.  accumulate_into: an
    existing fp32 [m, n] tensor the product is ADDED to (TMA reduce-add) and that is returned."""
    out = accumulate_into if accumulate_into is not None else torch.empty(m, n, dtype=torch.float32, device=a_hi.device)
    ws = workspace(size("etpgt_gemm_bf16x3_workspace_bytes", m, n, k, split_k), a_hi.device)
    call("etpgt_gemm_bf16x3_ex", ptr(a_hi), ptr(a_lo), ptr(b_hi), ptr(b_lo), m, n, k, lda, ldb, int(a_mn), int(b_mn),
         ptr(bias), int(accumulate_into is not None), ptr(out), n, split_k, ptr(ws), ws.numel(), stream())
    return out


class LinearTensorCore(torch.autograd.Function):
    """y = x @ W^T + b on the tcgen05 tensor cores with split-bf16 operands (fp32-grade accuracy,
    etpgt_gemm_bf16x3_ex).  The hi/lo splits of x and W made for the forward are kept for the backward,
    whose two GEMMs read them (and the split of dY) MN-major: dX = dY x W, dW = dY^T x X (K = nodes,
    deterministic split-K); db is the column sum produced while splitting dY.  Per layer and step:
    three split passes (x, W, dY) and three GEMMs, no transposed copies."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        _require_cuda(x, "node features")
        x, weight = _f32(x), _f32(weight)
        bias_c = _f32(bias) if bias is not None else None
        n, k = x.shape
        n_out = weight.size(0)
        x_hi, x_lo, _, _, _, _ = _split(x, True, False)
        w_hi, w_lo, _, _, _, _ = _split(weight, True, False)
        y = _gemm_x3(x_hi, x_lo, w_hi, w_lo, n, n_out, k, k, k, bias_c)
        ctx.save_for_backward(x_hi, x_lo, w_hi, w_lo)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, d_y):
        x_hi, x_lo, w_hi, w_lo = ctx.saved_tensors
        d_y = _f32(d_y)
        n, k = x_hi.shape
        n_out = w_hi.size(0)
        need_x, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        g_hi, g_lo, _, _, _, d_bias = _split(d_y, True, False, colsum=ctx.has_bias)
        d_x = d_w = None
        if need_x:   # dX[n, k] = dY[n, n_out] x W[n_out, k]: B = W^T given as W, MN-major
            d_x = _gemm_x3(g_hi, g_lo, w_hi, w_lo, n, k, n_out, n_out, k, None, b_mn=True)
        if need_w:   # dW[n_out, k] = dY^T x X: both operands given by their row-major [nodes, .] splits
            d_w = _gemm_x3(g_hi, g_lo, x_hi, x_lo, n_out, k, n, n_out, k, None, split_k=0, a_mn=True, b_mn=True)
        return d_x, d_w, d_bias


class TransformerConvLayer(torch.autograd.Function):
    """One whole TransformerConv layer (etpgt/model/graph_transformer.py:73-98,174): the fused
    query|key|value|skip projection on the tensor cores, then the fused attention / aggregation / gate
    kernel.  Joining the two lets the backward edge kernels write the projection gradient d(qkvs) directly
    as split-bf16 tensor-core operands together with its column sums (the bias gradient)
    (etpgt_tconv_bwd_split): the [N, 4*dim] fp32 gradient and its split pass never exist."""

    @staticmethod
    def forward(ctx, x, weight, bias, w_beta, alpha_mask, index: GraphIndex, heads: int):
        _require_cuda(x, "node features")
        x, weight, bias_c = _f32(x), _f32(weight), _f32(bias)
        n, k = x.shape
        width = weight.size(0)
        dim = width // 4
        dev = x.device
        x_hi, x_lo, _, _, _, _ = _split(x, True, False)
        w_hi, w_lo, _, _, _, _ = _split(weight, True, False)
        qkvs = _gemm_x3(x_hi, x_lo, w_hi, w_lo, n, width, k, k, k, bias_c)
        w_beta_c = _f32(w_beta).reshape(-1) if w_beta is not None else None
        mask_c = _f32(alpha_mask) if alpha_mask is not None else None
        f32 = dict(dtype=torch.float32, device=dev)
        out, agg = torch.empty(n, dim, **f32), torch.empty(n, dim, **f32)
        beta, m, inv_l = torch.empty(n, **f32), torch.empty(n, heads, **f32), torch.empty(n, heads, **f32)
        _tconv_fwd(qkvs, n, dim, heads, index, w_beta_c, mask_c, out, agg, beta, m, inv_l)
        ctx.save_for_backward(x_hi, x_lo, w_hi, w_lo, qkvs, w_beta_c, mask_c, agg, beta, m, inv_l)
        ctx.index, ctx.heads = index, heads
        ctx.w_beta_shape = None if w_beta is None else tuple(w_beta.shape)
        return out

    @staticmethod
    def backward(ctx, d_out):
        x_hi, x_lo, w_hi, w_lo, qkvs, w_beta, mask, agg, beta, m, inv_l = ctx.saved_tensors
        index, heads = ctx.index, ctx.heads
        d_out = _f32(d_out)
        n, k = x_hi.shape
        width = w_hi.size(0)
        dim = width // 4
        dev = d_out.device
        g_hi = torch.empty(n, width, dtype=torch.bfloat16, device=dev)
        g_lo = torch.empty(n, width, dtype=torch.bfloat16, device=dev)
        d_bias = torch.empty(width, dtype=torch.float32, device=dev)
        d_w_beta = torch.empty(3 * dim, dtype=torch.float32, device=dev) if w_beta is not None else None
        _tconv_bwd(qkvs, d_out, n, dim, heads, index, w_beta, mask, agg, beta, m, inv_l, None, g_hi, g_lo, d_bias,
                   d_w_beta)
        d_x = d_w = None
        if ctx.needs_input_grad[0]:
            d_x = _gemm_x3(g_hi, g_lo, w_hi, w_lo, n, k, width, width, k, None, b_mn=True)
        if ctx.needs_input_grad[1]:
            d_w = _gemm_x3(g_hi, g_lo, x_hi, x_lo, width, k, n, width, k, None, split_k=0, a_mn=True, b_mn=True)
        if d_w_beta is not None:
            d_w_beta = d_w_beta.view(ctx.w_beta_shape)
        return d_x, d_w, d_bias, d_w_beta, None, None, None


class TransformerLayer(torch.autograd.Function):
    """One whole layer of the optimized GraphTransformer (etpgt/model/graph_transformer.py:172-177):

        y = dropout_p( BatchNorm1d( TransformerConv(x, edges) ) + x )

    Forward: split(x) [skipped when the previous layer already produced it] -> projection GEMM ->
    fused conv -> BN statistics (all-reduced under data parallelism) -> one apply kernel doing affine +
    residual + Philox dropout and, when asked, the bf16 split of y for the next layer.
    Backward: BN statistics / apply with the regenerated dropout mask (also emitting the residual
    branch's gradient), the edge kernels writing split-bf16 d(qkvs) + bias column sums, then
    dX = d_res + dQKVS x W (accumulated by the GEMM's TMA reduce-add) and dW (split-K).
    No dropout mask, no fp32 d(qkvs), no autograd add for the residual ever touch HBM."""

    @staticmethod
    def forward(ctx, x, x_split, weight, bias, w_beta, alpha_mask, index: GraphIndex, heads, gamma, bn_bias,
                running_mean, running_var, training, momentum, eps, group, drop_p, drop_seed, want_split):
        _require_cuda(x, "node features")
        x, weight, bias_c = _f32(x), _f32(weight), _f32(bias)
        n, k = x.shape
        width = weight.size(0)
        dim = width // 4
        dev = x.device
        if x_split is None:
            x_hi, x_lo, _, _, _, _ = _split(x, True, False)
        else:
            x_hi, x_lo = x_split
        w_hi, w_lo, _, _, _, _ = _split(weight, True, False)
        qkvs = _gemm_x3(x_hi, x_lo, w_hi, w_lo, n, width, k, k, k, bias_c)
        w_beta_c = _f32(w_beta).reshape(-1) if w_beta is not None else None
        mask_c = _f32(alpha_mask) if alpha_mask is not None else None
        f32 = dict(dtype=torch.float32, device=dev)
        conv_out, agg = torch.empty(n, dim, **f32), torch.empty(n, dim, **f32)
        beta, m, inv_l = torch.empty(n, **f32), torch.empty(n, heads, **f32), torch.empty(n, heads, **f32)
        sums = torch.empty(2 * dim + 1, dtype=torch.float64, device=dev) if training else None
        # (training: the BatchNorm statistics of the conv output are taken by the conv kernel itself)
        _tconv_fwd(qkvs, n, dim, heads, index, w_beta_c, mask_c, conv_out, agg, beta, m, inv_l, bn_sums=sums)
        gamma_c, bn_bias_c = _f32(gamma), _f32(bn_bias)
        mean, invstd = torch.empty(dim, **f32), torch.empty(dim, **f32)
        count = float(n)
        if training:
            if _dist_ready(group):
                sums[2 * dim:].fill_(count)
                dist.all_reduce(sums, group=group or None)
                count = 0.0
            elif count < 2:
                raise ValueError("Expected more than 1 value per channel when training")
            call("etpgt_bn_finalize", ptr(sums), count, dim, float(eps), float(momentum), ptr(mean), ptr(invstd),
                 ptr(running_mean), ptr(running_var), stream())
        else:
            call("etpgt_bn_from_running", ptr(running_mean), ptr(running_var), dim, float(eps), ptr(mean),
                 ptr(invstd), stream())
        y = torch.empty(n, dim, **f32)
        y_hi = y_lo = None
        if want_split:
            y_hi = torch.empty(n, dim, dtype=torch.bfloat16, device=dev)
            y_lo = torch.empty(n, dim, dtype=torch.bfloat16, device=dev)
        call("etpgt_bn_apply_ex", ptr(conv_out), n, dim, ptr(mean), ptr(invstd), ptr(gamma_c), ptr(bn_bias_c), ptr(x),
             0, float(drop_p), int(drop_seed), ptr(y), ptr(y_hi), ptr(y_lo), stream())
        ctx.save_for_backward(x_hi, x_lo, w_hi, w_lo, qkvs, w_beta_c, mask_c, agg, beta, m, inv_l, conv_out, mean,
                              invstd, gamma_c)
        ctx.index, ctx.heads = index, heads
        ctx.meta = (bool(training), count, group, float(drop_p), int(drop_seed))
        ctx.w_beta_shape = None if w_beta is None else tuple(w_beta.shape)
        ctx.set_materialize_grads(False)   # no zero-filled "gradients" for the two bf16 hand-over outputs
        if want_split:
            ctx.mark_non_differentiable(y_hi, y_lo)
        return y, y_hi, y_lo

    @staticmethod
    def backward(ctx, d_y, _d_hi, _d_lo):
        (x_hi, x_lo, w_hi, w_lo, qkvs, w_beta, mask, agg, beta, m, inv_l, conv_out, mean, invstd,
         gamma) = ctx.saved_tensors
        index, heads = ctx.index, ctx.heads
        training, count, group, drop_p, drop_seed = ctx.meta
        n, k = x_hi.shape
        if d_y is None:   # the layer output was not used downstream
            d_y = torch.zeros(n, w_hi.size(0) // 4, dtype=torch.float32, device=x_hi.device)
        d_y = _f32(d_y)
        width = w_hi.size(0)
        dim = width // 4
        dev = d_y.device
        f32 = dict(dtype=torch.float32, device=dev)
        # BatchNorm backward (the dropout mask is regenerated from the seed)
        local = torch.empty(2 * dim + 1, dtype=torch.float64, device=dev)
        ws = workspace(size("etpgt_bn_workspace_bytes", n, dim), dev)
        call("etpgt_bn_bwd_stats_ex", ptr(conv_out), None, ptr(d_y), n, dim, ptr(mean), ptr(invstd), 0, drop_p,
             drop_seed, ptr(local), ptr(ws), ws.numel(), stream())
        sums = local
        if training and _dist_ready(group):
            local[2 * dim:].fill_(float(n))
            sums = local.clone()
            dist.all_reduce(sums, group=group or None)
        d_conv, d_res = torch.empty(n, dim, **f32), torch.empty(n, dim, **f32)
        d_gamma, d_bn_bias = torch.empty(dim, **f32), torch.empty(dim, **f32)
        call("etpgt_bn_bwd_apply_ex", ptr(conv_out), None, ptr(d_y), n, dim, ptr(mean), ptr(invstd), ptr(gamma), 0,
             int(training), ptr(sums), count, ptr(local), drop_p, drop_seed, ptr(d_conv), ptr(d_res), ptr(d_gamma),
             ptr(d_bn_bias), stream())
        # conv backward: split-bf16 d(qkvs) + its column sums (the fused bias gradient)
        g_hi = torch.empty(n, width, dtype=torch.bfloat16, device=dev)
        g_lo = torch.empty(n, width, dtype=torch.bfloat16, device=dev)
        d_bias = torch.empty(width, **f32)
        d_w_beta = torch.empty(3 * dim, **f32) if w_beta is not None else None
        _tconv_bwd(qkvs, d_conv, n, dim, heads, index, w_beta, mask, agg, beta, m, inv_l, None, g_hi, g_lo, d_bias,
                   d_w_beta)
        d_x = d_w = None
        if ctx.needs_input_grad[0]:   # residual branch + projection branch, summed by the GEMM epilogue
            d_x = _gemm_x3(g_hi, g_lo, w_hi, w_lo, n, k, width, width, k, None, b_mn=True, accumulate_into=d_res)
        if ctx.needs_input_grad[2]:
            d_w = _gemm_x3(g_hi, g_lo, x_hi, x_lo, width, k, n, width, k, None, split_k=0, a_mn=True, b_mn=True)
        if d_w_beta is not None:
            d_w_beta = d_w_beta.view(ctx.w_beta_shape)
        return (d_x, None, d_w, d_bias, d_w_beta, None, None, None, d_gamma, d_bn_bias, None, None, None, None, None,
                None, None, None, None)


def dropout_mask(n: int, p: float, device, seed: int | None = None) -> torch.Tensor:
    """[n] floats, 0 with probability p else 1/(1-p) (etpgt_dropout_mask); the seed comes from torch's
    CPU generator unless given, so torch.manual_seed makes runs reproducible."""
    if seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    out = torch.empty(n, dtype=torch.float32, device=device)
    call("etpgt_dropout_mask", int(seed), float(p), n, ptr(out), stream())
    return out


class FusedRows(torch.autograd.Function):
    """The row-concatenation of parameters that already ARE consecutive row blocks of one buffer
    (nn.TransformerConv.fused_parameters): forward is a view, backward hands each parameter its row
    block of the fused gradient as a view.  No kernel on either side (torch.cat would copy twice)."""

    @staticmethod
    def forward(ctx, fused, *parts):
        ctx.rows = [p.size(0) for p in parts]
        return fused.view_as(fused)

    @staticmethod
    def backward(ctx, d_fused):
        grads, row = [], 0
        for r in ctx.rows:
            grads.append(d_fused[row:row + r])
            row += r
        return (None, *grads)


def fused_conv_supported(x: torch.Tensor, in_channels: int, width: int) -> bool:
    return PROJECTION_BACKEND == "tcgen05" and x.is_cuda and x.size(0) > 0 and in_channels % 8 == 0 and \
        width % 32 == 0 and supported_dim(width // 4)


def supported_dim(dim: int) -> bool:
    return dim in (32, 64, 128, 256)


def embed_split_supported(table: torch.Tensor, embedding_dim: int, hidden_dim: int) -> bool:
    """Whether the embedding kernel should also write x0 as the bf16 operand pair of the first fused layer (the
    conditions under which that layer takes the tensor-core projection path for an [N, embedding_dim] input)."""
    return FUSED_LAYER and embedding_dim == hidden_dim and fused_conv_supported(table, embedding_dim, 4 * hidden_dim)


class FeedForward(torch.autograd.Function):
    """out = x + Dropout(Linear2(Dropout(GELU(Linear1(x))))) — the FFN block of the non-optimized GraphTransformer
    (etpgt/model/graph_transformer.py:109-124,157-168).  Forward: GEMM 1 with the GELU (+ Philox dropout) in its
    epilogue, which writes h directly as the split-bf16 operand pair of GEMM 2 next to the fp32 pre-activation u
    (etpgt_gemm_bf16x3_gelu); GEMM 2 adds its tiles onto a copy of x (TMA reduce-add) when no second dropout is
    active.  Backward: dH = dY W2, one element pass du = dH * mask * gelu'(u) that emits the split pair and the bias
    column sums (etpgt_gelu_bwd_split), dX = du W1 added onto the residual gradient, two split-K weight gradients."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2, p1: float, p2: float, seed1: int, seed2: int):
        _require_cuda(x, "node features")
        x, w1, w2, b1, b2 = _f32(x), _f32(w1), _f32(w2), _f32(b1), _f32(b2)
        n, d = x.shape
        f = w1.size(0)
        dev = x.device
        x_hi, x_lo, _, _, _, _ = _split(x, True, False)
        w1_hi, w1_lo, _, _, _, _ = _split(w1, True, False)
        w2_hi, w2_lo, _, _, _, _ = _split(w2, True, False)
        u = torch.empty(n, f, dtype=torch.float32, device=dev)
        h_hi = torch.empty(n, f, dtype=torch.bfloat16, device=dev)
        h_lo = torch.empty(n, f, dtype=torch.bfloat16, device=dev)
        ws = workspace(size("etpgt_gemm_bf16x3_workspace_bytes", n, f, d, 1), dev)
        call("etpgt_gemm_bf16x3_gelu", ptr(x_hi), ptr(x_lo), ptr(w1_hi), ptr(w1_lo), n, f, d, d, d, ptr(b1), ptr(u), f,
             ptr(h_hi), ptr(h_lo), f, float(p1), int(seed1), ptr(ws), ws.numel(), stream())
        mask2 = None
        if p2 > 0.0:
            mask2 = dropout_mask(n * d, p2, dev, seed=seed2).view(n, d)
            out = torch.addcmul(x, _gemm_x3(h_hi, h_lo, w2_hi, w2_lo, n, d, f, f, f, b2), mask2)
        else:
            out = _gemm_x3(h_hi, h_lo, w2_hi, w2_lo, n, d, f, f, f, b2, accumulate_into=x.clone())
        ctx.save_for_backward(x_hi, x_lo, w1_hi, w1_lo, w2_hi, w2_lo, u, h_hi, h_lo, mask2)
        ctx.p1, ctx.seed1 = float(p1), int(seed1)
        return out

    @staticmethod
    def backward(ctx, d_out):
        x_hi, x_lo, w1_hi, w1_lo, w2_hi, w2_lo, u, h_hi, h_lo, mask2 = ctx.saved_tensors
        d_out = _f32(d_out)
        n, d = x_hi.shape
        f = w1_hi.size(0)
        dev = d_out.device
        d_y = d_out if mask2 is None else d_out * mask2
        g_hi, g_lo, _, _, _, d_b2 = _split(d_y, True, False, colsum=True)
        d_h = _gemm_x3(g_hi, g_lo, w2_hi, w2_lo, n, f, d, d, f, None, b_mn=True)                    # dY W2
        d_w2 = _gemm_x3(g_hi, g_lo, h_hi, h_lo, d, f, n, d, f, None, split_k=0, a_mn=True, b_mn=True)  # dY^T H
        du_hi = torch.empty(n, f, dtype=torch.bfloat16, device=dev)
        du_lo = torch.empty(n, f, dtype=torch.bfloat16, device=dev)
        d_b1 = torch.empty(f, dtype=torch.float32, device=dev)
        ws = workspace(size("etpgt_split_bf16_workspace_bytes", n, f), dev)
        call("etpgt_gelu_bwd_split", ptr(d_h), ptr(u), n, f, ctx.p1, ctx.seed1, ptr(du_hi), ptr(du_lo), f, ptr(d_b1),
             ptr(ws), ws.numel(), stream())
        d_x = _gemm_x3(du_hi, du_lo, w1_hi, w1_lo, n, d, f, f, d, None, b_mn=True, accumulate_into=d_out.clone())
        d_w1 = _gemm_x3(du_hi, du_lo, x_hi, x_lo, f, d, n, f, d, None, split_k=0, a_mn=True, b_mn=True)
        return d_x, d_w1, d_b1, d_w2, d_b2, None, None, None, None


def feed_forward_supported(x: torch.Tensor, w1: torch.Tensor, w2: torch.Tensor) -> bool:
    return (PROJECTION_BACKEND == "tcgen05" and x.is_cuda and x.size(0) > 0 and x.size(1) % 8 == 0
            and w1.size(0) % 8 == 0 and w2.size(0) == x.size(1))


def linear(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor | None) -> torch.Tensor:
    """Dense projection of the path.  Tensor-core split-bf16 GEMM when the shape allows it
    (inner and outer widths multiples of 8), else a library fp32 GEMM."""
    if PROJECTION_BACKEND == "tcgen05" and x.is_cuda and x.size(1) % 8 == 0 and weight.size(0) % 8 == 0 \
            and x.size(0) > 0:
        return LinearTensorCore.apply(x, weight, bias)
    global _WARNED_LIBRARY_LINEAR
    if not _WARNED_LIBRARY_LINEAR and x.is_cuda:
        _WARNED_LIBRARY_LINEAR = True
        import warnings

        warnings.warn(f"etpgt_b200.ops.linear: widths {tuple(weight.shape)} are not multiples of 8 — this projection "
                      "runs on the library GEMM (torch.nn.functional.linear), not on etpgt_gemm_bf16x3", stacklevel=2)
    return torch.nn.functional.linear(x, weight, bias)


_WARNED_LIBRARY_LINEAR = False


import os as _os  # noqa: E402

PROJECTION_BACKEND = _os.environ.get("ETPGT_PROJECTION", "tcgen05")
FUSED_LAYER = _os.environ.get("ETPGT_FUSED_LAYER", "1") != "0"   # ops.TransformerLayer (conv + BN + residual + dropout)


# ------------------------------------------------------------------------------ GAT / GraphSAGE


def _edge_mask(mask_edges):
    """fp32 attention-dropout mask over the edges; an edgeless graph still needs a non-NULL pointer next to the
    self-loop mask (the kernels take both masks or neither)."""
    if mask_edges is None:
        return None
    me = _f32(mask_edges)
    return me if me.numel() > 0 else me.new_zeros(1)


class GatAggregateFn(torch.autograd.Function):
    """Edge softmax over leaky_relu(a_src[j] + a_dst[i]) and per-head aggregation of h_j, with the
    PyG self-loop rule (etpgt_gat_fwd / _bwd).  Returns the per-head result [N, heads*C]."""

    @staticmethod
    def forward(ctx, h, a_src, a_dst, mask_edges, mask_self, index: GraphIndex, heads: int, slope: float):
        _require_cuda(h, "node features")
        h, a_src, a_dst = _f32(h), _f32(a_src), _f32(a_dst)
        n, width = h.shape
        dev = h.device
        me = _edge_mask(mask_edges)
        ms = _f32(mask_self) if mask_self is not None else None
        agg = torch.empty(n, width, dtype=torch.float32, device=dev)
        m = torch.empty(n, heads, dtype=torch.float32, device=dev)
        inv_l = torch.empty(n, heads, dtype=torch.float32, device=dev)
        call("etpgt_gat_fwd", ptr(h), ptr(a_src), ptr(a_dst), n, width, heads, ptr(index.rowptr), ptr(index.col),
             ptr(index.eperm), float(slope), ptr(me), ptr(ms), ptr(agg), ptr(m), ptr(inv_l), stream())
        ctx.save_for_backward(h, a_src, a_dst, me, ms, agg, m, inv_l)
        ctx.index, ctx.heads, ctx.slope = index, heads, float(slope)
        return agg

    @staticmethod
    def backward(ctx, d_agg):
        h, a_src, a_dst, me, ms, agg, m, inv_l = ctx.saved_tensors
        index, heads = ctx.index, ctx.heads
        d_agg = _f32(d_agg)
        n, width = h.shape
        dev = h.device
        d_h = torch.empty_like(h)
        d_a_src = torch.empty_like(a_src)
        d_a_dst = torch.empty_like(a_dst)
        ws = workspace(size("etpgt_gat_bwd_workspace_bytes", n, index.num_edges, heads), dev)
        call("etpgt_gat_bwd", ptr(h), ptr(a_src), ptr(a_dst), ptr(d_agg), ptr(agg), n, width, heads,
             ptr(index.rowptr), ptr(index.col), ptr(index.eperm), ptr(index.colptr), ptr(index.row), ptr(index.cpos),
             index.num_edges, ctx.slope, ptr(me), ptr(ms), ptr(m), ptr(inv_l), ptr(d_h), ptr(d_a_src), ptr(d_a_dst),
             ptr(ws), ws.numel(), stream())
        return d_h, d_a_src, d_a_dst, None, None, None, None, None


class GatConvFn(torch.autograd.Function):
    """Everything of PyG GATConv(concat=False) after the projection as one autograd node: attention
    scalars (etpgt_gat_scores_fwd), edge softmax + aggregation with the head mean + bias in its epilogue
    (etpgt_gat_fwd_mean; etpgt_gat_fwd + etpgt_head_mean_fwd for narrow heads), and the matching backward chain
    (etpgt_gat_bwd_mean from d_out [N, C]) — etpgt/model/gat.py:49-109,137."""

    @staticmethod
    def forward(ctx, h, att_src, att_dst, bias, mask_edges, mask_self, index: GraphIndex, heads: int, slope: float):
        _require_cuda(h, "node features")
        h = _f32(h)
        n, width = h.shape
        c = width // heads
        dev = h.device
        att_s, att_d = _f32(att_src).reshape(-1), _f32(att_dst).reshape(-1)
        bias_c = _f32(bias) if bias is not None else None
        me = _edge_mask(mask_edges)
        ms = _f32(mask_self) if mask_self is not None else None
        f32 = dict(dtype=torch.float32, device=dev)
        a_src, a_dst = torch.empty(n, heads, **f32), torch.empty(n, heads, **f32)
        call("etpgt_gat_scores_fwd", ptr(h), ptr(att_s), ptr(att_d), n, width, heads, ptr(a_src), ptr(a_dst), stream())
        agg = torch.empty(n, width, **f32)
        m, inv_l = torch.empty(n, heads, **f32), torch.empty(n, heads, **f32)
        out = torch.empty(n, c, **f32)
        if size("etpgt_gat_mean_fused_supported", width, heads):
            # head mean + bias inside the edge kernel (bit-identical to the separate pass: same head order)
            call("etpgt_gat_fwd_mean", ptr(h), ptr(a_src), ptr(a_dst), n, width, heads, ptr(index.rowptr),
                 ptr(index.col), ptr(index.eperm), float(slope), ptr(me), ptr(ms), ptr(bias_c), ptr(agg), ptr(m),
                 ptr(inv_l), ptr(out), stream())
        else:
            call("etpgt_gat_fwd", ptr(h), ptr(a_src), ptr(a_dst), n, width, heads, ptr(index.rowptr), ptr(index.col),
                 ptr(index.eperm), float(slope), ptr(me), ptr(ms), ptr(agg), ptr(m), ptr(inv_l), stream())
            call("etpgt_head_mean_fwd", ptr(agg), ptr(bias_c), n, heads, c, ptr(out), stream())
        ctx.save_for_backward(h, att_s, att_d, a_src, a_dst, me, ms, agg, m, inv_l)
        ctx.index, ctx.heads, ctx.slope = index, heads, float(slope)
        ctx.shapes = (tuple(att_src.shape), tuple(att_dst.shape), bias is not None)
        return out

    @staticmethod
    def backward(ctx, d_out):
        h, att_s, att_d, a_src, a_dst, me, ms, agg, m, inv_l = ctx.saved_tensors
        index, heads = ctx.index, ctx.heads
        d_out = _f32(d_out)
        n, width = h.shape
        c = width // heads
        dev = h.device
        f32 = dict(dtype=torch.float32, device=dev)
        d_bias = torch.empty(c, **f32) if ctx.shapes[2] else None
        ws = workspace(size("etpgt_gat_aux_workspace_bytes", n, width), dev)
        d_h = torch.empty_like(h)
        d_a_src, d_a_dst = torch.empty_like(a_src), torch.empty_like(a_dst)
        ws2 = workspace(size("etpgt_gat_bwd_workspace_bytes", n, index.num_edges, heads), dev)
        # the edge kernels expand d_out / heads in registers: the [N, heads*C] gradient of the per-head result is
        # never written, and the source pass gathers C instead of heads*C floats per edge
        if d_bias is not None:
            call("etpgt_head_mean_bwd", ptr(d_out), n, heads, c, None, ptr(d_bias), ptr(ws), ws.numel(), stream())
        call("etpgt_gat_bwd_mean", ptr(h), ptr(a_src), ptr(a_dst), None, ptr(d_out), ptr(agg), n, width, heads,
             ptr(index.rowptr), ptr(index.col), ptr(index.eperm), ptr(index.colptr), ptr(index.row), ptr(index.cpos),
             index.num_edges, ctx.slope, ptr(me), ptr(ms), ptr(m), ptr(inv_l), ptr(d_h), None, None, ptr(d_a_src),
             ptr(d_a_dst), ptr(ws2), ws2.numel(), stream())
        d_att_s, d_att_d = torch.empty(width, **f32), torch.empty(width, **f32)
        call("etpgt_gat_scores_bwd", ptr(h), ptr(att_s), ptr(att_d), ptr(d_a_src), ptr(d_a_dst), n, width, heads,
             ptr(d_h), ptr(d_att_s), ptr(d_att_d), ptr(ws), ws.numel(), stream())
        return (d_h, d_att_s.view(ctx.shapes[0]), d_att_d.view(ctx.shapes[1]), d_bias, None, None, None, None, None)


class GatLayerFn(torch.autograd.Function):
    """A whole PyG GATConv(concat=False) layer — projection included — as one autograd node
    (etpgt/model/gat.py:49-109,137).  Compared with `linear` + GatConvFn:
      * the attention scalars come from the layer INPUT: a_src[n,h] = <x[n,:], u_src[h,:]> with the fold
        u_src[h,:] = W_h^T att_src[h,:] (etpgt_gat_input_scores_fwd reads [N, in] instead of [N, heads*C]);
      * their backward therefore no longer touches d(lin(x)) (d_x += d_a u, d_u = d_a^T x — one pass over x), so
      * the source pass of the edge backward writes d(lin(x)) directly as the split-bf16 operands of the two
        projection-gradient GEMMs (no fp32 [N, heads*C] gradient, no split pass over it);
      * head mean + bias sit in the forward edge kernel's epilogue, d_out / heads is expanded in registers.
    The folds and their gradients (d_W += att (x) d_u, d_att = W d_u) are element-wise work on parameter-sized
    tensors."""

    @staticmethod
    def forward(ctx, x, weight, att_src, att_dst, bias, mask_edges, mask_self, index: GraphIndex, heads: int,
                slope: float):
        _require_cuda(x, "node features")
        x, weight = _f32(x), _f32(weight)
        n, in_dim = x.shape
        width = weight.size(0)
        c = width // heads
        dev = x.device
        f32 = dict(dtype=torch.float32, device=dev)
        att_s, att_d = _f32(att_src).reshape(heads, c), _f32(att_dst).reshape(heads, c)
        bias_c = _f32(bias) if bias is not None else None
        me = _edge_mask(mask_edges)
        ms = _f32(mask_self) if mask_self is not None else None
        x_hi, x_lo, _, _, _, _ = _split(x, True, False)
        w_hi, w_lo, _, _, _, _ = _split(weight, True, False)
        h = _gemm_x3(x_hi, x_lo, w_hi, w_lo, n, width, in_dim, in_dim, in_dim, None)
        w3 = weight.view(heads, c, in_dim)
        u = torch.cat([(w3 * att_s.unsqueeze(-1)).sum(1), (w3 * att_d.unsqueeze(-1)).sum(1)]).contiguous()  # [2H, in]
        a_src, a_dst = torch.empty(n, heads, **f32), torch.empty(n, heads, **f32)
        call("etpgt_gat_input_scores_fwd", ptr(x), ptr(u), n, in_dim, heads, ptr(a_src), ptr(a_dst), stream())
        agg = torch.empty(n, width, **f32)
        m, inv_l = torch.empty(n, heads, **f32), torch.empty(n, heads, **f32)
        out = torch.empty(n, c, **f32)
        call("etpgt_gat_fwd_mean", ptr(h), ptr(a_src), ptr(a_dst), n, width, heads, ptr(index.rowptr), ptr(index.col),
             ptr(index.eperm), float(slope), ptr(me), ptr(ms), ptr(bias_c), ptr(agg), ptr(m), ptr(inv_l), ptr(out),
             stream())
        ctx.save_for_backward(x, x_hi, x_lo, weight, w_hi, w_lo, att_s, att_d, u, h, a_src, a_dst, me, ms, agg, m, inv_l)
        ctx.index, ctx.heads, ctx.slope = index, heads, float(slope)
        ctx.shapes = (tuple(att_src.shape), tuple(att_dst.shape), bias is not None)
        return out

    @staticmethod
    def backward(ctx, d_out):
        x, x_hi, x_lo, weight, w_hi, w_lo, att_s, att_d, u, h, a_src, a_dst, me, ms, agg, m, inv_l = ctx.saved_tensors
        index, heads = ctx.index, ctx.heads
        d_out = _f32(d_out)
        n, in_dim = x.shape
        width = weight.size(0)
        c = width // heads
        dev = x.device
        f32 = dict(dtype=torch.float32, device=dev)
        d_bias = None
        if ctx.shapes[2]:
            d_bias = torch.empty(c, **f32)
            ws = workspace(size("etpgt_gat_aux_workspace_bytes", n, width), dev)
            call("etpgt_head_mean_bwd", ptr(d_out), n, heads, c, None, ptr(d_bias), ptr(ws), ws.numel(), stream())
        g_hi = torch.empty(n, width, dtype=torch.bfloat16, device=dev)
        g_lo = torch.empty(n, width, dtype=torch.bfloat16, device=dev)
        d_a_src, d_a_dst = torch.empty_like(a_src), torch.empty_like(a_dst)
        ws2 = workspace(size("etpgt_gat_bwd_workspace_bytes", n, index.num_edges, heads), dev)
        call("etpgt_gat_bwd_mean", ptr(h), ptr(a_src), ptr(a_dst), None, ptr(d_out), ptr(agg), n, width, heads,
             ptr(index.rowptr), ptr(index.col), ptr(index.eperm), ptr(index.colptr), ptr(index.row), ptr(index.cpos),
             index.num_edges, ctx.slope, ptr(me), ptr(ms), ptr(m), ptr(inv_l), None, ptr(g_hi), ptr(g_lo), ptr(d_a_src),
             ptr(d_a_dst), ptr(ws2), ws2.numel(), stream())
        d_x = torch.empty_like(x)
        d_u = torch.empty_like(u)
        ws3 = workspace(size("etpgt_gat_input_scores_workspace_bytes", n, in_dim, heads), dev)
        call("etpgt_gat_input_scores_bwd", ptr(x), ptr(u), ptr(d_a_src), ptr(d_a_dst), n, in_dim, heads, ptr(d_x),
             ptr(d_u), ptr(ws3), ws3.numel(), stream())
        # dX = d(lin) W added onto the scores' share; dW = d(lin)^T X (+ the folds' share below)
        _gemm_x3(g_hi, g_lo, w_hi, w_lo, n, in_dim, width, width, in_dim, None, b_mn=True, accumulate_into=d_x)
        d_w = _gemm_x3(g_hi, g_lo, x_hi, x_lo, width, in_dim, n, width, in_dim, None, split_k=0, a_mn=True, b_mn=True)
        w3 = weight.view(heads, c, in_dim)
        du_s, du_d = d_u[:heads], d_u[heads:]
        d_w = d_w + (att_s.unsqueeze(-1) * du_s.unsqueeze(1) + att_d.unsqueeze(-1) * du_d.unsqueeze(1)).view(width, in_dim)
        d_att_s = (w3 * du_s.unsqueeze(1)).sum(2)
        d_att_d = (w3 * du_d.unsqueeze(1)).sum(2)
        return (d_x, d_w, d_att_s.view(ctx.shapes[0]), d_att_d.view(ctx.shapes[1]), d_bias, None, None, None, None,
                None)


class RowScores(torch.autograd.Function):
    """score[n] = <x[n, :], w> + b — the attention readout's nn.Linear(hidden, 1) (etpgt/model/base.py:175-189) as one
    pass over x on this library's kernels (etpgt_gat_input_scores_fwd/_bwd with one vector; the second vector of the
    pair is zero) instead of a library GEMV: d_x = d_score (x) w, d_w = d_score^T x (deterministic), d_b = sum."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        _require_cuda(x, "node features")
        x = _f32(x)
        n, dim = x.shape
        u = torch.zeros(2, dim, dtype=torch.float32, device=x.device)
        u[0] = _f32(weight).reshape(-1)
        score, unused = torch.empty(n, 1, dtype=torch.float32, device=x.device), torch.empty(n, 1, dtype=torch.float32,
                                                                                             device=x.device)
        call("etpgt_gat_input_scores_fwd", ptr(x), ptr(u), n, dim, 1, ptr(score), ptr(unused), stream())
        ctx.save_for_backward(x, u)
        ctx.has_bias = bias is not None
        ctx.w_shape = tuple(weight.shape)
        return score.view(n) + bias.reshape(()) if bias is not None else score.view(n)

    @staticmethod
    def backward(ctx, d_score):
        x, u = ctx.saved_tensors
        n, dim = x.shape
        d_s = _f32(d_score).reshape(n, 1)
        zeros = torch.zeros_like(d_s)
        d_x, d_u = torch.empty_like(x), torch.empty_like(u)
        ws = workspace(size("etpgt_gat_input_scores_workspace_bytes", n, dim, 1), x.device)
        call("etpgt_gat_input_scores_bwd", ptr(x), ptr(u), ptr(d_s), ptr(zeros), n, dim, 1, ptr(d_x), ptr(d_u), ptr(ws),
             ws.numel(), stream())
        d_b = d_s.sum().reshape(1) if ctx.has_bias else None
        return d_x, d_u[0].view(ctx.w_shape), d_b


def row_scores_supported(x: torch.Tensor) -> bool:
    return x.is_cuda and x.size(0) > 0 and x.size(1) % 4 == 0 and x.size(1) <= 1024


def gat_layer_supported(x: torch.Tensor, in_dim: int, width: int, heads: int) -> bool:
    return (PROJECTION_BACKEND == "tcgen05" and x.is_cuda and x.size(0) > 0 and in_dim % 8 == 0 and width % 8 == 0
            and in_dim <= 1024 and width <= 1024 and heads in (1, 2, 4, 8)
            and bool(size("etpgt_gat_mean_fused_supported", width, heads)))


class SageMeanFn(torch.autograd.Function):
    """Mean of in-neighbour rows (0 for isolated nodes) — PyG SAGEConv(aggr='mean') aggregation."""

    @staticmethod
    def forward(ctx, x, index: GraphIndex):
        _require_cuda(x, "node features")
        x = _f32(x)
        n, dim = x.shape
        mean = torch.empty_like(x)
        call("etpgt_sage_mean_fwd", ptr(x), n, dim, ptr(index.rowptr), ptr(index.col), ptr(mean), stream())
        ctx.index = index
        return mean

    @staticmethod
    def backward(ctx, d_mean):
        index = ctx.index
        d_mean = _f32(d_mean)
        n, dim = d_mean.shape
        d_x = torch.empty_like(d_mean)
        call("etpgt_sage_mean_bwd", ptr(d_mean), n, dim, ptr(index.rowptr), ptr(index.colptr), ptr(index.row),
             ptr(d_x), stream())
        return d_x, None


def _split_into(src: torch.Tensor, hi: torch.Tensor, lo: torch.Tensor, col0: int, colsum: bool = False):
    """fp32 [R, C] -> bf16 hi/lo written into columns [col0, col0 + C) of the wider row-major operands `hi` / `lo`."""
    r, c = src.shape
    ld = hi.size(1)
    sums = torch.empty(c, dtype=torch.float32, device=src.device) if colsum else None
    ws = workspace(size("etpgt_split_bf16_workspace_bytes", r, c) if colsum else 256, src.device)
    call("etpgt_split_bf16", ptr(src), r, c, c, ptr(hi.view(-1)[col0:]), ptr(lo.view(-1)[col0:]), ld, None, None, 0,
         ptr(sums), ptr(ws), ws.numel(), stream())
    return sums


class SageLayerFn(torch.autograd.Function):
    """A whole PyG SAGEConv(aggr="mean") layer, lin_l(mean_j x_j) + lin_r(x_i) (etpgt/model/graphsage.py:43-48,75),
    as ONE GEMM over the concatenated operand [mean | x] (K = 2*in) against [W_l | W_r]: the mean kernel's output and
    x are split straight into the two column halves of one bf16 operand pair.  Backward: dY is split once, one GEMM
    gives [d_mean | d_root] side by side (N = 2*in), the mean-backward kernel reads the left half with its pitch and
    adds the right half in (etpgt_sage_mean_bwd_ld), one split-K GEMM gives [dW_l | dW_r].  Per layer: 3 GEMMs
    instead of 6, 3 split passes instead of 6, no element-wise adds."""

    @staticmethod
    def forward(ctx, x, w_l, b_l, w_r, index: GraphIndex):
        _require_cuda(x, "node features")
        x, w_l, w_r = _f32(x), _f32(w_l), _f32(w_r)
        b_c = _f32(b_l) if b_l is not None else None
        n, in_dim = x.shape
        out_dim = w_l.size(0)
        dev = x.device
        bf = dict(dtype=torch.bfloat16, device=dev)
        a_hi, a_lo = torch.empty(n, 2 * in_dim, **bf), torch.empty(n, 2 * in_dim, **bf)
        # the mean goes straight into the left column half as a bf16 pair (no fp32 mean, no split pass over it)
        call("etpgt_sage_mean_fwd_split", ptr(x), n, in_dim, ptr(index.rowptr), ptr(index.col), None, ptr(a_hi),
             ptr(a_lo), 2 * in_dim, stream())
        _split_into(x, a_hi, a_lo, in_dim)
        w_hi, w_lo = torch.empty(out_dim, 2 * in_dim, **bf), torch.empty(out_dim, 2 * in_dim, **bf)
        _split_into(w_l, w_hi, w_lo, 0)
        _split_into(w_r, w_hi, w_lo, in_dim)
        y = _gemm_x3(a_hi, a_lo, w_hi, w_lo, n, out_dim, 2 * in_dim, 2 * in_dim, 2 * in_dim, b_c)
        ctx.save_for_backward(a_hi, a_lo, w_hi, w_lo)
        ctx.index, ctx.has_bias = index, b_l is not None
        return y

    @staticmethod
    def backward(ctx, d_y):
        a_hi, a_lo, w_hi, w_lo = ctx.saved_tensors
        index = ctx.index
        d_y = _f32(d_y)
        n, k2 = a_hi.shape
        in_dim = k2 // 2
        out_dim = w_hi.size(0)
        g_hi, g_lo, _, _, _, d_b = _split(d_y, True, False, colsum=ctx.has_bias)
        d_a = _gemm_x3(g_hi, g_lo, w_hi, w_lo, n, k2, out_dim, out_dim, k2, None, b_mn=True)   # [d_mean | d_root]
        d_x = torch.empty(n, in_dim, dtype=torch.float32, device=d_y.device)
        call("etpgt_sage_mean_bwd_ld", ptr(d_a), k2, ptr(d_a.view(-1)[in_dim:]), n, in_dim, ptr(index.rowptr),
             ptr(index.colptr), ptr(index.row), ptr(d_x), stream())
        d_w = _gemm_x3(g_hi, g_lo, a_hi, a_lo, out_dim, k2, n, out_dim, k2, None, split_k=0, a_mn=True, b_mn=True)
        return d_x, d_w[:, :in_dim].contiguous(), d_b, d_w[:, in_dim:].contiguous(), None


def sage_layer_supported(x: torch.Tensor, in_dim: int, out_dim: int) -> bool:
    return (PROJECTION_BACKEND == "tcgen05" and x.is_cuda and x.size(0) > 0 and in_dim in (32, 64, 128, 256)
            and out_dim % 8 == 0)


# ------------------------------------------------------------------------------ BatchNorm (+res, +relu)


def _dist_ready(group) -> bool:
    return group is not False and dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1


class BatchNormRows(torch.autograd.Function):
    """BatchNorm1d over all node rows of the (global) batch + residual (+ ReLU).
    etpgt/model/graph_transformer.py:175-176, gat.py:138-140, graphsage.py:76-77.  Under data
    parallelism the 2*dim partial sums are all-reduced so statistics cover every rank's nodes."""

    @staticmethod
    def forward(ctx, x, gamma, bias, residual, running_mean, running_var, training, momentum, eps, relu, group,
                drop_p=0.0, drop_seed=0):
        _require_cuda(x, "node features")
        x = _f32(x)
        n, dim = x.shape
        dev = x.device
        gamma_c, bias_c = _f32(gamma), _f32(bias)
        res_c = _f32(residual) if residual is not None else None
        mean = torch.empty(dim, dtype=torch.float32, device=dev)
        invstd = torch.empty(dim, dtype=torch.float32, device=dev)
        count = float(n)
        if training:
            # [sum x | sum x^2 | row count]: under data parallelism the whole vector is all-reduced and
            # the kernels read the GLOBAL count from its tail (count argument 0) — no host round trip
            sums = torch.empty(2 * dim + 1, dtype=torch.float64, device=dev)
            ws = workspace(size("etpgt_bn_workspace_bytes", n, dim), dev)
            call("etpgt_bn_stats", ptr(x), n, dim, ptr(sums), ptr(ws), ws.numel(), stream())
            if _dist_ready(group):
                sums[2 * dim:].fill_(count)
                dist.all_reduce(sums, group=group or None)
                count = 0.0
            elif count < 2:
                raise ValueError("Expected more than 1 value per channel when training")
            call("etpgt_bn_finalize", ptr(sums), count, dim, float(eps), float(momentum), ptr(mean), ptr(invstd),
                 ptr(running_mean), ptr(running_var), stream())
        else:
            call("etpgt_bn_from_running", ptr(running_mean), ptr(running_var), dim, float(eps), ptr(mean),
                 ptr(invstd), stream())
        y = torch.empty_like(x)
        # (+ the layer's dropout, Philox mask regenerated in backward: gat.py:139-141, graphsage.py:77-78)
        call("etpgt_bn_apply_ex", ptr(x), n, dim, ptr(mean), ptr(invstd), ptr(gamma_c), ptr(bias_c), ptr(res_c),
             int(bool(relu)), float(drop_p), int(drop_seed), ptr(y), None, None, stream())
        ctx.save_for_backward(x, y if relu else None, mean, invstd, gamma_c)
        ctx.meta = (bool(training), bool(relu), count, residual is not None, group, float(drop_p), int(drop_seed))
        return y

    @staticmethod
    def backward(ctx, d_y):
        x, y, mean, invstd, gamma = ctx.saved_tensors
        training, relu, count, has_res, group, drop_p, drop_seed = ctx.meta
        d_y = _f32(d_y)
        n, dim = x.shape
        dev = x.device
        local = torch.empty(2 * dim + 1, dtype=torch.float64, device=dev)
        ws = workspace(size("etpgt_bn_workspace_bytes", n, dim), dev)
        call("etpgt_bn_bwd_stats_ex", ptr(x), ptr(y), ptr(d_y), n, dim, ptr(mean), ptr(invstd), int(relu), drop_p,
             drop_seed, ptr(local), ptr(ws), ws.numel(), stream())
        sums = local
        if training and _dist_ready(group):
            local[2 * dim:].fill_(float(n))
            sums = local.clone()
            dist.all_reduce(sums, group=group or None)   # count == 0.0: read from the reduced tail
        d_x = torch.empty_like(x)
        d_gamma = torch.empty(dim, dtype=torch.float32, device=dev)
        d_bias = torch.empty(dim, dtype=torch.float32, device=dev)
        # the residual branch's gradient (d_y through the dropout mask and the ReLU gate) comes out of the same pass
        d_res = torch.empty_like(x) if has_res and (relu or drop_p > 0.0) else None
        call("etpgt_bn_bwd_apply_ex", ptr(x), ptr(y), ptr(d_y), n, dim, ptr(mean), ptr(invstd), ptr(gamma), int(relu),
             int(training), ptr(sums), count, ptr(local), drop_p, drop_seed, ptr(d_x), ptr(d_res), ptr(d_gamma),
             ptr(d_bias), stream())
        if has_res and d_res is None:
            d_res = d_y
        return d_x, d_gamma, d_bias, d_res, None, None, None, None, None, None, None, None, None


# ------------------------------------------------------------------------------ readout


class SegmentReadout(torch.autograd.Function):
    """Session readout over contiguous node ranges — etpgt/model/base.py:136-193."""

    @staticmethod
    def forward(ctx, x, scores, seg_ptr, mode: int):
        _require_cuda(x, "node embeddings")
        x = _f32(x)
        n, dim = x.shape
        s = seg_ptr.numel() - 1
        dev = x.device
        out = torch.empty(s, dim, dtype=torch.float32, device=dev)
        aux = None
        scores_c = None
        if mode == READOUT_MODES["max"]:
            aux = torch.empty(s, dim, dtype=torch.int32, device=dev)
        elif mode == READOUT_MODES["attention"]:
            aux = torch.empty(n, dtype=torch.float32, device=dev)
            scores_c = _f32(scores).reshape(-1)
        call("etpgt_readout_fwd", ptr(x), ptr(seg_ptr), s, dim, mode, ptr(scores_c), ptr(out), ptr(aux), stream())
        ctx.save_for_backward(x, out, seg_ptr, aux)
        ctx.mode = mode
        ctx.scores_shape = None if scores is None else tuple(scores.shape)
        return out

    @staticmethod
    def backward(ctx, d_out):
        x, out, seg_ptr, aux = ctx.saved_tensors
        mode = ctx.mode
        d_out = _f32(d_out)
        n, dim = x.shape
        d_x = torch.empty_like(x)
        d_scores = torch.empty(n, dtype=torch.float32, device=x.device) if mode == READOUT_MODES["attention"] else None
        call("etpgt_readout_bwd", ptr(x), ptr(out), ptr(d_out), ptr(seg_ptr), n, seg_ptr.numel() - 1, dim, mode,
             ptr(aux), ptr(d_x), ptr(d_scores), stream())
        if d_scores is not None:
            d_scores = d_scores.view(ctx.scores_shape)
        return d_x, d_scores, None, None


# ------------------------------------------------------------------------------ sampled losses


class SampledLoss(torch.autograd.Function):
    """BPR / listwise / dual loss over (target, negatives) — etpgt/train/losses.py:20-164.
    Returns a device tensor [3] = (total, listwise, bpr); only `[0]` carries gradient."""

    @staticmethod
    def forward(ctx, sess, table, targets, negatives, mode, alpha, temperature, total_sessions, padding_idx):
        _require_cuda(sess, "session embeddings")
        sess_c, table_c = _f32(sess), _f32(table)
        targets, negatives = _i64(targets), _i64(negatives)
        b, dim = sess_c.shape
        if negatives.dim() != 2 or negatives.size(0) != b:
            raise RuntimeError(f"negative_items must be [batch, num_negatives]; got {tuple(negatives.shape)}")
        num_neg = negatives.size(1)
        dev = sess_c.device
        total = float(total_sessions if total_sessions else b)
        scores = torch.empty(b, num_neg + 1, dtype=torch.float32, device=dev)
        losses = torch.empty(3, dtype=torch.float32, device=dev)
        ws = workspace(size("etpgt_sampled_loss_workspace_bytes", b, num_neg, dim), dev)
        call("etpgt_sampled_loss_fwd", ptr(sess_c), ptr(table_c), ptr(targets), ptr(negatives), b, num_neg, dim, mode,
             float(alpha), float(temperature), total, ptr(scores), ptr(losses), ptr(ws), ws.numel(), stream())
        ctx.save_for_backward(sess_c, table_c, targets, negatives, scores)
        ctx.table_ref = table
        ctx.plan = _find_plan(targets, negatives)
        ctx.meta = (mode, float(alpha), float(temperature), total, -1 if padding_idx is None else int(padding_idx))
        return losses

    @staticmethod
    def backward(ctx, d_losses):
        sess, table, targets, negatives, scores = ctx.saved_tensors
        mode, alpha, temperature, total, padding_idx = ctx.meta
        b, dim = sess.shape
        num_neg = negatives.size(1)
        dev = sess.device
        d_loss = _f32(d_losses)[0:1].contiguous()
        d_sess = torch.empty_like(sess)
        d_table, table_grad = _table_grad(ctx, table.shape, dev)
        ws = workspace(size("etpgt_sampled_loss_workspace_bytes", b, num_neg, dim), dev)
        plan = ctx.plan if d_table is not None and ctx.plan is not None and ctx.plan.m == b * (num_neg + 1) else None
        call("etpgt_sampled_loss_bwd_planned", ptr(sess), ptr(table), ptr(targets), ptr(negatives), b, num_neg, dim,
             mode, alpha, temperature, total, ptr(scores), ptr(d_loss), table.size(0), padding_idx,
             ptr(plan.sorted_key) if plan else None, ptr(plan.perm) if plan else None, ptr(d_sess),
             ptr(d_table), ptr(ws), ws.numel(), stream())
        return d_sess, table_grad, None, None, None, None, None, None, None


def sampled_loss(sess, item_embeddings, targets, negatives, kind: str, alpha=0.7, temperature=1.0,
                 total_sessions=None) -> torch.Tensor:
    """`item_embeddings` is the nn.Embedding the reference passes around (trainer.py:103)."""
    weight, padding_idx = _weight_and_padding(item_embeddings)
    return SampledLoss.apply(sess, weight, targets, negatives, LOSS_MODES[kind], alpha, temperature,
                             total_sessions, padding_idx)


# ------------------------------------------------------------------------------ full-catalogue softmax


def _softmax_inputs(name, sess, table, targets, *more_cuda):
    """Contiguous fp32 sess [B, D] and table [I, D] and int64 targets [B], checked as both softmax losses check them
    (`name` in the messages); the (tensor, what) pairs of `more_cuda` must be on the GPU too."""
    for t, what in ((sess, "session embeddings"), (table, "item embeddings"), (targets, "targets"), *more_cuda):
        _require_cuda(t, what)
    sess_c, table_c, targets = _f32(sess), _f32(table), _i64(targets)
    if sess_c.dim() != 2 or table_c.dim() != 2 or sess_c.size(1) != table_c.size(1):
        raise RuntimeError(f"{name}: sess [B, D] and table [I, D] expected; got "
                           f"{tuple(sess_c.shape)} and {tuple(table_c.shape)}")
    if targets.dim() != 1 or targets.size(0) != sess_c.size(0):
        raise RuntimeError(f"target_items must be [batch={sess_c.size(0)}]; got {tuple(targets.shape)}")
    return sess_c, table_c, targets


SOFTMAX_PRECISIONS = {"bf16x3": 0, "bf16": 1}     # ETPGT_SOFTMAX_BF16X3, ETPGT_SOFTMAX_BF16


def _softmax_precision(precision) -> int:
    """The ABI value of a softmax loss precision: "bf16x3" (split-bf16 products, ~1e-5 relative to fp64, the default)
    or "bf16" (S, E and G rounded once to bf16, one bf16 MMA per product, for training)."""
    if not isinstance(precision, str) or precision not in SOFTMAX_PRECISIONS:
        raise ValueError(f"softmax loss precision must be \"bf16x3\" or \"bf16\"; got {precision!r}")
    return SOFTMAX_PRECISIONS[precision]


class FullSoftmaxLoss(torch.autograd.Function):
    """Cross-entropy over every item of the table (the padding row left out), etpgt_full_softmax_fwd_ex / _bwd_ex:
    tcgen05 GEMMs with the softmax in the epilogue, so the [B, I] logits never exist.  `precision` "bf16x3" (default)
    makes every product split-bf16, "bf16" rounds S, E and G once to bf16.  Returns the scalar mean over
    `total_sessions` (default: the batch)."""

    @staticmethod
    def forward(ctx, sess, table, targets, temperature, total_sessions, padding_idx, precision="bf16x3"):
        prec = _softmax_precision(precision)
        sess_c, table_c, targets = _softmax_inputs("full_softmax_loss", sess, table, targets)
        b, dim = sess_c.shape
        dev = sess_c.device
        total = float(total_sessions if total_sessions else b)
        pad = -1 if padding_idx is None else int(padding_idx)
        lse = torch.empty(b, dtype=torch.float32, device=dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        ws = workspace(size("etpgt_full_softmax_workspace_bytes", b, table_c.size(0), dim), dev)
        call("etpgt_full_softmax_fwd_ex", ptr(sess_c), ptr(table_c), ptr(targets), b, table_c.size(0), dim,
             float(temperature), total, pad, ptr(lse), ptr(loss), ptr(ws), ws.numel(), stream(), prec)
        ctx.save_for_backward(sess_c, table_c, targets, lse)
        ctx.table_ref = table
        ctx.meta = (float(temperature), total, pad, prec)
        ctx.mark_non_differentiable(lse)
        return loss[0], lse

    @staticmethod
    def backward(ctx, d_loss, _d_lse):
        sess, table, targets, lse = ctx.saved_tensors
        temperature, total, pad, prec = ctx.meta
        b, dim = sess.shape
        dev = sess.device
        d_loss = _f32(d_loss).reshape(1).contiguous()
        d_sess = torch.empty_like(sess) if ctx.needs_input_grad[0] else None
        d_table, table_grad = _table_grad(ctx, table.shape, dev)
        ws = workspace(size("etpgt_full_softmax_workspace_bytes", b, table.size(0), dim), dev)
        call("etpgt_full_softmax_bwd_ex", ptr(sess), ptr(table), ptr(targets), ptr(lse), ptr(d_loss), b,
             table.size(0), dim, temperature, total, pad, ptr(d_sess), ptr(d_table), ptr(ws), ws.numel(), stream(),
             prec)
        return d_sess, table_grad, None, None, None, None, None


def full_softmax_loss(sess, item_embeddings, targets, temperature=1.0, total_sessions=None,
                      precision="bf16x3") -> torch.Tensor:
    """Softmax cross-entropy of `targets` over the whole catalogue.  `item_embeddings` is the nn.Embedding (its
    padding_idx column is left out of the softmax and its row gets no gradient) or a bare weight tensor.  The table
    gradient goes into the etpgt_b200.optim gradient sink when one is registered, else it is returned densely.
    precision "bf16x3" (default): split-bf16 products, ~1e-5 relative to fp64.  "bf16": the sessions, the table and
    the softmax gradient are rounded once to bf16 and every product is one bf16 MMA (fp32 accumulation); lse and the
    softmax stay fp32.  A different numerical contract for training, not the same result faster."""
    weight, padding_idx = _weight_and_padding(item_embeddings)
    return FullSoftmaxLoss.apply(sess, weight, targets, temperature, total_sessions, padding_idx, precision)[0]


# ------------------------------------------------------------------------------ shared-pool sampled softmax


def item_sampling_table(counts=None, power=0.75, padding_idx=0, *, num_items=None, device=None) -> torch.Tensor:
    """The proposal q(i) = w_i / W of `sample_item_pool` as int64 cumulative weights cum [I + 1] (cum[0] = 0,
    cum[i + 1] = cum[i] + w_i).  w_i = floor(count_i ** power * 2^s) in fp64, with s chosen so that W = cum[I] < 2^62;
    counts=None is uniform (w_i = 1 before the scaling; `num_items` then gives I).  The padding row and items with
    count 0 get weight 0 and are never drawn.  On `device` (default: that of `counts`, else CUDA)."""
    import math

    import numpy as np

    if counts is None:
        if num_items is None:
            raise ValueError("item_sampling_table: num_items is required when counts is None")
        w = np.ones(int(num_items), dtype=np.float64)
    else:
        if device is None and isinstance(counts, torch.Tensor):
            device = counts.device
        c = (counts.detach().double().cpu().numpy() if isinstance(counts, torch.Tensor)
             else np.asarray(counts, dtype=np.float64)).reshape(-1)
        if num_items is not None and c.size != int(num_items):
            raise ValueError(f"item_sampling_table: {c.size} counts for {num_items} items")
        if (c < 0).any() or not np.isfinite(c).all():
            raise ValueError("item_sampling_table: counts must be finite and >= 0")
        w = np.where(c > 0, np.power(c, float(power)), 0.0)
    if padding_idx is not None and 0 <= padding_idx < w.size:
        w[padding_idx] = 0.0
    total = float(w.sum())
    if not total > 0.0:
        raise ValueError("item_sampling_table: no item has a positive weight")
    s = 61 - math.ceil(math.log2(total))          # every w_i 2^s <= 2^61, so W <= 2^61 < 2^62
    wi = np.floor(np.ldexp(w, s)).astype(np.int64)
    cum = np.zeros(w.size + 1, dtype=np.int64)
    np.cumsum(wi, out=cum[1:])
    if cum[-1] <= 0:
        raise ValueError("item_sampling_table: no item has a positive weight")
    return torch.from_numpy(cum).to(device if device is not None else "cuda")


def sample_item_pool(cum: torch.Tensor, num_sampled: int, seed: int, step: int):
    """`num_sampled` item ids drawn with replacement from the proposal `cum` (item_sampling_table, on the device),
    sorted ascending, and log_q = log(num_sampled * q(id)) [num_sampled] fp32 (etpgt_sample_item_pool).  The pool
    depends on (seed, step) only, so data-parallel ranks draw the same one without communicating."""
    _require_cuda(cum, "cum")
    cum = _i64(cum)
    if cum.dim() != 1 or cum.numel() < 2:
        raise RuntimeError(f"sample_item_pool: cum must be [num_items + 1]; got {tuple(cum.shape)}")
    m = int(num_sampled)
    pool = torch.empty(max(m, 0), dtype=torch.int64, device=cum.device)
    log_q = torch.empty(max(m, 0), dtype=torch.float32, device=cum.device)
    ws = workspace(size("etpgt_sample_item_pool_workspace_bytes", max(m, 1)), cum.device)
    call("etpgt_sample_item_pool", ptr(cum), cum.numel() - 1, m, int(seed) & 0xFFFFFFFFFFFFFFFF,
         int(step) & 0xFFFFFFFF, ptr(pool), ptr(log_q), ptr(ws), ws.numel(), stream())
    return pool, log_q


class PoolSoftmaxLoss(torch.autograd.Function):
    """Sampled softmax over one pool of negatives shared by the batch, with the log-Q correction
    (etpgt_pool_softmax_fwd / _bwd, the tensor-core kernels of the full-catalogue loss with the pool rows as columns):
        z_pos[b] = s_b . e_{t_b} / T,   z[b, j] = s_b . e_{p_j} / T - log_q[j]  (-inf where p_j is t_b or padding)
        loss = sum_b (logsumexp(z_pos[b], z[b, :]) - z_pos[b]) / total_sessions
    `validate` checks the pool ids against the table and sorts an unsorted pool (one device-to-host copy); pools from
    `sample_item_pool` are sorted and in range already.  `precision` as FullSoftmaxLoss ("bf16": the positive is the
    fp32 dot of the rounded operands).  Returns (loss, lse)."""

    @staticmethod
    def forward(ctx, sess, table, targets, pool_ids, log_q, temperature, total_sessions, padding_idx, validate,
                precision="bf16x3"):
        prec = _softmax_precision(precision)
        sess_c, table_c, targets = _softmax_inputs("pool_softmax_loss", sess, table, targets, (pool_ids, "pool_ids"),
                                                   (log_q, "log_q"))
        pool, lq = _i64(pool_ids), _f32(log_q)
        b, dim = sess_c.shape
        items = table_c.size(0)
        if pool.dim() != 1 or pool.numel() == 0:
            raise RuntimeError(f"pool_softmax_loss: pool_ids must be a non-empty [M]; got {tuple(pool.shape)}")
        if lq.shape != pool.shape:
            raise RuntimeError(f"pool_softmax_loss: log_q {tuple(lq.shape)} must match pool_ids {tuple(pool.shape)}")
        if validate:
            lo, hi, unsorted = torch.stack([pool.min(), pool.max(), (pool[1:] < pool[:-1]).any().long()]).tolist()
            if lo < 0 or hi >= items:
                raise RuntimeError(f"pool_softmax_loss: pool id out of range [0, {items}) (min {lo}, max {hi})")
            if unsorted:
                pool, order = torch.sort(pool)
                lq = lq[order].contiguous()
        m = pool.numel()
        dev = sess_c.device
        total = float(total_sessions if total_sessions else b)
        pad = -1 if padding_idx is None else int(padding_idx)
        lse = torch.empty(b, dtype=torch.float32, device=dev)
        z_pos = torch.empty(b, dtype=torch.float32, device=dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        ws = workspace(size("etpgt_pool_softmax_workspace_bytes", b, m, dim), dev)
        call("etpgt_pool_softmax_fwd_ex", ptr(sess_c), ptr(table_c), ptr(targets), ptr(pool), ptr(lq), b, items, m,
             dim, float(temperature), total, pad, ptr(lse), ptr(z_pos), ptr(loss), ptr(ws), ws.numel(), stream(), prec)
        ctx.save_for_backward(sess_c, table_c, targets, pool, lq, lse, z_pos)
        ctx.table_ref = table
        ctx.meta = (float(temperature), total, pad, prec)
        ctx.mark_non_differentiable(lse)
        return loss[0], lse

    @staticmethod
    def backward(ctx, d_loss, _d_lse):
        sess, table, targets, pool, lq, lse, z_pos = ctx.saved_tensors
        temperature, total, pad, prec = ctx.meta
        b, dim = sess.shape
        m = pool.numel()
        dev = sess.device
        d_loss = _f32(d_loss).reshape(1).contiguous()
        d_sess = torch.empty_like(sess) if ctx.needs_input_grad[0] else None
        d_table, table_grad = _table_grad(ctx, table.shape, dev)
        ws = workspace(size("etpgt_pool_softmax_workspace_bytes", b, m, dim), dev)
        call("etpgt_pool_softmax_bwd_ex", ptr(sess), ptr(table), ptr(targets), ptr(pool), ptr(lq), ptr(lse),
             ptr(z_pos), ptr(d_loss), b, table.size(0), m, dim, temperature, total, pad, ptr(d_sess), ptr(d_table),
             ptr(ws), ws.numel(), stream(), prec)
        return d_sess, table_grad, None, None, None, None, None, None, None, None


def pool_softmax_loss(sess, item_embeddings, targets, pool_ids, log_q, temperature=1.0,
                      total_sessions=None, precision="bf16x3") -> torch.Tensor:
    """Sampled softmax cross-entropy of `targets` against the shared negative pool `pool_ids` [M] with its log-Q
    correction `log_q` [M] = log(M q(pool_ids)) (see PoolSoftmaxLoss; `sample_item_pool` draws both).  The pool is
    sorted (with its log_q) when it is not sorted already; ids outside the table raise.  `item_embeddings` is the
    nn.Embedding (its padding_idx never counts as a negative and its row gets no gradient) or a bare weight tensor.
    The table gradient goes into the etpgt_b200.optim gradient sink when one is registered, else it is returned
    densely (non-zero on the pool and target rows only).  `precision` "bf16x3" (default) or "bf16", as in
    full_softmax_loss."""
    weight, padding_idx = _weight_and_padding(item_embeddings)
    return PoolSoftmaxLoss.apply(sess, weight, targets, pool_ids, log_q, temperature, total_sessions, padding_idx,
                                 True, precision)[0]


def in_batch_columns(targets, freq, last, step, decay, padding_idx, pool_ids=None, pool_log_q=None):
    """The in-batch negatives of `targets` [B] as columns of PoolSoftmaxLoss (etpgt_in_batch_columns): (columns
    int64 [M + B] ascending, log_q fp32 [M + B]), the optional sorted pool `pool_ids` / `pool_log_q` [M]
    (sample_item_pool) merged in, pool entries first among equal ids, then the in-batch entries in session order.
    Updates the streaming estimate of each item's share of the targets in place first: for each distinct target i
    (in [0, I), not `padding_idx`) with n copies,
        freq[i] = freq[i] (1 - decay)^(step - last[i]) + decay n / B,   last[i] = step
    with freq fp64 [I] and last int64 [I] on the device; steps must increase from call to call.  An in-batch column
    gets log_q = log(B freq[t_b]) after the update; the padding id and ids outside the table get +inf (never a
    negative) and leave freq / last alone.  No host read, no synchronisation."""
    for t, what in ((targets, "targets"), (freq, "freq"), (last, "last")):
        _require_cuda(t, what)
    if freq.dtype != torch.float64 or last.dtype != torch.int64 or freq.dim() != 1 or last.shape != freq.shape \
            or not freq.is_contiguous() or not last.is_contiguous():
        raise ValueError("in_batch_columns: freq must be a contiguous fp64 [num_items] and last a contiguous int64 of "
                         f"the same shape; got {freq.dtype} {tuple(freq.shape)} and {last.dtype} {tuple(last.shape)}")
    targets = _i64(targets)
    if targets.dim() != 1 or targets.numel() == 0:
        raise ValueError(f"in_batch_columns: targets must be a non-empty [B]; got {tuple(targets.shape)}")
    if not 0.0 < float(decay) <= 1.0:
        raise ValueError(f"in_batch_columns: decay must be in (0, 1]; got {decay}")
    if int(step) < 0:
        raise ValueError(f"in_batch_columns: step must be >= 0; got {step}")
    if (pool_ids is None) != (pool_log_q is None):
        raise ValueError("in_batch_columns: pool_ids and pool_log_q go together")
    m = 0
    if pool_ids is not None:
        _require_cuda(pool_ids, "pool_ids")
        _require_cuda(pool_log_q, "pool_log_q")
        pool_ids, pool_log_q = _i64(pool_ids), _f32(pool_log_q)
        if pool_ids.dim() != 1 or pool_log_q.shape != pool_ids.shape:
            raise ValueError(f"in_batch_columns: pool_ids {tuple(pool_ids.shape)} and pool_log_q "
                             f"{tuple(pool_log_q.shape)} must be the same [M]")
        m = pool_ids.numel()
    b = targets.numel()
    columns = torch.empty(m + b, dtype=torch.int64, device=targets.device)
    log_q = torch.empty(m + b, dtype=torch.float32, device=targets.device)
    ws = workspace(size("etpgt_in_batch_columns_workspace_bytes", b, m), targets.device)
    call("etpgt_in_batch_columns", ptr(targets), b, ptr(pool_ids) if m else None, ptr(pool_log_q) if m else None, m,
         ptr(freq), ptr(last), freq.numel(), -1 if padding_idx is None else int(padding_idx), int(step), float(decay),
         ptr(columns), ptr(log_q), ptr(ws), ws.numel(), stream())
    return columns, log_q


# ------------------------------------------------------------------------------ scoring / top-k


def to_bf16(t: torch.Tensor) -> torch.Tensor:
    """Round-to-nearest-even fp32 -> bf16 copy (etpgt_f32_to_bf16)."""
    if t.dtype == torch.bfloat16:
        return t.contiguous()
    src = _f32(t.detach())
    dst = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    call("etpgt_f32_to_bf16", ptr(src), ptr(dst), src.numel(), stream())
    return dst


SCORE_MAX_K = 256        # ETPGT_SCORE_MAX_K: the tensor-core scorer and the merges
SCORE_F32_MAX_K = 64     # the fp32 CUDA-core scorer
_SCORE_WS_BUDGET = 4 << 30   # bf16 workspace per call for k > 32: larger batches are scored in row chunks


def score_row_chunks(batch: int, items: int, k: int, budget: int = _SCORE_WS_BUDGET) -> tuple[int, int]:
    """(rows per call, workspace bytes) of the bf16 scorer.  For k > 32 the workspace holds a slot for every 16-item
    piece of a row, so the batch is halved until one call's workspace fits `budget` (a single row may still exceed
    it).  The workspace is the larger of the full chunks' and the last chunk's need: the library's sizing is not
    monotone in the row count (the split plan depends on it).  k <= 32: one call for the whole batch."""
    def need(n):
        return size("etpgt_score_topk_bf16_workspace_bytes", n, items, k)

    rows = batch
    if k > 32:
        while rows > 1 and need(rows) > budget:
            rows = (rows + 1) // 2
    ws = need(max(rows, 0))
    last = batch - (batch - 1) // rows * rows if batch > rows else rows
    if last != rows:
        ws = max(ws, need(last))
    return rows, ws


def tensor_core_scoring_supported(dim: int, k: int) -> bool:
    return dim in (64, 128, 192, 256) and 1 <= k <= SCORE_MAX_K


def auto_score_precision(batch: int, dim: int, k: int) -> str:
    """The scorer `precision="auto"` picks (predict, sharded_predict): for k <= 32, the tensor-core scorer from 64 rows
    on and the fp32 CUDA-core scorer (the reference's arithmetic) below; for 33 <= k <= 64 the fp32 scorer; above 64
    the tensor-core scorer at every batch size, the only one there."""
    if k > SCORE_F32_MAX_K and tensor_core_scoring_supported(dim, k):
        return "bf16"
    return "bf16" if batch >= 64 and k <= 32 and tensor_core_scoring_supported(dim, k) else "fp32"


def _exclusion_rows(exclude: torch.Tensor, b: int, dev, rows_sorted: bool) -> torch.Tensor:
    """Checks an exclusion list ([B, L] int64 on the scoring device) and returns it with every row sorted."""
    if not torch.is_tensor(exclude) or not exclude.is_cuda or exclude.device != dev:
        raise RuntimeError("score_topk: `exclude` must be a CUDA tensor on the device of the session embeddings")
    if exclude.dtype != torch.int64 or exclude.dim() != 2 or exclude.size(0) != b:
        raise RuntimeError(f"score_topk: `exclude` must be int64 [B={b}, L], got {exclude.dtype} "
                           f"{tuple(exclude.shape)}")
    if exclude.size(1) == 0 or rows_sorted:
        return exclude.contiguous()
    return torch.sort(exclude, dim=1).values.contiguous()


@torch.no_grad()
def score_topk(sess: torch.Tensor, table: torch.Tensor, k: int, id_base: int = 0, precision: str = "fp32",
               out: tuple | None = None, targets: torch.Tensor | None = None, exclude: torch.Tensor | None = None,
               exclude_sorted: bool = False):
    """Top-k item ids by dot product, ties to the lower id — etpgt/model/base.py:59-78.

    precision "fp32": CUDA-core scorer with the reference's fp32 arithmetic.
    precision "bf16": tcgen05 tensor-core scorer (bf16 operands, fp32 accumulation in TMEM); `table`
    may already be a bf16 copy (an evaluation loop converts it once).
    out: (top_val [B, k] f32, top_idx [B, k] i64) to write into (contiguous), else fresh tensors.
    targets [B] (bf16 scorer): also returns hit_pos [B] int32 — the position of each target in its row's results or
    -1, taken inside the scorer's select epilogue (the input of `hit_metrics`): (top_val, top_idx, hit_pos).
    exclude [B, L] int64: ids each row must not receive (e.g. `seen_items(batch)`), ranked as if they were absent
    from the table.  Rows need not be sorted (they are sorted here); duplicates, -1 padding and ids outside
    [id_base, id_base + rows of `table`) are ignored, so an item shard takes the global list.  k may then exceed a
    row's eligible items: the missing slots are (-inf, INT64_MAX), and an excluded target has hit_pos -1.
    exclude_sorted: the rows are already ascending (`seen_items` returns them so): skips the sort, which at
    evaluation size costs about a third of the scoring time."""
    _require_cuda(sess, "session embeddings")
    b, dim = sess.shape
    items = table.size(0)
    dev = sess.device
    if exclude is not None:
        exclude = _exclusion_rows(exclude, b, dev, exclude_sorted)
    if out is not None:
        top_val, top_idx = out
        if tuple(top_val.shape) != (b, k) or tuple(top_idx.shape) != (b, k) or top_val.dtype != torch.float32 \
                or top_idx.dtype != torch.int64:
            raise RuntimeError("score_topk: `out` must be (float32 [B, k], int64 [B, k])")
    else:
        top_val = torch.empty(b, k, dtype=torch.float32, device=dev)
        top_idx = torch.empty(b, k, dtype=torch.int64, device=dev)
    if precision == "bf16":
        sess_h, table_h = to_bf16(sess), to_bf16(table)
        rows, ws_bytes = score_row_chunks(b, items, k)
        ws = workspace(ws_bytes, dev)
        hit_pos = None
        if targets is not None:
            targets = _i64(targets)
            hit_pos = torch.empty(b, dtype=torch.int32, device=dev)
        for r0 in range(0, b, rows) if b > 0 else [0]:   # rows == b == 0: one call that checks the arguments
            n = min(rows, b - r0)
            s_h = sess_h[r0:r0 + n]
            tv, ti = top_val[r0:r0 + n], top_idx[r0:r0 + n]
            tg = targets[r0:r0 + n] if targets is not None else None
            hp = hit_pos[r0:r0 + n] if hit_pos is not None else None
            if exclude is None:
                call("etpgt_score_topk_bf16_eval", ptr(s_h), ptr(table_h), n, items, dim, k, id_base, ptr(tv),
                     ptr(ti), ptr(tg), ptr(hp), ptr(ws), ws.numel(), stream())
            else:
                call("etpgt_score_topk_bf16_exclude", ptr(s_h), ptr(table_h), n, items, dim, k, id_base, ptr(tv),
                     ptr(ti), ptr(tg), ptr(hp), ptr(exclude[r0:r0 + n]), exclude.size(1), ptr(ws), ws.numel(),
                     stream())
        return (top_val, top_idx) if targets is None else (top_val, top_idx, hit_pos)
    if precision != "fp32":
        raise ValueError(f"Unknown scoring precision: {precision}")
    if k > SCORE_F32_MAX_K:
        raise RuntimeError(f"score_topk: k={k} exceeds the fp32 scorer's bound of {SCORE_F32_MAX_K}; "
                         f'precision="bf16" takes k <= {SCORE_MAX_K}')
    sess_c, table_c = _f32(sess.detach()), _f32(table.detach())
    ws = workspace(size("etpgt_score_topk_workspace_bytes", b, items, dim, k), dev)
    if exclude is None:
        call("etpgt_score_topk_f32", ptr(sess_c), ptr(table_c), b, items, dim, k, id_base, ptr(top_val),
             ptr(top_idx), ptr(ws), ws.numel(), stream())
    else:
        call("etpgt_score_topk_f32_exclude", ptr(sess_c), ptr(table_c), b, items, dim, k, id_base, ptr(top_val),
             ptr(top_idx), ptr(exclude), exclude.size(1), ptr(ws), ws.numel(), stream())
    if targets is None:
        return top_val, top_idx
    # the fp32 CUDA-core scorer (small batches) has no fused epilogue: positions from its id matrix
    match = top_idx == _i64(targets).view(-1, 1)
    hit_pos = torch.where(match.any(dim=1), match.float().argmax(dim=1), torch.full((b,), -1, device=dev)).int()
    return top_val, top_idx, hit_pos


@torch.no_grad()
def seen_items(batch, num_sessions: int | None = None, width: int | None = None,
               exclude_padding: bool = True) -> torch.Tensor:
    """Exclusion rows for `score_topk(exclude=...)`: [B, L] int64, row b = the item ids of session b's graph
    (`batch.x` grouped by `batch.ptr`, or by `batch.batch` when the batch has no ptr), plus the padding id 0 when
    `exclude_padding`, sorted, padded with -1.

    width: L.  A loader that cuts sessions to `max_session_length` items gives width = max_session_length + 1 (the +1
    for id 0), and then no value is read back to the host; a session with more than L (L - 1 with id 0) items keeps
    only its first ones in the list.  None: L is the longest session (+1), which costs one host read."""
    x, bvec = batch.x, batch.batch
    dev = x.device
    if num_sessions is None:
        n = getattr(batch, "num_graphs", None)
        num_sessions = int(n) if isinstance(n, int) else None
    node_ptr = getattr(batch, "ptr", None)
    if num_sessions is None:
        num_sessions = node_ptr.numel() - 1 if node_ptr is not None else (int(bvec.max().item()) + 1 if x.numel() else 0)
    if node_ptr is None:
        counts = torch.bincount(bvec, minlength=num_sessions)
        node_ptr = torch.zeros(num_sessions + 1, dtype=torch.int64, device=dev)
        torch.cumsum(counts, 0, out=node_ptr[1:])
    node_ptr = node_ptr.to(torch.int64)
    pad = 1 if exclude_padding else 0
    if width is None:
        longest = int((node_ptr[1:] - node_ptr[:-1]).max().item()) if num_sessions > 0 else 0
        width = longest + pad
    out = torch.full((num_sessions, max(int(width), pad)), -1, dtype=torch.int64, device=dev)
    if exclude_padding:
        out[:, 0] = 0
    if x.numel() and out.size(1) > pad:
        bvec = bvec.to(torch.int64)
        col = torch.arange(x.numel(), device=dev) - node_ptr[bvec] + pad
        keep = col < out.size(1)
        out.view(-1).index_put_(((bvec * out.size(1) + col)[keep],), x.to(torch.int64)[keep])
    return torch.sort(out, dim=1).values


@torch.no_grad()
def topk_merge(cand_val: torch.Tensor, cand_idx: torch.Tensor, k: int):
    """Exact merge of per-shard candidate lists [B, parts*k] (score desc, id asc)."""
    b = cand_val.size(0)
    parts = cand_val.size(1) // k
    cand_val, cand_idx = _f32(cand_val), _i64(cand_idx)
    top_val = torch.empty(b, k, dtype=torch.float32, device=cand_val.device)
    top_idx = torch.empty(b, k, dtype=torch.int64, device=cand_val.device)
    call("etpgt_topk_merge", ptr(cand_val), ptr(cand_idx), b, parts, k, ptr(top_val), ptr(top_idx), stream())
    return top_val, top_idx


@torch.no_grad()
def topk_metrics(top_idx: torch.Tensor, targets: torch.Tensor, k: int, acc: torch.Tensor | None = None):
    """Adds (#hits@k, sum of 1/log2(pos+2)) into `acc` (double[2]) without leaving the device."""
    top_idx, targets = _i64(top_idx), _i64(targets)
    if acc is None:
        acc = torch.zeros(2, dtype=torch.float64, device=top_idx.device)
    call("etpgt_topk_metrics", ptr(top_idx), ptr(targets), top_idx.size(0), top_idx.size(1), k, ptr(acc), stream())
    return acc


def launch_count() -> int:
    return _lib.launch_count()


@torch.no_grad()
def topk_merge_parts(parts: torch.Tensor, num_parts: int, part_stride: int, idx_offset: int, rows_total: int, k: int,
                     row_begin: int, rows: int, targets: torch.Tensor | None = None):
    """Exact merge of item-sharded candidates out of the rank-major layout one all-gather leaves them in
    (etpgt_topk_merge_parts).  Returns (top_val, top_idx, hit_pos or None)."""
    dev = parts.device
    top_val = torch.empty(rows, k, dtype=torch.float32, device=dev)
    top_idx = torch.empty(rows, k, dtype=torch.int64, device=dev)
    hit_pos = None
    if targets is not None:
        targets = _i64(targets)
        hit_pos = torch.empty(rows, dtype=torch.int32, device=dev)
    call("etpgt_topk_merge_parts", ptr(parts), int(num_parts), int(part_stride), int(idx_offset), int(rows_total), int(k),
         int(row_begin), int(rows), ptr(top_val), ptr(top_idx), ptr(targets), ptr(hit_pos), stream())
    return top_val, top_idx, hit_pos


@torch.no_grad()
def hit_metrics(hit_pos: torch.Tensor, k: int, acc: torch.Tensor | None = None):
    """Adds (#targets found within the first k positions, sum of 1/log2(pos+2)) into `acc` (double[2])."""
    if acc is None:
        acc = torch.zeros(2, dtype=torch.float64, device=hit_pos.device)
    call("etpgt_hit_metrics", ptr(hit_pos), hit_pos.numel(), int(k), ptr(acc), stream())
    return acc
