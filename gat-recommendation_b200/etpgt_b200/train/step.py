"""The training step through the C++ step driver (`etpgt_gt_step_run`, csrc/gt_step.cu).

`FusedTrainStep(model, loss)` does what the reference's trainer does between `optimizer.zero_grad()` and
`optimizer.step()` (etpgt/train/trainer.py:95-127: `model(batch)` -> loss -> `loss.backward()`) for a
GraphTransformer without FFN, in ONE host call: the driver launches the same kernels, in the same order and
with the same arguments as the autograd path of etpgt_b200/ops.py (results are bit-identical, tested), but
from compiled code and out of one arena, so the host cost of a step drops from ~1.6 ms of Python / autograd
dispatch to the ~80 kernel launches themselves.

    step = FusedTrainStep(model, "bpr")
    losses = step(batch)            # device tensor [3] = (total, listwise, bpr); parameter .grad are set
    optimizer.step()

Gradients follow torch's semantics (set when `.grad is None`, accumulated otherwise; the item table's rows go
into the optimizer's persistent gradient buffer when there is one).  Under data parallelism
(`parallel.enable_global_batch_norm`) the step runs phase by phase with the BatchNorm statistics all-reduced in
between, and `allreduce_gradients()` sums the dense gradients as one flat buffer plus the table gradient.
Configurations the driver does not cover (FFN, attention readout, per-node PE, eval-mode BN...) raise
`NotImplementedError` from `supported()`-guarded callers; use the per-operator path for those.
"""

from __future__ import annotations

import ctypes
import weakref
from ctypes import c_double, c_float, c_int32, c_int64, c_size_t, c_uint64, c_void_p

import torch
import torch.distributed as dist

from .. import _lib, ops
from .._lib import stream
from ..model.graph_transformer import GraphTransformer
from ..nn import TransformerConv

MAX_LAYERS = 4


class _GtLayer(ctypes.Structure):
    _fields_ = [(name, c_void_p) for name in (
        "weight", "bias", "w_beta", "bn_weight", "bn_bias", "running_mean", "running_var", "num_batches_tracked",
        "d_weight", "d_bias", "d_w_beta", "d_bn_weight", "d_bn_bias")] + [
        ("momentum", c_double), ("eps", c_double), ("alpha_seed", c_uint64), ("drop_seed", c_uint64)]


class _GtStep(ctypes.Structure):
    _fields_ = (
        [("struct_bytes", c_int64), ("num_nodes", c_int64), ("num_edges", c_int64), ("num_sessions", c_int64)]
        + [(name, c_void_p) for name in (
            "ids", "batch_vec", "rowptr", "col", "eperm", "colptr", "row", "cpos", "targets", "negatives",
            "plan_nodes_key", "plan_nodes_perm", "plan_loss_key", "plan_loss_perm")]
        + [("num_items", c_int64), ("padding_idx", c_int64)]
        + [(name, c_int32) for name in (
            "dim", "heads", "num_layers", "k_pe", "num_neg", "readout_mode", "loss_mode", "training", "backward",
            "distributed")]
        + [("alpha", c_float), ("temperature", c_float)]
        + [("total_sessions", c_double), ("alpha_p", c_double), ("drop_p", c_double)]
        + [(name, c_void_p) for name in ("table", "pe", "w_pe", "b_pe", "d_table", "d_w_pe", "d_b_pe")]
        + [("layer", _GtLayer * MAX_LAYERS)]
        + [("sess", c_void_p), ("losses", c_void_p), ("bn_sums", c_void_p), ("comm", c_void_p), ("arena", c_void_p),
           ("arena_bytes", c_size_t)])


def exchange_row(phase: int, layers: int) -> int | None:
    """Row of `bn_sums` that `phase` of the step driver produces and the next phase consumes (to be all-reduced in
    between under data parallelism), or None for phases that produce no BatchNorm statistics.  Phases 0..layers-1
    produce the forward sums of layers 0..layers-1 (rows 0..layers-1); phase layers+j (j = 0..layers-1) produces
    the backward sums of layer layers-1-j (row 2*layers-1-j); phases 2*layers and 2*layers+1 produce none (the
    table gradient is complete after phase 2*layers).  Mirrors csrc/gt_step.cu."""
    if 0 <= phase < layers:
        return phase
    if layers <= phase < 2 * layers:
        return layers + (2 * layers - 1 - phase)
    return None


def _addr(t: torch.Tensor | None):
    return None if t is None else t.data_ptr()


class FusedTrainStep:
    # batches up to this many nodes run as ONE CUDA graph launch (graph="auto"): below it the step is bound by the
    # gaps between its ~55 microsecond kernels, above it by the kernels themselves
    GRAPH_MAX_NODES = 24_576

    def __init__(self, model: GraphTransformer, loss: str = "bpr", alpha: float = 0.7, temperature: float = 1.0,
                 graph: bool | str = "auto"):
        """graph: True / False / "auto" — run the step's launches as one CUDA graph (etpgt_gt_step_run_graph;
        bit-identical results).  "auto": for batches of at most GRAPH_MAX_NODES nodes."""
        why = self.unsupported_reason(model)
        if why:
            raise NotImplementedError(f"FusedTrainStep: {why}")
        if loss not in ops.LOSS_MODES:
            raise ValueError(f"Unknown loss type: {loss}")
        self.model, self.loss, self.alpha, self.temperature = model, loss, float(alpha), float(temperature)
        self.session_embeddings = None      # [B, dim] of the last call (detached)
        self._flat = None
        self._arena, self._arena_stream = None, None
        self._table_work = None
        self._views: list[tuple[torch.nn.Parameter, torch.Tensor]] = []
        self._flat_key = None
        self._desc = _GtStep()
        self._desc.struct_bytes = ctypes.sizeof(_GtStep)
        self.graph = graph
        self._graph_cache, self._graph_stream = None, None
        self._tracked, self._bound_key, self._pe = None, None, None

    # ------------------------------------------------------------------ what the driver covers
    @staticmethod
    def unsupported_reason(model) -> str | None:
        if not isinstance(model, GraphTransformer):
            return "the step driver covers GraphTransformer models"
        if model.use_ffn:
            return "use_ffn=True is not driven (use the per-operator path)"
        if model.readout_type not in ("mean", "max", "last"):
            return f"readout '{model.readout_type}' is not driven"
        if not 1 <= len(model.convs) <= MAX_LAYERS:
            return f"1..{MAX_LAYERS} layers"
        dim = model.hidden_dim
        if model.embedding_dim != dim or not ops.supported_dim(dim) or not ops.FUSED_LAYER \
                or ops.PROJECTION_BACKEND != "tcgen05":
            return "embedding_dim == hidden_dim in {32, 64, 128, 256} on the tcgen05 projection path"
        for conv, bn in zip(model.convs, model.batch_norms):
            if not isinstance(conv, TransformerConv) or conv.heads * conv.out_channels != dim or conv.in_channels != dim:
                return "TransformerConv(dim -> dim) layers"
            if not (bn.affine and bn.track_running_stats):
                return "affine BatchNorm1d with running statistics"
        if not model.item_embedding.weight.is_cuda:
            return "CUDA parameters (no CPU fallback)"
        return None

    @classmethod
    def supported(cls, model) -> bool:
        return cls.unsupported_reason(model) is None

    # ------------------------------------------------------------------ gradient buffers
    def _dense_parameters(self):
        """[(parameters aliasing one gradient block, block numel)] in the flat gradient buffer's order."""
        model = self.model
        blocks = []
        for conv, bn in zip(model.convs, model.batch_norms):
            blocks.append(conv.fused_store("weight")[1])
            blocks.append(conv.fused_store("bias")[1])
            if conv.lin_beta is not None:
                blocks.append([conv.lin_beta.weight])
            blocks.append([bn.weight])
            blocks.append([bn.bias])
        if model.use_laplacian_pe:
            blocks.append([model.laplacian_pe.projection.weight])
            blocks.append([model.laplacian_pe.projection.bias])
        return blocks

    def _gradient_views(self):
        """One persistent flat fp32 buffer for every dense gradient (the driver's kernels OVERWRITE it); each
        parameter's .grad is a view of its slice, so the data-parallel all-reduce is one call on the buffer."""
        blocks = self._dense_parameters()
        peer = self._peer()
        key = tuple(p.data_ptr() for block in blocks for p in block) + (id(peer),)
        if key != self._flat_key:
            dev = self.model.item_embedding.weight.device
            total = sum(p.numel() for block in blocks for p in block)
            if peer is not None:
                # peer-memory data parallelism: the driver writes this rank's gradients into the peer region (the
                # other ranks read them); the parameters' .grad are views of the buffer that receives the SUM
                self._flat, shown = peer.flat[:total], peer.flat_reduced
                peer.flat_numel = total
            else:
                self._flat = shown = torch.zeros(total, dtype=torch.float32, device=dev)
            self._views, self._block_ptr, offset = [], [], 0
            for block in blocks:
                self._block_ptr.append(self._flat.data_ptr() + 4 * offset)
                for p in block:
                    self._views.append((p, shown[offset:offset + p.numel()].view_as(p)))
                    offset += p.numel()
            self._flat_key = key
        return self._block_ptr

    def _tracked_tensors(self):
        """Every tensor whose address the descriptor holds (parameters, BatchNorm buffers, the cached PE)."""
        model = self.model
        if self._tracked is None:
            tensors = [model.item_embedding.weight]
            for conv, bn in zip(model.convs, model.batch_norms):
                tensors += [conv.lin_query.weight, conv.lin_key.weight, conv.lin_value.weight, conv.lin_skip.weight,
                            conv.lin_query.bias, conv.lin_key.bias, conv.lin_value.bias, conv.lin_skip.bias]
                if conv.lin_beta is not None:
                    tensors.append(conv.lin_beta.weight)
                tensors += [bn.weight, bn.bias, bn.running_mean, bn.running_var]
                if bn.num_batches_tracked is not None:
                    tensors.append(bn.num_batches_tracked)
            if model.use_laplacian_pe:
                tensors += [model.laplacian_pe.projection.weight, model.laplacian_pe.projection.bias]
            self._tracked = tensors
        return self._tracked

    def _bind_model(self, backward: bool, peer) -> None:
        model, d = self.model, self._desc
        pe = model.laplacian_pe._cached_pe if model.use_laplacian_pe else None
        if model.use_laplacian_pe and pe is None:
            pe = model.laplacian_pe.cached()        # raises the reference's "not precomputed" error
        key = (tuple(t.data_ptr() for t in self._tracked_tensors()), None if pe is None else (pe.data_ptr(), pe.dtype),
               backward, id(peer), model.readout_type, self.loss, model.dropout_layer.p)
        if key == self._bound_key:
            return
        layers = len(model.convs)
        table = model.item_embedding.weight
        d.num_items = table.size(0)
        pad = model.item_embedding.padding_idx
        d.padding_idx = -1 if pad is None else int(pad)
        d.dim, d.heads, d.num_layers = model.hidden_dim, model.convs[0].heads, layers
        d.readout_mode, d.loss_mode = ops.READOUT_MODES[model.readout_type], ops.LOSS_MODES[self.loss]
        d.alpha, d.temperature = self.alpha, self.temperature
        d.table = table.data_ptr()
        w_pe = b_pe = None
        self._pe = None
        if model.use_laplacian_pe:
            self._pe = pe = ops._f32(pe)            # kept alive: a converted copy would otherwise be freed
            w_pe, b_pe = model.laplacian_pe.projection.weight, model.laplacian_pe.projection.bias
            d.k_pe = pe.size(1)
        else:
            d.k_pe = 0
        d.pe, d.w_pe, d.b_pe = _addr(pe), _addr(w_pe), _addr(b_pe)
        block_ptr = iter(self._gradient_views()) if backward else None
        for l, (conv, bn) in enumerate(zip(model.convs, model.batch_norms)):
            if conv.dropout != model.convs[0].dropout or conv.heads != model.convs[0].heads:
                raise NotImplementedError("FusedTrainStep: layers must share heads and attention dropout")
            layer = d.layer[l]
            layer.weight = conv.fused_store("weight")[0].data_ptr()
            layer.bias = conv.fused_store("bias")[0].data_ptr()
            layer.w_beta = _addr(conv.lin_beta.weight) if conv.lin_beta is not None else None
            layer.bn_weight, layer.bn_bias = bn.weight.data_ptr(), bn.bias.data_ptr()
            layer.running_mean, layer.running_var = bn.running_mean.data_ptr(), bn.running_var.data_ptr()
            layer.num_batches_tracked = _addr(bn.num_batches_tracked)
            if backward:
                layer.d_weight, layer.d_bias = next(block_ptr), next(block_ptr)
                layer.d_w_beta = next(block_ptr) if conv.lin_beta is not None else None
                layer.d_bn_weight, layer.d_bn_bias = next(block_ptr), next(block_ptr)
            layer.momentum = 0.1 if bn.momentum is None else float(bn.momentum)
            layer.eps = float(bn.eps)
            layer.alpha_seed = layer.drop_seed = 0
        if backward and model.use_laplacian_pe:
            d.d_w_pe, d.d_b_pe = next(block_ptr), next(block_ptr)
        else:
            d.d_w_pe = d.d_b_pe = None
        # fused_store() may have re-homed the four projection parameters of a layer: take the key again
        self._bound_key = (tuple(t.data_ptr() for t in self._tracked_tensors()),) + key[1:]

    def _peer(self):
        """The PeerDataParallel of the model when its exchanges run over peer memory (world > 1), else None."""
        peer = getattr(self.model, "_etpgt_peer", None)
        return peer if peer is not None and peer.world > 1 else None

    # ------------------------------------------------------------------ the step
    def __call__(self, batch, target_items=None, negative_items=None, total_sessions=None, backward: bool = True):
        model, d = self.model, self._desc
        ids, edge_index = batch.x, batch.edge_index
        if not ids.is_cuda:
            raise RuntimeError("etpgt_b200 models run on CUDA batches only (call batch.to('cuda')); "
                               "there is no CPU fallback")
        if getattr(batch, "laplacian_pe", None) is not None:
            raise NotImplementedError("FusedTrainStep: per-node batch.laplacian_pe is not driven")
        targets = batch.target_item if target_items is None else target_items
        negatives = batch.negative_items if negative_items is None else negative_items
        ids, targets, negatives = ops._i64(ids), ops._i64(targets), ops._i64(negatives)
        batch_vec = ops._i64(batch.batch)
        b = targets.numel()
        negatives = negatives.reshape(b, -1)     # trainer.py:87-89
        n, dim = ids.numel(), model.hidden_dim
        index = ops.graph_index_of(batch, edge_index, n)
        training = model.training
        peer = self._peer()
        distributed = training and (peer is not None or ops._dist_ready(model.bn_process_group))
        layers = len(model.convs)
        dev = ids.device
        table = model.item_embedding.weight
        if table.dtype != torch.float32 or not table.is_contiguous():
            raise RuntimeError("FusedTrainStep needs a contiguous fp32 item table")

        d.num_nodes, d.num_edges, d.num_sessions = n, index.num_edges, b
        d.ids, d.batch_vec = ids.data_ptr(), batch_vec.data_ptr()
        d.rowptr, d.col, d.eperm = index.rowptr.data_ptr(), index.col.data_ptr(), index.eperm.data_ptr()
        d.colptr, d.row, d.cpos = index.colptr.data_ptr(), index.row.data_ptr(), index.cpos.data_ptr()
        d.targets, d.negatives = targets.data_ptr(), negatives.data_ptr()
        plan_nodes, plan_loss = ops._find_plan(ids), ops._find_plan(targets, negatives)
        if plan_nodes is not None and plan_nodes.m != n:
            plan_nodes = None
        if plan_loss is not None and plan_loss.m != negatives.numel() + b:
            plan_loss = None
        d.plan_nodes_key = _addr(plan_nodes.sorted_key) if plan_nodes else None
        d.plan_nodes_perm = _addr(plan_nodes.perm) if plan_nodes else None
        d.plan_loss_key = _addr(plan_loss.sorted_key) if plan_loss else None
        d.plan_loss_perm = _addr(plan_loss.perm) if plan_loss else None
        d.num_neg = negatives.size(1)
        d.training, d.backward, d.distributed = int(training), int(backward), int(distributed)
        d.total_sessions = float(total_sessions if total_sessions else b)
        alpha_p = float(model.convs[0].dropout) if training else 0.0
        drop_p = float(model.dropout_layer.p) if training else 0.0
        d.alpha_p, d.drop_p = alpha_p, drop_p
        # everything of the descriptor that depends on the model only (parameter / buffer / gradient addresses,
        # hyper-parameters) is bound once and re-bound when an address changes (model.to(), a re-homed table, ...)
        self._bind_model(backward, peer)

        # gradients: dense ones into the flat buffer; the table's rows into the optimizer's sink or a dense .grad
        carried = []
        if backward:
            # gradients that were not cleared since the last backward: torch accumulates into them
            carried = [(p, p.grad.clone() if p.grad.data_ptr() == view.data_ptr() else p.grad)
                       for p, view in self._views if p.grad is not None]
            if carried and peer is not None:
                raise RuntimeError("FusedTrainStep under peer-memory data parallelism: gradients of the previous "
                                   "step are still set; call optimizer.zero_grad() before every step")
            sink = ops._grad_sink(table)
            if sink is None:
                if table.grad is None:
                    table.grad = torch.zeros_like(table)
                sink = table.grad
            d.d_table = sink.data_ptr()
        else:
            d.d_table = None
        # the same draws, in the same order, as the per-operator path (nn.transformer_layer)
        per_layer = int(alpha_p > 0.0) + int(drop_p > 0.0)
        if per_layer:
            seeds = iter(torch.randint(0, 2 ** 62, (per_layer * layers,)).tolist())
            for l in range(layers):
                layer = d.layer[l]
                layer.alpha_seed = next(seeds) if alpha_p > 0.0 else 0
                layer.drop_seed = next(seeds) if drop_p > 0.0 else 0

        sess = torch.empty(b, dim, dtype=torch.float32, device=dev)
        losses = torch.empty(3, dtype=torch.float32, device=dev)
        bn_sums = torch.empty(2 * layers, 2 * dim + 1, dtype=torch.float64, device=dev)
        d.sess, d.losses, d.bn_sums = sess.data_ptr(), losses.data_ptr(), bn_sums.data_ptr()
        d.comm = peer.comm.handle if (peer is not None and distributed) else None
        lib = _lib.load()
        d.arena, d.arena_bytes = None, 0
        arena_bytes = int(lib.etpgt_gt_step_arena_bytes(ctypes.byref(d)))
        if arena_bytes == 0:
            msg = _lib.last_error()
            raise (ValueError if msg.startswith(("Unknown", "Expected")) else RuntimeError)(msg)
        # the arena persists across steps (grown with head-room when a larger batch arrives): batches differ in
        # size, and a fresh GB-sized allocation per step would keep the caching allocator splitting and
        # re-growing its blocks.  It belongs to the stream that used it last.
        raw_stream = stream().value
        if self._arena is None or self._arena.numel() < arena_bytes or self._arena_stream != raw_stream \
                or self._arena.device != dev:
            self._arena = None
            self._arena = torch.empty(arena_bytes + arena_bytes // 8, dtype=torch.uint8, device=dev)
            self._arena_stream = raw_stream
        d.arena, d.arena_bytes = self._arena.data_ptr(), self._arena.numel()

        phases = 2 * layers + 2
        if self._table_work is not None:     # a previous step's table all-reduce nobody joined
            self._table_work.wait()
        self._table_work = None
        if not distributed or peer is not None:
            # one host call; under peer-memory data parallelism the driver exchanges the BatchNorm sums itself
            if self.graph is True or (self.graph == "auto" and n <= self.GRAPH_MAX_NODES):
                self._run_graph(phases)
            elif peer is not None and backward:
                # the table gradient is complete one phase before the end (the driver orders the backward tail that
                # way): mark that point, so that the optimizer can run the table's reduce-scatter + AdamW + all-gather
                # on its exchange stream UNDERNEATH the last phase (weight gradient of layer 0, PE projection gradient)
                _lib.call("etpgt_gt_step_run", ctypes.byref(d), 0, phases - 1, stream())
                peer.mark_table_ready()
                _lib.call("etpgt_gt_step_run", ctypes.byref(d), phases - 1, phases, stream())
            else:
                _lib.call("etpgt_gt_step_run", ctypes.byref(d), 0, phases, stream())
            if peer is not None and backward:
                peer.flat_dirty = True
        else:
            group = model.bn_process_group or None
            last = phases if backward else layers + 1
            for phase in range(last):
                _lib.call("etpgt_gt_step_run", ctypes.byref(d), phase, phase + 1, stream())
                row = exchange_row(phase, layers)
                if row is not None and phase < last - 1:
                    dist.all_reduce(bn_sums[row], group=group)
                elif phase == 2 * layers:
                    # the table gradient is complete: its all-reduce (the step's largest message) runs on NCCL's
                    # stream underneath the last phase; allreduce_gradients() joins it
                    self._table_work = dist.all_reduce(sink, group=group, async_op=True)
        if backward:
            for p, view in self._views:
                p.grad = view
            for p, old in carried:
                p.grad += old
        self.session_embeddings = sess
        return losses

    def _run_graph(self, phases: int) -> None:
        """All phases as one CUDA graph launch.  The legacy default stream cannot be captured, so from there the step
        runs on a stream of its own, ordered after and before the caller's stream."""
        if self._graph_cache is None:
            handle = ctypes.c_void_p()
            _lib.call("etpgt_graph_create", ctypes.byref(handle))
            self._graph_cache = handle
            self._graph_finalizer = weakref.finalize(self, _lib.load().etpgt_graph_destroy, handle)
        cur = torch.cuda.current_stream()
        if cur.cuda_stream != 0:
            _lib.call("etpgt_gt_step_run_graph", ctypes.byref(self._desc), 0, phases, self._graph_cache, stream())
            return
        if self._graph_stream is None or self._graph_stream.device != cur.device:
            self._graph_stream = torch.cuda.Stream(device=cur.device)
        side = self._graph_stream
        side.wait_stream(cur)
        _lib.call("etpgt_gt_step_run_graph", ctypes.byref(self._desc), 0, phases, self._graph_cache,
                  ctypes.c_void_p(side.cuda_stream))
        cur.wait_stream(side)

    def graph_rebuilds(self) -> int:
        """Instantiations of the executable graph so far (1 in a steady loop; every other step only updates it)."""
        return 0 if self._graph_cache is None else int(_lib.load().etpgt_graph_rebuilds(self._graph_cache))

    def allreduce_gradients(self, group=None) -> None:
        """Data parallelism: sums the dense gradients (one flat buffer) and the table gradient across ranks.
        Call it between the step and `optimizer.step()`: the table's all-reduce was started underneath the
        step's last phase and is joined here."""
        peer = self._peer()
        if peer is not None:
            # barrier + dense-gradient sum over the peers (the .grad views then show the global-batch gradient);
            # the table's reduce-scatter + update + all-gather is one kernel inside optimizer.step()
            peer.exchange_dense()
            return
        if not (dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1):
            return
        dist.all_reduce(self._flat, group=group)
        if self._table_work is not None:      # started by __call__ underneath the last phase
            self._table_work.wait()
            self._table_work = None
        else:
            dist.all_reduce(self.model.item_embedding.weight.grad, group=group)
