"""Session-batch data parallelism over one NVLink/NVSwitch box: one process per GPU,
`torch.distributed` (NCCL) for the plumbing (SURVEY.md §8e; the reference is single-GPU).

  * sessions are independent graph components -> contiguous session ranges per rank, balanced by
    a (nodes + edges)-like cost prefix sum, no data-path collective for the graph kernels;
  * the only couplings are (a) BatchNorm statistics (2*dim+1 doubles per layer and direction, so
    whole-batch semantics are kept), (b) the loss mean over the GLOBAL batch, (c) the parameter
    gradients (dense parameters, item table).  With `enable_data_parallel(model)` (PeerDataParallel) all
    three run as kernels of this library over peer memory — every rank maps every peer's region (CUDA IPC)
    and the BatchNorm sums, the dense-gradient sum and the table's reduce-scatter + AdamW + all-gather are
    loads / stores over NVLink ordered by system-scope flags (csrc/peer.cu, csrc/optim.cu), the training step
    stays ONE host call.  `enable_global_batch_norm` + `allreduce_gradients` is the plain NCCL variant
    (all-reduces between the phases of the step driver, replicated optimizer), kept as the comparison point
    and for the per-operator autograd path;
  * evaluation shards the item table by contiguous id ranges: every rank scores all sessions
    against its shard with the fused top-k kernel, candidates are all-gathered and merged exactly
    (score desc, id asc), so the result is identical for any GPU count.
"""

from __future__ import annotations

import ctypes
import weakref

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from ._lib import stream


def world() -> tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def partition_sessions(cost: np.ndarray, parts: int) -> np.ndarray:
    """Boundaries [parts+1] of contiguous session ranges with near-equal total cost
    (cost[s] ~ nodes + edges of session s)."""
    total = np.concatenate([[0], np.cumsum(cost, dtype=np.float64)])
    targets = total[-1] * np.arange(1, parts) / parts
    cuts = np.searchsorted(total, targets, side="left")
    return np.concatenate([[0], cuts, [len(cost)]]).astype(np.int64)


def item_shard(num_items: int, rank: int, world_size: int) -> tuple[int, int]:
    """Contiguous id range [lo, hi) of the item-table shard of `rank`."""
    per = (num_items + world_size - 1) // world_size
    lo = min(rank * per, num_items)
    return lo, min(lo + per, num_items)


def enable_global_batch_norm(model, group=None) -> None:
    """BatchNorm statistics (forward and backward) are summed over every rank's node rows."""
    model.bn_process_group = group if group is not None else dist.group.WORLD


def allreduce_gradients(params, group=None) -> None:
    """Sums gradients across ranks: one flat all-reduce for the dense parameters and one for each
    large (>= 4 MB) gradient such as the item table, in place.  The loss is already divided by the
    global batch, so SUM gives the global-batch gradient."""
    rank, size = world()
    if size == 1:
        return
    small, large = [], []
    for p in params:
        if p.grad is None:
            continue
        (large if p.grad.numel() * p.grad.element_size() >= (4 << 20) else small).append(p)
    if small:
        flat = torch.cat([p.grad.reshape(-1) for p in small])
        dist.all_reduce(flat, group=group)
        offset = 0
        for p in small:   # rebind .grad to its slice of the reduced buffer: no copy back
            n = p.grad.numel()
            p.grad = flat[offset:offset + n].view_as(p.grad)
            offset += n
    for p in large:
        dist.all_reduce(p.grad, group=group)


_GATHER_INDEX: dict = {}


def _compact_index(counts: tuple, device) -> torch.Tensor:
    """Row indices that drop the padding of an all-gather of max(counts)-row blocks (cached per counts tuple)."""
    key = (counts, str(device))
    idx = _GATHER_INDEX.get(key)
    if idx is None:
        width = max(counts)
        idx = torch.from_numpy(np.concatenate([r * width + np.arange(c) for r, c in enumerate(counts)])).to(device)
        if len(_GATHER_INDEX) > 64:
            _GATHER_INDEX.clear()
        _GATHER_INDEX[key] = idx
    return idx


@torch.no_grad()
def sharded_predict(model, session_embeddings: torch.Tensor, k: int = 20, group=None, counts=None, targets=None,
                    precision: str = "auto", exclude=None, exclude_sorted: bool = False):
    """Item-sharded full-catalogue top-k (SURVEY.md section 8e): one all-gather of the session vectors, ONE scoring
    call of this rank's contiguous id range for all sessions (fused top-k), one all-gather of the packed
    (value, id) candidates, one exact merge kernel that reads the gathered layout directly.  Returns the top-k ids
    of THIS rank's sessions — identical to single-GPU scoring for any GPU count; with `targets` [B] returns
    (ids, hit_pos) where hit_pos[b] is the position of the target in the top-k or -1 (input of ops.hit_metrics).

    counts: every rank's session count (host ints), when the caller knows them (a sharding loader does);
    otherwise they are exchanged, which costs one host read.
    group=False: score on this process alone even when a process group is initialised (a single-process replica
    inside a data-parallel job: no collective is entered).

    exclude [B, L] int64 (ops.score_topk's format, e.g. ops.seen_items(batch)): ids each of this rank's sessions must
    not receive.  The rows travel with the session vectors (same padding and compaction) and every shard filters
    against the global ids.  With `counts` given every rank passes the same L (a loader's max_session_length + 1);
    without, the widths are exchanged together with the counts.  exclude_sorted: the rows are already ascending."""
    from . import ops

    rank, size = (0, 1) if group is False else world()
    table = model.get_item_embeddings()
    b_local, width = session_embeddings.shape
    dev = session_embeddings.device
    if precision == "auto":
        precision = getattr(model, "score_precision", "auto")
    if size == 1:
        if precision == "auto":
            precision = "bf16" if b_local >= 64 and ops.tensor_core_scoring_supported(width, k) else "fp32"
        if targets is None:
            return ops.score_topk(session_embeddings, table, k, precision=precision, exclude=exclude,
                                  exclude_sorted=exclude_sorted)[1]
        _, top, hit = ops.score_topk(session_embeddings, table, k, precision=precision, targets=targets,
                                     exclude=exclude, exclude_sorted=exclude_sorted)
        return top, hit
    ex_width = int(exclude.size(1)) if exclude is not None else 0
    if counts is None:
        mine = torch.tensor([b_local, ex_width], dtype=torch.int64, device=dev)
        everyone_counts = torch.empty(2 * size, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(everyone_counts, mine, group=group)
        exchanged = everyone_counts.tolist()
        counts, ex_width = exchanged[0::2], max(exchanged[1::2])
    counts = tuple(int(c) for c in counts)
    total, widest = sum(counts), max(counts)
    send = ops._f32(session_embeddings)
    if b_local != widest:
        padded = torch.zeros(widest, width, dtype=torch.float32, device=dev)
        padded[:b_local] = send
        send = padded
    gathered = torch.empty(size * widest, width, dtype=torch.float32, device=dev)
    dist.all_gather_into_tensor(gathered, send, group=group)
    everyone = gathered if total == size * widest else gathered.index_select(0, _compact_index(counts, dev))
    everyone_ex = None
    if exclude is not None:   # the exclusion rows of all sessions, gathered like the session vectors (-1: no id)
        send_ex = torch.full((widest, ex_width), -1, dtype=torch.int64, device=dev)
        send_ex[:b_local, :exclude.size(1)] = exclude
        gathered_ex = torch.empty(size * widest, ex_width, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(gathered_ex, send_ex, group=group)
        everyone_ex = gathered_ex if total == size * widest else \
            gathered_ex.index_select(0, _compact_index(counts, dev))
        if not exclude_sorted:   # sorted once here rather than by every scoring call below
            everyone_ex = torch.sort(everyone_ex, dim=1).values
    if precision == "auto":
        precision = "bf16" if total >= 64 and ops.tensor_core_scoring_supported(width, k) else "fp32"
    # this rank's candidates for ALL sessions, packed as one block: val [total, k] f32 | idx [total, k] i64
    lo, hi = item_shard(table.size(0), rank, size)
    kk = min(k, hi - lo)
    val_bytes = _align(total * k * 4)
    block = torch.empty(val_bytes + total * k * 8, dtype=torch.uint8, device=dev)
    val = block[: total * k * 4].view(torch.float32).view(total, k)
    idx = block[val_bytes:].view(torch.int64).view(total, k)
    if kk == k:
        ops.score_topk(everyone, table[lo:hi], k, id_base=lo, precision=precision, out=(val, idx), exclude=everyone_ex,
                       exclude_sorted=True)
    else:   # a shard with fewer than k items: pad with sentinels that lose every comparison
        val.fill_(float("-inf"))
        idx.fill_(torch.iinfo(torch.int64).max)
        if kk > 0:
            v, i = ops.score_topk(everyone, table[lo:hi], kk, id_base=lo, precision=precision, exclude=everyone_ex,
                                  exclude_sorted=True)
            val[:, :kk], idx[:, :kk] = v, i
    parts = torch.empty(size * block.numel(), dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(parts, block, group=group)
    start = sum(counts[:rank])
    _, top, hit = ops.topk_merge_parts(parts, size, block.numel(), val_bytes, total, k, start, b_local, targets)
    return top if targets is None else (top, hit)


# ------------------------------------------------------------------------------ peer memory


class _RawDeviceMemory:
    """`nbytes` of device memory at `address` for torch.as_tensor (CUDA array interface); `owner` is kept alive."""

    def __init__(self, address: int, nbytes: int, owner):
        self.owner = owner
        self.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(address), False),
                                         "version": 2}


class PeerComm:
    """One rank's end of the peer-memory communicator (include/etpgt_b200.h, `etpgt_comm_*`): a device region
    that every peer maps, a barrier, a small fp64 all-reduce and a sum over the peers' fp32 buffers.

    `PeerComm(region_bytes, group=...)` is collective over the torch.distributed group (handles travel through
    `all_gather_object`; the data path never touches torch.distributed).  `PeerComm.local_group(world, bytes)`
    builds `world` ranks inside ONE process on the current device (plain pointers, no IPC) — every kernel
    behaves as across GPUs, which is how the single-GPU tests cover the protocol."""

    def __init__(self, region_bytes: int, group=None, rank: int | None = None, world: int | None = None,
                 connect: bool = True):
        if rank is None:
            if dist.is_available() and dist.is_initialized():
                rank, world = dist.get_rank(group), dist.get_world_size(group)
            else:
                rank, world = 0, 1
        self.rank, self.world, self.group = int(rank), int(world), group
        self.control_bytes = int(_lib.size("etpgt_comm_control_bytes"))
        self.region_bytes = max(int(region_bytes), self.control_bytes)
        handle = ctypes.c_void_p()
        _lib.call("etpgt_comm_create", self.rank, self.world, self.region_bytes, ctypes.byref(handle))
        self.handle = handle
        self.device = torch.device("cuda", torch.cuda.current_device())
        self._finalizer = weakref.finalize(self, _lib.load().etpgt_comm_destroy, handle)
        if connect:
            self._connect_ipc()

    def _connect_ipc(self) -> None:
        if self.world == 1:
            return
        mine = (ctypes.c_ubyte * 64)()
        _lib.call("etpgt_comm_ipc_handle", self.handle, mine)
        gathered = [None] * self.world
        dist.all_gather_object(gathered, bytes(mine), group=self.group)
        _lib.call("etpgt_comm_connect_ipc", self.handle, b"".join(gathered))
        dist.barrier(group=self.group)      # every rank has mapped every region before anyone writes to a peer

    @classmethod
    def local_group(cls, world: int, region_bytes: int) -> list["PeerComm"]:
        comms = [cls(region_bytes, rank=r, world=world, connect=False) for r in range(world)]
        bases = (ctypes.c_void_p * world)(*[c.base(c.rank) for c in comms])
        for c in comms:
            _lib.call("etpgt_comm_connect_ptrs", c.handle, bases)
        return comms

    def base(self, rank: int | None = None) -> int:
        """Address (in this process) of `rank`'s region."""
        return int(_lib.load().etpgt_comm_region(self.handle, self.rank if rank is None else rank) or 0)

    def tensor(self, offset: int, shape, dtype=torch.float32, rank: int | None = None) -> torch.Tensor:
        """A tensor over [offset, offset + bytes) of `rank`'s region (default: this rank's own)."""
        shape = tuple(int(v) for v in (shape if isinstance(shape, (tuple, list, torch.Size)) else (shape,)))
        nbytes = int(np.prod(shape, dtype=np.int64)) * torch.empty(0, dtype=dtype).element_size()
        if offset < self.control_bytes or offset % 256 or offset + nbytes > self.region_bytes:
            raise ValueError(f"peer region: [{offset}, {offset + nbytes}) is outside the caller's part of the region")
        raw = torch.as_tensor(_RawDeviceMemory(self.base(rank) + offset, max(nbytes, 1), self), device=self.device)
        return raw[:nbytes].view(dtype).view(shape)

    def barrier(self, channel: int = 0) -> None:
        _lib.call("etpgt_comm_barrier", self.handle, int(channel), stream())

    def allreduce_f64(self, inp: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        out = inp if out is None else out
        _lib.call("etpgt_comm_allreduce_f64", self.handle, _lib.ptr(inp), _lib.ptr(out), inp.numel(), stream())
        return out

    def sum_f32(self, offset: int, numel: int, out: torch.Tensor) -> torch.Tensor:
        _lib.call("etpgt_comm_sum_f32", self.handle, int(offset), int(numel), _lib.ptr(out), stream())
        return out

    def set_timeout(self, seconds: float) -> None:
        _lib.call("etpgt_comm_set_timeout", self.handle, float(seconds))

    def status(self) -> int:
        """0, or the code of a wait that gave up (1 barrier, 2 all-reduce).  Synchronises the device."""
        value = ctypes.c_int(0)
        _lib.call("etpgt_comm_status", self.handle, ctypes.byref(value))
        return int(value.value)

    def check(self) -> None:
        code = self.status()
        if code:
            raise RuntimeError(f"etpgt_b200 peer communicator: a wait for a peer timed out (code {code}); "
                               "results of this step are invalid")


# item table storage address -> weak reference to the PeerDataParallel that owns it
_PEERS: dict[int, "weakref.ReferenceType[PeerDataParallel]"] = {}


def peer_for(table: torch.Tensor):
    """The PeerDataParallel whose region holds `table` (a parameter or its data), or None."""
    ref = _PEERS.get(table.data_ptr())
    peer = ref() if ref is not None else None
    if peer is None or peer.table.data_ptr() != table.data_ptr():
        return None
    return peer


def _align(n: int, a: int = 256) -> int:
    return (int(n) + a - 1) // a * a


class PeerDataParallel:
    """Data-parallel state of one model replica with the exchanges over peer memory.

    Re-homes the item table into this rank's region (peers WRITE updated rows into it), and places the table's
    gradient buffer and the flat dense-gradient buffer of the step driver there as well (peers READ them).
    Create it BEFORE the optimizer (etpgt_b200.optim picks the region's gradient buffer up as its sink) and do
    not move the model afterwards.  Per step:

        losses = fused(batch, total_sessions=global_batch)   # ONE host call; BatchNorm sums exchanged in-kernel
        optimizer.step()    # barrier | dense-gradient sum | table reduce-scatter+AdamW+all-gather | barrier

    Every rank owns the contiguous row range `item_shard(num_items, rank, world)` of the table: it keeps those
    rows' AdamW moments current (`gather_optimizer_state` collects them for a checkpoint)."""

    def __init__(self, model, group=None, comm: PeerComm | None = None, broadcast: bool = True):
        table = model.item_embedding.weight
        if not table.is_cuda or table.dtype != torch.float32:
            raise RuntimeError("PeerDataParallel needs a CUDA fp32 model (no CPU fallback)")
        self.dense = [p for p in model.parameters() if p is not table]
        dense_numel = sum(p.numel() for p in self.dense)
        control = int(_lib.size("etpgt_comm_control_bytes"))
        self.flat_offset = control
        self.grad_offset = self.flat_offset + _align(4 * dense_numel)
        self.param_offset = self.grad_offset + _align(4 * table.numel())
        total = self.param_offset + _align(4 * table.numel())
        self.comm = comm if comm is not None else PeerComm(total, group=group)
        if self.comm.region_bytes < total:
            raise ValueError(f"peer region of {self.comm.region_bytes} bytes < {total} needed for this model")
        self.rank, self.world, self.group = self.comm.rank, self.comm.world, group
        self.table = self.comm.tensor(self.param_offset, table.shape)
        with torch.no_grad():
            self.table.copy_(table.data)
            table.data = self.table
        self.table_grad = self.comm.tensor(self.grad_offset, table.shape).zero_()
        self.flat = self.comm.tensor(self.flat_offset, (max(dense_numel, 1),)).zero_()
        self.flat_reduced = torch.zeros(max(dense_numel, 1), dtype=torch.float32, device=table.device)
        self.flat_numel = 0            # elements of `flat` the step driver fills (set by FusedTrainStep)
        self.flat_dirty = False        # the driver wrote local gradients that are not summed yet
        self.rows = item_shard(table.size(0), self.rank, self.world)
        self.num_items, self.dim = int(table.size(0)), int(table.size(1))
        _PEERS[self.table.data_ptr()] = weakref.ref(self)
        model._etpgt_peer = self
        ready = dist.is_available() and dist.is_initialized()
        if ready and self.world > 1:
            model.bn_process_group = group if group is not None else dist.group.WORLD
            if broadcast:
                for t in list(model.parameters()) + list(model.buffers()):
                    dist.broadcast(t.data, dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        torch.cuda.current_stream().synchronize()
        if ready and self.world > 1:
            dist.barrier(group=group)

    # ------------------------------------------------------------------ the exchanges
    def exchange_dense(self) -> bool:
        """Dense gradients: barrier (every rank's backward is complete), then flat_reduced = sum over ranks of
        their flat buffers, in rank order.  The parameters' .grad are views of flat_reduced.  Returns False when
        the step driver did not fill the flat buffer (per-operator autograd path: the caller reduces those
        gradients through torch.distributed)."""
        if getattr(self, "_entered", False):     # allreduce_gradients() already ran for this step
            return self._reduced
        self.comm.barrier()
        self._reduced = bool(self.flat_dirty and self.flat_numel)
        if self._reduced:
            self.comm.sum_f32(self.flat_offset, self.flat_numel, self.flat_reduced)
        self.flat_dirty = False
        self._entered = True
        return self._reduced

    def mark_table_ready(self) -> None:
        """Called by the step driver where this rank's table gradient is complete (one phase before the end of the
        backward pass): `update_table` then runs on the exchange stream from that point on."""
        self.table_ready = torch.cuda.Event()
        self.table_ready.record()

    def update_table(self, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, weight_decay, decoupled, step) -> None:
        """Reduce-scatter + AdamW + all-gather of the table (etpgt_dp_adam_table) between two barriers, then the
        local gradient buffer is cleared (every peer has read its rows by then).

        When the step driver marked the point where the table gradient was complete, all of this runs on the
        exchange stream from that point — underneath the driver's last phase and the dense-parameter exchange —
        with its own barrier channel; the caller's stream joins it at the end (the next step reads the table).
        What keeps a peer from overwriting the flat dense-gradient buffer while this rank still sums it is the
        next step's first in-kernel BatchNorm all-reduce, which every rank enters after its dense sum."""
        lo, hi = self.rows
        args = (self.comm.handle, self.param_offset, self.grad_offset, _lib.ptr(exp_avg), _lib.ptr(exp_avg_sq),
                self.num_items, self.dim, lo, hi, float(lr), float(beta1), float(beta2), float(eps), float(weight_decay),
                int(decoupled), int(step))
        ready = getattr(self, "table_ready", None)
        self.table_ready = None
        if ready is None:
            if not getattr(self, "_entered", False):
                self.comm.barrier()
            _lib.call("etpgt_dp_adam_table", *args, stream())
            self.comm.barrier()
            self.table_grad.zero_()
            return
        main = torch.cuda.current_stream()
        if getattr(self, "_exchange_stream", None) is None:
            self._exchange_stream = torch.cuda.Stream(device=self.table.device)
        side = self._exchange_stream
        side.wait_event(ready)
        with torch.cuda.stream(side):
            self.comm.barrier(1)
            _lib.call("etpgt_dp_adam_table", *args, stream())
            self.comm.barrier(1)
            self.table_grad.zero_()
        main.wait_stream(side)

    def end_exchange(self) -> None:
        """The optimizer step that consumed this exchange is queued: the next exchange_dense() starts a new one."""
        self._entered = False

    def reduced_table_gradient(self) -> torch.Tensor:
        """The summed table gradient as a fresh tensor (diagnostics / tests; the training path never forms it)."""
        out = torch.empty(self.num_items, self.dim, dtype=torch.float32, device=self.table.device)
        self.comm.barrier()
        self.comm.sum_f32(self.grad_offset, self.num_items * self.dim, out)
        self.comm.barrier()
        return out

    def gather_optimizer_state(self, optimizer) -> None:
        """Collects the table's AdamW moments (each rank keeps only its own rows current) into the full tensors
        of every rank's optimizer state, so that `optimizer.state_dict()` is a complete checkpoint.  Collective."""
        if self.world == 1 or not (dist.is_available() and dist.is_initialized()):
            return
        state = optimizer.state.get(_parameter_of(optimizer, self.table))
        if not state:
            return
        per = (self.num_items + self.world - 1) // self.world
        for name in ("exp_avg", "exp_avg_sq"):
            full = state[name]
            padded = torch.zeros(per * self.world, self.dim, dtype=full.dtype, device=full.device)
            lo, hi = self.rows
            dist.all_gather_into_tensor(padded, torch.nn.functional.pad(full[lo:hi], (0, 0, 0, per - (hi - lo))),
                                        group=self.group)
            full.copy_(padded[: self.num_items])


def _parameter_of(optimizer, data: torch.Tensor):
    for group in optimizer.param_groups:
        for p in group["params"]:
            if p.data_ptr() == data.data_ptr():
                return p
    return None


def enable_data_parallel(model, group=None, exchange: str = "peer", broadcast: bool = True):
    """Makes `model` one replica of a session-batch data-parallel job.  exchange="peer": the exchanges run over
    peer memory (returns the PeerDataParallel); exchange="nccl": BatchNorm sums and gradients go through
    torch.distributed all-reduces (returns None).  Call before creating the optimizer."""
    if exchange == "peer":
        return PeerDataParallel(model, group=group, broadcast=broadcast)
    if exchange != "nccl":
        raise ValueError(f"Unknown exchange: {exchange}")
    enable_global_batch_norm(model, group)
    if broadcast and dist.is_available() and dist.is_initialized():
        for t in list(model.parameters()) + list(model.buffers()):
            dist.broadcast(t.data, dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    return None
