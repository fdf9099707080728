#!/usr/bin/env python3
"""bench.py — the driver-facing benchmark of the etpgt_b200 hot path.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the CPU oracle port, same model / data / optimizer
    python bench.py ... --dump-outputs DIR                   # + the outputs of the last timed step as DIR/*.npy

Workloads
  rr      (default, BASELINE.json configs[1]) graph_transformer_optimized (D=256, L=2, H=2, k_pe=16), BPR loss,
          AdamW(1e-3, 1e-5), session batches of the synthetic RetailRocket-shaped data (82,174 items, ~740k edges).
  scaled  (BASELINE.json configs[4]) the same model on 1,000,000 items / ~20.6M co-occurrence edges (built on the
          device from ~8M Yoochoose-shaped sessions), data parallel at 1/2/4/8 GPUs.

One step = optimizer.zero_grad() + forward + loss + backward (the C++ step driver etpgt_gt_step_run through
etpgt_b200.train.step.FusedTrainStep) + gradient exchange (N > 1) + optimizer step over one batch of `--batch`
sessions per GPU (weak scaling; default 32,768).  Every step also prepares its batch (CSR + CSC index, scatter plans:
etpgt_batch_prepare) inside the timed region, one step ahead on a side stream.  N > 1: the exchanges run over peer
memory (`--exchange peer`: in-kernel BatchNorm all-reduce, dense-gradient sum, fused reduce-scatter + AdamW +
all-gather of the item table; no NCCL call on the step) or over NCCL (`--exchange nccl`, the comparison point).
Prints ONE JSON line (rank 0).

  value   sessions/s with the batch tensors already resident in HBM;
  e2e     rr: the same step driven from pinned HOST batch tensors (H2D of x / edge_index / batch / targets /
          negatives inside the timed region), loss read back every step; scaled: driven from pinned host SESSION IDS
          (H2D of the ids, session subgraphs + collate + Philox negatives built on the device — rows a1-a3);
  e2e_from_sessions   (rr) that second form next to the first;
  roofline  the dominant kernel group (fused TransformerConv fwd+bwd) timed alone with CUDA events: algorithmic
          bytes of SURVEY.md section 8(d) / time vs the measured HBM peak; `traffic` = DRAM bytes of the same launches
          from the ncu capture committed under profiles/ (this round's);
  scoring   full-catalogue evaluation scoring + top-20 (23,861 x 82,174 x 256): dense flops / time vs the measured bf16
          peak, with the GEMM kernel's tensor-pipe activity from the committed ncu capture;
  baseline_models   BASELINE.json configs[2]: GAT / GraphSAGE training steps (+ the FFN variant of the transformer) and
          their edge kernels alone; laplacian_pe_device: the one-off eigen solver on the co-occurrence graph;
  cpu_baseline  the oracle port (oracle/model_ref.py, a restatement of the reference's PyTorch/PyG path) on this
          box's host cores, on a bounded sample of the same workload, at the batch size printed with it.
"""

from __future__ import annotations

import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT / "gat-recommendation_b200"))
sys.path.insert(0, str(ROOT))

METRIC = "train sessions/sec/GPU at 1/2/4/8 B200; TransformerConv edges/sec & HBM GB/s"
DIM, LAYERS, HEADS, K_PE, NUM_NEG = 256, 2, 2, 16, 5
WORKLOADS = {
    "rr": {"items": 82_174, "label": "graph_transformer_optimized training step (fwd+BPR+bwd+AdamW), RR-synth sessions"},
    "scaled": {"items": 1_000_000, "label": "graph_transformer_optimized training step (fwd+BPR+bwd+AdamW), 1M items / "
                                            "20M edges, Yoochoose-shaped sessions"},
}
DUMP_ROWS, DUMP_MAX_BYTES = 8192, 64 << 20     # --dump-outputs: rows kept of a larger array, bytes in all


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="rr", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=32768, help="sessions per GPU per step")
    ap.add_argument("--cpu-batch", type=int, default=1024,
                    help="sessions per step of the CPU arm (the reference's per-session readout loop is O(B*N): a "
                         "32,768-session step takes minutes on the host cores, 1,024 is near the CPU's best rate)")
    ap.add_argument("--rotate", type=int, default=4, help="distinct batches rotated through the timed steps")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: gradient / BatchNorm exchange over peer memory (this library's kernels) or NCCL")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--step-only", action="store_true",
                    help="only the training-step measurements (for profiler runs): no sweep, rooflines or baselines")
    ap.add_argument("--sweep-batches", type=str, default="32,1024,16384,65536,120436",
                    help="extra device-resident measurements at these batch sizes (rank 0, 1 GPU; '' = off)")
    ap.add_argument("--scaled-sessions", type=int, default=8_000_000, help="sessions of the scaled workload")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of `value`, write what the last of them computed as DIR/<name>.npy: "
                         "the loss, the session embeddings, every parameter after the optimizer step, the dense "
                         f"gradients and the BatchNorm running statistics; an array of more than {DUMP_ROWS} rows as "
                         "a fixed, seeded sample of its rows (rank 0, b200 arm)")
    return ap.parse_args()


# ------------------------------------------------------------------------------ helpers


def load_synth():
    """etpgt_b200/synth.py by file path: the generator is host-only numpy, and loading it this way keeps the
    reference arm from importing the product package (whose __init__ loads the CUDA library)."""
    name = "etpgt_synth"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, ROOT / "gat-recommendation_b200" / "etpgt_b200" / "synth.py")
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def peaks() -> dict:
    path = ROOT / "MEASURED_PEAKS.json"
    if path.exists():
        d = json.loads(path.read_text())
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback"}


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.samples, self.proc = gpu_index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            # wait for the first sample: nvidia-smi's start-up (process spawn + NVML initialisation, 0.1-1 s, with the
            # driver lock held for part of it) must not land inside the first timed loop — under data parallelism
            # eight of them start at once
            deadline = time.time() + 5.0
            while not self.samples and self.proc.poll() is None and time.time() < deadline:
                time.sleep(0.01)
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([f.strip() for f in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None:
            self.proc.terminate()

    def summary(self) -> dict:
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.samples:
            try:
                sm.append(float(row[0])), mx.append(float(row[1]))
            except (ValueError, IndexError):
                continue
            for name, flag in zip(names, row[2:6]):
                if flag.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def sample_negatives_host(rng, members, num_items, num_neg):
    """Host negatives with the reference's acceptance rule (dataloader.py:116-124): uniform in
    [1, num_items), never a session item, duplicates allowed.  Setup only (the device sampler is the
    production path: see e2e_from_sessions)."""
    out = rng.integers(1, num_items, size=(len(members), num_neg))
    for b, items in enumerate(members):
        bad = np.isin(out[b], items)
        while bad.any():
            out[b, bad] = rng.integers(1, num_items, size=int(bad.sum()))
            bad = np.isin(out[b], items)
    return out.astype(np.int64)


class HostBatch:
    """One batch as pinned host tensors, the way the reference's DataLoader hands it over."""

    FIELDS = ("x", "edge_index", "batch", "target", "negatives")

    def __init__(self, arrays: dict, pin: bool):
        self.t = {k: torch.from_numpy(np.ascontiguousarray(arrays[k])) for k in self.FIELDS}
        if pin:
            self.t = {k: v.pin_memory() for k, v in self.t.items()}
        self.num_graphs = int(arrays["target"].shape[0])
        self.nodes, self.edges = int(arrays["x"].shape[0]), int(arrays["edge_index"].shape[1])

    def nbytes(self) -> int:
        return sum(v.numel() * v.element_size() for v in self.t.values())

    def to_device(self, device):
        return DeviceBatch({k: v.to(device, non_blocking=True) for k, v in self.t.items()}, self.num_graphs)


class DeviceBatch:
    def __init__(self, t: dict, num_graphs: int):
        self.x, self.edge_index, self.batch = t["x"], t["edge_index"], t["batch"]
        self.target_item, self.negative_items = t["target"], t["negatives"]
        self.num_graphs = num_graphs

    def fresh(self):
        """The same resident tensors behind a new batch object (nothing derived is carried along)."""
        return DeviceBatch({"x": self.x, "edge_index": self.edge_index, "batch": self.batch,
                            "target": self.target_item, "negatives": self.negative_items}, self.num_graphs)

    @classmethod
    def of(cls, b):
        """From a data.SessionBatch built on the device."""
        return cls({"x": b.x, "edge_index": b.edge_index, "batch": b.batch, "target": b.target_item,
                    "negatives": b.negative_items}, int(b.num_graphs))


def make_host_batches(data, edge_keys, first_session, batch, count, seed, pin):
    synth = load_synth()
    rng = np.random.default_rng(seed)
    out = []
    for i in range(count):
        ids = (first_session + i * batch + np.arange(batch)) % data.num_sessions
        arrays = synth.build_batch(data, ids, edge_keys=edge_keys)
        arrays["negatives"] = sample_negatives_host(rng, arrays["members"], data.num_items, NUM_NEG)
        out.append(HostBatch(arrays, pin))
    return out


def dump_outputs(path, model, last):
    """--dump-outputs: the step's outputs as float32 / float64 .npy files; inputs are seeded, so two builds given the
    same arguments can be compared file by file."""
    arrays = {"loss": last["loss"], "session_embeddings": last["session_embeddings"]}
    for name, p in model.named_parameters():
        arrays[f"param.{name}"] = p
        if p.grad is not None:
            arrays[f"grad.{name}"] = p.grad
    arrays.update({f"buffer.{name}": b for name, b in model.named_buffers() if "running" in name})
    out = {}
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy() if t.dtype != torch.float64 else t.detach().cpu().numpy()
        if a.ndim and a.shape[0] > DUMP_ROWS:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], DUMP_ROWS, replace=False))]
        out[name] = a
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_MAX_BYTES})")
    Path(path).mkdir(parents=True, exist_ok=True)
    for name, a in out.items():
        np.save(Path(path) / f"{name}.npy", a)


def cached_pe(num_items):
    return torch.randn(num_items, K_PE, generator=torch.Generator().manual_seed(7)).abs()


def workload_data(args, need_graph: bool):
    synth = load_synth()
    if args.workload == "scaled":
        return synth.generate_scaled(num_sessions=args.scaled_sessions, build_graph=need_graph)
    return synth.generate()


def workload_config(args, stats, sessions_per_step=None, exchange=None):
    return {"workload": WORKLOADS[args.workload]["label"], "name": args.workload,
            "dim": DIM, "layers": LAYERS, "heads": HEADS, "k_pe": K_PE, "negatives": NUM_NEG,
            "sessions_per_gpu_per_step": int(sessions_per_step or args.batch), "items": stats["items"],
            "graph_edges": stats["graph_edges"], "graph_nodes": stats["graph_nodes"],
            "parallelism": f"dp{args.gpus}", "exchange": exchange or (args.exchange if args.gpus > 1 else "none"),
            "l2_policy": "inputs larger than L2 (rotating batches, 84 MB+ table, >300 MB activations)"}


# ------------------------------------------------------------------------------ reference arm


def oracle_training_steps(data, edge_keys, num_items, batch, steps, warmup):
    """The CPU oracle port of the same step (embedding + PE, 2x TransformerConv/BN/residual, mean
    readout, BPR, AdamW over every parameter incl. the dense item table) on all host cores."""
    from oracle import model_ref

    torch.set_num_threads(os.cpu_count() or 1)
    g = torch.Generator().manual_seed(0)
    state = {"item_embedding.weight": torch.randn(num_items, DIM, generator=g) * 0.05,
             "laplacian_pe.projection.weight": torch.randn(DIM, K_PE, generator=g) * 0.1,
             "laplacian_pe.projection.bias": torch.zeros(DIM), "laplacian_pe._cached_pe": cached_pe(num_items)}
    state["item_embedding.weight"][0] = 0
    for layer in range(LAYERS):
        for lin in ("query", "key", "value", "skip"):
            state[f"convs.{layer}.lin_{lin}.weight"] = torch.randn(DIM, DIM, generator=g) / DIM ** 0.5
            state[f"convs.{layer}.lin_{lin}.bias"] = torch.zeros(DIM)
        state[f"convs.{layer}.lin_beta.weight"] = torch.randn(1, 3 * DIM, generator=g) * 0.05
        state[f"batch_norms.{layer}.weight"] = torch.ones(DIM)
        state[f"batch_norms.{layer}.bias"] = torch.zeros(DIM)
        state[f"batch_norms.{layer}.running_mean"] = torch.zeros(DIM)
        state[f"batch_norms.{layer}.running_var"] = torch.ones(DIM)
    params = [k for k in state if "running" not in k and "_cached_pe" not in k]
    for k in params:
        state[k].requires_grad_(True)
    opt = torch.optim.AdamW([state[k] for k in params], lr=1e-3, weight_decay=1e-5)
    batches = make_host_batches(data, edge_keys, 0, batch, 2, seed=1, pin=False)
    times = []
    for step in range(warmup + steps):
        hb = batches[step % len(batches)]
        t0 = time.perf_counter()
        sess = model_ref.graph_transformer_forward(state, hb.t["x"], hb.t["edge_index"], hb.t["batch"],
                                                   num_layers=LAYERS, num_heads=HEADS, training=True)
        loss = model_ref.bpr_loss(sess, state["item_embedding.weight"], hb.t["target"], hb.t["negatives"])
        opt.zero_grad()
        loss.backward()
        opt.step()
        loss.item()
        if step >= warmup:
            times.append(time.perf_counter() - t0)
    return batch / (sum(times) / len(times)), sum(times) / len(times)


CPU_BATCH_NOTE = ("the CPU arm steps over its own batch size: the reference's readout loops over the sessions of a "
                  "batch with a boolean mask over all nodes (etpgt/model/base.py:136-193, restated by the oracle), so a "
                  "step costs O(B*N) and the host cores' rate FALLS with the batch (measured: 1,024 -> 4,096 sessions "
                  "per step lowers sessions/s by ~40%); a 32,768-session step would take minutes")


def run_reference(args, rank):
    """The reference's CPU path (oracle port) on the host cores: same model, data and optimizer as the GPU arm, at the
    batch size `--cpu-batch` (printed in `config`; see CPU_BATCH_NOTE), a bounded number of steps.  Does not import the
    product package or load its CUDA library."""
    if rank != 0:
        return
    synth = load_synth()
    data = workload_data(args, need_graph=True)
    edge_keys = synth.sorted_edge_keys(data)
    steps, warmup = max(1, min(args.steps, 30)), min(args.warmup, 3)
    value, sec = oracle_training_steps(data, edge_keys, WORKLOADS[args.workload]["items"], args.cpu_batch, steps, warmup)
    cores = os.cpu_count() or 1
    sample = (f"{steps} steps of {args.cpu_batch} sessions after {warmup} warm-up (oracle port of the reference "
              f"PyTorch/PyG path, fp32, CPU, {cores} threads)")
    config = workload_config(args, data.stats(), sessions_per_step=args.cpu_batch, exchange="none")
    config["same_batch_as_gpu_arm"] = args.cpu_batch == args.batch
    config["batch_note"] = CPU_BATCH_NOTE
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "sessions/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
        "cpu_baseline": {"value": value, "unit": "sessions/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "sessions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------ B200 arm


def run_b200(args, rank, world_size, local_rank):
    import torch.distributed as dist

    import etpgt_b200  # noqa: F401
    from etpgt_b200 import _lib, data as ddata, ops, optim, parallel
    from etpgt_b200.model import create_graph_transformer_optimized
    from etpgt_b200.train.step import FusedTrainStep

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the etpgt_b200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    distributed = world_size > 1
    if distributed:
        dist.init_process_group("nccl", device_id=device)
    synth = load_synth()
    num_items = WORKLOADS[args.workload]["items"]
    scaled = args.workload == "scaled"

    # ---- data: sessions (host generator) -> resident device arrays; the scaled workload builds its co-occurrence
    # graph on the device (etpgt_cooc_graph_build), the rr workload takes the generator's (the reference's CSV order)
    data = workload_data(args, need_graph=not scaled)
    store = ddata.SessionStore(data.sess_ptr, data.sess_items, device)
    if scaled:
        gi, gj, _, _ = ddata.build_co_event_graph(data.sess_ptr, data.sess_items, None, 5, num_items, device)
        graph = ddata.ItemGraph(gi, gj, num_items, device)
        stats = data.stats()
        stats["graph_edges"], stats["graph_nodes"] = int(gi.numel()), int(torch.unique(torch.cat([gi, gj])).numel())
        del gi, gj
    else:
        graph = ddata.ItemGraph(data.item_i, data.item_j, num_items, device)
        stats = data.stats()

    def session_ids(first, batch, count):
        return [(first + i * batch + np.arange(batch)) % data.num_sessions for i in range(count)]

    def device_built(ids, step):
        """Rows a1-a3 on the device: session subgraphs + collate layout + Philox negatives from session ids."""
        batch = ddata.build_batch(graph, store, ids, 50, False, False)
        batch.negative_items = ddata.sample_negatives(store, ids, num_items, NUM_NEG, seed=3, step=step)
        return batch

    args.rotate = max(args.rotate, 2)   # step i + 1 is prepared while step i runs: they must be different batches
    first = rank * args.batch * args.rotate
    id_batches = session_ids(first, args.batch, args.rotate)
    ids_pinned = [torch.from_numpy(ids.astype(np.int64)).pin_memory() for ids in id_batches]
    host_batches = None
    if scaled:
        dev_batches = [DeviceBatch.of(device_built(torch.from_numpy(ids).to(device), i)) for i, ids in enumerate(id_batches)]
    else:
        edge_keys = synth.sorted_edge_keys(data)
        host_batches = make_host_batches(data, edge_keys, first, args.batch, args.rotate, seed=100 + rank, pin=True)
        dev_batches = [hb.to_device(device) for hb in host_batches]

    torch.manual_seed(0)
    model = create_graph_transformer_optimized(num_items, DIM, DIM, LAYERS, HEADS, dropout=0.1).to(device)
    model.laplacian_pe._cached_pe = cached_pe(num_items).to(device)
    peer = None
    if distributed:
        # before the optimizer: with the peer exchange the item table and its gradient buffer move into this rank's
        # peer region (parallel.PeerDataParallel); parameters are broadcast from rank 0
        peer = parallel.enable_data_parallel(model, exchange=args.exchange)
    opt = optim.AdamW(model.parameters(), lr=1e-3, weight_decay=1e-5)   # etpgt_adam_step, table-gradient sink
    params = list(model.parameters())
    total_sessions = args.batch * world_size
    model.train()

    # forward + BPR loss + backward through the C++ step driver (etpgt_gt_step_run: the same kernels as the
    # per-operator autograd path, bit-identical results, one host call); ETPGT_BENCH_AUTOGRAD=1 times that path
    fused = None if os.environ.get("ETPGT_BENCH_AUTOGRAD") else FusedTrainStep(model, "bpr")
    last = {}       # what the latest step handed its caller besides the updated model (for --dump-outputs)

    def step(batch):
        opt.zero_grad()
        if fused is not None:
            loss = fused(batch, total_sessions=total_sessions)[0]
            sess = fused.session_embeddings
            if distributed and peer is None:
                fused.allreduce_gradients()      # NCCL variant; the peer exchange is part of opt.step()
        else:
            sess = model(batch)
            loss = ops.sampled_loss(sess, model.item_embedding, batch.target_item, batch.negative_items, "bpr",
                                    total_sessions=total_sessions)[0]
            loss.backward()
            if distributed and peer is None:
                parallel.allreduce_gradients(params)
        opt.step()
        last["loss"], last["session_embeddings"] = loss, sess
        return loss

    def sync():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    step_stats = {}

    def timed(fn, steps, label="value"):
        import gc

        # the cyclic collector off inside the timed region (as timeit does): a generation-2 pass over the process's
        # objects takes milliseconds on one rank, and under data parallelism every rank then waits for it
        gc.collect()
        gc.disable()
        sync()
        mallocs = torch.cuda.memory_stats(device).get("num_device_alloc", 0)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        marks[0].record()
        for i in range(steps):
            fn(i)
            marks[i + 1].record()
        sync()
        gc.enable()
        mallocs = torch.cuda.memory_stats(device).get("num_device_alloc", 0) - mallocs
        if mallocs and rank == 0:   # a cudaMalloc inside the timed region means the warm-up was too short
            print(f"bench.py: {mallocs} device allocations inside the timed region '{label}'", file=sys.stderr)
        per_step = [marks[i].elapsed_time(marks[i + 1]) for i in range(steps)]
        step_stats[label] = {"min": min(per_step), "median": float(np.median(per_step)), "max": max(per_step),
                             "device_allocations": int(mallocs)}
        ms = torch.tensor([marks[0].elapsed_time(marks[-1])], device=device)
        if distributed:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    losses = []
    # Batch preparation runs one step ahead on a side stream, the way the reference's DataLoader (prefetching
    # workers + pinned memory) feeds its trainer: the H2D copy of batch i+1 (or of its session ids + the device
    # build of the batch), and for every source its integer preparation (ops.prepare_batch: CSR + CSC index, the
    # sorts of the two table-gradient scatters — all functions of the batch's inputs only), overlap step i.  Every
    # step still prepares (and copies in / builds) its own batch inside the timed region; nothing is cached from
    # one visit of a batch to the next.  The loss of step i is read back (pinned buffer + event) after step i+1 has
    # been queued, so the device never waits for the host.
    copy_stream = torch.cuda.Stream(device=device)
    pool = ops.BatchPreparer(depth=4)     # ring of preparation buffers: a steady loop allocates nothing
    loss_host = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    pending = {"batch": None, "ready": None, "prepared": None, "loss_event": None, "slot": 0}

    def from_host(i):
        return host_batches[i % len(host_batches)].to_device(device)

    def from_sessions(i):
        ids = ids_pinned[i % len(ids_pinned)].to(device, non_blocking=True)
        return DeviceBatch.of(device_built(ids, i))

    def resident(batches):
        # same resident tensors, a fresh batch object: no index / plans carried over from its last visit
        return lambda i: batches[i % len(batches)].fresh()

    def prefetch(i, source):
        with torch.cuda.stream(copy_stream):
            batch = source(i)
            prepared = ops.prepare_batch(batch, num_items, pool=pool)
            ready = torch.cuda.Event()
            ready.record(copy_stream)
        pending["batch"], pending["ready"], pending["prepared"] = batch, ready, prepared

    def take(i, source):
        """The prepared batch of step i (made one step ahead), handed over to the compute stream; queues the
        preparation of step i + 1."""
        if pending["batch"] is None:
            prefetch(i, source)
        batch, ready, prepared = pending["batch"], pending["ready"], pending["prepared"]
        cur = torch.cuda.current_stream()
        cur.wait_event(ready)
        for t in [batch.x, batch.edge_index, batch.batch, batch.target_item, batch.negative_items] + prepared.tensors():
            t.record_stream(cur)
        prefetch(i + 1, source)
        return batch, prepared

    def drop_pending():
        if pending["prepared"] is not None:
            pending["prepared"].release()
        pending["batch"] = pending["prepared"] = None

    def drain_loss():
        if pending["loss_event"] is not None:
            pending["loss_event"].synchronize()
            losses.append(float(loss_host[pending["slot"] ^ 1][0]))
            pending["loss_event"] = None

    resident_source = resident(dev_batches)
    in_flight = []

    def throttle():
        """Keeps the host at most two steps ahead of the device (a loop that logs its loss is never further
        ahead either).  Buffers handed from the preparation stream to the compute stream return to the
        allocator only when the device has passed them; an unbounded run-ahead would make it grow instead."""
        event = torch.cuda.Event()
        event.record()
        in_flight.append(event)
        if len(in_flight) > 2:
            in_flight.pop(0).synchronize()

    def value_step(i, source=None):
        batch, prepared = take(i, source or resident_source)
        step(batch)
        prepared.release()
        throttle()

    def read_back_step(source):
        def run(i):
            batch, prepared = take(i, source)
            loss = step(batch)
            prepared.release()
            slot = pending["slot"]
            loss_host[slot].copy_(loss.detach().reshape(1), non_blocking=True)
            event = torch.cuda.Event()
            event.record()
            drain_loss()                      # the PREVIOUS step's loss: its copy finished long ago
            pending["loss_event"], pending["slot"] = event, slot ^ 1
        return run

    def measure_read_back(source, label, warm):
        run = read_back_step(source)
        for i in range(warm):
            run(i)
        drain_loss()
        drop_pending()

        def all_steps(i):
            run(i)
            if i == args.steps - 1:
                drain_loss()              # the last loss is read inside the timed region too
        ms = timed(all_steps, args.steps, label)
        drop_pending()
        return ms

    # W untimed warm-up steps, and never fewer than 24: the first timed loop of a process (`value`) showed one step of
    # 4.6 ms (1 GPU) / 8.2 ms (8 GPUs) among 20 of ~2.9 / ~3.1 ms with nine warm-up steps, none of the later loops did
    warm = max(args.warmup, 2 * args.rotate + 1, 24)
    with ClockSampler(local_rank) as clocks:
        # ---- device-resident timing (value); the warm-up visits every rotating batch so that the caching
        # allocator and the preparation ring have seen every shape before the clock starts
        for i in range(warm):
            value_step(i)
        drop_pending()
        # the first dist.barrier of a process sets up its collective (tens of ms, and the ranks leave it far apart):
        # do that here, not at the start of the first timed region — under data parallelism a step is as slow as the
        # rank that starts last
        sync()
        sync()
        _lib.reset_launch_count()
        ms_total = timed(value_step, args.steps)
        launches = _lib.launch_count()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, model, last)
        drop_pending()
        value = total_sessions * args.steps / (ms_total / 1e3)
        # ---- end to end (e2e): host batches (rr) / host session ids + device batch build (scaled)
        e2e_extra = None
        if scaled:
            ms_e2e = measure_read_back(from_sessions, "e2e", warm)
            h2d = int(ids_pinned[0].numel() * 8)
        else:
            ms_e2e = measure_read_back(from_host, "e2e", warm)
            h2d = int(np.mean([hb.nbytes() for hb in host_batches]))
            if not args.step_only:
                ms_sess = measure_read_back(from_sessions, "e2e_from_sessions", warm)
                e2e_extra = {"value": total_sessions * args.steps / (ms_sess / 1e3), "unit": "sessions/s",
                             "ms_per_step": ms_sess / args.steps, "h2d_bytes_per_step": int(ids_pinned[0].numel() * 8),
                             "d2h_bytes_per_step": 4 + 8,
                             "what": "pinned host session ids -> H2D -> etpgt_session_subgraphs_count/_fill (a1, a2) + "
                                     "etpgt_sample_negatives (a3) + etpgt_batch_prepare + the step, all inside the "
                                     "timed region (the two batch totals are read back to size the batch tensors)"}
        e2e_value = total_sessions * args.steps / (ms_e2e / 1e3)
        # ---- >= 1 s of back-to-back steps: the short timed region above against a sustained one
        sustained = None
        if not args.step_only:
            long_steps = max(args.steps, int(1100.0 / (ms_total / args.steps)))
            ms_long = timed(value_step, long_steps, "sustained")
            drop_pending()
            sustained = {"steps": long_steps, "ms_per_step": ms_long / long_steps,
                         "value": total_sessions * long_steps / (ms_long / 1e3), "unit": "sessions/s"}
    if peer is not None:
        peer.comm.check()

    out = {
        "metric": METRIC, "value": value, "unit": "sessions/s", "n_gpus": world_size, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, stats),
        "e2e": {"value": e2e_value, "unit": "sessions/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4 + (8 if scaled else 0), "ms_per_step": ms_e2e / args.steps,
                "source": "pinned host session ids, batch built on the device" if scaled else
                          "pinned host batch tensors (x, edge_index, batch, targets, negatives)"},
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
        "step_ms": step_stats,      # device time between the ends of consecutive steps (rank 0)
        "final_loss": losses[-1] if losses else None,
        "batch_shape": {"nodes": int(dev_batches[0].x.numel()), "edges": int(dev_batches[0].edge_index.size(1))},
        "warmup_steps_run": int(warm),      # untimed steps before the first timed loop: max(W, 24)
    }
    if e2e_extra is not None:
        out["e2e_from_sessions"] = e2e_extra
    if sustained is not None:
        out["sustained"] = sustained
    if args.step_only:
        if rank == 0:
            print(json.dumps(out))
        if distributed:
            dist.destroy_process_group()
        return
    # ---- item-sharded full-catalogue evaluation (BASELINE.json configs[3]): every rank takes part
    out["sharded_eval"] = sharded_eval(model, device, rank, world_size, num_items, distributed)
    if rank == 0 and world_size == 1 and args.sweep_batches and not scaled:
        # the same step on either side of the default batch, down to the reference's own operating point (B = 32,
        # params.yaml:6) and up to a whole 120,436-session epoch as ONE batch
        out["batch_sweep"] = []
        for sweep in [int(v) for v in args.sweep_batches.split(",") if v]:
            if sweep == args.batch:
                continue
            big = [DeviceBatch.of(device_built(torch.from_numpy(ids).to(device), 50 + j))
                   for j, ids in enumerate(session_ids(0, sweep, 2))]
            total_sessions = sweep
            big_source = resident(big)
            drop_pending()
            for i in range(6):
                value_step(i, big_source)
            drop_pending()
            sweep_steps = max(args.steps // 2, 4) if sweep >= 16384 else 10 * args.steps
            ms_big = timed(lambda i: value_step(i, big_source), sweep_steps, f"sweep_{sweep}")
            drop_pending()
            out["batch_sweep"].append({"sessions_per_step": sweep, "ms_per_step": ms_big / sweep_steps,
                                       "value": sweep * sweep_steps / (ms_big / 1e3), "unit": "sessions/s",
                                       "nodes": big[0].x.numel(), "edges": big[0].edge_index.size(1)})
            del big
        total_sessions = args.batch * world_size
    if rank == 0:
        out["scoring"] = scoring_roofline(model, device, num_items)
        out["roofline"] = tconv_roofline(model, dev_batches[0], data, device, num_items, global_graph=not scaled)
        out["edges_per_s_tconv_fwd_bwd"] = out["roofline"].pop("edges_per_s")
        if world_size == 1 and not scaled:
            out["baseline_models"] = baseline_models(dev_batches, device, num_items)
            out["laplacian_pe_device"] = laplacian_pe_device(data, device, num_items)
        if world_size == 1 and not args.skip_cpu_baseline and not scaled:
            # the oracle port on the host cores, 10-25 s: at the CPU arm's batch and at 4x that (its rate falls with
            # the batch, see CPU_BATCH_NOTE); the better of the two is the baseline
            edge_keys = synth.sorted_edge_keys(data)
            cores = os.cpu_count() or 1
            v1, sec1 = oracle_training_steps(data, edge_keys, num_items, args.cpu_batch, 8, 1)
            v4, sec4 = oracle_training_steps(data, edge_keys, num_items, 4 * args.cpu_batch, 1, 1)
            out["cpu_baseline"] = {"value": max(v1, v4), "unit": "sessions/s", "cores": cores, "kind": "port",
                                   "sample": f"oracle port, fp32 CPU, {cores} threads: 8 steps of {args.cpu_batch} "
                                             f"sessions ({sec1:.2f} s/step, {v1:.0f} sessions/s) and 1 step of "
                                             f"{4 * args.cpu_batch} ({sec4:.2f} s/step, {v4:.0f} sessions/s), one "
                                             f"warm-up each; value = the better rate",
                                   "batch_note": CPU_BATCH_NOTE}
        print(json.dumps(out))
    if distributed:
        dist.destroy_process_group()


def sharded_eval(model, device, rank, world_size, num_items, distributed, sessions=23_861, k=20, reps=5):
    """BASELINE.json configs[3]: full-catalogue top-20 of 23,861 validation-sized session vectors with the item
    table sharded by contiguous id ranges over the ranks (parallel.sharded_predict: all-gather of the session
    vectors, ONE fused scoring + top-k call per rank, one all-gather of the packed candidates, one merge kernel).
    Device time, max over ranks; every rank holds a contiguous share of the sessions."""
    import torch.distributed as dist

    from etpgt_b200 import parallel

    counts = [sessions // world_size + (1 if r < sessions % world_size else 0) for r in range(world_size)]
    g = torch.Generator(device=device).manual_seed(1234 + rank)
    sess = torch.randn(counts[rank], DIM, device=device, generator=g) * 0.1
    model.eval()
    for _ in range(2):
        parallel.sharded_predict(model, sess, k=k, counts=counts)
    torch.cuda.synchronize()
    if distributed:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        parallel.sharded_predict(model, sess, k=k, counts=counts)
    b.record()
    torch.cuda.synchronize()
    ms = torch.tensor([a.elapsed_time(b) / reps], device=device)
    if distributed:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    model.train()
    ms = float(ms.item())
    flops = 2.0 * sessions * num_items * DIM
    return {"sessions": sessions, "items": num_items, "k": k, "shards": world_size, "ms": ms,
            "sessions_per_s": sessions / (ms / 1e3), "tflops": flops / (ms / 1e3) / 1e12,
            "includes": "bf16 conversion of the table shard + session gather + scoring + candidate gather + merge"}


def baseline_models(dev_batches, device, num_items, steps=10):
    """BASELINE.json configs[2]: the GAT and GraphSAGE baselines (scripts/evaluate_local.py:33-58 shapes:
    3 layers, GAT with 4 averaged heads) on the same session batches: training-step sessions/s with the
    edge-softmax / mean-aggregation kernels, BPR loss and the device optimizer; plus the edge kernels timed alone
    against the HBM roofline."""
    from etpgt_b200 import ops, optim
    from etpgt_b200.model import create_gat, create_graphsage

    out = {}
    sessions = dev_batches[0].num_graphs
    def ffn_variant():
        # the non-optimized GraphTransformer (graph_transformer.py:185-227: 3 layers, 4 heads, FFN x4): its FFN blocks
        # run as GEMM -> GELU (+ Philox dropout) in the epilogue -> GEMM (ops.FeedForward, SURVEY.md section 8 f4)
        from etpgt_b200.model import create_graph_transformer

        model = create_graph_transformer(num_items, DIM, DIM, 3, 4, dropout=0.1, laplacian_k=K_PE)
        model.laplacian_pe._cached_pe = cached_pe(num_items)
        return model

    for name, make in (("gat_l3_h4", lambda: create_gat(num_items, DIM, DIM, 3, 4, dropout=0.1)),
                       ("graphsage_l3_mean", lambda: create_graphsage(num_items, DIM, DIM, 3, dropout=0.1)),
                       ("graph_transformer_ffn_l3_h4", ffn_variant)):
        torch.manual_seed(0)
        model = make().to(device)
        opt = optim.AdamW(model.parameters(), lr=1e-3, weight_decay=1e-5)
        model.train()

        def step(batch):
            loss = ops.sampled_loss(model(batch), model.item_embedding, batch.target_item, batch.negative_items, "bpr")[0]
            opt.zero_grad()
            loss.backward()
            opt.step()

        # fresh batch objects: the graph index is rebuilt (inline, on the compute stream) in every step
        for i in range(4):
            step(dev_batches[i % len(dev_batches)].fresh())
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(steps):
            step(dev_batches[i % len(dev_batches)].fresh())
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / steps
        out[name] = {"ms_per_step": ms, "value": sessions / (ms / 1e3), "unit": "sessions/s"}
        del model, opt
    out["edge_kernels"] = edge_kernel_rooflines(dev_batches[0], device)
    return out


def laplacian_pe_device(data, device, num_items):
    """SURVEY.md section 8 f4: the one-off Laplacian-PE eigendecomposition (etpgt/encodings/laplacian_pe.py:19-66) of the
    co-occurrence graph on the device — the 17 smallest eigenpairs of the sym-normalised Laplacian of the undirected
    graph (Chebyshev-filtered subspace iteration over etpgt_lap_sym_block), timed with the setup (CSR build)."""
    from etpgt_b200.encodings.laplacian_pe import compute_laplacian_pe_device

    ei = torch.from_numpy(np.stack([data.item_i, data.item_j])).to(device)
    compute_laplacian_pe_device(ei, num_items, k=K_PE)          # warm-up (cuSOLVER handles, workspace)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pe, info = compute_laplacian_pe_device(ei, num_items, k=K_PE, return_info=True)
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    return {"seconds": sec, "nodes": num_items, "undirected_edges": int(ei.size(1)), "k": K_PE,
            "outer_iterations": int(info["iterations"]), "max_residual": float(info["residuals"].max()),
            "zero_eigenvalues": int((info["eigenvalues"].abs() < 1e-9).sum())}


def _time_launches(fn, flush, reps=20):
    for _ in range(3):
        fn()
    total = 0.0
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        total += a.elapsed_time(b)
    return total / reps


def edge_kernel_rooflines(batch, device):
    """GAT edge softmax + aggregation (W = 4 heads x 256) and GraphSAGE mean aggregation (D = 256) forward + backward
    alone on the step's own batch, L2 flushed: algorithmic bytes (SURVEY.md section 8d "other kernels": the gathered
    neighbour rows + one read / write of every node row the kernel touches + indices) / time vs the HBM peak."""
    from etpgt_b200 import ops
    from etpgt_b200._lib import call, ptr, size, stream, workspace

    pk = peaks()
    index = ops.graph_index_of(batch, batch.edge_index, batch.x.numel())
    n, e = index.num_nodes, index.num_edges
    f32 = dict(dtype=torch.float32, device=device)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    heads, width = 4, 4 * DIM
    h = torch.randn(n, width, **f32)
    a_src, a_dst = torch.randn(n, heads, **f32), torch.randn(n, heads, **f32)
    agg, m, inv_l = torch.empty(n, width, **f32), torch.empty(n, heads, **f32), torch.empty(n, heads, **f32)
    d_agg, d_h = torch.randn(n, width, **f32), torch.empty(n, width, **f32)
    d_as, d_ad = torch.empty(n, heads, **f32), torch.empty(n, heads, **f32)
    ws = workspace(size("etpgt_gat_bwd_workspace_bytes", n, e, heads), device)

    def gat_fwd():
        call("etpgt_gat_fwd", ptr(h), ptr(a_src), ptr(a_dst), n, width, heads, ptr(index.rowptr), ptr(index.col),
             ptr(index.eperm), 0.2, None, None, ptr(agg), ptr(m), ptr(inv_l), stream())

    def gat_bwd():
        call("etpgt_gat_bwd", ptr(h), ptr(a_src), ptr(a_dst), ptr(d_agg), ptr(agg), n, width, heads, ptr(index.rowptr),
             ptr(index.col), ptr(index.eperm), ptr(index.colptr), ptr(index.row), ptr(index.cpos), e, 0.2, None, None,
             ptr(m), ptr(inv_l), ptr(d_h), ptr(d_as), ptr(d_ad), ptr(ws), ws.numel(), stream())

    x = torch.randn(n, DIM, **f32)
    mean, d_mean, d_x = torch.empty(n, DIM, **f32), torch.randn(n, DIM, **f32), torch.empty(n, DIM, **f32)

    def sage_fwd():
        call("etpgt_sage_mean_fwd", ptr(x), n, DIM, ptr(index.rowptr), ptr(index.col), ptr(mean), stream())

    def sage_bwd():
        call("etpgt_sage_mean_bwd", ptr(d_mean), n, DIM, ptr(index.rowptr), ptr(index.colptr), ptr(index.row), ptr(d_x),
             stream())

    s = 4
    # GAT: forward gathers h_j per edge (+ the self loop), writes agg; backward gathers h_j and d_agg_i per edge
    # (destination pass) and again per out-edge (source pass), reads h / agg / d_agg rows, writes d_h
    bytes_gat = (e * (width * s + 4) + n * (2 * width * s + heads * 16 + 4)) + \
                (e * (3 * width * s + 12) + n * (4 * width * s + heads * 24))
    bytes_sage = (e * (DIM * s + 4) + n * (DIM * s + 4)) + (e * (DIM * s + 4) + n * (2 * DIM * s + 8))
    ms_gat = _time_launches(gat_fwd, flush) + _time_launches(gat_bwd, flush)
    ms_sage = _time_launches(sage_fwd, flush) + _time_launches(sage_bwd, flush)
    out = {}
    for name, nbytes, ms in (("gat_fwd_bwd_w1024_h4", bytes_gat, ms_gat), ("sage_mean_fwd_bwd_d256", bytes_sage, ms_sage)):
        achieved = nbytes / (ms / 1e3) / 1e9
        out[name] = {"bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s",
                     "frac": achieved / pk["hbm_gbs"], "ms": ms, "nodes": n, "edges": e, "traffic": None}
    return out


def scoring_roofline(model, device, num_items, sessions=23_861, k=20, reps=10):
    """Full-catalogue evaluation scoring (BASELINE.json config 4 shape: every validation session
    against the whole item table, top-20) on the tcgen05 kernel: dense flops / time vs the measured
    bf16 tensor peak.  The item table is converted to bf16 once, as an evaluation loop does."""
    from etpgt_b200 import ops

    pk = peaks()
    table = ops.to_bf16(model.item_embedding.weight)
    sess = torch.randn(sessions, DIM, device=device) * 0.1
    sess_h = ops.to_bf16(sess)
    for _ in range(3):
        ops.score_topk(sess_h, table, k, precision="bf16")
    torch.cuda.synchronize()
    # back-to-back launches between one pair of events: the host side of a call (tensor-map encode,
    # workspace hand-out) is hidden behind the previous call's kernels, so this is device time.  The
    # working set (54 MB operands + ~1.5 GB dump buffers) is far larger than L2.
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        ops.score_topk(sess_h, table, k, precision="bf16")
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    flops = 2.0 * sessions * num_items * DIM
    achieved = flops / (ms / 1e3) / 1e12
    out = {"bound": "tensor", "kernel": "score_dump_tc (tcgen05 bf16 GEMM on CTA pairs + fused piece dump) + score_select",
           "achieved": achieved, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": achieved / pk["bf16_tflops"],
           "peak_source": pk["source"], "ms": ms, "sessions": sessions, "items": num_items, "k": k,
           "sessions_per_s": sessions / (ms / 1e3)}
    out.update(scoring_ncu_capture())
    return out


def scoring_ncu_capture() -> dict:
    """Tensor-pipe utilisation of the scoring GEMM kernel from the committed `ncu --set full` capture of this shape
    (profiles/r02_score_ncu_full.csv; tools/prof_scoring.py under ncu) — a profiler figure, not measured in this run."""
    import csv

    path = ROOT / "profiles" / "r02_score_ncu_full.csv"
    if not path.exists():
        return {"tensor_pipe_active_pct_ncu": None}
    rows = list(csv.reader(path.open()))
    hdr = rows[0]
    for r in rows[2:]:
        d = dict(zip(hdr, r))
        if "score_dump_tc" in d.get("Kernel Name", ""):
            return {"tensor_pipe_active_pct_ncu": float(d["sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"]),
                    "gemm_kernel_us_ncu": float(d["gpu__time_duration.sum"]),
                    "ncu_capture": "profiles/r02_score_ncu_full.csv (ncu --set full --clock-control none, 23,861 x 82,174 x 256)"}
    return {"tensor_pipe_active_pct_ncu": None}


def time_tconv(qkvs, w_beta, index, device, reps=20, hubs=True):
    """Average CUDA-event time (ms) of the fused TransformerConv forward and backward launches on
    torch's current stream, L2 flushed between repetitions.  hubs: rows of more than 256 edges go through the
    hub-row kernels (the product path whenever a graph has such rows); False times the plain row kernels."""
    from etpgt_b200._lib import call, ptr, size, stream, workspace

    n, e = index.num_nodes, index.num_edges
    f32 = dict(dtype=torch.float32, device=device)
    out, agg = torch.empty(n, DIM, **f32), torch.empty(n, DIM, **f32)
    beta, m, inv_l = torch.empty(n, **f32), torch.empty(n, HEADS, **f32), torch.empty(n, HEADS, **f32)
    d_out, d_qkvs, d_wb = torch.randn(n, DIM, **f32), torch.empty_like(qkvs), torch.empty(3 * DIM, **f32)
    ws = workspace(size("etpgt_tconv_bwd_workspace_bytes", n, e, DIM, HEADS), device)
    plan = index.hub_plan() if hubs else None
    hub_ws = workspace(size("etpgt_tconv_hub_workspace_bytes", e, DIM), device) if plan is not None else None
    hub_bytes = hub_ws.numel() if hub_ws is not None else 0
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)

    def fwd():
        call("etpgt_tconv_fwd_hub", ptr(qkvs), n, DIM, HEADS, ptr(index.rowptr), ptr(index.col), ptr(index.eperm), e,
             ptr(w_beta), None, ptr(out), ptr(agg), ptr(beta), ptr(m), ptr(inv_l), ptr(plan), ptr(hub_ws), hub_bytes,
             stream())

    def bwd():
        call("etpgt_tconv_bwd_split_hub", ptr(qkvs), ptr(d_out), n, DIM, HEADS, ptr(index.rowptr), ptr(index.col),
             ptr(index.eperm), ptr(index.colptr), ptr(index.row), ptr(index.cpos), e, ptr(w_beta), None, ptr(agg),
             ptr(beta), ptr(m), ptr(inv_l), ptr(d_qkvs), None, None, None, ptr(d_wb), ptr(ws), ws.numel(), ptr(plan),
             ptr(hub_ws), hub_bytes, stream())

    return _time_launches(fwd, flush, reps), _time_launches(bwd, flush, reps)


def tconv_bytes(n, e):
    """Algorithmic bytes of one layer, SURVEY.md section 8(d), fp32, D = 256, H = 2:
    forward  E*(2*D*s) + N*(3*D*s) + E*4 + (N+1)*4 + N*H*8      = 2,052 B/edge + 3,092 B/node
    backward E*(4*D*s + 16 + 8) + N*(9*D*s)                      = 4,120 B/edge + 9,216 B/node"""
    s = 4
    fwd = e * (2 * DIM * s) + n * (3 * DIM * s) + e * 4 + (n + 1) * 4 + n * HEADS * 8
    bwd = e * (4 * DIM * s + 16 + 8) + n * (9 * DIM * s)
    return fwd, bwd


def tconv_traffic(n, e):
    """DRAM bytes (read + write) of tconv_fwd + tconv_bwd_dst + tconv_bwd_src for this batch shape from the ncu
    --set full capture committed under profiles/ (newest matching entry of profiles/tconv_traffic.json).  A shape
    without a capture is reported loudly instead of silently printing null."""
    tfile = ROOT / "profiles" / "tconv_traffic.json"
    if not tfile.exists():
        print("bench.py: profiles/tconv_traffic.json is missing: roofline.traffic = null", file=sys.stderr)
        return None, None
    entries = json.loads(tfile.read_text())
    entries = entries if isinstance(entries, list) else [entries]
    for entry in reversed(entries):
        if entry.get("nodes") == n and entry.get("edges") == e:
            return entry["dram_bytes_fwd_bwd"], entry.get("capture")
    print(f"bench.py: no ncu capture for the batch shape (nodes={n}, edges={e}) in profiles/tconv_traffic.json "
          f"(has {[(x.get('nodes'), x.get('edges')) for x in entries]}): roofline.traffic = null — re-capture with "
          "tools/prof_tconv.sh", file=sys.stderr)
    return None, None


def tconv_roofline(model, batch, data, device, num_items, global_graph=True):
    """The dominant edge-kernel group timed alone: (a) on the step's own layer-0 tensors (session batch:
    millions of tiny segments) and (b) on the whole symmetrised co-occurrence graph as ONE graph (power-law
    rows; the notebook's "whole graph as one session" case, SURVEY.md section 0)."""
    from etpgt_b200 import ops

    pk = peaks()
    index = ops.graph_index_of(batch, batch.edge_index, batch.x.numel())
    n, e = index.num_nodes, index.num_edges
    conv = model.convs[0]
    with torch.no_grad():
        x = ops.EmbedPE.apply(batch.x, model.item_embedding.weight, model.laplacian_pe.cached(), False,
                              model.laplacian_pe.projection.weight, model.laplacian_pe.projection.bias, 0)
        qkvs = conv.project(x).contiguous()
        w_beta = conv.lin_beta.weight.detach().reshape(-1).contiguous()
    ms_f, ms_b = time_tconv(qkvs, w_beta, index, device)
    bytes_f, bytes_b = tconv_bytes(n, e)
    achieved = (bytes_f + bytes_b) / ((ms_f + ms_b) / 1e3) / 1e9
    traffic, capture = tconv_traffic(n, e)
    out = {"bound": "hbm", "kernel": "tconv_fwd + tconv_bwd_dst + tconv_bwd_src (layer 0, session batch)",
           "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": achieved / pk["hbm_gbs"],
           "peak_source": pk["source"], "traffic": traffic, "traffic_capture": capture,
           "bytes_model": "SURVEY.md 8(d): fwd 2,052 B/edge + 3,092 B/node, bwd 4,120 B/edge + 9,216 B/node",
           "algorithmic_bytes": bytes_f + bytes_b, "ms_fwd": ms_f, "ms_bwd": ms_b,
           "gbs_fwd": bytes_f / (ms_f / 1e3) / 1e9, "gbs_bwd": bytes_b / (ms_b / 1e3) / 1e9,
           "nodes": n, "edges": e, "edges_per_s": e / ((ms_f + ms_b) / 1e3)}
    if traffic:
        # what actually crossed the HBM interface (ncu): below the algorithmic bytes because the neighbour rows
        # of a session are adjacent and are served by L1 / L2 — which is also how `frac` can exceed 1
        out["achieved_dram"] = traffic / ((ms_f + ms_b) / 1e3) / 1e9
        out["frac_dram"] = out["achieved_dram"] / pk["hbm_gbs"]
        out["note"] = ("achieved = algorithmic bytes / time; measured DRAM traffic is lower (L1/L2 reuse of "
                       "neighbour rows), see achieved_dram / frac_dram; global_graph is the same kernel group on a "
                       "working set larger than L2")
    if not global_graph:
        return out
    # (b) the whole graph, both directions of every stored pair
    src = torch.from_numpy(np.concatenate([data.item_i, data.item_j])).to(device)
    dst = torch.from_numpy(np.concatenate([data.item_j, data.item_i])).to(device)
    gindex = ops.GraphIndex(torch.stack([src, dst]), data.num_items)
    with torch.no_grad():
        gq = conv.project(model.item_embedding.weight.detach()).contiguous()
    gf, gb = time_tconv(gq, w_beta, gindex, device, reps=10)
    gbf, gbb = tconv_bytes(gindex.num_nodes, gindex.num_edges)
    g_ach = (gbf + gbb) / ((gf + gb) / 1e3) / 1e9
    out["global_graph"] = {"nodes": gindex.num_nodes, "edges": gindex.num_edges, "ms_fwd": gf, "ms_bwd": gb,
                           "achieved": g_ach, "frac": g_ach / pk["hbm_gbs"],
                           "edges_per_s_fwd": gindex.num_edges / (gf / 1e3),
                           "edges_per_s_fwd_bwd": gindex.num_edges / ((gf + gb) / 1e3),
                           "max_degree": int(torch.diff(gindex.rowptr).max().item()),
                           "hub_rows": gindex.hub_plan() is not None}
    # (c) the same node / edge counts with the popularity law of the reference's generator (zipf(1.5) weights,
    # scripts/data/00_generate_synthetic_data.py:53): rows of 10,000+ edges, cut into chunks by the hub-row kernels;
    # `serial_rows` is the same graph through the plain row kernels (one lane group per row)
    zi, zj = load_synth().zipf_graph(data.num_items, len(data.item_i))
    zsrc = torch.from_numpy(np.concatenate([zi, zj])).to(device)
    zdst = torch.from_numpy(np.concatenate([zj, zi])).to(device)
    zindex = ops.GraphIndex(torch.stack([zsrc, zdst]), data.num_items)
    zf, zb = time_tconv(gq, w_beta, zindex, device, reps=10)
    sf, sb = time_tconv(gq, w_beta, zindex, device, reps=3, hubs=False)
    zbf, zbb = tconv_bytes(zindex.num_nodes, zindex.num_edges)
    z_ach = (zbf + zbb) / ((zf + zb) / 1e3) / 1e9
    counts = zindex.hub_plan()[:16].view(torch.int32).tolist() if zindex.hub_plan() is not None else [0, 0, 0, 0]
    out["zipf_graph"] = {"nodes": zindex.num_nodes, "edges": zindex.num_edges, "ms_fwd": zf, "ms_bwd": zb,
                         "achieved": z_ach, "frac": z_ach / pk["hbm_gbs"], "vs_global_graph": z_ach / g_ach,
                         "max_degree": int(torch.diff(zindex.rowptr).max().item()),
                         "hub_destinations": counts[0], "hub_chunks": counts[1],
                         "serial_rows": {"ms_fwd": sf, "ms_bwd": sb,
                                         "achieved": (zbf + zbb) / ((sf + sb) / 1e3) / 1e9}}
    return out


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs writes the outputs of the b200 arm only")
        run_reference(args, rank)
        return
    if world_size == 1 and args.gpus > 1:
        # launched without torchrun: N independent ranks are not available; measure one GPU
        print(f"bench.py: --gpus {args.gpus} without torchrun env; running a single rank", file=sys.stderr)
    run_b200(args, rank, world_size, local_rank)


if __name__ == "__main__":
    main()
