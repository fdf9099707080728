"""GPU-resident replacement of the reference data loader with the same entry point
(`create_dataloader(sessions_path, graph_edges_path, batch_size, num_negatives, max_session_length,
shuffle, num_workers)`, etpgt/train/dataloader.py:205-241).

The reference re-scans the 738k-row edge frame with pandas for every sample and remaps edges in a
Python loop; here the two CSVs are read ONCE into device arrays (`data.ItemGraph`, `data.SessionStore`)
and every batch — session subgraphs, PyG-collate layout, targets, Philox negatives — is produced by
device kernels (`etpgt_session_subgraphs_*`, `etpgt_sample_negatives`).  Iterating yields objects with
the attributes of the PyG `Batch` the reference trainer consumes (`x, edge_index, batch, ptr,
target_item, negative_items [B*num_neg], num_graphs`), already on the GPU.
"""

from __future__ import annotations

from pathlib import Path

import numpy as np
import torch

from .. import data, ops


def load_sessions(sessions_path) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """train.csv / val.csv (columns session_id, timestamp, itemid, ...) -> (session ids in the
    reference's group order, ptr, items ordered by timestamp inside a session) — dataloader.py:35-40,78-82."""
    import pandas as pd

    df = pd.read_csv(sessions_path, usecols=["session_id", "timestamp", "itemid"])
    df = df.sort_values(["session_id", "timestamp"], kind="stable")
    ids, counts = np.unique(df["session_id"].to_numpy(), return_counts=True)
    ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    return ids, ptr, df["itemid"].to_numpy().astype(np.int64)


class DeviceSessionLoader:
    """Iterable over GPU-built batches; `len()` = number of batches, `.num_items` as the reference dataset."""

    def __init__(self, sessions_path, graph_edges_path, batch_size=32, num_negatives=5, max_session_length=50,
                 shuffle=True, seed=0, device="cuda", symmetrize=False, self_loop_if_empty=False,
                 flatten_negatives=True, rank: int = 0, world_size: int = 1):
        import pandas as pd

        self.session_ids, ptr, items = load_sessions(Path(sessions_path))
        edges = pd.read_csv(graph_edges_path, usecols=["item_i", "item_j"])
        item_i, item_j = edges["item_i"].to_numpy(), edges["item_j"].to_numpy()
        # dataloader.py:50-58
        self.num_items = int(max(items.max(initial=0), item_i.max(initial=0), item_j.max(initial=0))) + 1
        if min(items.min(initial=0), item_i.min(initial=0), item_j.min(initial=0)) < 0:
            raise IndexError("index out of range in self: negative item id in the session / edge files")
        self._lengths = np.minimum(np.diff(ptr), max_session_length).astype(np.float64)   # per-session cost
        self.rank, self.world_size = int(rank), int(world_size)
        self._pool = ops.BatchPreparer()
        self.graph = data.ItemGraph(item_i, item_j, self.num_items, device)
        self.sessions = data.SessionStore(ptr, items, device)
        self.batch_size, self.num_negatives, self.max_session_length = batch_size, num_negatives, max_session_length
        self.shuffle, self.seed, self.epoch, self.step = shuffle, seed, 0, 0
        self.symmetrize, self.self_loop_if_empty = symmetrize, self_loop_if_empty
        self.flatten_negatives = flatten_negatives
        self.device = device

    def __len__(self) -> int:
        return (self.sessions.num_sessions + self.batch_size - 1) // self.batch_size

    def item_counts(self) -> torch.Tensor:
        """Occurrences of every item id over all stored sessions, int64 [num_items] on the device: the counts of
        the popularity proposal of train.losses.SharedPoolSoftmaxLoss."""
        return torch.bincount(self.sessions.items, minlength=self.num_items)

    def _share(self, ids: np.ndarray):
        """This rank's contiguous share of one global batch (balanced by session length), every rank's session
        count, and whether the batch is replicated: a global batch too small to give every rank two sessions is
        processed WHOLE by every rank with total_sessions = B * world — the sums every rank contributes are then
        identical, so losses, BatchNorm statistics and gradients equal those of the single batch."""
        from .. import parallel

        world = self.world_size
        if world == 1:
            return ids, (len(ids),), False
        if len(ids) < 2 * world:
            return ids, (len(ids),) * world, True
        cuts = parallel.partition_sessions(self._lengths[ids], world)
        cuts = np.maximum.accumulate(np.maximum(cuts, 2 * np.arange(world + 1)))   # >= 2 sessions for every rank
        cuts = np.minimum(cuts, len(ids) - 2 * (world - np.arange(world + 1)))
        counts = tuple(int(c) for c in np.diff(cuts))
        return ids[cuts[self.rank]:cuts[self.rank + 1]], counts, False

    def __iter__(self):
        n = self.sessions.num_sessions
        if self.shuffle:    # the same permutation on every rank (seeded CPU generator)
            order = torch.randperm(n, generator=torch.Generator().manual_seed(self.seed + self.epoch)).numpy()
        else:
            order = np.arange(n)
        self.epoch += 1
        for start in range(0, n, self.batch_size):
            whole = order[start:start + self.batch_size]
            mine, counts, replicated = self._share(whole)
            ids = torch.from_numpy(np.ascontiguousarray(mine)).to(self.device)
            batch = data.build_batch(self.graph, self.sessions, ids, self.max_session_length, self.symmetrize,
                                     self.self_loop_if_empty)
            neg = data.sample_negatives(self.sessions, ids, self.num_items, self.num_negatives, self.seed, self.step,
                                        max_len=self.max_session_length)
            # PyG collate concatenates the per-sample [num_neg] tensors (trainer.py:87-89 reshapes them back)
            batch.negative_items = neg.reshape(-1) if self.flatten_negatives else neg
            # data parallelism: the global batch this share belongs to
            batch.total_sessions = len(whole) * (self.world_size if replicated else 1)
            batch.rank_sessions, batch.replicated = counts, replicated
            # the rest of "collate": CSR / CSC index and the sorts of the two table-gradient scatters
            batch.prepared = ops.prepare_batch(batch, self.num_items, pool=self._pool)
            self.step += 1
            yield batch


def create_dataloader(sessions_path, graph_edges_path, batch_size: int = 32, num_negatives: int = 5,
                      max_session_length: int = 50, shuffle: bool = True, num_workers: int = 0,
                      rank: int = 0, world_size: int = 1) -> DeviceSessionLoader:
    """Same signature as the reference; `num_workers` is accepted and ignored (no host workers: the batch
    is built on the device).  rank / world_size (data parallelism): every rank iterates the same global batches
    and builds only its contiguous share of each."""
    del num_workers
    return DeviceSessionLoader(sessions_path, graph_edges_path, batch_size, num_negatives, max_session_length, shuffle,
                               rank=rank, world_size=world_size)
