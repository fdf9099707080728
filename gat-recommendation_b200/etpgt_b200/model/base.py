"""Base class and session readout with the reference's public surface
(etpgt/model/base.py): `item_embedding`, `get_item_embeddings`, `predict`, `compute_loss`,
`SessionReadout(hidden_dim, readout_type)`."""

from __future__ import annotations

from abc import ABC, abstractmethod

import torch
import torch.nn as nn

from .. import ops


class BaseRecommendationModel(nn.Module, ABC):
    def __init__(self, num_items: int, embedding_dim: int = 256, hidden_dim: int = 256, num_layers: int = 3,
                 dropout: float = 0.1):
        super().__init__()
        self.num_items, self.embedding_dim, self.hidden_dim = num_items, embedding_dim, hidden_dim
        self.num_layers, self.dropout = num_layers, dropout
        # id 0 is the padding item: zero row, zero gradient, never initialised (base.py:36-37)
        self.item_embedding = nn.Embedding(num_items, embedding_dim, padding_idx=0)
        nn.init.xavier_uniform_(self.item_embedding.weight[1:])
        self.bn_process_group = None  # set by the data-parallel wrapper
        self.score_precision = "auto"  # "auto" | "fp32" | "bf16" for predict()

    @abstractmethod
    def forward(self, batch):
        """batch.x [N] item ids, batch.edge_index [2,E], batch.batch [N] -> [num_sessions, hidden]."""

    def get_item_embeddings(self) -> torch.Tensor:
        return self.item_embedding.weight

    def predict(self, session_embeddings: torch.Tensor, k: int = 20, exclude_items: torch.Tensor | None = None,
                exclude_sorted: bool = False) -> torch.Tensor:
        """Top-k item ids per session by dot product against the whole table; the [B, I] score
        matrix is never materialised (fused scoring + top-k kernel).

        exclude_items [B, L] int64 (e.g. `ops.seen_items(batch)`): ids each session must not receive, filtered inside
        the scorer; slots a session has no eligible item for hold INT64_MAX.  None ranks every id, like the
        reference's offline predict (base.py:73-76).  exclude_sorted: rows already ascending (skips a sort)."""
        precision = self.score_precision
        if precision == "auto":
            # small batches: fp32 CUDA-core scorer (the reference's arithmetic); evaluation-sized batches and k > 64:
            # tcgen05 bf16 scorer (BASELINE.json: bf16 GEMM within 1e-2, ties to the lower id)
            precision = ops.auto_score_precision(session_embeddings.size(0), session_embeddings.size(1), k)
        _, top = ops.score_topk(session_embeddings, self.get_item_embeddings(), k, precision=precision,
                                exclude=exclude_items, exclude_sorted=exclude_sorted)
        return top

    @torch.no_grad()
    def recommend(self, batch, k: int = 20, exclude_seen: bool = True) -> torch.Tensor:
        """What each session of `batch` should see next: forward pass, then the top-k items leaving out the session's
        own items and the padding id 0 (exclude_seen) — the batched form of the reference's serving path
        (recommender.py:133-134).  Like the reference it leaves train / eval mode to the caller."""
        sess = self(batch)
        exclude = ops.seen_items(batch, num_sessions=sess.size(0)) if exclude_seen else None
        return self.predict(sess, k, exclude_items=exclude, exclude_sorted=True)

    def compute_loss(self, session_embeddings, target_items, negative_items) -> torch.Tensor:
        """The model's default (BPR) loss — base.py:80-113."""
        return ops.sampled_loss(session_embeddings, self.item_embedding, target_items, negative_items, "bpr")[0]

    # helpers shared by the three model families -------------------------------------------------
    def _graph(self, batch):
        ids, edge_index = batch.x, batch.edge_index
        if not ids.is_cuda:
            raise RuntimeError("etpgt_b200 models run on CUDA batches only (call batch.to('cuda')); "
                               "there is no CPU fallback")
        return ids, ops.graph_index_of(batch, edge_index, ids.numel())

    @staticmethod
    def _num_sessions(batch):
        n = getattr(batch, "num_graphs", None)
        return int(n) if isinstance(n, int) else None


class SessionReadout(nn.Module):
    def __init__(self, hidden_dim: int = 256, readout_type: str = "mean"):
        super().__init__()
        self.hidden_dim, self.readout_type = hidden_dim, readout_type
        if readout_type == "attention":
            self.attention = nn.Linear(hidden_dim, 1)
            nn.init.xavier_uniform_(self.attention.weight)
            nn.init.zeros_(self.attention.bias)

    def forward(self, node_embeddings: torch.Tensor, batch_indices: torch.Tensor, num_sessions: int | None = None):
        if self.readout_type not in ops.READOUT_MODES:
            raise ValueError(f"Unknown readout type: {self.readout_type}")
        if num_sessions is None:  # the reference syncs here as well (base.py:146)
            num_sessions = int(batch_indices.max().item()) + 1
        seg_ptr = ops.segment_ptr(batch_indices, num_sessions)
        scores = None
        if self.readout_type == "attention":      # nn.Linear(hidden, 1): one pass over the rows, no library GEMV
            if ops.row_scores_supported(node_embeddings):
                scores = ops.RowScores.apply(node_embeddings, self.attention.weight, self.attention.bias)
            else:
                scores = self.attention(node_embeddings).squeeze(-1)
        return ops.SegmentReadout.apply(node_embeddings, scores, seg_ptr, ops.READOUT_MODES[self.readout_type])
