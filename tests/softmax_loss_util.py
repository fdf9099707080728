"""Helpers shared by the GPU tests of the full-catalogue and shared-pool softmax losses."""

import numpy as np
import torch


def err(got, want):
    """max|got - want| / max|want|."""
    got, want = torch.as_tensor(got).double(), torch.as_tensor(want).double().to(torch.as_tensor(got).device)
    return float((got - want).abs().max() / want.abs().max().clamp_min(1e-300))


def model_and_batch(dim=64, sessions=256):
    """A 2-layer GraphTransformer on cuda over 400 synth items, a batch of its first `sessions` sessions and the
    (data, graph, store) it came from."""
    from etpgt_b200 import data, synth
    from etpgt_b200.model import create_graph_transformer_optimized

    d = synth.generate(num_sessions=1200, graph_sessions=900, num_items=400, clusters=16, seed=5)
    graph = data.ItemGraph(d.item_i, d.item_j, d.num_items)
    store = data.SessionStore(d.sess_ptr, d.sess_items)
    torch.manual_seed(1)
    model = create_graph_transformer_optimized(d.num_items, dim, dim, num_layers=2, num_heads=2, dropout=0.0,
                                               use_laplacian_pe=False).cuda()
    batch = data.build_batch(graph, store, np.arange(sessions), 50, False, False)
    return model, batch, (d, graph, store)


def grads(model):
    return {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
