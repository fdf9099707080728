"""Helpers shared by the parity tests: load a tests/golden fixture written by
oracle/make_golden.py and the error measure the tolerances are stated in.

A fixture at production width (D = 256) would take megabytes, so make_golden.py may store it compact:
no `state/*` arrays but the seeds they were drawn from and a SHA-256 of the arrays (the state is
re-drawn here and checked against it), and a fixed sample of the entries of every large gradient
(`grad/<name>` values at the flat positions `grad_index/<name>`)."""

import hashlib
from pathlib import Path

import numpy as np
import torch

GOLDEN = Path(__file__).resolve().parent / "golden"
GRAD_SAMPLE = 8192      # entries kept of a gradient larger than this in a compact fixture


def reference_init_state(cfg, seed, pe_seed, pe_k=16):
    """The state dict of the reference's `create_graph_transformer_optimized(**cfg)` (mean readout, Laplacian
    PE) after `torch.manual_seed(seed)`, with `_cached_pe = randn(num_items, pe_k, seed pe_seed).abs()` and the
    BatchNorm parameters and running statistics drawn as oracle/make_golden.py draws them: the constructor's
    draws replayed in its order (etpgt/model/base.py, encodings/laplacian_pe.py, model/graph_transformer.py;
    torch_geometric TransformerConv creates lin_key, lin_query, lin_value, lin_skip, lin_beta)."""
    nn = torch.nn
    items, emb, hid = int(cfg["num_items"]), int(cfg["embedding_dim"]), int(cfg["hidden_dim"])
    layers = int(cfg["num_layers"])
    state = {}
    with torch.random.fork_rng(devices=[]), torch.no_grad():      # the caller's generator state is left as it was
        torch.manual_seed(seed)
        table = nn.Embedding(items, emb, padding_idx=0)
        nn.init.xavier_uniform_(table.weight[1:])
        state["item_embedding.weight"] = table.weight
        proj = nn.Linear(pe_k, emb)
        nn.init.xavier_uniform_(proj.weight)
        nn.init.zeros_(proj.bias)
        state["laplacian_pe._cached_pe"] = torch.randn(items, pe_k, generator=torch.Generator().manual_seed(pe_seed)).abs()
        state["laplacian_pe.projection.weight"], state["laplacian_pe.projection.bias"] = proj.weight, proj.bias
        for layer, width in enumerate([emb] + [hid] * (layers - 1)):
            for lin in ("key", "query", "value", "skip"):
                m = nn.Linear(width, hid)
                state[f"convs.{layer}.lin_{lin}.weight"], state[f"convs.{layer}.lin_{lin}.bias"] = m.weight, m.bias
            state[f"convs.{layer}.lin_beta.weight"] = nn.Linear(3 * hid, 1, bias=False).weight
        for layer in range(layers):
            bn = nn.BatchNorm1d(hid)
            bn.weight.uniform_(0.5, 1.5)
            bn.bias.uniform_(-0.2, 0.2)
            bn.running_mean.uniform_(-0.1, 0.1)
            bn.running_var.uniform_(0.5, 1.5)
            for k, v in bn.state_dict().items():
                state[f"batch_norms.{layer}.{k}"] = v
    return {k: v.detach().numpy().copy() for k, v in state.items()}


def state_digest(state):
    """SHA-256 over the names, dtypes, shapes and bytes of a state dict of numpy arrays."""
    h = hashlib.sha256()
    for k in sorted(state):
        v = np.ascontiguousarray(state[k])
        h.update(f"{k}|{v.dtype.str}|{v.shape}|".encode())
        h.update(v.tobytes())
    return h.hexdigest()


def compact(out, seed, pe_seed):
    """A fixture dict written by oracle/make_golden.py, made compact (see the module docstring)."""
    state = {k[6:]: v for k, v in out.items() if k.startswith("state/")}
    cfg = {k[4:]: v for k, v in out.items() if k.startswith("cfg_")}
    digest = state_digest(state)
    assert state_digest(reference_init_state(cfg, seed, pe_seed)) == digest, "the state replay differs"
    res = {k: v for k, v in out.items() if not k.startswith("state/")}
    res.update(state_seed=np.asarray(seed), pe_seed=np.asarray(pe_seed), state_sha256=np.asarray(digest))
    rng = np.random.default_rng(0)
    for k in sorted(k for k in out if k.startswith("grad/")):
        if out[k].size > GRAD_SAMPLE:
            index = np.sort(rng.choice(out[k].size, GRAD_SAMPLE, replace=False)).astype(np.int32)
            res[k], res["grad_index/" + k[5:]] = out[k].reshape(-1)[index], index
    return res


class Golden:
    def __init__(self, name):
        self.raw = dict(np.load(GOLDEN / f"{name}.npz"))
        if "state_seed" in self.raw:
            state = reference_init_state(self.cfg(), int(self.raw["state_seed"]), int(self.raw["pe_seed"]))
            assert state_digest(state) == str(self.raw["state_sha256"]), f"{name}: the re-drawn state differs"
            self.raw.update({"state/" + k: v for k, v in state.items()})

    def gradients(self):
        """{parameter: (want, flat positions or None)}; `pick(grad, positions)` gives what `want` holds."""
        index = self.group("grad_index")
        return {k: (v, index.get(k)) for k, v in self.group("grad").items()}

    def tensor(self, key, dtype=None):
        t = torch.from_numpy(np.asarray(self.raw[key]))
        return t if dtype is None else t.to(dtype)

    def group(self, prefix, dtype=None):
        n = len(prefix) + 1
        return {k[n:]: self.tensor(k, dtype) for k in self.raw if k.startswith(prefix + "/")}

    def cfg(self):
        out = {}
        for k, v in self.raw.items():
            if k.startswith("cfg_"):
                out[k[4:]] = v.item() if hasattr(v, "item") else v
        return out


def pick(t, index):
    """The entries of `t` at the flat positions `index` (all of `t` for None)."""
    return t if index is None else t.reshape(-1)[index.to(t.device).long()]


def rel_err(got, want, floor=1e-9):
    """max |got - want| / max(|want|): the 'relative' of BASELINE.json's 1e-4 bound.  `floor`
    keeps analytically-zero tensors (e.g. the key-bias gradient, which the per-destination
    softmax cancels exactly) from dividing rounding noise by rounding noise."""
    got = torch.as_tensor(got).double().cpu()
    want = torch.as_tensor(want).double().cpu()
    assert got.shape == want.shape, (got.shape, want.shape)
    if want.numel() == 0:
        return 0.0
    denom = want.abs().max().item()
    return (got - want).abs().max().item() / max(denom, floor)
