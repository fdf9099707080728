"""TEST INFRASTRUCTURE — fp64 reference of the row-sparse ("lazy") AdamW / Adam update of etpgt_b200.optim.

Built on the dense oracle (oracle/optim_ref.adam_step, pinned to torch.optim in tests/test_optim_oracle.py):
a row whose gradient row has an element != 0 (or a NaN) gets exactly the dense update with the global step;
every other row keeps its parameter and moments.
"""

from __future__ import annotations

import numpy as np

from oracle import optim_ref


def touched_rows(grad) -> np.ndarray:
    """Boolean mask of the rows of a [rows, dim] gradient that the lazy step updates."""
    g = np.asarray(grad)
    return ((g != 0) | np.isnan(g)).any(axis=1)


def lazy_adam_step(param, grad, exp_avg, exp_avg_sq, step, **kw):
    """One lazy update; returns new (param, exp_avg, exp_avg_sq) as float64 arrays and the touched-row mask."""
    p = np.asarray(param, dtype=np.float64).copy()
    m = np.asarray(exp_avg, dtype=np.float64).copy()
    v = np.asarray(exp_avg_sq, dtype=np.float64).copy()
    hit = touched_rows(grad)
    if hit.any():
        p[hit], m[hit], v[hit] = optim_ref.adam_step(p[hit], np.asarray(grad, dtype=np.float64)[hit], m[hit], v[hit],
                                                     step, **kw)
    return p, m, v, hit
