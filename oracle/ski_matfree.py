"""Pixel-coordinate GP regression of oracle/ski.py on grids too large for its dense definition (grid_size 300: G = 90 000).
Test infrastructure only.

The model is oracle/ski.py's.  This restatement is matrix-free and works in the n x n data space, not in the product's
eigen-coordinates on the grid (package ski.py, csrc/ski_kron.cu), so a check of one against the other is not circular.
"""
from __future__ import annotations

import numpy as np

from .ski import keys, make_grid


def ski_posterior_matfree(X, y, Xq, bounds=(0.0, 224.0), grid_size=300, length_scale=1.0, outputscale=1.0, noise=1.0,
                          const_mean=0.0, likelihood=True, var_idx=(), tol=1e-12, max_iter=200000):
    """The same posterior for grids too large for the dense definition, matrix-free: K = os K1 (x) K1 applied by
    reshaping a grid vector to gs x gs (K1 V K1), W as a scipy sparse matrix, and plain (unpreconditioned) conjugate
    gradients on the n x n system (W K W^T + s2 I) alpha = rhs, all right-hand sides at once with per-column scalars.
    Returns the mean at every row of Xq, the variance at the rows Xq[var_idx], and the CG iteration count."""
    import scipy.sparse as sp
    g0, h = make_grid(bounds[0], bounds[1], grid_size)
    gs = grid_size
    c = g0 + h * np.arange(gs)
    K1 = np.exp(-0.5 * (c[:, None] - c[None, :]) ** 2 / (length_scale * length_scale))

    def sparse_w(P):
        P = np.asarray(P, dtype=np.float64)
        n = P.shape[0]
        u = (P - g0) / h
        base = np.floor(u).astype(int) - 1
        rows, cols, vals = [], [], []
        for a in range(4):
            for b in range(4):
                rows.append(np.arange(n))
                cols.append(np.clip(base[:, 0] + a, 0, gs - 1) * gs + np.clip(base[:, 1] + b, 0, gs - 1))
                vals.append(keys(u[:, 0] - (base[:, 0] + a)) * keys(u[:, 1] - (base[:, 1] + b)))
        return sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, gs * gs))

    def kmul(V):                                            # V [G, k] -> K V
        k = V.shape[1]
        B = V.T.reshape(k, gs, gs)
        return (outputscale * (K1 @ B @ K1)).reshape(k, gs * gs).T

    W, Wq = sparse_w(X), sparse_w(Xq)
    var_idx = np.asarray(var_idx, dtype=int)
    Wv = Wq[var_idx]
    Kqv = W @ kmul(Wv.T.toarray()) if var_idx.size else np.zeros((W.shape[0], 0))   # k(X, x*) per variance query
    rhs = np.concatenate([(np.asarray(y, dtype=np.float64) - const_mean)[:, None], Kqv], axis=1)
    op = lambda V: W @ kmul(np.asarray(W.T @ V)) + noise * V
    x = np.zeros_like(rhs)
    r = rhs.copy()
    p = r.copy()
    rr = (r * r).sum(0)
    bn = np.sqrt(rr)
    it = 0
    active = np.sqrt(rr) > tol * bn
    while active.any():
        if it >= max_iter:
            raise RuntimeError(f"matrix-free CG: relative residual {np.max(np.sqrt(rr) / bn):.2e} after {it} iterations")
        q = op(p[:, active])
        alpha = rr[active] / (p[:, active] * q).sum(0)
        x[:, active] += alpha * p[:, active]
        r[:, active] -= alpha * q
        rr_new = (r[:, active] ** 2).sum(0)
        p[:, active] = r[:, active] + (rr_new / rr[active]) * p[:, active]
        rr[active] = rr_new
        active = np.sqrt(rr) > tol * bn
        it += 1
    mean = const_mean + Wq @ kmul(np.asarray(W.T @ x[:, :1]))[:, 0]
    prior = (Wv @ kmul(Wv.T.toarray())).diagonal() if var_idx.size else np.zeros(0)
    var = prior - (Kqv * x[:, 1:]).sum(0)
    return mean, var + (noise if likelihood else 0.0), it
