"""Greedy Kriging-believer batch acquisition in dense numpy fp64 (test infrastructure only).

Reference for ActiveMaskGP.select_batch / nib_gp_kb_select.  Each pick is fantasised at its posterior mean; that leaves
every other posterior mean unchanged, so the mean is computed once (gp.gp_fit / gp.gp_predict on the real training set)
and only the variance is recomputed after each pick:

    var_k(x) = y_std^2 * max(0, 1 - k_x^T (K_k + alpha I)^-1 k_x)      K_k: training set + the first k picks

with y_std frozen at the real training set's.  EI is gp.expected_improvement's with the incumbent b updated to
max(b, mu_j) (min when not greater_is_better) after each pick; picked candidates get sigma = NaN; the pick is the
arg-max of the non-NaN EI, lowest index on ties; no non-NaN EI left stops the batch.
"""
from __future__ import annotations

import numpy as np
from scipy.linalg import cho_factor, cholesky, solve_triangular

from . import gp as ogp


def _pick(mu, var, y_std, used, best, greater_is_better):
    sd = np.sqrt(var * y_std ** 2)
    sd[used] = np.nan
    ei = -ogp.expected_improvement(mu, sd, np.array([best]), greater_is_better)
    if np.isnan(ei).all():
        return -1, ei
    return int(np.nanargmax(ei)), ei


def kriging_believer_batch(Ztrain, y, cand, q, ell, alpha=1e-5, greater_is_better=True, bordered=False, follow=None):
    """Ztrain [n, S] and cand [m, S] 0/1 design matrices, y [n].  Returns a dict:
      picks      the oracle's pick at each step (its own arg-max)
      ei         [k, m] EI of every candidate at each step (NaN for used ones)
      ei_at_pick EI of the candidate conditioned on at each step (the oracle's pick, or follow[k])
      var        [k+1, m] normalised variance max(0, 1 - k^T (K + alpha I)^-1 k) after 0, 1, .., k picks
      mu, y_std  the fixed posterior mean and the frozen y scale
    `follow`: candidate indices to condition on instead of the oracle's own picks (so a caller whose pick differs by an
    EI tie can keep comparing along its own path).  bordered=False factors K_k from scratch with cho_factor at every step;
    bordered=True factors the training set once and borders the factor by one solve_triangular per pick."""
    Ztrain, cand = np.asarray(Ztrain, np.float64), np.asarray(cand, np.float64)
    fit = ogp.gp_fit(Ztrain, y, ell, alpha)
    mu, _, _ = ogp.gp_predict(fit, cand)
    y_std = fit["y_std"]
    y = np.asarray(y, np.float64)
    best = float(y.max() if greater_is_better else y.min())
    m, n = cand.shape[0], Ztrain.shape[0]
    used = np.zeros(m, bool)
    T = Ztrain
    if bordered:
        L = np.zeros((n + q, n + q))
        L[:n, :n] = cholesky(ogp.rbf_gram(T, None, ell) + alpha * np.eye(n), lower=True, check_finite=False)
        V = np.empty((n + q, m))
        V[:n] = solve_triangular(L[:n, :n], ogp.rbf_gram(T, cand, ell), lower=True, check_finite=False)
        ssq = np.einsum("ij,ij->j", V[:n], V[:n])

    def variance():
        if bordered:
            return np.maximum(0.0, 1.0 - ssq)
        c, _ = cho_factor(ogp.rbf_gram(T, None, ell) + alpha * np.eye(T.shape[0]), lower=True, check_finite=False)
        W = solve_triangular(c, ogp.rbf_gram(T, cand, ell), lower=True, check_finite=False)
        return np.maximum(0.0, 1.0 - np.einsum("ij,ij->j", W, W))

    picks, eis, ei_at, vars_ = [], [], [], [variance()]
    for k in range(q):
        j, ei = _pick(mu, vars_[-1], y_std, used, best, greater_is_better)
        if j < 0 or (follow is not None and k >= len(follow)):
            break
        picks.append(j)
        eis.append(ei)
        if follow is not None:
            j = int(follow[k])
        ei_at.append(ei[j])
        z = cand[j:j + 1]
        if bordered:
            nk = n + k
            l = solve_triangular(L[:nk, :nk], ogp.rbf_gram(T, z, ell)[:, 0], lower=True, check_finite=False)
            d2 = 1.0 + alpha - l @ l
            if not d2 > 0.0:
                raise np.linalg.LinAlgError(f"pick {k}: bordered factor lost positive definiteness")
            L[nk, :nk], L[nk, nk] = l, np.sqrt(d2)
            V[nk] = (ogp.rbf_gram(cand, z, ell)[:, 0] - V[:nk].T @ l) / L[nk, nk]
            ssq = ssq + V[nk] * V[nk]
        T = np.vstack([T, z])
        used[j] = True
        best = max(best, mu[j]) if greater_is_better else min(best, mu[j])
        vars_.append(variance())
    return dict(picks=np.asarray(picks, np.int64), ei=np.asarray(eis), ei_at_pick=np.asarray(ei_at),
                var=np.asarray(vars_), mu=mu, y_std=y_std)
