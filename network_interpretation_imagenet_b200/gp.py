"""Stage 3 host mirror: Gaussian-process surrogate + Expected Improvement on the device.

Duck-types the estimator the reference builds at BayesianOptimization.py:154-159
(`GaussianProcessRegressor(kernel=RBF(), alpha=1e-5, n_restarts_optimizer=10, normalize_y=True)`):
`fit(X, y)` (:166) and `predict(X, return_std=True)` (:39) with numpy fp64 in/out, plus
`log_marginal_likelihood(theta, eval_gradient=True)` following sklearn/gaussian_process/_gpr.py:588-655.
The hyper-parameter search keeps scikit-learn's host control flow (scipy L-BFGS-B on theta = log l from
the initial l and `n_restarts_optimizer` log-uniform restarts, _gpr.py:298-339) while every O(n^2)/O(n^3)
step — Gram, Cholesky, solves, K^-1, posterior, EI — runs in libnib.so kernels.

X may be (a) selection bit-vectors [n, words] uint64 (the scaled-up spec: masks as inputs, SURVEY.md §8a8),
(b) a 0/1 matrix [n, S], converted to (a), or (c) any real matrix [n, d] (the reference's 1-D firstIndex GP).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
from scipy.optimize import minimize

from . import _lib


def _is_bits(X) -> bool:
    return isinstance(X, np.ndarray) and X.dtype == np.uint64


def pack_bits(X01: np.ndarray) -> np.ndarray:
    X01 = np.asarray(X01)
    n, S = X01.shape
    words = (S + 63) // 64
    out = np.zeros((n, words), dtype=np.uint64)
    for s in range(S):
        out[:, s >> 6] |= (X01[:, s] != 0).astype(np.uint64) << np.uint64(s & 63)
    return out


class GaussianProcessRegressor:
    def __init__(self, alpha: float = 1e-5, normalize_y: bool = True, length_scale: float = 1.0,
                 length_scale_bounds=(1e-5, 1e5), n_restarts_optimizer: int = 0, optimizer: str | None = "fmin_l_bfgs_b",
                 random_state=None, kernel=None, device="cuda", query_chunk: int = 8192):
        # `kernel` is accepted for signature compatibility with gp_params passthrough (BayesianOptimization.py:150-151);
        # only RBF is implemented, its length_scale / bounds are read if present.
        if kernel is not None:
            length_scale = float(getattr(kernel, "length_scale", length_scale))
            length_scale_bounds = tuple(getattr(kernel, "length_scale_bounds", length_scale_bounds))
        self.alpha = float(alpha)
        self.normalize_y = normalize_y
        self.length_scale0 = float(length_scale)
        self.length_scale_bounds = length_scale_bounds
        self.n_restarts_optimizer = int(n_restarts_optimizer)
        self.optimizer = optimizer
        self.random_state = random_state
        self.device = torch.device(device)
        self.query_chunk = int(query_chunk)
        self.lib = _lib.load()
        self.length_scale_ = self.length_scale0
        self.n = 0
        self.stats = {"lml_evals": 0}

    # ---- helpers -------------------------------------------------------------------------------
    def _upload_X(self, X):
        X = np.asarray(X)
        if _is_bits(X):
            bits = np.ascontiguousarray(X)
            return "bits", torch.from_numpy(bits.view(np.int64)).to(self.device), bits.shape[1]
        if X.ndim == 2 and X.shape[1] > 1 and np.isin(X, (0, 1)).all():
            bits = pack_bits(X)
            return "bits", torch.from_numpy(bits.view(np.int64)).to(self.device), bits.shape[1]
        Xr = np.ascontiguousarray(np.atleast_2d(X), dtype=np.float64)
        return "real", torch.from_numpy(Xr).to(self.device), Xr.shape[1]

    def _gram(self, kind, A, na, B, nb, dim, ell, jitter, same, out):
        st = _lib.stream_handle()
        if kind == "bits":
            a_ptr, b_ptr = A.data_ptr(), (A.data_ptr() if same else B.data_ptr())
            _lib.check(self.lib.nib_gp_gram_binary(a_ptr, na, b_ptr, nb, dim, ell, jitter, out.data_ptr(),
                                                   out.stride(0), st), "nib_gp_gram_binary")
        else:
            _lib.check(self.lib.nib_gp_gram_rbf(A.data_ptr(), na, B.data_ptr(), nb, dim, ell, jitter, int(same),
                                                out.data_ptr(), out.stride(0), st), "nib_gp_gram_rbf")

    def _factor(self, ell: float):
        """K(+alpha I) -> L (in place), alpha_vec = K^-1 y.  Raises LinAlgError like _gpr.py:352-361."""
        n = self.n
        st = _lib.stream_handle()
        self._gram(self.kind, self.X_d, n, self.X_d, n, self.dim, ell, self.alpha, True, self.L)
        _lib.check(self.lib.nib_gp_cholesky(self.L.data_ptr(), n, self.L.stride(0), self.info.data_ptr(), st),
                   "nib_gp_cholesky")
        self.alpha_vec.copy_(self.y_d)
        for trans in (0, 1):
            _lib.check(self.lib.nib_gp_trsm(self.L.data_ptr(), n, self.L.stride(0), self.alpha_vec.data_ptr(), 1, 1,
                                            trans, st), "nib_gp_trsm")
        info = int(self.info.item())
        if info != 0:
            raise np.linalg.LinAlgError(
                f"The kernel is not returning a positive definite matrix (pivot {info}). "
                "Try gradually increasing the 'alpha' parameter of your GaussianProcessRegressor estimator.")

    # ---- sklearn surface -------------------------------------------------------------------------
    def fit(self, X, y):
        y = np.asarray(y, dtype=np.float64).reshape(-1)
        self.kind, self.X_d, self.dim = self._upload_X(X)
        self.n = n = int(self.X_d.shape[0])
        if y.shape[0] != n:
            raise ValueError("X and y have inconsistent lengths")
        if self.normalize_y:   # _gpr.py:276-280
            self._y_train_mean = float(np.mean(y))
            std = float(np.std(y))
            self._y_train_std = std if std != 0.0 else 1.0
        else:
            self._y_train_mean, self._y_train_std = 0.0, 1.0
        yn = (y - self._y_train_mean) / self._y_train_std
        dev = self.device
        self.y_d = torch.from_numpy(yn).to(dev)
        self.L = torch.empty(n, n, dtype=torch.float64, device=dev)
        self.alpha_vec = torch.empty(n, dtype=torch.float64, device=dev)
        self.info = torch.zeros(1, dtype=torch.int32, device=dev)
        self._K0 = self._Kinv = None
        self._fitted = False

        if self.optimizer is not None:
            lo, hi = np.log(self.length_scale_bounds[0]), np.log(self.length_scale_bounds[1])

            def obj(theta):
                lml, g = self.log_marginal_likelihood(theta, eval_gradient=True, _keep=False)
                return -lml, -np.atleast_1d(g)

            def run(theta0):
                r = minimize(obj, theta0, method="L-BFGS-B", jac=True, bounds=[(lo, hi)])
                return r.x, r.fun

            optima = [run(np.array([np.log(self.length_scale0)]))]
            if self.n_restarts_optimizer > 0:
                rng = np.random.RandomState(self.random_state) if not isinstance(self.random_state, np.random.RandomState) else self.random_state
                for _ in range(self.n_restarts_optimizer):
                    theta0 = rng.uniform(lo, hi, size=1)   # _gpr.py:324-327
                    optima.append(run(theta0))
            best = min(optima, key=lambda t: t[1])
            self.length_scale_ = float(np.exp(best[0][0]))
            self.log_marginal_likelihood_value_ = -float(best[1])
        else:
            self.length_scale_ = self.length_scale0
        self._factor(self.length_scale_)
        self._K0 = self._Kinv = None   # free optimiser scratch
        self._fitted = True
        return self

    def log_marginal_likelihood(self, theta=None, eval_gradient: bool = False, _keep: bool = True):
        """_gpr.py:538-655 for theta = log(length_scale).  Side-effect free like scikit-learn's: the factor lives in
        the model's own L / alpha buffers (no second n x n allocation), so a query at another theta on a fitted model
        (`_keep`, the default; `fit` passes False while it searches) re-factors at the fitted length scale afterwards."""
        ell = self.length_scale_ if theta is None else float(np.exp(np.atleast_1d(theta)[0]))
        restore = _keep and getattr(self, "_fitted", False) and ell != self.length_scale_
        try:
            return self._lml(ell, eval_gradient)
        finally:
            if restore:
                self._factor(self.length_scale_)

    def _lml(self, ell: float, eval_gradient: bool):
        n = self.n
        st = _lib.stream_handle()
        self.stats["lml_evals"] += 1
        try:
            self._factor(ell)
        except np.linalg.LinAlgError:
            return (-np.inf, np.zeros(1)) if eval_gradient else -np.inf
        lml = C.c_double()
        _lib.check(self.lib.nib_gp_lml(self.L.data_ptr(), n, self.L.stride(0), self.y_d.data_ptr(),
                                       self.alpha_vec.data_ptr(), C.byref(lml), st), "nib_gp_lml")
        if not eval_gradient:
            return lml.value
        dev = self.device
        if self._K0 is None:
            self._K0 = torch.empty(n, n, dtype=torch.float64, device=dev)
            self._Kinv = torch.empty(n, n, dtype=torch.float64, device=dev)
        self._gram(self.kind, self.X_d, n, self.X_d, n, self.dim, ell, 0.0, True, self._K0)
        self._Kinv.zero_()
        self._Kinv.diagonal().fill_(1.0)
        for trans in (0, 1):   # K^-1 = L^-T L^-1 I  (cho_solve(L, eye), _gpr.py:631)
            _lib.check(self.lib.nib_gp_trsm(self.L.data_ptr(), n, self.L.stride(0), self._Kinv.data_ptr(), n, n, trans, st),
                       "nib_gp_trsm")
        g = C.c_double()
        if self.kind == "bits":
            _lib.check(self.lib.nib_gp_lml_grad(self._K0.data_ptr(), self._Kinv.data_ptr(), self.alpha_vec.data_ptr(),
                                                self.X_d.data_ptr(), self.dim, n, n, ell, C.byref(g), st), "nib_gp_lml_grad")
        else:
            _lib.check(self.lib.nib_gp_lml_grad_rbf(self._K0.data_ptr(), self._Kinv.data_ptr(),
                                                    self.alpha_vec.data_ptr(), self.X_d.data_ptr(), self.dim, n, n, ell,
                                                    C.byref(g), st), "nib_gp_lml_grad_rbf")
        return lml.value, np.array([g.value])

    def predict_device(self, Xq):
        """(mu, var, std) as fp64 CUDA tensors for all queries (chunked so scratch stays bounded)."""
        kind, Q, dim = self._upload_X(Xq)
        if kind != self.kind or dim != self.dim:
            raise ValueError("query inputs do not match the training inputs")
        m = int(Q.shape[0])
        dev = self.device
        mu = torch.empty(m, dtype=torch.float64, device=dev)
        var = torch.empty(m, dtype=torch.float64, device=dev)
        sd = torch.empty(m, dtype=torch.float64, device=dev)
        n = self.n
        st = _lib.stream_handle()
        ch = min(m, self.query_chunk)
        Ks = torch.empty(ch, n, dtype=torch.float64, device=dev)
        work = torch.empty(n * ch, dtype=torch.float64, device=dev)
        for i in range(0, m, ch):
            c = min(ch, m - i)
            self._gram(kind, Q[i:i + c], c, self.X_d, n, dim, self.length_scale_, 0.0, False, Ks)
            _lib.check(self.lib.nib_gp_posterior(self.L.data_ptr(), n, self.L.stride(0), self.alpha_vec.data_ptr(),
                                                 Ks.data_ptr(), c, Ks.stride(0), self._y_train_mean, self._y_train_std,
                                                 1.0, work.data_ptr(), mu[i:i + c].data_ptr(), var[i:i + c].data_ptr(),
                                                 sd[i:i + c].data_ptr(), st), "nib_gp_posterior")
        return mu, var, sd

    def predict(self, X, return_std: bool = False):
        mu, _, sd = self.predict_device(X)
        if return_std:
            return mu.cpu().numpy(), sd.cpu().numpy()
        return mu.cpu().numpy()


class ActiveMaskGP:
    """The GP of an acquisition loop over a FIXED candidate pool, maintained by rank-one updates.

    The reference's loop (BayesianOptimization.py:140-185, bayesian_active_learning_imagenet.py) refits the GP and
    re-predicts every candidate each round: O(n^3 + m n^2).  With a fixed length scale the Gram matrix of the first n
    points never changes, so adding the chosen candidate only borders the Cholesky factor by one row, and the posterior
    workspace V = L^-1 K*^T gains one row:

        l = L^-1 k(X, z)          d = sqrt(1 + alpha - l.l)          L <- [[L, 0], [l^T, d]]
        V <- [V; (k*(z) - l^T V) / d]        ssq += (new row)^2        u <- [u; (y - l.u)/d]    w <- [w; (1 - l.w)/d]

    and   mu = ybar + V^T (u - ybar w),   var = ystd^2 max(0, 1 - ssq)   (u = L^-1 y, w = L^-1 1: y-normalisation,
    _gpr.py:276-280, changes every round but stays an O(n) correction).  O(n^2 + m n) per round; same posterior as a
    refit up to rounding (tests/test_gpu_gp.py compares the two and the scikit-learn oracle).

    `select_batch(q)` picks q candidates at once by greedy Kriging believer (nib_gp_kb_select): each pick is fantasised
    at its posterior mean, which leaves every other mean unchanged and only shrinks variances, so the q picks cost q new
    rows of L and V and no host round trip.  `set_batch_values(scores)` then puts the measured values in place of the
    fantasies."""

    def __init__(self, candidate_bits, alpha: float = 1e-5, length_scale: float = 1.0, normalize_y: bool = True,
                 capacity: int = 64, device="cuda"):
        self.lib = _lib.load()
        self.device = torch.device(device)
        self.alpha, self.ell, self.normalize_y, self.capacity = float(alpha), float(length_scale), normalize_y, int(capacity)
        cand = np.ascontiguousarray(candidate_bits, dtype=np.uint64)
        self.m, self.words = int(cand.shape[0]), int(cand.shape[1])
        self.cand_host = cand
        self.cand_d = torch.from_numpy(cand.view(np.int64)).to(self.device)
        self.alive = torch.ones(self.m, dtype=torch.bool, device=self.device)
        self._pending = None     # the last select_batch() while its values are outstanding
        self.stats = {}

    def _gram(self, A, na, B, nb, jitter, out, ld):
        _lib.check(self.lib.nib_gp_gram_binary(A.data_ptr(), na, B.data_ptr(), nb, self.words, self.ell, jitter,
                                               out.data_ptr(), ld, _lib.stream_handle()), "nib_gp_gram_binary")

    def fit(self, Z_bits, y):
        Z = np.ascontiguousarray(Z_bits, dtype=np.uint64)
        n, cap, m, dev = int(Z.shape[0]), int(Z.shape[0]) + self.capacity, self.m, self.device
        st = _lib.stream_handle()
        self.n, self.cap = n, cap
        self.X_d = torch.zeros(cap, self.words, dtype=torch.int64, device=dev)
        self.X_d[:n] = torch.from_numpy(Z.view(np.int64)).to(dev)
        self.y_host = list(np.asarray(y, dtype=np.float64).reshape(-1))
        self.L = torch.zeros(cap, cap, dtype=torch.float64, device=dev)
        self.V = torch.empty(cap, m, dtype=torch.float64, device=dev)
        self.info = torch.zeros(1, dtype=torch.int32, device=dev)
        self._gram(self.X_d, n, self.X_d, n, self.alpha, self.L, cap)
        _lib.check(self.lib.nib_gp_cholesky(self.L.data_ptr(), n, cap, self.info.data_ptr(), st), "nib_gp_cholesky")
        if int(self.info.item()) != 0:
            raise np.linalg.LinAlgError("The kernel is not returning a positive definite matrix")
        self._gram(self.X_d, n, self.cand_d, m, 0.0, self.V, m)                       # K*^T  [n x m]
        _lib.check(self.lib.nib_gp_trsm(self.L.data_ptr(), n, cap, self.V.data_ptr(), m, m, 0, st), "nib_gp_trsm")
        self.ssq = torch.empty(m, dtype=torch.float64, device=dev)
        _lib.check(self.lib.nib_gp_colsumsq(self.V.data_ptr(), n, m, m, self.ssq.data_ptr(), st), "nib_gp_colsumsq")
        self.uw = torch.zeros(2, cap, dtype=torch.float64, device=dev)               # u = L^-1 y, w = L^-1 1
        self.uw[0, :n] = torch.as_tensor(np.asarray(self.y_host), device=dev)
        self.uw[1, :n] = 1.0
        for r in range(2):
            _lib.check(self.lib.nib_gp_trsm(self.L.data_ptr(), n, cap, self.uw[r].data_ptr(), 1, 1, 0, st), "nib_gp_trsm")
        self._tmp = torch.empty(3, max(m, cap), dtype=torch.float64, device=dev)
        self._pending = None
        return self

    def _ystats(self):
        y = np.asarray(self.y_host)
        if not self.normalize_y:
            return 0.0, 1.0
        sd = float(np.std(y))
        return float(np.mean(y)), (sd if sd != 0.0 else 1.0)

    def posterior(self):
        """(mu, var, std) over the whole candidate pool, fp64 on the device; candidates already used carry std = NaN so
        that Expected Improvement skips them (the reference's duplicate guard, BayesianOptimization.py:178-180).
        While a batch awaits set_batch_values() this is the posterior given its fantasies: the mean the batch was
        selected with and the variances after its rows, both at the y-normalisation of that moment."""
        if self._pending is not None:
            ystd = self._pending["ystats"][1]
            var = (1.0 - self.ssq).clamp_(min=0.0) * (ystd * ystd)
            sd = var.sqrt()
            sd[~self.alive] = float("nan")
            return self._pending["mu"].clone(), var, sd
        n, m, st = self.n, self.m, _lib.stream_handle()
        ybar, ystd = self._ystats()
        z = self._tmp[0, :n]
        torch.sub(self.uw[0, :n], self.uw[1, :n], alpha=ybar, out=z)                  # ystd * L^-1 y_normalised
        mu = torch.empty(m, dtype=torch.float64, device=self.device)
        _lib.check(self.lib.nib_gp_gemv_t(self.V.data_ptr(), n, m, m, z.data_ptr(), mu.data_ptr(), st), "nib_gp_gemv_t")
        mu += ybar
        var = (1.0 - self.ssq).clamp_(min=0.0) * (ystd * ystd)
        sd = var.sqrt()
        sd[~self.alive] = float("nan")
        return mu, var, sd

    def append(self, index: int, y_new: float):
        """Candidate `index` has been evaluated: it joins the training set (and leaves the pool)."""
        if self._pending is not None:
            raise RuntimeError("ActiveMaskGP: the last select_batch() awaits set_batch_values()")
        if self.n >= self.cap:
            raise RuntimeError("ActiveMaskGP capacity exhausted: construct with a larger `capacity`")
        n, m, cap, st = self.n, self.m, self.cap, _lib.stream_handle()
        znew = self.cand_d[index:index + 1]
        l = self.L[n, :n]                                                            # row n of L, filled in place
        self._gram(znew, 1, self.X_d, n, 0.0, l, cap)                                # k(z, X)  [1 x n]
        _lib.check(self.lib.nib_gp_trsm(self.L.data_ptr(), n, cap, l.data_ptr(), 1, 1, 0, st), "nib_gp_trsm")
        d2 = 1.0 + self.alpha - float(torch.dot(l, l).item())
        if not d2 > 0.0:
            raise np.linalg.LinAlgError("rank-one update lost positive definiteness (duplicate mask with alpha too small?)")
        d = float(np.sqrt(d2))
        self.L[n, n] = d
        ks, dot = self._tmp[1, :m], self._tmp[2, :m]
        self._gram(self.cand_d, m, znew, 1, 0.0, ks, 1)                              # k*(z)  [m x 1]
        _lib.check(self.lib.nib_gp_gemv_t(self.V.data_ptr(), n, m, m, l.data_ptr(), dot.data_ptr(), st), "nib_gp_gemv_t")
        _lib.check(self.lib.nib_gp_append_row(ks.data_ptr(), dot.data_ptr(), d, self.V[n].data_ptr(),
                                              self.ssq.data_ptr(), m, st), "nib_gp_append_row")
        lu = torch.mv(self.uw[:, :n], l)                                              # (l.u, l.w)
        self.uw[0, n] = (float(y_new) - lu[0]) / d
        self.uw[1, n] = (1.0 - lu[1]) / d
        self.X_d[n] = self.cand_d[index]
        self.y_host.append(float(y_new))
        self.alive[index] = False
        self.n = n + 1

    def select_batch(self, q: int, greater_is_better: bool = True):
        """Up to q candidates to evaluate next, by greedy Kriging believer on the device: pick the EI arg-max, condition on
        a fantasy observation equal to its posterior mean (the incumbent becomes max(incumbent, that mean)), repeat.
        The mean is computed once, at the current y-normalisation.  Returns (picks int64, EI at each pick); fewer than q
        when no candidate with a defined EI is left.  The picks join the training set with their fantasies until
        set_batch_values() supplies the measured values."""
        q = int(q)
        if q < 1:
            raise ValueError("select_batch: q must be >= 1")
        if self._pending is not None:
            raise RuntimeError("ActiveMaskGP: the last select_batch() awaits set_batch_values()")
        if self.n + q > self.cap:
            raise RuntimeError("ActiveMaskGP capacity exhausted: construct with a larger `capacity`")
        mu, _, _ = self.posterior()
        ystats = self._ystats()
        y = np.asarray(self.y_host)
        best = float(y.max() if greater_is_better else y.min())
        ssq0, alive0 = self.ssq.clone(), self.alive.clone()
        dev, n = self.device, self.n
        picks = torch.empty(q, dtype=torch.int64, device=dev)
        ei = torch.empty(q, dtype=torch.float64, device=dev)
        status = torch.empty(1, dtype=torch.int32, device=dev)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        _lib.check(self.lib.nib_gp_kb_select(self.L.data_ptr(), self.cap, self.V.data_ptr(), self.m, self.ssq.data_ptr(),
                                             self.alive.data_ptr(), self.cand_d.data_ptr(), self.m, self.words,
                                             self.X_d.data_ptr(), n, q, mu.data_ptr(), ystats[1], best,
                                             int(greater_is_better), self.ell, self.alpha, picks.data_ptr(),
                                             ei.data_ptr(), status.data_ptr(), _lib.stream_handle()), "nib_gp_kb_select")
        ev[1].record()
        ev[1].synchronize()
        self.stats["select_ms"] = ev[0].elapsed_time(ev[1])       # the q picks' kernels, device time
        picks, ei, status = picks.cpu().numpy(), ei.cpu().numpy(), int(status.item())
        if status != 0:
            self.ssq.copy_(ssq0)
            self.alive.copy_(alive0)
            raise np.linalg.LinAlgError(f"Kriging-believer pick {status - 1} lost positive definiteness "
                                        "(duplicate mask with alpha too small?)")
        p = int(np.count_nonzero(picks >= 0))
        if p:
            self.n = n + p
            self._pending = {"n0": n, "mu": mu, "ystats": ystats}
        return picks[:p].astype(np.int64), ei[:p].copy()

    def set_batch_values(self, scores):
        """The measured values of the last select_batch(), in pick order: they replace the fantasies in u = L^-1 y and
        w = L^-1 1 (rows n0 .. n0+p-1 of L solve L_bb u_b = y_b - L_ba u_a) and join y.  Afterwards posterior() equals a
        fit from scratch on the grown training set."""
        if self._pending is None:
            raise RuntimeError("ActiveMaskGP.set_batch_values: no batch is pending")
        n0, n = self._pending["n0"], self.n
        p = n - n0
        s = np.asarray(scores, dtype=np.float64).reshape(-1)
        if s.shape[0] != p:
            raise ValueError(f"set_batch_values: {p} values expected, got {s.shape[0]}")
        dev, cap = self.device, self.cap
        rhs = torch.empty(p, 2, dtype=torch.float64, device=dev)
        rhs[:, 0] = torch.from_numpy(s).to(dev)
        rhs[:, 1] = 1.0
        rhs -= self.L[n0:n, :n0] @ self.uw[:, :n0].t()                                 # (y_b, 1) - L_ba (u_a, w_a)
        Lbb = self.L[n0:, n0:]
        _lib.check(self.lib.nib_gp_trsm(Lbb.data_ptr(), p, cap, rhs.data_ptr(), 2, 2, 0, _lib.stream_handle()),
                   "nib_gp_trsm")
        self.uw[:, n0:n] = rhs.t()
        self.y_host.extend(float(v) for v in s)
        self._pending = None


def expected_improvement_device(mu: torch.Tensor, sigma: torch.Tensor, best: float, greater_is_better: bool = False):
    """+EI and its argmax on the device (BayesianOptimization.py:37-54 returns -EI)."""
    lib = _lib.load()
    m = int(mu.shape[0])
    ei = torch.empty(m, dtype=torch.float64, device=mu.device)
    arg = torch.empty(1, dtype=torch.int64, device=mu.device)
    _lib.check(lib.nib_gp_ei(mu.data_ptr(), sigma.data_ptr(), m, float(best), int(greater_is_better), ei.data_ptr(),
                             arg.data_ptr(), _lib.stream_handle()), "nib_gp_ei")
    return ei, arg


def expected_improvement(x, gaussian_process, evaluated_loss, greater_is_better=False, n_params=1):
    """Drop-in for BayesianOptimization.py:16-54 (same signature, returns -EI as numpy)."""
    x_to_predict = np.asarray(x).reshape(-1, n_params)
    mu, _, sd = gaussian_process.predict_device(x_to_predict)
    best = np.max(evaluated_loss) if greater_is_better else np.min(evaluated_loss)
    ei, _ = expected_improvement_device(mu, sd, float(best), greater_is_better)
    return -1 * ei.cpu().numpy()
