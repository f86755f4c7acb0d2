"""Host mirror of the pixel-coordinate GP regression of gp_regression.py (SURVEY.md §8f row 2) over libnib.so.

`GridGPRegression` stands where the reference's `GPRegressionModel` (ExactGP + GridInterpolationKernel(RBF, grid_size=30,
grid_bounds=[(0, n), (0, n)]) + outputscale, gp_regression.py:160-176) and its prediction loop (:244-261) stand:
`fit(train_x, train_y)` then `predict(test_x)` -> (mean, variance) for every query pixel.  Arithmetic in csrc/ski.cu + gp.cu:

    K = L L^T (grid Gram, G = grid_size^2)        A = W^T W, b = W^T (y - c)   (sparse accumulation over the n pixels)
    B = s2 I + L^T A L = C C^T                    mean_U = L B^-1 L^T b         var(x*) = s2 |C^-1 L^T w*|^2 (+ s2)

i.e. the exact posterior of the SKI model in its inducing-weight form: two G x G Cholesky factorizations instead of an
n x n solve (n up to 224^2 = 50 176), and well conditioned whatever the length scale (cond(B) <= 1 + |A| |K| / s2).
Above grid_size 100 (solver="auto"; grid_size 300 has G = 90 000 and 65 GB per G x G matrix) the same posterior is
solved without any G x G matrix: K = L L^T is replaced by the Kronecker square root S = M_R (x) M_C of `kron_factors`, A is
kept in band form and B is solved by preconditioned CG (csrc/ski_kron.cu, DESIGN.md §4).
`heatmap_from_masks` replaces the O(N * 224^2) Python dictionary loop of prepare_training_data (:63-104).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib

KRON_ABOVE = 100                 # solver="auto": the dense G x G path up to this grid size, the Kronecker solver above
KRON_BLOCK_BYTES = 4 << 30       # device memory of one block of variance right-hand sides (PCG vectors and workspace)
PCG_CHECK_EVERY = 4              # PCG iterations between host reads of the convergence state


def heatmap_from_masks(masks_u8, labels, on_value: int = 255, device="cuda") -> torch.Tensor:
    """H[p] = sum_i labels[i] * [masks[i][p] == on_value]  (gp_regression.py:82-94).  masks [N,H,W] uint8 (numpy or
    CUDA tensor), labels [N].  Returns fp32 [H,W] on the device."""
    lib = _lib.load()
    m = torch.as_tensor(masks_u8).to(device=device, dtype=torch.uint8).contiguous()
    N, H, W = (int(v) for v in m.shape)
    y = torch.as_tensor(np.asarray(labels, dtype=np.float32)).to(device)
    heat = torch.zeros(H, W, dtype=torch.float32, device=device)
    _lib.check(lib.nib_heatmap_pixels(m.data_ptr(), y.data_ptr(), N, H * W, int(on_value), heat.data_ptr(),
                                      _lib.stream_handle()), "nib_heatmap_pixels")
    return heat


def interp_1d(x, g0: float, h: float, gs: int) -> np.ndarray:
    """Cubic-convolution weights of coordinates x on one grid axis, W [len(x), gs] (host): the per-axis factor of the W
    of csrc/ski.cu (indices clamped to the grid, weights of a clamped index added)."""
    u = (np.asarray(x, dtype=np.float64) - g0) / h
    a = np.floor(u).astype(np.int64) - 1
    W = np.zeros((u.shape[0], gs))
    for k in range(4):
        s = np.abs(u - (a + k))
        w = np.where(s <= 1.0, (1.5 * s - 2.5) * s * s + 1.0, np.where(s < 2.0, ((-0.5 * s + 2.5) * s - 4.0) * s + 2.0, 0.0))
        np.add.at(W, (np.arange(u.shape[0]), np.clip(a + k, 0, gs - 1)), w)
    return W


def kron_factors(gs: int, g0: float, h: float, length_scale: float, outputscale: float, rows, cols):
    """Host part of the Kronecker solver: (M_R, M_C, theta_R, theta_C) for the grid g0 + k h (k < gs) and the distinct
    training coordinates `rows` / `cols` of the two axes.

    K1 = Q Lam Q^T is the 1-D Gram of the grid coordinates (negative eigenvalues from rounding clipped to 0), and per axis
    M = os^(1/4) Q Lam^(1/2) V with V Theta V^T = Lam^(1/2) Q^T A_axis Q Lam^(1/2), A_axis = W_axis^T W_axis.  Then
    (M_R (x) M_C)(M_R (x) M_C)^T = os K1 (x) K1 = K, and on the training lattice rows x cols, where A = A_R (x) A_C,
    (M_R (x) M_C)^T A (M_R (x) M_C) = os Theta_R (x) Theta_C is diagonal.  Nothing factors K, so no jitter is added."""
    c = g0 + h * np.arange(gs)
    K1 = np.exp(-0.5 * (c[:, None] / length_scale - c[None, :] / length_scale) ** 2)
    lam, Q = np.linalg.eigh(K1)
    P = Q * np.sqrt(np.clip(lam, 0.0, None))
    out = []
    for coords in (rows, cols):
        Wa = interp_1d(coords, g0, h, gs)
        theta, V = np.linalg.eigh(P.T @ (Wa.T @ Wa) @ P)
        out.append((outputscale ** 0.25 * (P @ V), np.clip(theta, 0.0, None)))
    (MR, thR), (MC, thC) = out
    return MR, MC, thR, thC


class GridGPRegression:
    def __init__(self, grid_size: int = 30, grid_bounds=((0.0, 224.0), (0.0, 224.0)), length_scale: float = 1.0,
                 outputscale: float = 1.0, noise: float = 1.0, const_mean: float = 0.0, jitter: float = 1e-8, device="cuda",
                 solver: str = "auto", cg_tol: float = 1e-10, max_iter: int = 1000):
        """solver: "dense" (two G x G Cholesky factorizations, G = grid_size^2), "kron" (matrix-free preconditioned CG on
        the Kronecker structure, csrc/ski_kron.cu; no jitter) or "auto" (dense up to grid_size 100, kron above).  cg_tol /
        max_iter: relative residual and iteration cap of each kron solve; `fit` / `predict` raise when the cap is hit."""
        (lo0, hi0), (lo1, hi1) = grid_bounds
        if (lo0, hi0) != (lo1, hi1):
            raise ValueError("both dimensions must share their bounds (gp_regression.py:168 uses [(0, n), (0, n)])")
        if solver not in ("auto", "dense", "kron"):
            raise ValueError(f"solver must be 'auto', 'dense' or 'kron', not {solver!r}")
        self.gs = int(grid_size)
        self.solver = ("dense" if self.gs <= KRON_ABOVE else "kron") if solver == "auto" else solver
        self.cg_tol, self.max_iter = float(cg_tol), int(max_iter)
        self.mean_iters, self.var_iters = None, []      # PCG iterations of the kron mean solve / of each variance block
        d = (hi0 - lo0) / (self.gs - 2)                 # one spacing of margin on either side (cubic stencil)
        self.g0 = float(lo0 - d)
        self.h = float((hi0 - lo0 + 2 * d) / (self.gs - 1))
        self.ell, self.os, self.noise, self.c, self.jitter = float(length_scale), float(outputscale), float(noise), float(const_mean), float(jitter)
        self.device = torch.device(device)
        self.lib = _lib.load()

    def _dev64(self, a):
        if torch.is_tensor(a):
            return a.detach().to(device=self.device, dtype=torch.float64).contiguous()
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(self.device)

    def _chol(self, M, what):
        G = M.shape[0]
        info = torch.zeros(1, dtype=torch.int32, device=self.device)
        _lib.check(self.lib.nib_gp_cholesky(M.data_ptr(), G, G, info.data_ptr(), _lib.stream_handle()), "nib_gp_cholesky")
        if int(info.item()) != 0:
            raise np.linalg.LinAlgError(f"{what} is not positive definite (pivot {int(info.item())})")

    def fit(self, X, y):
        lib, st, dev = self.lib, _lib.stream_handle(), self.device
        X, y = self._dev64(X), self._dev64(y).reshape(-1)
        n, gs, G = int(X.shape[0]), self.gs, self.gs * self.gs
        if X.shape[1] != 2 or y.shape[0] != n:
            raise ValueError("train_x must be [n, 2] pixel coordinates and train_y [n]")
        if self.solver == "kron":
            return self._fit_kron(X, y)
        c = self.g0 + self.h * torch.arange(gs, dtype=torch.float64, device=dev)
        U = torch.stack(torch.meshgrid(c, c, indexing="ij"), -1).reshape(G, 2).contiguous()
        L = torch.empty(G, G, dtype=torch.float64, device=dev)
        _lib.check(lib.nib_gp_gram_rbf(U.data_ptr(), G, U.data_ptr(), G, 2, self.ell, 0.0, 1, L.data_ptr(), G, st), "nib_gp_gram_rbf")
        L.mul_(self.os)
        L.diagonal().add_(self.jitter * self.os)
        self._chol(L, "the grid kernel K_UU")
        L.tril_()
        A = torch.zeros(G, G, dtype=torch.float64, device=dev)
        b = torch.zeros(G, dtype=torch.float64, device=dev)
        _lib.check(lib.nib_ski_accumulate(X.data_ptr(), y.data_ptr(), n, self.g0, self.h, gs, self.c, A.data_ptr(),
                                          b.data_ptr(), st), "nib_ski_accumulate")
        T = torch.zeros(G, G, dtype=torch.float64, device=dev)
        _lib.check(lib.nib_gp_dgemm_sub(A.data_ptr(), L.data_ptr(), T.data_ptr(), G, G, G, st), "nib_gp_dgemm_sub")   # T = -A L
        LT = L.t().contiguous()
        B = torch.zeros(G, G, dtype=torch.float64, device=dev)
        B.diagonal().fill_(self.noise)
        _lib.check(lib.nib_gp_dgemm_sub(LT.data_ptr(), T.data_ptr(), B.data_ptr(), G, G, G, st), "nib_gp_dgemm_sub")  # B = s2 I + L^T A L
        self._chol(B, "s2 I + L^T W^T W L")
        w = torch.empty(G, dtype=torch.float64, device=dev)
        _lib.check(lib.nib_gp_gemv_t(L.data_ptr(), G, G, G, b.data_ptr(), w.data_ptr(), st), "nib_gp_gemv_t")         # L^T b
        for trans in (0, 1):
            _lib.check(lib.nib_gp_trsm(B.data_ptr(), G, G, w.data_ptr(), 1, 1, trans, st), "nib_gp_trsm")
        self.mean_u = torch.empty(G, dtype=torch.float64, device=dev)
        _lib.check(lib.nib_gp_gemv_t(LT.data_ptr(), G, G, G, w.data_ptr(), self.mean_u.data_ptr(), st), "nib_gp_gemv_t")  # L w
        self.Gm = LT                                                                                                       # C^-1 L^T
        _lib.check(lib.nib_gp_trsm(B.data_ptr(), G, G, self.Gm.data_ptr(), G, G, 0, st), "nib_gp_trsm")
        self.n = n
        return self

    def predict(self, Xq, return_var: bool = True, likelihood: bool = True):
        """Posterior mean (and variance; with the Gaussian likelihood's noise when `likelihood`, as `likelihood(model(x))`
        at gp_regression.py:254) at pixel coordinates Xq [m, 2].  fp64 CUDA tensors."""
        Xq = self._dev64(Xq)
        m = int(Xq.shape[0])
        mean = torch.empty(m, dtype=torch.float64, device=self.device)
        var = torch.empty(m, dtype=torch.float64, device=self.device) if return_var else None
        if self.solver == "kron":
            return self._predict_kron(Xq, mean, var, likelihood)
        _lib.check(self.lib.nib_ski_predict(Xq.data_ptr(), m, self.g0, self.h, self.gs, self.c, self.mean_u.data_ptr(),
                                            self.Gm.data_ptr(), self.noise, int(likelihood), mean.data_ptr(),
                                            var.data_ptr() if var is not None else None, _lib.stream_handle()), "nib_ski_predict")
        return (mean, var) if return_var else mean

    # ---- Kronecker-structured solver (csrc/ski_kron.cu) ------------------------------------------------------------------
    # S = M_R (x) M_C from kron_factors; CG on B = s2 I + S^T A S preconditioned by s2 + coef Theta_R (x) Theta_C, exact on
    # a lattice of training pixels; for other point sets coef = os n / (|R| |C|) matches the density of points.  The gs x gs
    # eigenproblems run on the host in numpy, everything of order G on the device.

    def _fit_kron(self, X, y):
        lib, st, dev = self.lib, _lib.stream_handle(), self.device
        n, gs, G = int(X.shape[0]), self.gs, self.gs * self.gs
        rows, cols = (torch.unique(X[:, d]).cpu().numpy() for d in (0, 1))
        MR, MC, thR, thC = kron_factors(gs, self.g0, self.h, self.ell, self.os, rows, cols)
        to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        self.MR, self.MC, self.thR, self.thC = (to_dev(a) for a in (MR, MC, thR, thC))
        self.coef = self.os * n / (len(rows) * len(cols))
        self.A = torch.empty(G * 49, dtype=torch.float64, device=dev)
        b = torch.empty(G, dtype=torch.float64, device=dev)
        work = torch.empty((4 * (2 * n + 3 * G + 2) + 72 * n + 7) // 8, dtype=torch.float64, device=dev)
        _lib.check(lib.nib_ski_band_accumulate(X.data_ptr(), y.data_ptr(), n, self.g0, self.h, gs, self.c, self.A.data_ptr(),
                                               b.data_ptr(), work.data_ptr(), st), "nib_ski_band_accumulate")
        rhs = torch.empty(G, dtype=torch.float64, device=dev)
        _lib.check(lib.nib_ski_kron_apply(b.data_ptr(), rhs.data_ptr(), 1, gs, self.MR.data_ptr(), self.MC.data_ptr(), 1,
                                          work.data_ptr(), st), "nib_ski_kron_apply")               # S^T b
        z = torch.empty(G, dtype=torch.float64, device=dev)
        self.mean_iters = self._pcg(rhs, z, 1, "the mean solve")
        self.mean_u = torch.empty(G, dtype=torch.float64, device=dev)
        _lib.check(lib.nib_ski_kron_apply(z.data_ptr(), self.mean_u.data_ptr(), 1, gs, self.MR.data_ptr(),
                                          self.MC.data_ptr(), 0, work.data_ptr(), st), "nib_ski_kron_apply")   # S z
        self.Gm = None
        self.var_iters = []
        self.n = n
        return self

    def _pcg(self, rhs, x, r, what):
        G = self.gs * self.gs
        work = torch.empty(5 * r * G + 5 * r + 4, dtype=torch.float64, device=self.device)
        iters, relres = C.c_int(0), C.c_double(0.0)
        _lib.check(self.lib.nib_ski_kron_pcg(self.A.data_ptr(), self.gs, self.MR.data_ptr(), self.MC.data_ptr(),
                                             self.thR.data_ptr(), self.thC.data_ptr(), self.coef, self.noise, rhs.data_ptr(),
                                             x.data_ptr(), r, self.cg_tol, self.max_iter, PCG_CHECK_EVERY, work.data_ptr(),
                                             C.byref(iters), C.byref(relres), _lib.stream_handle()), "nib_ski_kron_pcg")
        if not relres.value <= self.cg_tol:
            raise np.linalg.LinAlgError(f"preconditioned CG of {what} did not converge in max_iter={self.max_iter} "
                                        f"iterations: relative residual {relres.value:.3e} > cg_tol={self.cg_tol:.1e}")
        return int(iters.value)

    def _predict_kron(self, Xq, mean, var, likelihood):
        lib, st, gs, G = self.lib, _lib.stream_handle(), self.gs, self.gs * self.gs
        m = int(Xq.shape[0])
        _lib.check(lib.nib_ski_predict(Xq.data_ptr(), m, self.g0, self.h, gs, self.c, self.mean_u.data_ptr(), None,
                                       self.noise, int(likelihood), mean.data_ptr(), None, st), "nib_ski_predict")
        if var is None:
            return mean
        rb = int(max(1, min(m, 65535, KRON_BLOCK_BYTES // (8 * 7 * G))))   # rhs, x and the 5 PCG work vectors
        rhs = torch.empty(rb * G, dtype=torch.float64, device=self.device)
        x = torch.empty(rb * G, dtype=torch.float64, device=self.device)
        self.var_iters = []
        for q0 in range(0, m, rb):
            r = min(rb, m - q0)
            Xb = Xq[q0:q0 + r]
            _lib.check(lib.nib_ski_kron_var_rhs(Xb.data_ptr(), r, self.g0, self.h, gs, self.MR.data_ptr(), self.MC.data_ptr(),
                                                rhs.data_ptr(), st), "nib_ski_kron_var_rhs")
            self.var_iters.append(self._pcg(rhs, x, r, f"the variance of queries {q0}..{q0 + r - 1}"))
            _lib.check(lib.nib_ski_kron_var_reduce(rhs.data_ptr(), x.data_ptr(), r, gs, self.noise, int(likelihood),
                                                   var.data_ptr() + 8 * q0, st), "nib_ski_kron_var_reduce")
        return mean, var
