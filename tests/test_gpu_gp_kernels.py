"""GPU: the fp64 GP kernels (csrc/gp.cu) called one by one through the C ABI, against plain fp64 library references
(scipy.linalg / LAPACK dpotrf / numpy / oracle.gp).

Inputs are well conditioned (A A^T / n + I, eigenvalues in [1, 5]), so a correct kernel lands within a few hundred ulps
of the reference; every tolerance below is stated where it is used and sits many orders of magnitude under what an
indexing or blocking error produces.  Buffers carry poison around the operands: NaN in the strict upper triangle the
kernels are documented not to read, and a sentinel NaN bit pattern in padding columns and spare rows that must come back
bit for bit.

`test_core_*` is a compact subset of the Cholesky / failing-pivot / TRSM / GEMM checks.  `test_solver_variant` reruns it
in a child process under each environment switch that selects another shipped solver path (DESIGN §4): the switches
are read once per process, so they can only be exercised that way.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from scipy.linalg import cho_solve, cholesky, solve_triangular
from scipy.linalg.lapack import dpotrf
from scipy.spatial.distance import cdist

from oracle import gp as ogp

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = np.finfo(np.float64).eps
SENT = np.uint64(0x7FF4DEADBEEF0001)   # a signalling-NaN bit pattern no kernel produces
# diagonal-block (64), GEMM-tile (64 / 128) and Cholesky super-block (512) edges
CHOL_NS = [1, 2, 63, 64, 65, 127, 128, 129, 255, 256, 257, 511, 512, 513, 575, 577, 1023, 1025, 1537]


class _Gp:
    def __init__(self, nib):
        self.nl = nib._lib
        self.lib = self.nl.load()

    def __call__(self, name, *args, stream=None):
        self.nl.check(getattr(self.lib, name)(*args, self.nl.stream_handle(stream)), name)


@pytest.fixture(scope="module")
def gp(nib):
    return _Gp(nib)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _host(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def _spd(n, seed):
    A = np.random.default_rng(seed).standard_normal((n, n))
    return A @ A.T / n + np.eye(n)


def _rand_bits(rng, n, S):
    words = (S + 63) // 64
    Z = rng.integers(0, np.iinfo(np.uint64).max, size=(n, words), dtype=np.uint64, endpoint=True)
    tail = S - 64 * (words - 1)
    if tail < 64:
        Z[:, -1] &= np.uint64((1 << tail) - 1)
    return Z


# ---- 1. Cholesky at block edges --------------------------------------------------------------------------------------
def _cholesky(gp, buf, n, ldk):
    d = _dev(buf)
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    gp("nib_gp_cholesky", d.data_ptr(), n, ldk, info.data_ptr())
    return _host(d), int(_host(info)[0])


def _check_cholesky(gp, n, ldk):
    K = _spd(n, n)
    # poisoned: strict upper triangle NaN, padding columns [n, ldk) and one spare row n = sentinel
    buf = np.empty((n + 1, ldk))
    _bits(buf)[:] = SENT
    body = K.copy()
    body[np.triu_indices(n, 1)] = np.nan
    buf[:n, :n] = body
    out, info = _cholesky(gp, buf, n, ldk)
    assert info == 0
    L = np.tril(out[:n, :n])
    Lref = cholesky(K, lower=True)
    kmax = np.abs(K).max()
    err = np.abs(L - Lref).max()
    assert err <= 1e-11 * kmax, f"max|L - L_scipy| = {err:.3e}"
    back = np.abs(L @ L.T - K).max()
    assert back <= 64 * n * EPS * kmax, f"max|L L^T - K| = {back:.3e}"
    iu = np.triu_indices(n, 1)
    assert np.array_equal(_bits(out[:n, :n])[iu], _bits(buf[:n, :n])[iu]), "strict upper triangle written"
    assert np.array_equal(_bits(out[:, n:]), _bits(buf[:, n:])), "padding columns written"
    assert np.array_equal(_bits(out[n]), _bits(buf[n])), "spare row written"
    # the same matrix stored in full, no poison: the factor must not depend on anything above the diagonal
    clean = np.zeros((n, ldk))
    clean[:, :n] = K
    out2, info2 = _cholesky(gp, clean, n, ldk)
    il = np.tril_indices(n)
    assert info2 == 0 and np.array_equal(_bits(out2[:n, :n])[il], _bits(out[:n, :n])[il])


@pytest.mark.parametrize("ldpad", [0, 3])   # ldk = n + 3: odd leading dimension, the GEMM's scalar epilogue
@pytest.mark.parametrize("n", CHOL_NS)
def test_cholesky_block_edges(gp, n, ldpad):
    _check_cholesky(gp, n, n + ldpad)


@pytest.mark.parametrize("ldpad", [0, 3])
@pytest.mark.parametrize("n", [1, 65, 129, 577, 1025])
def test_core_cholesky(gp, n, ldpad):
    _check_cholesky(gp, n, n + ldpad)


# ---- 2. failing pivots -----------------------------------------------------------------------------------------------
PIVOTS = [0, 1, 63, 64, 127, 255, 256, 511, 512, 513]
PIVOT_CASES = [(n, j) for n in (130, 700, 1100) for j in sorted(set(PIVOTS + [n - 1])) if j < n]


def _make_indefinite(K, j, how):
    """Leading minors of order <= j stay positive definite; the one of order j+1 gets pivot -0.5 (or NaN)."""
    K = K.copy()
    if how == "nan":
        K[j, j] = np.nan
    else:
        K[j, j] -= cholesky(K, lower=True)[j, j] ** 2 + 0.5
    return K


def _lapack_info(K, how):
    """LAPACK's pivot number.  For a NaN pivot the reference routines (dpotrf2 / dpotf2: `AJJ.LE.ZERO .OR. DISNAN(AJJ)`)
    report it, but an optimised dpotrf (OpenBLAS's own, which scipy may link) can return info = 0 with a NaN factor, so
    there the reference's answer is stated directly."""
    return None if how == "nan" else int(dpotrf(K, lower=1)[1])


def _check_pivot(gp, nib, n, j, how):
    K = _make_indefinite(_spd(n, 7 * n + j), j, how)
    want = j + 1
    assert _lapack_info(K, how) in (None, want)
    _, info = _cholesky(gp, K, n, n)
    assert info == want, f"info {info}, LAPACK {want}"
    # the same through GaussianProcessRegressor.fit: its Gram (RBF + alpha) edited on the device before factorising
    rng = np.random.default_rng(n + j)
    X = rng.uniform(0.0, 4.0, size=(n, 3))
    alpha, ell = 1e-2, 1.0
    Kf = ogp.rbf_gram(X, None, ell) + alpha * np.eye(n)
    delta = cholesky(Kf, lower=True)[j, j] ** 2 + 0.5
    Kf = _make_indefinite(Kf, j, how)
    assert _lapack_info(Kf, how) in (None, want)

    class Edited(nib.GaussianProcessRegressor):
        def _gram(self, kind, A, na, B, nb, dim, ell_, jitter, same, out):
            super()._gram(kind, A, na, B, nb, dim, ell_, jitter, same, out)
            if same:
                out[j, j] = float("nan") if how == "nan" else out[j, j] - delta

    model = Edited(alpha=alpha, length_scale=ell, optimizer=None)
    with pytest.raises(np.linalg.LinAlgError, match=rf"\(pivot {want}\)"):
        model.fit(X, rng.standard_normal(n))


@pytest.mark.parametrize("n,j", PIVOT_CASES)
def test_failing_pivot_reports_lapack_info(gp, nib, n, j):
    _check_pivot(gp, nib, n, j, "negative")


@pytest.mark.parametrize("n,j", [(130, 0), (130, 64), (700, 63), (700, 512), (1100, 1099)])
def test_nan_pivot_reports_lapack_info(gp, nib, n, j):
    _check_pivot(gp, nib, n, j, "nan")


@pytest.mark.parametrize("how", ["negative", "nan"])
@pytest.mark.parametrize("j", [0, 64, 513, 699])
def test_core_failing_pivot(gp, nib, j, how):
    _check_pivot(gp, nib, 700, j, how)


# ---- 3. TRSM / TRSV --------------------------------------------------------------------------------------------------
RHS = [(1, 1), (1, 2)] + [(r, r + p) for r in (1, 2, 127, 129, 1000) for p in (0, 5) if (r, r + p) != (1, 1)]


def _check_trsm(gp, n, shapes):
    K = _spd(n, 1000 + n)
    L = cholesky(K, lower=True)
    ldl = n + 2
    Lbuf = np.full((n, ldl), np.nan)            # NaN above the diagonal and in the padding: read only the lower part
    Lbuf[:, :n] = np.where(np.tri(n, dtype=bool), L, np.nan)
    dL = _dev(Lbuf)
    rng = np.random.default_rng(n)
    for nrhs, ldb in shapes:
        for trans in (0, 1):
            B = rng.standard_normal((n, nrhs))
            buf = np.empty((n, ldb))
            _bits(buf)[:] = SENT
            buf[:, :nrhs] = B
            d = _dev(buf)
            gp("nib_gp_trsm", dL.data_ptr(), n, ldl, d.data_ptr(), nrhs, ldb, trans)
            out = _host(d)
            ref = solve_triangular(L, B, lower=True, trans=trans)
            err = np.abs(out[:, :nrhs] - ref).max()
            # forward error of a solve with cond(L) <= sqrt(5): ~n eps; 1e-11 leaves > 30x margin at n = 1537
            assert err <= 1e-11 * max(1.0, np.abs(ref).max()), f"nrhs={nrhs} ldb={ldb} trans={trans}: {err:.3e}"
            assert np.array_equal(_bits(out[:, nrhs:]), _bits(buf[:, nrhs:])), f"padding written (ldb={ldb})"


@pytest.mark.parametrize("n", CHOL_NS)
def test_trsm_vs_solve_triangular(gp, n):
    _check_trsm(gp, n, RHS)


@pytest.mark.parametrize("n", [65, 577, 1025])
def test_core_trsm(gp, n):
    _check_trsm(gp, n, [(1, 1), (1, 2), (129, 134)])


# ---- 4. the DMMA GEMM ------------------------------------------------------------------------------------------------
DG = [1, 15, 16, 17, 63, 65, 127, 129, 200]   # straddle GK = 16, GTM = 64 / 128, GT = 128


def _check_dgemm(gp, M, Ns, Ks, seed):
    rng = np.random.default_rng(seed)
    for N in Ns:
        for K in Ks:
            A = rng.standard_normal((M, K))
            B = rng.standard_normal((K, N))
            C0 = rng.standard_normal((M, N))
            ref = C0 - A @ B
            bound = 2 * (K + 2) * EPS * (np.abs(A) @ np.abs(B) + np.abs(C0))
            # C at offset 2 (16-byte aligned: paired stores) and at offset 1 (scalar stores), sentinel guards around it
            for off in (1, 2):
                buf = np.empty(M * N + 4)
                _bits(buf)[:] = SENT
                buf[off:off + M * N] = C0.ravel()
                dA, dB, dC = _dev(A), _dev(B), _dev(buf)
                gp("nib_gp_dgemm_sub", dA.data_ptr(), dB.data_ptr(), dC.data_ptr() + 8 * off, M, N, K)
                out = _host(dC)
                got = out[off:off + M * N].reshape(M, N)
                assert (np.abs(got - ref) <= bound).all(), f"M={M} N={N} K={K} off={off}: {np.abs(got - ref).max():.3e}"
                assert np.array_equal(_bits(out[:off]), _bits(buf[:off]))
                tail = off + M * N
                assert np.array_equal(_bits(out[tail:]), _bits(buf[tail:])), f"M={M} N={N} K={K}: wrote past C"


@pytest.mark.parametrize("M", DG)
def test_dgemm_sub_vs_numpy(gp, M):
    _check_dgemm(gp, M, DG, DG, M)


@pytest.mark.parametrize("M", [1, 129, 200])
def test_core_dgemm(gp, M):
    _check_dgemm(gp, M, [15, 129, 200], [17, 129], M)


# ---- 5. posterior pieces ---------------------------------------------------------------------------------------------
def _posterior(gp, L, alpha_vec, Ks, y_mean, y_std, ldl, ldks):
    n, m = L.shape[0], Ks.shape[0]
    Lbuf = np.full((n, ldl), np.nan)
    Lbuf[:, :n] = np.where(np.tri(n, dtype=bool), L, np.nan)
    Kbuf = np.full((m, ldks), np.nan)
    Kbuf[:, :n] = Ks
    dL, da, dK = _dev(Lbuf), _dev(alpha_vec), _dev(Kbuf)
    work = torch.empty(n * m, dtype=torch.float64, device="cuda")
    mu, var, sd = (torch.empty(m, dtype=torch.float64, device="cuda") for _ in range(3))
    gp("nib_gp_posterior", dL.data_ptr(), n, ldl, da.data_ptr(), dK.data_ptr(), m, ldks, y_mean, y_std, 1.0,
       work.data_ptr(), mu.data_ptr(), var.data_ptr(), sd.data_ptr())
    return _host(mu), _host(var), _host(sd)


@pytest.mark.parametrize("n,m", [(300, 257), (1025, 1000), (129, 300)])
def test_posterior_vs_oracle(gp, n, m):
    rng = np.random.default_rng(n * m)
    X = rng.uniform(0.0, 3.0, size=(n + m, 3))
    fit = ogp.gp_fit(X[:n], rng.standard_normal(n), 1.0, alpha=1e-2)
    mu0, var0, sd0 = ogp.gp_predict(fit, X[n:])
    Ks = ogp.rbf_gram(X[n:], X[:n], 1.0)
    mu, var, sd = _posterior(gp, fit["L"], fit["alpha"], Ks, fit["y_mean"], fit["y_std"], n + 3, n + 5)
    mscale = fit["y_std"] * (np.abs(Ks) @ np.abs(fit["alpha"])).max() + abs(fit["y_mean"])
    assert np.abs(mu - mu0).max() <= 1e-11 * mscale
    assert np.abs(var - var0).max() <= 1e-11 * fit["y_std"] ** 2
    assert np.array_equal(sd, np.sqrt(var))


def test_posterior_variance_clips_to_zero(gp):
    """Queries equal to training points with a tiny negative jitter (alpha = -1e-9): the exact posterior variance there
    is 1 - k^T K^-1 k = alpha + O(alpha^2) < 0, far beyond rounding, so both implementations clip it to exactly 0."""
    n, m = 40, 37
    rng = np.random.default_rng(40)
    X = rng.uniform(0.0, 20.0, size=(n, 3))
    Xq = np.concatenate([X[:5], rng.uniform(0.0, 20.0, size=(m - 5, 3))])
    fit = ogp.gp_fit(X, rng.standard_normal(n), 1.0, alpha=-1e-9)
    mu0, var0, _ = ogp.gp_predict(fit, Xq)
    Ks = ogp.rbf_gram(Xq, X, 1.0)
    mu, var, sd = _posterior(gp, fit["L"], fit["alpha"], Ks, fit["y_mean"], fit["y_std"], n + 1, n + 1)
    assert (var0[:5] == 0.0).all()
    assert (var[:5] == 0.0).all() and (sd[:5] == 0.0).all()
    assert (var[5:] > 0.0).all()
    np.testing.assert_allclose(mu, mu0, rtol=1e-10, atol=1e-10)
    assert np.abs(var - var0).max() <= 1e-11 * fit["y_std"] ** 2


@pytest.mark.parametrize("n,m", [(1, 1), (7, 300), (131, 257), (1027, 1000), (2050, 513)])
def test_gemv_t_and_colsumsq(gp, n, m):
    rng = np.random.default_rng(n + m)
    ldv = m + 3
    V = rng.standard_normal((n, m))
    x = rng.standard_normal(n)
    buf = np.full((n + 1, ldv), np.nan)   # NaN padding columns and a NaN spare row: neither may be read
    buf[:n, :m] = V
    dV, dx = _dev(buf), _dev(x)
    out = torch.empty(m, dtype=torch.float64, device="cuda")
    gp("nib_gp_gemv_t", dV.data_ptr(), n, m, ldv, dx.data_ptr(), out.data_ptr())
    got = _host(out)
    assert (np.abs(got - V.T @ x) <= 2 * n * EPS * (np.abs(V.T) @ np.abs(x))).all()
    gp("nib_gp_colsumsq", dV.data_ptr(), n, m, ldv, out.data_ptr())
    got = _host(out)
    ref = (V * V).sum(0)
    assert (np.abs(got - ref) <= 2 * n * EPS * ref).all()


@pytest.mark.parametrize("m", [1, 255, 257, 1000])
def test_append_row(gp, m):
    rng = np.random.default_rng(m)
    ks, dot, ssq0 = rng.standard_normal(m), rng.standard_normal(m), rng.uniform(0.0, 1.0, m)
    d = 1.7
    row = np.empty(m + 2)
    _bits(row)[:] = SENT
    dks, ddot, drow, dssq = _dev(ks), _dev(dot), _dev(row), _dev(ssq0)
    gp("nib_gp_append_row", dks.data_ptr(), ddot.data_ptr(), d, drow.data_ptr() + 8, dssq.data_ptr(), m)
    out, ssq = _host(drow), _host(dssq)
    v = (ks - dot) / d
    assert np.array_equal(out[1:-1], v)             # one IEEE subtraction and division: exact
    assert _bits(out)[0] == SENT and _bits(out)[-1] == SENT
    ref = ssq0 + v * v
    assert (np.abs(ssq - ref) <= 2 * EPS * ref).all()


# ---- 6. Gram kernels -------------------------------------------------------------------------------------------------
def _gram_binary(gp, Za, Zb, words, ell, jitter, ldk, same=False):
    na, nb = Za.shape[0], Zb.shape[0]
    dA = _dev(Za.view(np.int64))
    dB = dA if same else _dev(Zb.view(np.int64))
    buf = np.empty((na + 1, ldk))
    _bits(buf)[:] = SENT
    dK = _dev(buf)
    gp("nib_gp_gram_binary", dA.data_ptr(), na, dB.data_ptr(), nb, words, ell, jitter, dK.data_ptr(), ldk)
    out = _host(dK)
    assert np.array_equal(_bits(out[:, nb:]), _bits(buf[:, nb:])) and np.array_equal(_bits(out[na]), _bits(buf[na]))
    return out[:na, :nb]


@pytest.mark.parametrize("S", [63, 64, 65, 128, 129])   # words = 1, 1, 2, 2, 3
def test_gram_binary_vs_rbf(gp, S):
    rng = np.random.default_rng(S)
    words, ell = (S + 63) // 64, 2.5
    Za, Zb = _rand_bits(rng, 70, S), _rand_bits(rng, 45, S)
    K = _gram_binary(gp, Za, Zb, words, ell, 0.0, 45 + 3)
    ref = ogp.rbf_gram(ogp.bits_to_matrix(Za, S), ogp.bits_to_matrix(Zb, S), ell)
    # the LUT holds exp(-h / (2 l^2)); the reference sums h squared differences of X / l: ulps of an argument <= 11
    np.testing.assert_allclose(K, ref, rtol=1e-12, atol=0)
    jitter = 1e-3
    Ks = _gram_binary(gp, Za, Za, words, ell, jitter, 70 + 5, same=True)
    assert (np.diag(Ks) == 1.0 + jitter).all()
    assert np.array_equal(_bits(Ks), _bits(Ks.T))
    ref = ogp.rbf_gram(ogp.bits_to_matrix(Za, S), None, ell)
    off = ~np.eye(70, dtype=bool)
    np.testing.assert_allclose(Ks[off], ref[off], rtol=1e-12, atol=0)


@pytest.mark.parametrize("d", [1, 3, 7])
def test_gram_rbf_vs_oracle(gp, d):
    rng = np.random.default_rng(d)
    ell = 1.3
    Xa, Xb = rng.uniform(0.0, 3.0, size=(70, d)), rng.uniform(0.0, 3.0, size=(45, d))
    for A, B, same, jitter in ((Xa, Xb, 0, 0.0), (Xa, Xa, 1, 1e-3)):
        na, nb = A.shape[0], B.shape[0]
        ldk = nb + 3
        dA = _dev(A)
        dB = dA if same else _dev(B)
        buf = np.empty((na + 1, ldk))
        _bits(buf)[:] = SENT
        dK = _dev(buf)
        gp("nib_gp_gram_rbf", dA.data_ptr(), na, dB.data_ptr(), nb, d, ell, jitter, same, dK.data_ptr(), ldk)
        out = _host(dK)
        K = out[:na, :nb]
        ref = ogp.rbf_gram(A, None if same else B, ell)
        if same:
            ref = ref + jitter * np.eye(na)
            assert (np.diag(K) == 1.0 + jitter).all()
        np.testing.assert_allclose(K, ref, rtol=1e-12, atol=0)
        assert np.array_equal(_bits(out[:, nb:]), _bits(buf[:, nb:])) and np.array_equal(_bits(out[na]), _bits(buf[na]))


# ---- 7. LML and its gradient -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1100, 1537])   # n > 1024: the LML kernel's single block of 1024 threads loops
def test_lml_and_gradients_vs_oracle(gp, n):
    rng = np.random.default_rng(n)
    S, ell, alpha = 50, 3.0, 1e-2
    ld = n + 3

    def padded(M):
        buf = np.full((n, ld), np.nan)
        buf[:, :n] = M
        return _dev(buf)

    for kind in ("bits", "real"):
        if kind == "bits":
            Z = _rand_bits(rng, n, S)
            X = ogp.bits_to_matrix(Z, S)
        else:
            X = rng.uniform(0.0, 3.0, size=(n, 3))
        yn = rng.standard_normal(n)
        K0 = ogp.rbf_gram(X, None, ell)
        L = cholesky(K0 + alpha * np.eye(n), lower=True)
        a = cho_solve((L, True), yn)
        Kinv = cho_solve((L, True), np.eye(n))
        lml0, g0 = ogp.lml_and_grad(X, yn, ell, alpha)
        dL, dK0, dKi, dy, da = padded(np.tril(L)), padded(K0), padded(Kinv), _dev(yn), _dev(a)
        out = C.c_double()
        gp("nib_gp_lml", dL.data_ptr(), n, ld, dy.data_ptr(), da.data_ptr(), C.byref(out))
        lscale = 0.5 * np.abs(yn @ a) + np.abs(np.log(np.diag(L))).sum() + n
        assert abs(out.value - lml0) <= 1e-12 * lscale, (out.value, lml0)
        # the gradient restated from cdist: 0.5 sum((a a^T - K^-1) .* K0 .* D2), D2 = sqeuclidean(X / l)
        D2 = cdist(X / ell, X / ell, metric="sqeuclidean")
        terms = (np.outer(a, a) - Kinv) * K0 * D2
        g_ref = 0.5 * terms.sum()
        gscale = 0.5 * np.abs(terms).sum()
        assert abs(g_ref - g0) <= 1e-12 * gscale
        if kind == "bits":
            dZ = _dev(Z.view(np.int64))
            gp("nib_gp_lml_grad", dK0.data_ptr(), dKi.data_ptr(), da.data_ptr(), dZ.data_ptr(), 1, n, ld, ell,
               C.byref(out))
        else:
            dX = _dev(X)
            gp("nib_gp_lml_grad_rbf", dK0.data_ptr(), dKi.data_ptr(), da.data_ptr(), dX.data_ptr(), 3, n, ld, ell,
               C.byref(out))
        assert abs(out.value - g_ref) <= 1e-11 * gscale, (kind, out.value, g_ref)


# ---- 8. EI and its argmax --------------------------------------------------------------------------------------------
def _ei(gp, mu, sigma, best, gib):
    m = mu.shape[0]
    dmu, dsg = _dev(mu), _dev(sigma)
    ei = torch.empty(m, dtype=torch.float64, device="cuda")
    arg = torch.full((1,), -7, dtype=torch.int64, device="cuda")
    gp("nib_gp_ei", dmu.data_ptr(), dsg.data_ptr(), m, float(best), int(gib), ei.data_ptr(), arg.data_ptr())
    return _host(ei), int(_host(arg)[0])


@pytest.mark.parametrize("gib", [False, True])
@pytest.mark.parametrize("m", [1, 1023, 1025, 5000])
def test_ei_and_argmax_vs_reference(gp, m, gib):
    rng = np.random.default_rng(m + gib)
    mu, sigma = rng.standard_normal(m), rng.uniform(0.05, 1.0, m)
    losses = rng.standard_normal(20)
    best = losses.max() if gib else losses.min()
    if m > 1:
        z = rng.choice(m, size=max(2, m // 50), replace=False)
        sigma[z] = 0.0                          # sigma = 0: finite where mu != best ...
        mu[z[::2]] = best                       # ... and 0/0 = NaN where mu == best
    ei, arg = _ei(gp, mu, sigma, best, gib)
    want = -ogp.expected_improvement(mu, sigma, losses, greater_is_better=gib)
    assert np.array_equal(np.isnan(ei), np.isnan(want))
    ok = ~np.isnan(want)
    np.testing.assert_allclose(ei[ok], want[ok], rtol=1e-12, atol=1e-15)
    assert arg == int(np.nanargmax(want))


@pytest.mark.parametrize("ties", [[4999, 1030, 9, 7, 40], [1030, 6], [3071, 2047, 1023], [4095]])
def test_argmax_ties_pick_the_lowest_index(gp, ties):
    """Duplicate (mu, sigma) pairs give bitwise-equal EI; the argmax is the lowest such index, like np.nanargmax.
    The first list puts tied entries in lanes of one warp (thread 6 holds 1030, threads 7 and 9 their own)."""
    m = 5000
    rng = np.random.default_rng(len(ties))
    mu, sigma = rng.uniform(-1.0, 0.0, m), rng.uniform(0.1, 0.5, m)
    mu[ties], sigma[ties] = 2.0, 0.3
    sigma[[0, 3, 1029]] = 0.0
    mu[[0, 3, 1029]] = 0.0                      # NaN (0/0) entries mixed in, one of them next to a tie
    ei, arg = _ei(gp, mu, sigma, 0.0, True)
    want = -ogp.expected_improvement(mu, sigma, np.array([0.0]), greater_is_better=True)
    assert np.isnan(ei[[0, 3, 1029]]).all()
    assert len(set(_bits(ei[ties]).tolist())) == 1
    assert arg == min(ties) == int(np.nanargmax(want))


# ---- 10. two streams -------------------------------------------------------------------------------------------------
def test_two_streams_match_one_stream(gp):
    """Two fits + posteriors of different sizes enqueued alternately on two streams without synchronising in between
    (the library's scratch is per stream) equal, bit for bit, the same calls run one after the other on one stream."""
    S, ell, alpha = 50, 3.0, 1e-2
    jobs = []
    for n, m, seed in ((700, 300, 1), (1100, 513, 2)):
        rng = np.random.default_rng(seed)
        Z, Q = _rand_bits(rng, n, S), _rand_bits(rng, m, S)
        jobs.append(dict(n=n, m=m, Z=_dev(Z.view(np.int64)), Q=_dev(Q.view(np.int64)), y=rng.standard_normal(n)))

    def buffers(job):
        n, m, f = job["n"], job["m"], dict(dtype=torch.float64, device="cuda")
        return dict(K=torch.empty(n, n, **f), Ks=torch.empty(m, n, **f), a=_dev(job["y"]), work=torch.empty(n * m, **f),
                    mu=torch.empty(m, **f), var=torch.empty(m, **f), sd=torch.empty(m, **f),
                    info=torch.zeros(1, dtype=torch.int32, device="cuda"))

    def calls(job, b, st):
        n, m = job["n"], job["m"]
        return [
            lambda: gp("nib_gp_gram_binary", job["Z"].data_ptr(), n, job["Z"].data_ptr(), n, 1, ell, alpha,
                       b["K"].data_ptr(), n, stream=st),
            lambda: gp("nib_gp_cholesky", b["K"].data_ptr(), n, n, b["info"].data_ptr(), stream=st),
            lambda: gp("nib_gp_trsm", b["K"].data_ptr(), n, n, b["a"].data_ptr(), 1, 1, 0, stream=st),
            lambda: gp("nib_gp_trsm", b["K"].data_ptr(), n, n, b["a"].data_ptr(), 1, 1, 1, stream=st),
            lambda: gp("nib_gp_gram_binary", job["Q"].data_ptr(), m, job["Z"].data_ptr(), n, 1, ell, 0.0,
                       b["Ks"].data_ptr(), n, stream=st),
            lambda: gp("nib_gp_posterior", b["K"].data_ptr(), n, n, b["a"].data_ptr(), b["Ks"].data_ptr(), m, n, 0.0,
                       1.0, 1.0, b["work"].data_ptr(), b["mu"].data_ptr(), b["var"].data_ptr(), b["sd"].data_ptr(),
                       stream=st),
        ]

    keys = ("K", "a", "mu", "var", "sd", "info")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    serial = [buffers(j) for j in jobs]
    torch.cuda.synchronize()
    for j, b in zip(jobs, serial):
        for c in calls(j, b, s1):
            c()
    torch.cuda.synchronize()
    want = [{k: b[k].cpu().numpy() for k in keys} for b in serial]
    for _ in range(2):
        conc = [buffers(j) for j in jobs]
        torch.cuda.synchronize()
        for c1, c2 in zip(calls(jobs[0], conc[0], s1), calls(jobs[1], conc[1], s2)):
            c1()
            c2()
        torch.cuda.synchronize()
        for w, b in zip(want, conc):
            assert int(w["info"][0]) == 0
            for k in keys:
                assert np.array_equal(w[k].view(np.uint8), b[k].cpu().numpy().view(np.uint8)), k


# ---- 11. a C of more than 2^31 elements ------------------------------------------------------------------------------
def test_dgemm_sub_c_beyond_2_31_elements(gp):
    """M * N = 2^31 + 261952 (C = 17.2 GB): rows on both sides of element 2^31 (row 65552) against numpy."""
    if torch.cuda.mem_get_info()[0] < 24 * 2 ** 30:
        pytest.skip("needs 24 GB of free device memory")
    M, N, K = 65560, 32760, 17
    assert M * N > 2 ** 31
    rng = np.random.default_rng(31)
    A, B = rng.standard_normal((M, K)), rng.standard_normal((K, N))
    dA, dB = _dev(A), _dev(B)
    dC = torch.full((M, N), 0.5, dtype=torch.float64, device="cuda")
    try:
        gp("nib_gp_dgemm_sub", dA.data_ptr(), dB.data_ptr(), dC.data_ptr(), M, N, K)
        rows = [0, 1, 63, 32767, 65535] + list(range(65548, M))
        got = _host(dC[rows])
    finally:
        del dC
        torch.cuda.empty_cache()
    ref = 0.5 - A[rows] @ B
    bound = 2 * (K + 2) * EPS * (np.abs(A[rows]) @ np.abs(B) + 0.5)
    assert (np.abs(got - ref) <= bound).all(), np.abs(got - ref).max()


# ---- 9. solver variants ----------------------------------------------------------------------------------------------
VARIANTS = {
    "v1": {"NIB_GP_V1": "1"},
    "trsv_steps": {"NIB_GP_TRSV_STEPS": "1"},
    "nbc64": {"NIB_GP_NBC": "64"},
    "nbc128": {"NIB_GP_NBC": "128"},
    "tile_m128": {"NIB_GP_TILE_M": "128"},
    "chol_rec": {"NIB_GP_CHOL_REC": "1"},
    "lookahead": {"NIB_GP_LOOKAHEAD": "1"},
}
SWITCHES = sorted({k for v in VARIANTS.values() for k in v})


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_solver_variant(nib, variant):
    """The test_core_* subset, each checked against scipy / LAPACK, in a child process with one switch set."""
    env = {k: v for k, v in os.environ.items() if k not in SWITCHES}
    env.update(VARIANTS[variant])
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [
        "-m", "pytest", os.path.abspath(__file__), "-q", "-m", "gpu", "-k", "core", "-p", "no:cacheprovider"]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    tail = r.stdout[-6000:] + r.stderr[-2000:]
    assert r.returncode == 0, tail
    assert " passed" in r.stdout and "skipped" not in r.stdout and "deselected" in r.stdout, tail
