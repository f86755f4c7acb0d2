"""GPU: the Kronecker-structured SKI solver (solver="kron", csrc/ski_kron.cu) against the dense definition, the product's
dense solver and the matrix-free oracle at grid_size 300; its kernels at the C ABI; the drop-in at grid_size 300."""
import numpy as np
import pytest
import torch

from oracle import ski as oski
from oracle import ski_matfree

pytestmark = pytest.mark.gpu

FULL = np.stack(np.meshgrid(np.arange(224.0), np.arange(224.0), indexing="ij"), -1).reshape(-1, 2)
STRIP = (150, 194)                                                  # 44 uncovered columns


def _strip_set():
    keep = (FULL[:, 1] < STRIP[0]) | (FULL[:, 1] >= STRIP[1])
    X = FULL[keep]
    y = 20.0 * np.exp(-((X[:, 0] - 100) ** 2 + (X[:, 1] - 120) ** 2) / (2 * 40.0 ** 2))
    return X, y


def _square_hole_set():
    hole = (FULL[:, 0] >= 90) & (FULL[:, 0] < 134) & (FULL[:, 1] >= 90) & (FULL[:, 1] < 134)
    X = FULL[~hole]
    return X, np.sin(X[:, 0] / 17.0) * 10.0 + X[:, 1] / 50.0


@pytest.mark.parametrize("n,gs,ell,noise,os_", [(300, 12, 1.0, 1.0, 1.0), (500, 30, 1.0, 1.0, 1.0), (400, 16, 25.0, 0.1, 2.0),
                                                (600, 64, 3.0, 1.0, 1.0)])
def test_kron_solver_equals_dense_ski_definition(nib, n, gs, ell, noise, os_):
    from network_interpretation_imagenet_b200.ski import GridGPRegression
    rng = np.random.RandomState(n)
    X = rng.randint(0, 224, size=(n, 2)).astype(np.float64)          # duplicates allowed: not a lattice
    y = rng.rand(n) * 40.0
    Xq = np.stack(np.meshgrid(np.arange(0, 224, 9.0), np.arange(0, 224, 7.0), indexing="ij"), -1).reshape(-1, 2)
    mean0, var0 = oski.ski_posterior(X, y, Xq, (0.0, 224.0), gs, ell, os_, noise, const_mean=0.5)
    args = (gs, ((0.0, 224.0), (0.0, 224.0)), ell, os_, noise)
    gp = GridGPRegression(*args, const_mean=0.5, solver="kron").fit(X, y)
    mean, var = (t.cpu().numpy() for t in gp.predict(Xq))
    assert gp.solver == "kron" and gp.mean_iters >= 1 and len(gp.var_iters) == 1
    assert np.abs(mean - mean0).max() <= 1e-8 * np.abs(mean0).max()
    assert np.abs(var - var0).max() <= 1e-8 * np.abs(var0).max()
    dense = GridGPRegression(*args, const_mean=0.5, solver="dense").fit(X, y)
    dmean, dvar = (t.cpu().numpy() for t in dense.predict(Xq))
    assert np.abs(mean - dmean).max() <= 1e-6 * np.abs(dmean).max()
    assert np.abs(var - dvar).max() <= 1e-6 * np.abs(dvar).max()
    lat = gp.predict(Xq, likelihood=False)[1].cpu().numpy()
    np.testing.assert_allclose(lat + noise, var, rtol=1e-12)
    np.testing.assert_array_equal(gp.predict(Xq, return_var=False).cpu().numpy(), mean)


def test_auto_picks_dense_up_to_grid_100_and_kron_above(nib):
    from network_interpretation_imagenet_b200.ski import GridGPRegression
    assert GridGPRegression(30).solver == "dense" and GridGPRegression(100).solver == "dense"
    assert GridGPRegression(101).solver == "kron" and GridGPRegression(300).solver == "kron"
    with pytest.raises(ValueError):
        GridGPRegression(30, solver="cholesky")


def test_full_lattice_mean_solve_takes_at_most_two_iterations_at_grid_300(nib):
    from network_interpretation_imagenet_b200.ski import GridGPRegression
    y = np.cos(FULL[:, 0] / 30.0) * 5.0 + FULL[:, 1] / 20.0
    gp = GridGPRegression(300, ((0.0, 224.0), (0.0, 224.0)), 1.0, 1.0, 1.0).fit(FULL, y)
    assert gp.solver == "kron" and 1 <= gp.mean_iters <= 2, gp.mean_iters


@pytest.mark.parametrize("ell,os_", [(1.0, 1.0), (1.0, 50.0), (10.0, 1.0), (10.0, 50.0)])
def test_grid_300_equals_matrix_free_oracle_on_a_lattice_with_an_uncovered_strip(nib, ell, os_):
    """n = 224^2 minus 44 uncovered columns.  Mean at every pixel, variance at 32 seeded pixels on both sides of the strip's
    edges and inside it (8 at l = 10, os = 50, where the oracle's unpreconditioned CG needs thousands of iterations)."""
    from network_interpretation_imagenet_b200.ski import GridGPRegression
    X, y = _strip_set()
    rng = np.random.RandomState(7)
    nv = 8 if (ell, os_) == (10.0, 50.0) else 32
    cols = np.concatenate([rng.randint(STRIP[0] - 6, STRIP[0] + 6, nv // 4), rng.randint(STRIP[1] - 6, STRIP[1] + 6, nv // 4),
                           rng.randint(STRIP[0] + 8, STRIP[1] - 8, nv // 4), rng.randint(0, STRIP[0] - 20, nv // 4)])
    idx = rng.randint(0, 224, nv) * 224 + cols
    mean0, var0, _ = ski_matfree.ski_posterior_matfree(X, y, FULL, (0.0, 224.0), 300, ell, os_, 1.0, var_idx=idx)
    gp = GridGPRegression(300, ((0.0, 224.0), (0.0, 224.0)), ell, os_, 1.0).fit(X, y)
    mean = gp.predict(FULL, return_var=False).cpu().numpy()
    var = gp.predict(FULL[idx])[1].cpu().numpy()
    assert np.abs(mean - mean0).max() <= 1e-6 * np.abs(mean0).max()
    np.testing.assert_allclose(var, var0, rtol=1e-6)
    inside = (cols >= STRIP[0] + 8) & (cols < STRIP[1] - 8)
    far = cols < STRIP[0] - 20
    assert var[inside].min() > var[far].max()


def test_iteration_cap_raises_and_names_the_residual(nib):
    from network_interpretation_imagenet_b200.ski import GridGPRegression
    X, y = _square_hole_set()
    gp = GridGPRegression(300, ((0.0, 224.0), (0.0, 224.0)), 1.0, 1.0, 1.0, max_iter=1)
    with pytest.raises(np.linalg.LinAlgError, match=r"relative residual \d\.\d+e[-+]\d+ > cg_tol"):
        gp.fit(X, y)


def test_two_streams_are_bitwise_equal_to_one(nib):
    from network_interpretation_imagenet_b200.ski import GridGPRegression
    X, y = _square_hole_set()
    q = FULL[np.random.RandomState(3).choice(FULL.shape[0], 1500, replace=False)]

    def run():
        gp = GridGPRegression(300, ((0.0, 224.0), (0.0, 224.0)), 1.0, 1.0, 1.0).fit(X, y)
        mean, var = gp.predict(q)
        return gp.mean_u.clone(), mean.clone(), var.clone(), gp.mean_iters

    ref = run()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    got = []
    for s in (s1, s2, s1):
        with torch.cuda.stream(s):
            got.append(run())
    torch.cuda.synchronize()
    assert ref[3] > 2                                     # the holed lattice takes several PCG iterations
    for g in got:
        assert all(torch.equal(a, b) for a, b in zip(ref[:3], g[:3])) and g[3] == ref[3]


# ---- kernels at the C ABI -------------------------------------------------------------------------------------------------

def _call(nib, name, *args):
    nib._lib.check(getattr(nib._lib.load(), name)(*args, torch.cuda.current_stream().cuda_stream), name)


@pytest.mark.parametrize("gs", [1, 7, 64, 65, 300])
@pytest.mark.parametrize("r", [1, 3, 1024])
def test_kron_apply_equals_numpy(nib, gs, r):
    rng = np.random.RandomState(gs * 7 + r)
    MR, MC = rng.randn(gs, gs), rng.randn(gs, gs)
    X = rng.randn(r, gs, gs)
    dX, dMR, dMC = (torch.from_numpy(a).cuda() for a in (X, MR, MC))
    for trans in (0, 1):
        want = MR @ X @ MC.T if trans == 0 else MR.T @ X @ MC
        dY = torch.full((r, gs, gs), np.nan, dtype=torch.float64, device="cuda")
        work = torch.empty(r * gs * gs, dtype=torch.float64, device="cuda")
        _call(nib, "nib_ski_kron_apply", dX.data_ptr(), dY.data_ptr(), r, gs, dMR.data_ptr(), dMC.data_ptr(), trans,
              work.data_ptr())
        scale = np.abs(MR).max() * np.abs(MC).max() * np.abs(X).max() * gs * gs
        assert np.abs(dY.cpu().numpy() - want).max() <= 1e-14 * scale


def _band_accumulate(nib, X, y, gs, c=0.5):
    g0, h = oski.make_grid(0.0, 224.0, gs)
    n, G = X.shape[0], gs * gs
    dX, dy = torch.from_numpy(X).cuda(), torch.from_numpy(y).cuda()
    A = torch.full((G * 49,), np.nan, dtype=torch.float64, device="cuda")
    b = torch.full((G,), np.nan, dtype=torch.float64, device="cuda")
    work = torch.empty((4 * (2 * n + 3 * G + 2) + 72 * n + 7) // 8, dtype=torch.float64, device="cuda")
    _call(nib, "nib_ski_band_accumulate", dX.data_ptr(), dy.data_ptr(), n, g0, h, gs, c, A.data_ptr(), b.data_ptr(),
          work.data_ptr())
    return A, b


def _band_to_dense(A, gs):
    A = A.reshape(gs, gs, 7, 7)
    D = np.zeros((gs, gs, gs, gs))
    for d0 in range(-3, 4):
        for d1 in range(-3, 4):
            for i in range(gs):
                for j in range(gs):
                    if 0 <= i + d0 < gs and 0 <= j + d1 < gs:
                        D[i, j, i + d0, j + d1] = A[i, j, d0 + 3, d1 + 3]
                    else:
                        assert A[i, j, d0 + 3, d1 + 3] == 0.0
    return D.reshape(gs * gs, gs * gs)


@pytest.mark.parametrize("gs", [4, 9, 16])
def test_band_accumulate_and_spmv_equal_dense_wtw(nib, gs):
    rng = np.random.RandomState(gs)
    X = np.concatenate([rng.randint(0, 224, size=(700, 2)), [[0, 0], [223, 223], [0, 223], [5, 5], [5, 5]]]).astype(np.float64)
    y = rng.randn(X.shape[0])
    g0, h = oski.make_grid(0.0, 224.0, gs)
    W = oski.interp_matrix(X, g0, h, gs)
    A, b = _band_accumulate(nib, X, y, gs)
    Ad = _band_to_dense(A.cpu().numpy(), gs)
    assert np.abs(Ad - W.T @ W).max() <= 1e-13 * np.abs(W.T @ W).max()
    assert np.abs(b.cpu().numpy() - W.T @ (y - 0.5)).max() <= 1e-13 * np.abs(W.T @ (y - 0.5)).max()
    r = 5
    V = rng.randn(r, gs * gs)
    dV = torch.from_numpy(V).cuda()
    dY = torch.full((r, gs * gs), np.nan, dtype=torch.float64, device="cuda")
    _call(nib, "nib_ski_band_spmv", A.data_ptr(), gs, dV.data_ptr(), dY.data_ptr(), r)
    want = V @ (W.T @ W)
    assert np.abs(dY.cpu().numpy() - want).max() <= 1e-13 * np.abs(want).max()


def test_band_accumulate_is_bitwise_reproducible(nib):
    rng = np.random.RandomState(11)
    X = np.concatenate([FULL, FULL[rng.choice(FULL.shape[0], 20000)]])       # duplicates: buckets of several points
    X = X[rng.permutation(X.shape[0])]
    y = rng.randn(X.shape[0])
    for gs in (30, 300):
        A1, b1 = _band_accumulate(nib, X, y, gs)
        A2, b2 = _band_accumulate(nib, X, y, gs)
        assert torch.equal(A1, A2) and torch.equal(b1, b2)


def test_gp_regression_entry_point_round_trip_at_grid_300(nib, tmp_path, monkeypatch):
    """The drop-in gp_regression.py with GPRegressionModel(..., grid_size=300) on a ./masks directory whose masks cover
    every pixel: fits, saves grid_size in the checkpoint, predicts all 224^2 pixels and writes the PNGs."""
    import cv2
    import importlib
    monkeypatch.chdir(tmp_path)
    (tmp_path / "masks").mkdir()
    rng = np.random.RandomState(2)
    i = 0
    for y0 in range(0, 224, 56):
        for x0 in range(0, 224, 56):
            for _ in range(3):
                m = np.zeros((224, 224), np.uint8)
                dy, dx = rng.randint(0, 20, size=2)
                m[max(0, y0 - dy):y0 + 74, max(0, x0 - dx):x0 + 74] = 255
                cv2.imwrite(str(tmp_path / "masks" / f"mask_{i}_{int(rng.rand() < 0.5)}.png"), m)
                i += 1
    import gp_regression as gpr
    gpr = importlib.reload(gpr)
    tx, ty = gpr.prepare_training_data()
    assert tx.shape == (224 * 224, 2)
    lik = gpr.GaussianLikelihood().cuda()
    model = gpr.GPRegressionModel(tx, ty, lik, grid_size=300).cuda()
    gpr.train(tx, ty, model)
    assert torch.load(gpr.CHECKPOINT)["grid_size"] == 300
    pred = gpr.eval_superpixels(gpr.GPRegressionModel(tx, ty, lik), lik)        # grid_size comes from the checkpoint
    assert pred.shape == (224 * 224,) and np.isfinite(pred).all()
    var = gpr.eval_superpixels.last_variance
    assert var.shape == (224 * 224,) and np.isfinite(var).all() and (var > 0).all()
    gpr.plot_result(pred)
    for f in ("predicted_mask_heatmap.png", "predicted_variance_heatmap.png", "summed_label_training_heatmap.png"):
        assert (tmp_path / "weighted_mask" / f).exists()
