"""CPU: the matrix-free SKI oracle against the dense definition, and the lattice algebra the Kronecker solver rests on."""
import numpy as np
import pytest

from oracle import ski as oski
from oracle import ski_matfree


@pytest.mark.parametrize("n,gs,ell,noise,os_", [(300, 12, 1.0, 1.0, 1.0), (500, 30, 1.0, 1.0, 1.0), (400, 12, 25.0, 0.1, 2.0)])
def test_matrix_free_oracle_equals_dense_definition(n, gs, ell, noise, os_):
    rng = np.random.RandomState(n)
    X = rng.randint(0, 224, size=(n, 2)).astype(np.float64)          # duplicates allowed, pixel 0 included
    X[0] = (0.0, 0.0)
    y = rng.rand(n) * 40.0
    Xq = np.stack(np.meshgrid(np.arange(0, 224, 9.0), np.arange(0, 224, 7.0), indexing="ij"), -1).reshape(-1, 2)
    mean0, var0 = oski.ski_posterior(X, y, Xq, (0.0, 224.0), gs, ell, os_, noise, const_mean=0.5)
    mean, var, _ = ski_matfree.ski_posterior_matfree(X, y, Xq, (0.0, 224.0), gs, ell, os_, noise, const_mean=0.5,
                                                     var_idx=np.arange(Xq.shape[0]))
    assert np.abs(mean - mean0).max() <= 1e-10 * np.abs(mean0).max()
    assert np.abs(var - var0).max() <= 1e-10 * np.abs(var0).max()


@pytest.mark.parametrize("gs,ell,os_", [(12, 1.0, 1.0), (20, 10.0, 50.0)])
def test_lattice_training_set_makes_the_eigen_coordinate_system_diagonal(gs, ell, os_):
    """Training pixels R x C, each once: A = A_R (x) A_C, and in the coordinates of kron_factors B - s2 I is diagonal."""
    from network_interpretation_imagenet_b200.ski import interp_1d, kron_factors
    rows, cols = np.arange(0.0, 224.0, 3.0), np.arange(1.0, 224.0, 5.0)
    X = np.stack(np.meshgrid(rows, cols, indexing="ij"), -1).reshape(-1, 2)
    g0, h = oski.make_grid(0.0, 224.0, gs)
    W = oski.interp_matrix(X, g0, h, gs)
    A = W.T @ W
    WR, WC = interp_1d(rows, g0, h, gs), interp_1d(cols, g0, h, gs)
    assert np.abs(A - np.kron(WR.T @ WR, WC.T @ WC)).max() <= 1e-12 * np.abs(A).max()
    MR, MC, thR, thC = kron_factors(gs, g0, h, ell, os_, rows, cols)
    S = np.kron(MR, MC)
    K = oski.grid_kernel(g0, h, gs, ell, os_)
    assert np.abs(S @ S.T - K).max() <= 1e-12 * np.abs(K).max()
    Bh = S.T @ A @ S
    D = os_ * np.outer(thR, thC).reshape(-1)
    assert np.abs(Bh - np.diag(D)).max() <= 1e-12 * np.abs(D).max()


def test_interp_1d_is_the_axis_factor_of_the_grid_interpolation():
    from network_interpretation_imagenet_b200.ski import interp_1d
    gs = 30
    g0, h = oski.make_grid(0.0, 224.0, gs)
    X = np.array([[0.0, 223.0], [0.5, 100.25], [17.0, 0.0], [223.0, 223.0]])
    W = oski.interp_matrix(X, g0, h, gs).reshape(-1, gs, gs)
    want = np.einsum("pi,pj->pij", interp_1d(X[:, 0], g0, h, gs), interp_1d(X[:, 1], g0, h, gs))
    assert np.abs(W - want).max() <= 1e-15
