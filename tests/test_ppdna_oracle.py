"""The numpy restatement of PPDNA (oracle/ppdna_oracle.py): the Jacobian identities it relies on, its Hessian
against finite differences of its gradient, and its solution against ADMM run to a tight KKT tolerance."""
import numpy as np
import pytest

from oracle import admm_oracle as orc
from oracle import ppdna_oracle as po


@pytest.mark.parametrize("sigma", [1e-3, 1.0, 10.0, 1e4])
def test_gamma_identity_equals_divided_differences(sigma):
    rng = np.random.default_rng(1)
    d = np.concatenate([rng.standard_normal(12) * 5, [0.7, 0.7, -3.0, -3.0, 0.0]])   # ties: phi' on the diagonal
    G1 = po.gamma_dense(po.phi_of(d, sigma), sigma)
    G2 = po.gamma_divided(d, sigma)
    assert np.abs(G1 - G2).max() <= 1e-12 * max(1.0, np.abs(G2).max())


def _random_point(K, p, reg, seed):
    """a random (Omega_t, Theta_t, X, S) whose V entries stay away from the kinks of prox_p"""
    rng = np.random.default_rng(seed)
    S = np.stack([np.cov(rng.standard_normal((p, 3 * p)), bias=True) for _ in range(K)])
    A = rng.standard_normal((K, p, p))
    X = 0.3 * (A + A.transpose(0, 2, 1))
    Om = np.stack([np.eye(p) + 0.1 * (B + B.T) for B in rng.standard_normal((K, p, p))])
    Th = Om.copy()
    return S, Om, Th, X


@pytest.mark.parametrize("reg", ["GGL", "FGL"])
@pytest.mark.parametrize("K", [1, 3, 5])
def test_hessian_matches_finite_differences_of_the_gradient(reg, K):
    p, sigma, l1, l2 = 6, 0.7, 0.05, 0.1
    S, Om, Th, X = _random_point(K, p, reg, seed=K)

    def point(Xn):
        return po.Point(Xn, S, Om, Th, sigma, l1, l2, reg)
    pt = point(X)
    rng = np.random.default_rng(10 + K)
    B = rng.standard_normal((K, p, p))
    Dm = B + B.transpose(0, 2, 1)
    h = 1e-6
    fd = (point(X + h * Dm).grad - point(X - h * Dm).grad) / (2 * h)
    # the central difference is exact only where no entry of V crosses a kink in [-h, h]
    assert np.abs(pt.hess(Dm) - fd).max() <= 1e-6 * max(1.0, np.abs(fd).max())
    # and the gradient is the derivative of Phi
    dphi = (point(X + h * Dm).Phi - point(X - h * Dm).Phi) / (2 * h)
    assert abs(dphi - float(np.sum(pt.grad * Dm))) <= 1e-6 * max(1.0, abs(dphi))


@pytest.mark.parametrize("reg", ["GGL", "FGL"])
def test_hessian_is_symmetric_positive_definite(reg):
    K, p = 3, 6
    S, Om, Th, X = _random_point(K, p, reg, seed=7)
    pt = po.Point(X, S, Om, Th, 2.0, 0.05, 0.1, reg)
    rng = np.random.default_rng(3)
    sym = lambda B: B + B.transpose(0, 2, 1)  # noqa: E731
    A, B = sym(rng.standard_normal((K, p, p))), sym(rng.standard_normal((K, p, p)))
    assert abs(np.sum(A * pt.hess(B)) - np.sum(pt.hess(A) * B)) <= 1e-12 * np.abs(np.sum(A * pt.hess(B))) + 1e-12
    for _ in range(5):
        C = sym(rng.standard_normal((K, p, p)))
        assert np.sum(C * pt.hess(C)) > 0


@pytest.mark.parametrize("name", ["mgl_ggl_K3_p50", "mgl_fgl_K3_p50"])
def test_oracle_ppdna_matches_tight_admm(golden, name):
    g = golden(name)
    S, reg = g["S"], str(g["reg"])
    K, p, _ = S.shape
    Om0 = np.repeat(np.eye(p)[None], K, 0)
    sol, info = po.ppdna(S, 0.05, 0.01, reg, Om0, eps_ppdna=1e-9, measure=True)
    assert info["status"] == "optimal"
    eta = orc.kkt_residual_mgl(sol["Omega"], sol["Theta"], np.zeros_like(S), sol["X"], S, 0.05, 0.01,
                               np.ones((K, 1, 1)), reg)
    assert eta <= 1e-9
    ref, rinfo = orc.admm_mgl(S, 0.05, 0.01, reg, Om0, stopping_criterion="kkt", tol=1e-10, max_iter=5000)
    assert rinfo["status"] == "optimal"
    assert np.abs(sol["Theta"] - ref["Theta"]).max() <= 1e-6
    assert np.array_equal(sol["Theta"] != 0, ref["Theta"] != 0)
