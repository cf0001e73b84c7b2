"""The host references of oracle/kernel_refs.py (used by tests/test_gpu_kernel_units.py) checked on hand-computed
cases and against the oracle's own statement of the same operations."""
import math
from fractions import Fraction

import numpy as np
import pytest

from oracle import admm_oracle as orc
from oracle import kernel_refs as kr


def _sym(rng, n, p, scale=1.0):
    A = rng.standard_normal((n, p, p)) * scale
    return A + A.transpose(0, 2, 1)


def test_fsum_and_exact_gershgorin_hand_cases():
    assert kr.fsum([1e16, 1.0, -1e16]) == 1.0
    assert kr.fsum(np.full(10, 0.1)) == 1.0
    A = np.array([[[4.0, -1.0, 2.0], [-1.0, 3.0, 0.5], [2.0, 0.5, 2.0]]])
    assert kr.gershgorin_exact(A) == [Fraction(-1, 2)]              # row 2: 2 - 2 - 0.5
    assert kr.gershgorin_exact(np.array([[[7.0]]])) == [Fraction(7)]
    # 0.1 + 0.2 is not 0.3 in binary: the exact bound of this row is not zero
    B = np.array([[[0.3, 0.1, 0.2], [0.1, 5.0, 0.0], [0.2, 0.0, 5.0]]])
    assert kr.gershgorin_exact(B)[0] == Fraction(0.3) - Fraction(0.1) - Fraction(0.2) != 0
    assert 0.3 - (0.1 + 0.2) != float(kr.gershgorin_exact(B)[0])


def test_soft_threshold_matches_oracle():
    v = np.array([-2.0, -0.5, -0.0, 0.0, 0.3, 0.5, 3.0])
    np.testing.assert_array_equal(kr.soft(v, 0.5), orc.soft_threshold(v, 0.5))


def test_stop_update_restatement_against_oracle_trajectory():
    """replaying the oracle's recorded ADMM_MGL trajectory through the host stopping test gives its r, s, eps and rho
    sequence and stops at the same iteration"""
    from gglasso_b200 import _lib as C
    rng = np.random.default_rng(3)
    K, p = 3, 8
    S = np.stack([np.cov(rng.standard_normal((p, 30)), bias=True) for _ in range(K)])
    Om0 = np.repeat(np.eye(p)[None], K, 0)
    trace = []
    _, info = orc.admm_mgl(S, 0.05, 0.02, "GGL", Om0, rho=1.0, max_iter=200, tol=1e-6, rtol=1e-5, trace=trace)
    assert info["status"] == "optimal" and len(trace) > 5
    rhos = {t["rho"] for t in trace}
    assert len(rhos) > 1, "the trajectory must exercise the rho update"
    ctrl = np.zeros((1, C.CTRL_STRIDE))
    ctrl[0, C.C_RHO], ctrl[0, C.C_XSCALE] = 1.0, 1.0
    hist = np.zeros((1, len(trace), 5))
    prev = Om0
    for it, t in enumerate(trace):
        assert ctrl[0, C.C_DONE] == 0 and ctrl[0, C.C_RHO] == t["rho"]
        # X in the trace is the scaled dual before the rescaling: the device holds the same value
        tl, res, d2 = t["Theta"] - t["L"], t["Omega"] - t["Theta"] + t["L"], t["Omega"] - prev
        sums = np.array([[kr.fsum(a * a) for a in (t["Omega"], tl, t["X"], res, d2)]])
        kr.stop_update(sums, ctrl, hist, len(trace), [K * (p * p + p) / 2], 1e-6, 1e-5, 1, C)
        np.testing.assert_allclose(hist[0, it, :4], [t["r"], t["s"], t["e_pri"], t["e_dual"]], rtol=1e-12)
        prev = t["Omega"]
    assert ctrl[0, C.C_DONE] == 1 and ctrl[0, C.C_STATUS] == 1 and ctrl[0, C.C_ITER] == len(trace)
    assert ctrl[0, C.C_RHO] == info["rho"]


def test_stop_update_boundaries():
    from gglasso_b200 import _lib as C

    def one(sums, rho=1.0, update=1, pdim=1.0, tol=0.0, rtol=0.0):
        ctrl = np.zeros((1, C.CTRL_STRIDE))
        ctrl[0, C.C_RHO], ctrl[0, C.C_XSCALE] = rho, 1.0
        kr.stop_update(np.array([sums], dtype=float), ctrl, np.zeros((1, 1, 5)), 1, [pdim], tol, rtol, update, C)
        return ctrl[0]
    assert one([0, 0, 0, 100, 1])[C.C_RHO] == 2.0           # r = 10 = 10 s
    assert one([0, 0, 0, 1, 100])[C.C_RHO] == 0.5           # s = 10 = 10 r
    assert one([0, 0, 0, 1, 100], update=0)[C.C_RHO] == 1.0
    c = one([0, 0, 0, 4, 9], pdim=3.0, tol=1.0)             # r = 2 <= 3, s = 3 <= 3
    assert c[C.C_DONE] == 1 and c[C.C_STATUS] == 1
    c = one([0, 0, 0, math.inf, 1])
    assert c[C.C_DONE] == 1 and c[C.C_STATUS] == -1


@pytest.mark.parametrize("Mblk,nb", [(1, 9), (2, 5), (3, 4), (5, 3), (7, 2)])
@pytest.mark.parametrize("latent", [False, True])
def test_fsgl_reference_against_oracle(Mblk, nb, latent):
    rng = np.random.default_rng(Mblk * 10 + nb)
    p, M = Mblk * nb, 2
    Om, Omp, X = _sym(rng, M, p, 0.4), _sym(rng, M, p), _sym(rng, M, p, 0.2)
    L = _sym(rng, M, p, 0.05) if latent else None
    rho = np.array([0.8, 1.7])
    th, out2, parts = kr.prox_fsgl(Om, Omp, L, X, 0.3, rho, Mblk, latent=latent)
    for m in range(M):
        A = Om[m] + (L[m] if latent else 0.0) + X[m]
        ref = orc.prox_sum_frob(A, Mblk, 0.3 / rho[m])
        np.testing.assert_allclose(th[m], ref, rtol=1e-14, atol=1e-15)
        np.testing.assert_allclose(th[m], kr.prox_sum_frob(A, Mblk, (1 / rho[m]) * 0.3), rtol=1e-14, atol=1e-15)
        if latent:
            np.testing.assert_allclose(out2[m], th[m] - X[m] - Om[m], rtol=1e-14, atol=1e-14)
        else:
            np.testing.assert_allclose(out2[m], X[m] + Om[m] - th[m], rtol=1e-14, atol=1e-14)
            r, s, _, _ = orc.boyd_residuals(Om[m], Omp[m], th[m], np.zeros((p, p)), out2[m], 1.0, 0, 0)
            np.testing.assert_allclose([math.sqrt(parts[m, 3]), math.sqrt(parts[m, 4])], [r, s], rtol=1e-13)
    if Mblk == 1:
        th1, _, _ = kr.prox_sgl(Om, Omp, L, X, 0.3, rho, latent=latent)
        np.testing.assert_array_max_ulp(th, th1, maxulp=1)


def test_block_norms_against_numpy():
    rng = np.random.default_rng(0)
    for Mblk in (1, 5, 6, 9):
        A = rng.standard_normal((2, Mblk * 3, Mblk * 3))
        n = kr.block_norms(A, Mblk)
        for i in range(3):
            for j in range(3):
                blk = A[:, i * Mblk:(i + 1) * Mblk, j * Mblk:(j + 1) * Mblk]
                np.testing.assert_allclose(n[:, i, j], np.linalg.norm(blk, axis=(1, 2)), rtol=1e-15)


@pytest.mark.parametrize("latent", [False, True])
def test_ext_references_against_oracle(latent):
    """the ext kernels' references reproduce one iteration of admm_oracle.ext_admm_mgl's Theta / Lambda / dual step"""
    from gglasso_b200.solver.ext_admm_solver import check_G
    rng = np.random.default_rng(5)
    pvec = [9, 4, 12, 7, 1]
    K, P = len(pvec), max(pvec)
    G = kr.ext_groups(pvec, rng)
    check_G(G, np.array(pvec))
    members = (G[0] >= 0).sum(axis=1)
    assert members.min() == 1 and members.max() > 1, "G must have singleton groups and shared ones"

    def padded(scale):
        A = np.zeros((K, P, P))
        for k, pk in enumerate(pvec):
            A[k, :pk, :pk] = _sym(rng, 1, pk, scale)[0]
        return A
    Om, X0, Lam, X1, Omp, Lamp = (padded(s) for s in (0.5, 0.1, 0.3, 0.1, 0.5, 0.3))
    L = padded(0.05) if latent else None
    lam1, lambda2, rho = np.array([0.1, 0.2, 0.05, 0.3, 0.1]), 0.07, 1.3
    th, C = kr.ext_theta(Om, L, X0, Lam, X1, lam1, rho)
    lam = kr.ext_lambda(th, X1, G, lambda2, rho)
    ref = orc.prox_2norm_G({k: th[k] + X1[k] for k in range(K)}, G, lambda2 / rho)
    x0, x1, parts = kr.ext_dual(X0, X1, Om, Omp, th, L, lam, Lamp, pvec)
    for k, pk in enumerate(pvec):
        s = (slice(0, pk), slice(0, pk))
        Lk = L[k][s] if latent else 0.0
        V = (Om[k][s] + Lk + X0[k][s] + Lam[k][s] - X1[k][s]) * 0.5
        np.testing.assert_allclose(th[k][s], orc.prox_od_1norm(V, lam1[k] / (2 * rho)), rtol=1e-15, atol=1e-16)
        np.testing.assert_allclose(C[k][s], th[k][s] - X0[k][s] - Om[k][s], rtol=1e-14, atol=1e-15)
        np.testing.assert_allclose(lam[k][s], ref[k][s], rtol=1e-14, atol=1e-16)
        np.testing.assert_allclose(x0[k][s], X0[k][s] + (Om[k][s] - th[k][s] + Lk), rtol=1e-14, atol=1e-15)
    nr = np.linalg.norm
    sl = lambda A, k: A[k, :pvec[k], :pvec[k]]  # noqa: E731
    tot = parts.sum(axis=0)
    Lz = L if latent else np.zeros_like(Om)
    r = math.sqrt(sum(nr(sl(Om, k) - sl(th, k) + sl(Lz, k)) ** 2 + nr(sl(lam, k) - sl(th, k)) ** 2 for k in range(K)))
    s = math.sqrt(sum(nr(sl(Om, k) - sl(Omp, k)) ** 2 + nr(sl(lam, k) - sl(Lamp, k)) ** 2 for k in range(K)))
    np.testing.assert_allclose([math.sqrt(tot[3]), math.sqrt(tot[4])], [r, s], rtol=1e-13)


def test_objective_reference_against_oracle():
    rng = np.random.default_rng(2)
    K, p = 4, 9
    Om, S, Th = _sym(rng, K, p), _sym(rng, K, p), _sym(rng, K, p)
    for reg, name in ((0, "GGL"), (1, "FGL")):
        ip, _, P = kr.objective_parts(Om, S, Th, 0.3, 0.2, reg)
        assert ip == pytest.approx(float(np.sum(Om * S)), rel=1e-14)
        assert P == pytest.approx(orc.P_val(Th, 0.3, 0.2, name), rel=1e-14)
