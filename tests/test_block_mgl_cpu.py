"""block_MGL without a GPU: the exact screen against its closed forms, the bitmask -> components conversion, the
decomposition theorem on the numpy restatement, and the argument checks of the public callables."""
import inspect

import numpy as np
import pytest

from gglasso_b200 import block_MGL, mgl_connected_components
from gglasso_b200.solver.admm_solver import _components_from_bitmask
from oracle import admm_oracle as orc
from oracle import screen_refs as sr


def _sym_entries(rng, K, p, scale):
    """(K,p,p) symmetric stack, unit diagonal, off-diagonal entries uniform in [-scale, scale]"""
    A = rng.uniform(-scale, scale, (K, p, p))
    A = np.triu(A, 1)
    A = A + A.transpose(0, 2, 1)
    A[:, np.arange(p), np.arange(p)] = 1.0
    return A


@pytest.mark.parametrize("K", [1, 3, 20])
def test_screen_ggl_closed_form(K):
    rng = np.random.default_rng(K)
    l1, l2 = 0.3, 0.28 * np.sqrt(K)                   # l2^2 near the mean of the sum: both outcomes occur
    S = _sym_entries(rng, K, 40, 0.9)
    A = sr.mgl_screen(S, l1, l2, "GGL")
    iu = np.triu_indices(40, 1)
    V = S[:, iu[0], iu[1]]
    sig = (np.maximum(np.abs(V) - l1, 0.0) ** 2).sum(axis=0)
    away = np.abs(sig - l2 ** 2) > 1e-9
    assert away.sum() > 700
    assert 0 < A[iu].sum() < len(iu[0])                 # both outcomes occur
    np.testing.assert_array_equal(A[iu][away], (sig > l2 ** 2)[away])


def test_screen_fgl_closed_form_K2():
    """Danaher, Wang & Witten (2014), Theorem 1: for K = 2 no edge iff |s1|, |s2| <= l1 + l2 and |s1 + s2| <= 2 l1"""
    rng = np.random.default_rng(7)
    l1, l2 = 0.2, 0.15
    S = _sym_entries(rng, 2, 60, 0.6)
    A = sr.mgl_screen(S, l1, l2, "FGL")
    iu = np.triu_indices(60, 1)
    s1, s2 = S[0][iu], S[1][iu]
    margins = np.stack([l1 + l2 - np.abs(s1), l1 + l2 - np.abs(s2), 2 * l1 - np.abs(s1 + s2)])
    away = (np.abs(margins) > 1e-9).all(axis=0)
    no_edge = (margins >= 0).all(axis=0)
    assert 0 < no_edge.sum() < len(s1)
    np.testing.assert_array_equal(A[iu][away], ~no_edge[away])


@pytest.mark.parametrize("p", [1, 31, 32, 33, 200])
def test_bitmask_components_match_scipy(p):
    rng = np.random.default_rng(p)
    for density in (0.0, 1.0 / max(p, 1), 3.0 / max(p, 1), 0.5):
        A = np.triu(rng.random((p, p)) < density, 1)
        words = sr.screen_words(A)
        assert words.shape == (p, (p + 31) // 32) and words.dtype == np.uint32
        numC, allC = _components_from_bitmask(words, p)
        n_ref, C_ref = sr.components(A)
        assert numC == n_ref == len(allC)
        for a, b in zip(allC, C_ref):
            np.testing.assert_array_equal(a, b)


def _blocky_cov(rng, K, sizes, N=2000):
    """K sample covariances of data with one strong common factor per block of ``sizes``: dense within blocks,
    small (sampling noise only) across blocks"""
    p = sum(sizes)
    out = []
    for _ in range(K):
        Z = rng.standard_normal((N, p))
        o = 0
        for n in sizes:
            Z[:, o:o + n] += 0.9 * rng.standard_normal((N, 1))
            o += n
        out.append(np.cov(Z, rowvar=False, bias=True))
    return np.stack(out)


# The two runs stop at the Boyd test with tol = rtol = 1e-10: primal and dual residuals of at most
# dim * 1e-10 + 1e-10 * |.| ~ 1e-7 (dim = K (p^2 + p) / 2 = 1395).  The objective is strongly convex on the level set
# (-log det has Hessian >= 1 / lambda_max(Theta)^2 ~ 0.1 here), so each iterate is within ~1e-6 of the solution;
# relative to |Theta| ~ 10 that is below 1e-6.
THEOREM_RTOL = 1e-6


@pytest.mark.parametrize("reg", ["GGL", "FGL"])
def test_block_decomposition_matches_full_problem_numpy(reg):
    rng = np.random.default_rng(11)
    K, sizes = 3, [1, 2, 4, 8, 15]
    S = _blocky_cov(rng, K, sizes)
    p = S.shape[1]
    l1, l2 = 0.2, 0.05
    Om0 = np.repeat(np.eye(p)[None], K, 0)
    kw = dict(tol=1e-10, rtol=1e-10, max_iter=20000)
    blk, comps = sr.block_mgl(S, l1, l2, reg, Om0, **kw)
    assert sum(len(C) > 1 for C in comps) >= 3, [len(C) for C in comps]
    full, info = orc.admm_mgl(S, l1, l2, reg, Om0, **kw)
    assert info["status"] == "optimal"
    np.testing.assert_array_equal(blk["Theta"] != 0, full["Theta"] != 0)
    err = np.linalg.norm(blk["Theta"] - full["Theta"]) / np.linalg.norm(full["Theta"])
    assert err < THEOREM_RTOL, err
    # the full problem's solution is zero off the components
    lab = np.empty(p, dtype=int)
    for c, C in enumerate(comps):
        lab[C] = c
    off = lab[:, None] != lab[None, :]
    assert np.all(full["Theta"][:, off] == 0)


def _args(K=3, p=5):
    S = np.repeat(np.eye(p)[None], K, 0)
    return S, S.copy()


def test_block_mgl_argument_checks():
    S, Om0 = _args()
    with pytest.raises(NotImplementedError):
        block_MGL(S, 0.1, 0.1, "GGL", Om0, latent=True)
    S91, Om91 = _args(K=91, p=3)
    with pytest.raises(NotImplementedError):
        block_MGL(S91, 0.1, 0.1, "GGL", Om91)
    with pytest.raises(NotImplementedError):
        mgl_connected_components(S91, 0.1, 0.1, "FGL")
    with pytest.raises(AssertionError):
        block_MGL(S, 0.1, 0.1, "GGL", Om0[:, :4, :4])
    with pytest.raises(AssertionError):
        block_MGL(S[:, :, :4], 0.1, 0.1, "GGL", Om0[:, :, :4])
    with pytest.raises(AssertionError):
        block_MGL(S, 0.1, 0.1, "SGL", Om0)
    with pytest.raises(AssertionError):
        block_MGL(S, 0.0, 0.1, "GGL", Om0)
    with pytest.raises(AssertionError):
        block_MGL(S, 0.1, -1.0, "FGL", Om0)
    with pytest.raises(AssertionError):
        block_MGL(S, 0.1, 0.1, "GGL", Om0, rho=0.0)
    params = inspect.signature(block_MGL).parameters
    assert "stopping_criterion" not in params and "measure" not in params
    with pytest.raises(TypeError):
        block_MGL(S, 0.1, 0.1, "GGL", Om0, stopping_criterion="kkt")
    with pytest.raises(TypeError):
        block_MGL(S, 0.1, 0.1, "GGL", Om0, measure=True)
