"""stability_selection on the GPU: the three kernels against numpy (with sentinel regions around every output), the
driver against ADMM_MGL_batch / ADMM_SGL with numpy counting, chunking, reproducibility and the refit."""
import contextlib
import ctypes
import io

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GUARD = 4096          # elements of sentinel before and after every output buffer
FILL = -7.25          # sentinel value (doubles)
IFILL = -123457       # sentinel value (int32)


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _guarded(n, dtype=torch.float64, init=None):
    buf = torch.full((n + 2 * GUARD,), FILL if dtype == torch.float64 else IFILL, dtype=dtype, device="cuda")
    if init is not None:
        buf[GUARD:GUARD + n].copy_(init.reshape(-1))
    return buf


def _inner(buf):
    return buf[GUARD:-GUARD]


def _guards_intact(buf):
    f = FILL if buf.dtype == torch.float64 else IFILL
    return bool((buf[:GUARD] == f).all()) and bool((buf[-GUARD:] == f).all())


def _quiet(fn, *a, **kw):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **kw)


def _samples(K, p, n, seed, kind="group"):
    """Gaussian draws from the generator's sparse precision matrices: K classes of n (or n[k]) samples"""
    from gglasso_b200 import datagen
    Th = datagen.instance_precisions(K, p, n_blocks=next(b for b in (10, 5, 2, 1) if p % b == 0 and p // b >= 2),
                                     seed=seed, kind=kind)
    rng = np.random.default_rng(seed + 7)
    ns = [n] * K if np.ndim(n) == 0 else list(n)
    out = []
    for k in range(K):
        Lc = np.linalg.cholesky(Th[k])
        out.append(np.linalg.solve(Lc.T, rng.standard_normal((p, ns[k]))).T.copy())
    return out


# --------------------------------------------------------------------------------------------
# gg_subsample_cov against np.cov(..., bias=True)
# --------------------------------------------------------------------------------------------
COV_CASES = [(7, [2]), (7, [3, 17, 2]), (48, [17]), (48, [64, 3, 150]), (50, [64]), (50, [2, 316, 17]),
             (130, [150]), (130, [3, 64, 316]), (500, [316]), (500, [150, 17, 64])]


def _run_cov(X, rowoff, idx, boff, nsub, K, p, scale):
    from gglasso_b200 import _lib
    lib = _lib.load()
    S = _guarded(nsub * K * p * p)
    mean = _guarded(nsub * K * p)
    zc = _guarded(nsub * K, torch.int32)
    _lib.check(lib.gg_subsample_cov(_p(X), _p(rowoff), _p(idx), _p(boff), nsub, K, p, int(scale), _p(_inner(mean)),
                                    _p(_inner(S)), _p(_inner(zc)), torch.cuda.current_stream().cuda_stream),
               "gg_subsample_cov")
    torch.cuda.synchronize()
    assert _guards_intact(S) and _guards_intact(mean) and _guards_intact(zc)
    return _inner(S).reshape(nsub, K, p, p).cpu().numpy(), _inner(zc).cpu().numpy()


@pytest.mark.parametrize("scale", [False, True])
@pytest.mark.parametrize("p, b", COV_CASES)
def test_subsample_cov_matches_numpy(p, b, scale):
    from gglasso_b200 import stability as stars
    rng = np.random.default_rng(p * 7 + len(b))
    K, nsub = len(b), 3
    n = [bk + 11 for bk in b]
    classes = [rng.standard_normal((n[k], p)) * rng.uniform(0.5, 3.0, p) + rng.uniform(-5, 5, p) for k in range(K)]
    idx = stars.draw_indices(n, b, nsub, seed=p)
    res = stars._Resident(classes, idx, torch.device("cuda"))
    S, zc = _run_cov(res.X, res.rowoff, res.idx, res.boff, nsub, K, p, scale)
    assert np.all(zc >= p)
    for s in range(nsub):
        for k in range(K):
            ref = stars.sample_covariance(classes[k][idx[k][s]], scale)
            err = np.max(np.abs(S[s, k] - ref)) / np.max(np.abs(ref))
            assert err <= 1e-13, (s, k, err)
            assert np.array_equal(S[s, k], S[s, k].T)
            if scale:
                assert np.max(np.abs(np.diag(S[s, k]) - 1.0)) <= 1e-15
    S2, _ = _run_cov(res.X, res.rowoff, res.idx, res.boff, nsub, K, p, scale)
    assert np.array_equal(S, S2)
    # the driver's private helper forms the same covariances
    assert np.array_equal(stars._device_covariances(classes, idx, scale).cpu().numpy(), S)


def test_zero_variance_column_raises():
    from gglasso_b200 import stability as stars
    from gglasso_b200 import stability_selection
    rng = np.random.default_rng(5)
    p = 9
    classes = [rng.standard_normal((40, p)) for _ in range(2)]
    classes[1][:20, 4] = 2.5                       # constant on the first 20 rows of class 1
    idx = [np.array([[0, 1, 2, 3], [5, 9, 30, 31]]), np.array([[20, 21, 22, 23], [1, 2, 3, 4]])]
    S = stars._device_covariances(classes, idx, False)     # unscaled: no error
    assert torch.isfinite(S).all()
    with pytest.raises(ValueError, match=r"subsample 1, class 1: column 4"):
        stars._device_covariances(classes, idx, True)
    full = [rng.standard_normal((40, p))]
    full[0][:, 2] = -1.0
    with pytest.raises(ValueError, match="column 2"):
        stability_selection(full[0], [0.3], n_subsamples=2, refit=False)
    with pytest.raises(ValueError, match="column 2"):
        stability_selection(full[0], [0.3], n_subsamples=2, refit=True)


# --------------------------------------------------------------------------------------------
# gg_edge_count / gg_stars_instability against numpy
# --------------------------------------------------------------------------------------------
def _np_instability(counts, B):
    """exact reference: sum_{i<j} 2 theta (1 - theta) / C(p,2) as a rational number, rounded once.  (Summing the
    rounded terms 2 theta (1 - theta) in floating point is off by up to ~6e-14 relative at these counts: the rounding
    of theta = c/B has the same sign in every term of one value of c.)"""
    from fractions import Fraction
    p = counts.shape[-1]
    iu = np.triu_indices(p, 1)
    c = counts[..., iu[0], iu[1]].astype(np.int64)
    sv = (c * (B - c)).sum(-1)
    D = np.vectorize(lambda v: float(Fraction(2 * int(v), B * B * p * (p - 1) // 2)))(sv)
    return D, c.sum(-1) / B


@pytest.mark.parametrize("p, L, K", [(7, 3, 2), (37, 4, 3), (130, 2, 1)])
def test_edge_count_and_instability_match_numpy(p, L, K):
    from gglasso_b200 import _lib
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(p)
    B = 5
    Th = rng.standard_normal((B, L, K, p, p)) * (rng.random((B, L, K, p, p)) < 0.3)
    Th[..., np.arange(p), np.arange(p)] = 1.0
    Th[0, 0, 0, 0, 1] = -0.0                       # a negative zero is not an edge
    Thd = torch.from_numpy(Th.reshape(-1, p, p)).cuda()
    iu = np.triu_indices(p, 1)
    ref = np.zeros((L, K, p, p), dtype=np.int64)
    ref[..., iu[0], iu[1]] = (Th[..., iu[0], iu[1]] != 0).sum(0)

    def counts_after(chunks):
        cnt = _guarded(L * K * p * p, torch.int32, torch.zeros(L * K * p * p, dtype=torch.int32))
        s0 = 0
        for ns in chunks:
            part = Thd[s0 * L * K:(s0 + ns) * L * K]
            _lib.check(lib.gg_edge_count(_p(part), ns, L, K, p, _p(_inner(cnt)), st), "gg_edge_count")
            s0 += ns
        torch.cuda.synchronize()
        assert _guards_intact(cnt)
        return cnt

    one = counts_after([B])
    two = counts_after([2, 3])
    assert torch.equal(one, two)
    C = _inner(one).reshape(L, K, p, p).cpu().numpy()
    assert np.array_equal(C, ref)
    out = _guarded(L * K * 2)
    _lib.check(lib.gg_stars_instability(_p(_inner(one)), L, K, p, B, _p(_inner(out)), st), "gg_stars_instability")
    torch.cuda.synchronize()
    assert _guards_intact(out)
    o = _inner(out).reshape(L, K, 2).cpu().numpy()
    D, E = _np_instability(ref, B)
    assert np.all(np.abs(o[..., 0] - D) <= 1e-14 * np.maximum(np.abs(D), 1e-300))
    assert np.all(np.abs(o[..., 1] - E) <= 1e-14 * np.maximum(np.abs(E), 1e-300))
    out2 = torch.empty(L * K * 2, dtype=torch.float64, device="cuda")
    _lib.check(lib.gg_stars_instability(_p(_inner(two)), L, K, p, B, _p(out2), st), "gg_stars_instability")
    assert torch.equal(out2, _inner(out))


# --------------------------------------------------------------------------------------------
# end to end against ADMM_MGL_batch / ADMM_SGL and numpy counting
# --------------------------------------------------------------------------------------------
B_SUB = 6
LAMS = np.array([0.08, 0.5, 0.15, 0.3])            # unsorted on purpose
TOL = dict(tol=1e-7, rtol=1e-7, max_iter=1000)


def _counts_np(Thetas):
    """Thetas: (B, L, K, p, p) -> counts (L, K, p, p) over i < j"""
    p = Thetas.shape[-1]
    iu = np.triu_indices(p, 1)
    C = np.zeros(Thetas.shape[1:], dtype=np.int64)
    C[..., iu[0], iu[1]] = (Thetas[..., iu[0], iu[1]] != 0).sum(0)
    return C


def _check_against_counts(res, C, B):
    L = C.shape[0]
    D_k, E = _np_instability(C, B)
    D = D_k.mean(axis=1)
    assert np.all(np.abs(res["instability"] - D) <= 1e-14 * np.maximum(np.abs(D), 1e-300))
    assert np.allclose(res["mean_edges"], E, rtol=1e-14, atol=0)
    from gglasso_b200 import stability as stars
    assert res["best_index"] == stars.select(D, 0.05)[1]
    Cb = C[res["best_index"]]
    F = (Cb + Cb.transpose(0, 2, 1)) / B
    ef = res["edge_frequency"]
    ef = ef[None] if ef.ndim == 2 else ef
    assert np.array_equal(ef * B, F * B)
    assert np.array_equal(ef, ef.transpose(0, 2, 1)) and np.all(np.diagonal(ef, axis1=1, axis2=2) == 0)
    assert res["n_not_optimal"].shape == (L,) and not res["n_not_optimal"].any()


@pytest.mark.parametrize("reg", ["GGL", "FGL"])
@pytest.mark.parametrize("K, p", [(3, 50), (5, 100)])
def test_mgl_end_to_end_against_batch_and_numpy(K, p, reg):
    from gglasso_b200 import ADMM_MGL_batch, stability_selection
    from gglasso_b200 import stability as stars
    data = _samples(K, p, 200, seed=K + p, kind="group" if reg == "GGL" else "fused")
    res = stability_selection(data, LAMS, lambda2=0.02, reg=reg, n_subsamples=B_SUB, refit=False, **TOL)
    lam = res["lambda1"]
    assert np.array_equal(lam, np.sort(LAMS)[::-1]) and res["lambda2"] == 0.02
    assert [ix.shape for ix in res["indices"]] == [(B_SUB, 141)] * K
    S = stars._device_covariances(data, res["indices"], True).cpu().numpy()
    L = len(lam)
    out = ADMM_MGL_batch(np.repeat(S, L, axis=0), np.tile(lam, B_SUB), 0.02, reg,
                         np.repeat(np.eye(p)[None], K, 0), **TOL)
    Th = np.stack([sol["Theta"] for sol, _ in out]).reshape(B_SUB, L, K, p, p)
    _check_against_counts(res, _counts_np(Th), B_SUB)


@pytest.mark.parametrize("p", [50, 130])
def test_sgl_end_to_end_against_admm_sgl_and_numpy(p):
    from gglasso_b200 import ADMM_SGL, stability_selection
    from gglasso_b200 import stability as stars
    data = _samples(1, p, 300, seed=p)[0]
    res = stability_selection(data, LAMS, n_subsamples=B_SUB, refit=False, **TOL)
    lam, L = res["lambda1"], len(LAMS)
    assert res["lambda2"] is None and res["edge_frequency"].shape == (p, p)
    Sd = stars._device_covariances([data], res["indices"], True).reshape(B_SUB, p, p)
    st, _ = stars._solve_chunk(Sd, 1, lam, None, None, **TOL)
    Tb = st.Theta.reshape(B_SUB, L, p, p).cpu().numpy()
    S = Sd.cpu().numpy()
    Th = np.empty((B_SUB, L, 1, p, p))
    for s in range(B_SUB):
        for l in range(L):
            sol, _ = _quiet(ADMM_SGL, S[s], lam[l], np.eye(p), **TOL)
            Th[s, l, 0] = sol["Theta"]
            rel = np.linalg.norm(Tb[s, l] - sol["Theta"]) / np.linalg.norm(sol["Theta"])
            assert rel <= 1e-10, (s, l, rel)
    C = _counts_np(Th)
    assert np.array_equal(C, _counts_np(Tb[:, :, None]))
    _check_against_counts(res, C, B_SUB)


def _same(r1, r2):
    for key in ("lambda1", "instability", "instability_bar", "instability_per_class", "mean_edges", "edge_frequency",
                "n_not_optimal"):
        assert np.array_equal(r1[key], r2[key]), key
    assert r1["best_index"] == r2["best_index"] and r1["best_lambda1"] == r2["best_lambda1"]
    assert all(np.array_equal(a, b) for a, b in zip(r1["indices"], r2["indices"]))


@pytest.mark.parametrize("case", ["GGL", "FGL", "SGL50", "SGL130"])
def test_chunking_and_reproducibility(case):
    from gglasso_b200 import _lib, stability_selection
    if case.startswith("SGL"):
        p = int(case[3:])
        data, kw = _samples(1, p, 300, seed=3)[0], {}
    else:
        p = 50
        data, kw = _samples(3, p, [150, 200, 170], seed=4), dict(reg=case, lambda2=0.02)
    full = stability_selection(data, LAMS, n_subsamples=B_SUB, refit=False, **kw, **TOL)
    again = stability_selection(data, LAMS, n_subsamples=B_SUB, refit=False, **kw, **TOL)
    _same(full, again)
    one = stability_selection(data, LAMS, n_subsamples=B_SUB, refit=False, max_batch=len(LAMS), **kw, **TOL)
    two = stability_selection(data, LAMS, n_subsamples=B_SUB, refit=False, max_batch=2 * len(LAMS) + 1, **kw, **TOL)
    lib = _lib.load()
    if case.startswith("SGL") and lib.gg_sgl_nparts(p, B_SUB * len(LAMS)) != lib.gg_sgl_nparts(p, len(LAMS)):
        # the SGL residual sums are split over a number of CTAs that depends on the batch (DESIGN.md section 11)
        for r in (one, two):
            assert np.array_equal(r["edge_frequency"], full["edge_frequency"])
            assert np.allclose(r["instability"], full["instability"], rtol=1e-14, atol=0)
    else:
        _same(full, one)
        _same(full, two)


@pytest.mark.parametrize("case", ["FGL", "SGL"])
def test_refit_equals_direct_call(case):
    from gglasso_b200 import ADMM_MGL, ADMM_SGL, stability_selection
    from gglasso_b200 import stability as stars
    if case == "SGL":
        p = 50
        data = _samples(1, p, 250, seed=9)[0]
        res = stability_selection(data, LAMS, n_subsamples=4, **TOL)
        S = stars.sample_covariance(data, True)
        sol, info = _quiet(ADMM_SGL, S, res["best_lambda1"], np.eye(p), **TOL)
    else:
        K, p = 3, 50
        data = _samples(K, p, 200, seed=10, kind="fused")
        res = stability_selection(data, LAMS, lambda2=0.02, reg="FGL", n_subsamples=4, **TOL)
        S = np.stack([stars.sample_covariance(x, True) for x in data])
        sol, info = _quiet(ADMM_MGL, S, res["best_lambda1"], 0.02, "FGL", np.repeat(np.eye(p)[None], K, 0), **TOL)
    assert res["info"] == info
    assert sol.keys() == res["sol"].keys()
    for key in sol:
        assert np.array_equal(sol[key], res["sol"][key]), key


def test_max_iter_warning_names_problems():
    from gglasso_b200 import stability_selection
    data = _samples(1, 20, 100, seed=12)[0]
    with pytest.warns(UserWarning, match="reached max_iter"):
        res = stability_selection(data, [0.05, 0.2], n_subsamples=3, refit=False, max_iter=2)
    assert np.array_equal(res["n_not_optimal"], [3, 3])
