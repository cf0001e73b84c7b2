"""block_MGL on the device: the screen kernel bit for bit against the oracle's prox, the ragged MGL prox against the
batched one and exact sums, and block_MGL against ADMM_MGL per component and on the full problem."""
import contextlib
import ctypes
import io

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from gglasso_b200 import ADMM_MGL, block_MGL, mgl_connected_components  # noqa: E402
from gglasso_b200 import _lib  # noqa: E402
from oracle import screen_refs as sr  # noqa: E402

pytestmark = pytest.mark.gpu

SENTINEL = 0x5A5A5A5A


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def dev_screen(S, l1, l2, reg, nk=None, pad=5):
    """gg_mgl_screen into a buffer with ``pad`` sentinel words on either side; checks the sentinels"""
    lib = _lib.load()
    K, p, _ = S.shape
    nw = (p + 31) // 32
    buf = torch.full((p * nw + 2 * pad,), SENTINEL, dtype=torch.int32, device="cuda")
    Sd = torch.from_numpy(np.ascontiguousarray(S)).cuda()
    nkd = None if nk is None else torch.from_numpy(np.asarray(nk, dtype=np.float64)).cuda()
    rc = lib.gg_mgl_screen(_ptr(Sd), _ptr(nkd), float(l1), float(l2), 0 if reg == "GGL" else 1, K, p,
                           ctypes.c_void_p(buf.data_ptr() + 4 * pad), torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    h = buf.cpu().numpy().view(np.uint32)
    assert np.all(h[:pad] == SENTINEL) and np.all(h[pad + p * nw:] == SENTINEL)
    return h[pad:pad + p * nw].reshape(p, nw)


def _sparse_sym(rng, K, p, scale=0.9, keep=0.5):
    """symmetric (K,p,p): about half of the entries are zero in every class, the others uniform in [-scale, scale]"""
    A = rng.uniform(-scale, scale, (K, p, p)) * (rng.random((p, p)) < keep)
    A = np.triu(A, 1)
    A = A + A.transpose(0, 2, 1)
    A[:, np.arange(p), np.arange(p)] = 1.0 + rng.random((K, p))
    return A


def _lams(reg, K):
    return (0.3, 0.28 * np.sqrt(K)) if reg == "GGL" else (0.3, 0.1)


@pytest.mark.parametrize("reg", ["GGL", "FGL"])
@pytest.mark.parametrize("K", [1, 2, 3, 5, 20, 90])
def test_screen_bitwise_vs_oracle(reg, K):
    rng = np.random.default_rng(1000 + K)
    l1, l2 = _lams(reg, K)
    for p in (2, 31, 32, 33, 100, 257):
        S = _sparse_sym(rng, K, p)
        A = sr.mgl_screen(S, l1, l2, reg)
        got = dev_screen(S, l1, l2, reg)
        np.testing.assert_array_equal(got, sr.screen_words(A), err_msg=f"p={p}")
        if p >= 31:
            assert 0 < A.sum() < p * (p - 1) // 2
        np.testing.assert_array_equal(dev_screen(S, l1, l2, reg), got)      # deterministic


@pytest.mark.parametrize("reg", ["GGL", "FGL"])
def test_screen_weights(reg):
    rng = np.random.default_rng(5)
    K, p = 3, 100
    nk = np.array([3.0, 0.5, 1.25])
    l1, l2 = _lams(reg, K)
    S = _sparse_sym(rng, K, p, scale=0.5)
    A1 = sr.mgl_screen(S, l1, l2, reg)
    Aw = sr.mgl_screen(S, l1, l2, reg, n_samples=nk)
    assert np.any(A1 != Aw)                                       # the weights flip edges
    np.testing.assert_array_equal(dev_screen(S, l1, l2, reg), sr.screen_words(A1))
    np.testing.assert_array_equal(dev_screen(S, l1, l2, reg, nk=nk), sr.screen_words(Aw))
    # int n_samples = the same weight for every class
    A7 = sr.mgl_screen(S, l1, l2, reg, n_samples=7)
    np.testing.assert_array_equal(dev_screen(S, l1, l2, reg, nk=np.full(K, 7.0)), sr.screen_words(A7))


@pytest.mark.parametrize("reg", ["GGL", "FGL"])
def test_screen_exact_ties(reg):
    """entries placed exactly on |s_k| = l1 and (GGL) sum_k (|s_k| - l1)_+^2 = l2^2, (FGL) Danaher's K = 2 bounds"""
    K, p = 3, 40
    l1, l2 = 0.5, 1.25
    rng = np.random.default_rng(9)
    S = _sparse_sym(rng, K, p, scale=2.0)
    ties = [(0.5, -0.5, 0.5),                       # every |s_k| = l1
            (1.25, 1.5, 0.0),                       # u = (0.75, 1.0, 0): |u| = 1.25 = l2 exactly
            (-1.25, 0.5, -1.5),                     # the same with signs and an entry on l1
            (1.75, 1.75, 1.75),                     # |s_k| = l1 + l2
            (1.75, -1.75, 0.5), (0.5, 1.0, 1.5)]
    rows = rng.permutation(p)
    for n, t in enumerate(ties * 3):                 # 18 entries on distinct node pairs
        i, j = rows[2 * n], rows[2 * n + 1]
        S[:, i, j] = S[:, j, i] = t
    A = sr.mgl_screen(S, l1, l2, reg)
    np.testing.assert_array_equal(dev_screen(S, l1, l2, reg), sr.screen_words(A))
    if reg == "GGL":
        i, j = 3, 17
        S[:, i, j] = S[:, j, i] = (1.25, 1.5, 0.0)
        assert not sr.mgl_screen(S, l1, l2, reg)[min(i, j), max(i, j)]
        assert not (dev_screen(S, l1, l2, reg)[min(i, j), max(i, j) // 32] >> (max(i, j) % 32)) & 1


# ---- ragged prox --------------------------------------------------------------------------------------------------
def _ragged_stacks(rng, K, p, pvec):
    B = len(pvec)
    Om = np.broadcast_to(np.eye(p), (B, K, p, p)).copy()
    Omp, X = Om.copy(), np.zeros((B, K, p, p))
    for q, n in enumerate(pvec):
        for A, s in ((Om, 0.3), (Omp, 0.3), (X, 0.2)):
            R = rng.uniform(-s, s, (K, n, n))
            R = R + R.transpose(0, 2, 1)
            if A is not X:
                R[:, np.arange(n), np.arange(n)] += 2.0
            A[q, :, :n, :n] = R
    return [a.reshape(B * K, p, p) for a in (Om, Omp, X)]


def _ragged_call(fn, Om, Omp, X, Th, ctrl, parts, reg, K, p, B, pvec_d=None):
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    if fn == "ragged":
        rc = lib.gg_prox_mgl_ragged(_ptr(Om), _ptr(Omp), _ptr(X), _ptr(Th), _ptr(ctrl), 0.1, 0.05, reg, K, p, B,
                                    _ptr(pvec_d), _ptr(parts), st)
    else:
        rc = lib.gg_prox_mgl_batch(_ptr(Om), _ptr(Omp), None, _ptr(X), _ptr(Th), None, _ptr(ctrl), 0.1, 0.05, reg, K,
                                   p, B, _ptr(parts), st)
    assert rc == 0
    torch.cuda.synchronize()


@pytest.mark.parametrize("reg", [0, 1])
def test_prox_mgl_ragged(reg):
    rng = np.random.default_rng(3 + reg)
    K, p, pvec = 3, 40, [40, 23, 7, 1]
    B = len(pvec)
    Om, Omp, X = _ragged_stacks(rng, K, p, pvec)
    rho = np.array([1.0, 2.0, 0.5, 4.0])
    lam1, lam2 = 0.3, 0.2
    ctrl = np.zeros((B, _lib.CTRL_STRIDE))
    ctrl[:, _lib.C_RHO], ctrl[:, _lib.C_XSCALE] = rho, 1.0
    ctrl[:, _lib.C_LAM1], ctrl[:, _lib.C_LAM2] = lam1, lam2
    nt = _lib.load().gg_mgl_ntile(p)
    d = {n: torch.from_numpy(a).cuda() for n, a in (("Om", Om), ("Omp", Omp), ("ctrl", ctrl))}
    pvec_d = torch.tensor(pvec, dtype=torch.int32, device="cuda")
    out = {}
    for fn in ("batch", "ragged"):
        Xd, Th = torch.from_numpy(X).cuda(), torch.zeros_like(d["Om"])
        parts = torch.zeros((B, nt * nt, _lib.NPART), dtype=torch.float64, device="cuda")
        _ragged_call(fn, d["Om"], d["Omp"], Xd, Th, d["ctrl"], parts, reg, K, p, B, pvec_d)
        out[fn] = (Th.cpu().numpy(), Xd.cpu().numpy(), parts.cpu().numpy().sum(axis=1))
    np.testing.assert_array_equal(out["ragged"][0], out["batch"][0])
    np.testing.assert_array_equal(out["ragged"][1], out["batch"][1])
    Th_ref, X_ref, parts_ref = sr.prox_mgl_ragged(Om, Omp, X, lam1, lam2, ["GGL", "FGL"][reg], rho, K, pvec)
    np.testing.assert_allclose(out["ragged"][0], Th_ref, rtol=0, atol=1e-15)
    np.testing.assert_allclose(out["ragged"][1], X_ref, rtol=0, atol=1e-15)
    np.testing.assert_allclose(out["ragged"][2], parts_ref, rtol=1e-13, atol=0)
    # the batched kernel counts the padding; the ragged one does not
    assert np.all(out["batch"][2][1:, 0] > parts_ref[1:, 0])

    # a problem marked done is left untouched: Theta, X and its partial sums
    ctrl_done = ctrl.copy()
    ctrl_done[1, _lib.C_DONE] = 1.0
    Xd = torch.from_numpy(X).cuda()
    Th = torch.full_like(d["Om"], 7.0)
    parts = torch.full((B, nt * nt, _lib.NPART), -1.0, dtype=torch.float64, device="cuda")
    _ragged_call("ragged", d["Om"], d["Omp"], Xd, Th, torch.from_numpy(ctrl_done).cuda(), parts, reg, K, p, B, pvec_d)
    s = slice(K, 2 * K)
    assert np.all(Th.cpu().numpy()[s] == 7.0)
    np.testing.assert_array_equal(Xd.cpu().numpy()[s], X[s])
    assert np.all(parts.cpu().numpy()[1] == -1.0)
    np.testing.assert_array_equal(Th.cpu().numpy()[:K], out["ragged"][0][:K])


# ---- block_MGL ----------------------------------------------------------------------------------------------------
SIZES = [1, 1, 2, 3, 5, 9, 17, 33, 70, 130, 200]        # singletons, buckets 2 .. 160, one component above 160


def _block_problem(K, sizes, seed=0, N=1000):
    """(K,p,p) block-diagonal covariances (a strong common factor per block, exact zeros across blocks) with the
    nodes randomly permuted; returns S and the components as index arrays"""
    rng = np.random.default_rng(seed)
    p = sum(sizes)
    S = np.zeros((K, p, p))
    for k in range(K):
        o = 0
        for n in sizes:
            Z = rng.standard_normal((N, n)) + 0.9 * rng.standard_normal((N, 1))
            S[k, o:o + n, o:o + n] = np.cov(Z, rowvar=False, bias=True).reshape(n, n)
            o += n
    perm = rng.permutation(p)
    S = np.ascontiguousarray(S[:, perm][:, :, perm])
    inv = np.argsort(perm)
    comps, o = [], 0
    for n in sizes:
        comps.append(np.sort(inv[o:o + n]))
        o += n
    comps.sort(key=lambda C: C[0])
    return S, comps


def _quiet(fn, *a, **kw):
    with contextlib.redirect_stdout(io.StringIO()) as buf:
        r = fn(*a, **kw)
    return r, buf.getvalue()


@pytest.mark.parametrize("reg,n_samples", [("GGL", None), ("FGL", np.array([2.0, 1.0, 1.5]))])
def test_block_mgl_per_component(reg, n_samples):
    K = 3
    S, comps = _block_problem(K, SIZES)
    p = S.shape[1]
    l1, l2 = 0.2, 0.05
    numC, allC = mgl_connected_components(S, l1, l2, reg, n_samples=n_samples)
    assert numC == len(comps)
    for a, b in zip(allC, comps):
        np.testing.assert_array_equal(a, b)
    Om0 = np.repeat(np.eye(p)[None], K, 0)
    kw = dict(tol=1e-10, rtol=1e-10, max_iter=5000)
    (sol, info), printed = _quiet(block_MGL, S, l1, l2, reg, Om0, n_samples=n_samples, **kw)
    assert printed == ""
    assert info["status"] == "optimal"
    assert len(info["components"]) == numC
    for ci, C in enumerate(comps):
        ix = (slice(None), C[:, None], C[None, :])
        if len(C) == 1:
            np.testing.assert_array_equal(sol["Theta"][ix], 1 / S[ix])
            assert info["component_iters"][ci] == 0
            continue
        (ref, rinfo), _ = _quiet(ADMM_MGL, np.ascontiguousarray(S[ix]), l1, l2, reg,
                                 np.ascontiguousarray(Om0[ix]), n_samples=n_samples, **kw)
        assert info["component_status"][ci] == rinfo["status"], (ci, len(C))
        err = np.linalg.norm(sol["Theta"][ix] - ref["Theta"]) / np.linalg.norm(ref["Theta"])
        assert err < 1e-9, (ci, len(C), err)
        np.testing.assert_array_equal(sol["Theta"][ix] != 0, ref["Theta"] != 0)
        assert info["component_iters"][ci] > 0
    assert np.all(sol["L"] == 0)
    (_, info_v), printed = _quiet(block_MGL, S, l1, l2, reg, Om0, n_samples=n_samples, verbose=True, max_iter=50)
    assert len(printed.splitlines()) == sum(len(C) > 1 for C in comps)


# Both runs stop at the Boyd test with tol = rtol = 1e-10, residuals of at most dim * 1e-10 + 1e-10 |.| ~ 3e-5 for the
# full problem (dim = K (p^2 + p) / 2 ~ 3.3e5); with the strong convexity of -log det on the level set (Hessian
# >= 1 / lambda_max(Theta)^2) each solution is within ~1e-5 of the optimum, ~1e-6 relative to |Theta| ~ 30.
FULL_RTOL = 1e-5


@pytest.mark.parametrize("reg", ["GGL", "FGL"])
def test_block_mgl_matches_full_problem(reg):
    K = 3
    S, comps = _block_problem(K, SIZES, seed=1)
    p = S.shape[1]
    l1, l2 = 0.2, 0.05
    Om0 = np.repeat(np.eye(p)[None], K, 0)
    kw = dict(tol=1e-10, rtol=1e-10, max_iter=5000)
    (sol, info), _ = _quiet(block_MGL, S, l1, l2, reg, Om0, **kw)
    (full, finfo), _ = _quiet(ADMM_MGL, S, l1, l2, reg, Om0, **kw)
    assert info["status"] == finfo["status"] == "optimal"
    np.testing.assert_array_equal(sol["Theta"] != 0, full["Theta"] != 0)
    err = np.linalg.norm(sol["Theta"] - full["Theta"]) / np.linalg.norm(full["Theta"])
    assert err < FULL_RTOL, err
    lab = np.empty(p, dtype=int)
    for c, C in enumerate(comps):
        lab[C] = c
    off = lab[:, None] != lab[None, :]
    assert np.all(full["Theta"][:, off] == 0)
    assert np.all(sol["Theta"][:, off] == 0)


@pytest.mark.parametrize("reg", ["GGL", "FGL"])
def test_block_mgl_single_component(reg):
    rng = np.random.default_rng(2)
    K, p = 3, 60
    S = np.stack([np.cov(rng.standard_normal((p, 300)), bias=True) for _ in range(K)])
    l1, l2 = 0.01, 0.005
    numC, _ = mgl_connected_components(S, l1, l2, reg)
    assert numC == 1
    Om0 = np.repeat(np.eye(p)[None], K, 0)
    (sol, info), _ = _quiet(block_MGL, S, l1, l2, reg, Om0, tol=1e-8, rtol=1e-8)
    (ref, rinfo), _ = _quiet(ADMM_MGL, S, l1, l2, reg, Om0, tol=1e-8, rtol=1e-8)
    assert info["status"] == rinfo["status"]
    np.testing.assert_array_equal(sol["Theta"] != 0, ref["Theta"] != 0)
    np.testing.assert_allclose(sol["Theta"], ref["Theta"], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(sol["X"], ref["X"], rtol=1e-12, atol=1e-14)
