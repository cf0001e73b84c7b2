"""ADMM_MGL_batch on the GPU: the batch entry points of the three MGL kernels against the single-problem ones (bitwise),
every problem of a batch against its own ADMM_MGL call, the reference fixtures, errors and concurrent host threads."""
import contextlib
import ctypes
import io
import threading

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GUARD = 4096          # elements of sentinel before and after every output buffer
FILL = -7.25          # sentinel value


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _sym(rng, n, p, scale=1.0):
    A = rng.standard_normal((n, p, p)) * scale
    return A + A.transpose(0, 2, 1)


def _quiet(fn, *a, **kw):
    with contextlib.redirect_stdout(io.StringIO()) as buf:
        out = fn(*a, **kw)
    return out, buf.getvalue()


def _rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def _guarded(n, init=None):
    buf = torch.full((n + 2 * GUARD,), FILL, dtype=torch.float64, device="cuda")
    if init is not None:
        buf[GUARD:GUARD + n].copy_(init.reshape(-1))
    return buf


def _inner(buf):
    return buf[GUARD:-GUARD]


def _guards_intact(buf):
    return bool((buf[:GUARD] == FILL).all()) and bool((buf[-GUARD:] == FILL).all())


# --------------------------------------------------------------------------------------------
# kernel level: gg_*_batch(nprob = 3) vs the single-problem entry point on each slice
# --------------------------------------------------------------------------------------------
NPROB = 3
DONE = 1              # problem 1 is marked done


def _ctrl(rng):
    from gglasso_b200._lib import CTRL_STRIDE, C_RHO, C_XSCALE, C_DONE, C_LAM1, C_LAM2
    c = np.zeros((NPROB, CTRL_STRIDE))
    c[:, C_RHO] = [1.0, 0.7, 2.5]
    c[:, C_XSCALE] = [1.0, 1.0, 0.4]                   # problem 2 carries a pending dual rescale
    c[:, C_LAM1] = [0.05, 0.2, 0.11]
    c[:, C_LAM2] = [0.3, 0.01, 0.07]
    c[DONE, C_DONE] = 1.0
    return torch.from_numpy(c).cuda()


def _kernel_inputs(K, p, seed):
    rng = np.random.default_rng(seed)
    M = NPROB * K
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    Om = dev(_sym(rng, M, p, 0.3) + 2 * np.eye(p))
    return dict(Om=Om, Omp=dev(_sym(rng, M, p, 0.3)), L=dev(_sym(rng, M, p, 0.05)), X=dev(_sym(rng, M, p, 0.1)),
                S=dev(_sym(rng, M, p)), Th=dev(_sym(rng, M, p, 0.2)), nk=dev(rng.uniform(50, 200, M)),
                ctrl=_ctrl(rng))


def _run_kernel(kind, reg, K, p, inp, nprob, sl=slice(None), ctrl=None, latent=False):
    """one call of the kernel under test on matrices ``sl``; returns {output name: guarded buffer}"""
    from gglasso_b200 import _lib
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    regi = 0 if reg == "GGL" else 1
    ctrl = inp["ctrl"] if ctrl is None else ctrl
    g = {k: inp[k][sl].contiguous() for k in ("Om", "Omp", "L", "X", "S", "Th")}
    nk = inp["nk"][sl].contiguous()
    n = g["Om"].numel()
    if kind == "build_w_upper":
        out = {"X": _guarded(n, g["X"]), "W": _guarded(n)}
        args = (_p(g["Th"]), _p(_inner(out["X"])), _p(g["S"]), _p(nk), _p(ctrl), K, p)
        if nprob is None:
            rc = lib.gg_build_w_upper(*args, _p(_inner(out["W"])), st)
        else:
            rc = lib.gg_build_w_upper_batch(*args, nprob, _p(_inner(out["W"])), st)
        _lib.check(rc, kind)
        return out
    if kind == "prox_mgl_upper":
        nparts = lib.gg_mgl_upper_nparts(p)
        out = {"X": _guarded(n, g["X"]), "Theta": _guarded(n), "partials": _guarded((nprob or 1) * nparts * 5)}
        args = (_p(g["Om"]), _p(g["Omp"]), _p(_inner(out["X"])), _p(_inner(out["Theta"])), _p(ctrl), 1.0, 1.0, regi, K,
                p)
        if nprob is None:
            rc = lib.gg_prox_mgl_upper(*args, _p(_inner(out["partials"])), st)
        else:
            rc = lib.gg_prox_mgl_upper_batch(*args, nprob, _p(_inner(out["partials"])), st)
        _lib.check(rc, kind)
        return out
    nparts = lib.gg_mgl_ntile(p) ** 2
    out = {"X": _guarded(n, g["X"]), "Theta": _guarded(n)}
    if latent:
        out["C"] = _guarded(n)
    else:
        out["partials"] = _guarded((nprob or 1) * nparts * 5)
    args = (_p(g["Om"]), _p(g["Omp"]), _p(g["L"] if latent else None), _p(_inner(out["X"])), _p(_inner(out["Theta"])),
            _p(_inner(out["C"]) if latent else None), _p(ctrl), 1.0, 1.0, regi, K, p)
    parts = None if latent else _p(_inner(out["partials"]))
    if nprob is None:
        rc = lib.gg_prox_mgl(*args, parts, st)
    else:
        rc = lib.gg_prox_mgl_batch(*args, nprob, parts, st)
    _lib.check(rc, kind)
    return out


KERNELS = [("prox_mgl", False), ("prox_mgl", True), ("prox_mgl_upper", False), ("build_w_upper", False)]


@pytest.mark.parametrize("kind,latent", KERNELS)
@pytest.mark.parametrize("reg", ["GGL", "FGL"])
@pytest.mark.parametrize("K", [1, 3, 90])
@pytest.mark.parametrize("p", [7, 48, 50, 130])
def test_batch_kernels_match_single_problem_bitwise(kind, latent, reg, K, p):
    """nprob = 3 with a different rho, lambda1, lambda2 (and pending X scale) per problem and problem 1 marked done:
    each not-done problem's output slices and partial sums are bitwise those of the single-problem entry point on
    that slice, the done problem's slices come back untouched, and nothing is written outside the outputs."""
    if kind == "build_w_upper" and reg == "FGL":
        pytest.skip("build_w_upper has no regulariser")
    from gglasso_b200 import _lib
    lib = _lib.load()
    inp = _kernel_inputs(K, p, seed=1000 * K + p)
    batch = _run_kernel(kind, reg, K, p, inp, NPROB, latent=latent)
    pp = p * p
    nparts = lib.gg_mgl_upper_nparts(p) if kind == "prox_mgl_upper" else lib.gg_mgl_ntile(p) ** 2
    for q in range(NPROB):
        single = _run_kernel(kind, reg, K, p, inp, None, sl=slice(q * K, (q + 1) * K),
                             ctrl=inp["ctrl"][q:q + 1].contiguous(), latent=latent)
        torch.cuda.synchronize()
        for name, buf in batch.items():
            assert _guards_intact(buf), name
            per = nparts * 5 if name == "partials" else K * pp
            got = _inner(buf)[q * per:(q + 1) * per].cpu().numpy()
            if q == DONE:
                init = inp["X"][q * K:(q + 1) * K].reshape(-1).cpu().numpy() if name == "X" else np.full(per, FILL)
                assert np.array_equal(got, init), f"done problem: {name} was written"
            else:
                assert _guards_intact(single[name]), name
                ref = _inner(single[name]).cpu().numpy()
                assert np.array_equal(got, ref, equal_nan=True), f"problem {q}: {name} differs"
        if q != DONE and "partials" in batch:
            assert np.abs(_inner(batch["partials"])[q * nparts * 5:(q + 1) * nparts * 5].cpu().numpy()).sum() > 0


# --------------------------------------------------------------------------------------------
# solver level: every problem of a batch vs its own ADMM_MGL call
# --------------------------------------------------------------------------------------------
def _problem_set(K, p, B, seed, N=200):
    rng = np.random.default_rng(seed)
    Sig = []
    for k in range(K):
        A = rng.standard_normal((p, p)) * (rng.random((p, p)) < 3.0 / p)
        Sig.append(np.linalg.inv(np.eye(p) + 0.25 * (A + A.T) / max(1.0, np.abs(A + A.T).sum(1).max())))
    S = np.empty((B, K, p, p))
    for b in range(B):
        for k in range(K):
            Z = rng.multivariate_normal(np.zeros(p), Sig[k], size=N)
            S[b, k] = np.cov(Z, rowvar=False, bias=True)
    return S


def _assert_same(sol_b, info_b, sol, info, n_iter, latent, what):
    assert info_b["status"] == info["status"], what
    assert len(info_b["residual"]) == n_iter, what
    assert np.array_equal(sol_b["Theta"] != 0, sol["Theta"] != 0), what + ": sparsity pattern of Theta differs"
    for k in ("Omega", "Theta", "X") + (("L",) if latent else ()):
        assert np.linalg.norm(sol_b[k] - sol[k]) <= 1e-12 * max(np.linalg.norm(sol[k]), 1e-300), f"{what}: {k}"
    if not latent:
        assert not np.any(sol_b["L"])


VARIANTS = {
    "shared_S_shared_Omega0": dict(),
    "per_problem_S_and_Omega0_nsamples": dict(per_S=True, per_Om=True, n_samples=150),
    "rho_2.5_fixed_rho": dict(per_S=True, rho=2.5, update_rho=False),
    "per_problem_start_points": dict(per_Om=True, start=True),
}


def _solve_both(reg, latent, p, variant, K=3, B=5, seed=7, tol=1e-7, max_iter=1000):
    from gglasso_b200 import ADMM_MGL, ADMM_MGL_batch
    v = VARIANTS[variant]
    S_all = _problem_set(K, p, B, seed + p)
    S = S_all if v.get("per_S") else S_all[0]
    rng = np.random.default_rng(seed)
    l1 = np.round(rng.uniform(0.02, 0.12, B), 4)
    l2 = np.round(rng.uniform(0.005, 0.08, B), 4)
    eye = np.repeat(np.eye(p)[None], K, 0)
    Om0 = np.stack([eye * (1.0 + 0.1 * b) for b in range(B)]) if v.get("per_Om") else eye
    kw = dict(tol=tol, rtol=tol, max_iter=max_iter, rho=v.get("rho", 1.0), update_rho=v.get("update_rho", True),
              n_samples=v.get("n_samples"))
    Th0 = X0 = None
    if v.get("start"):
        Th0 = Om0 * 0.9
        X0 = np.stack([0.01 * b * eye for b in range(B)])
    mu = None
    if latent:
        mu = np.stack([np.full(K, 0.5 + 0.1 * b) for b in range(B)])
        kw.update(latent=True)
    res = ADMM_MGL_batch(S, l1, l2, reg, Om0, Theta_0=Th0, X_0=X0, mu1=mu, **kw)
    singles = []
    for b in range(B):
        a = dict(kw)
        if latent:
            a["mu1"] = mu[b]
        Sb = S[b] if S.ndim == 4 else S
        Ob = Om0[b] if Om0.ndim == 4 else Om0
        extra = {}
        if Th0 is not None:
            extra = dict(Theta_0=Th0[b], X_0=X0[b])
        (sol, info), out = _quiet(ADMM_MGL, Sb, float(l1[b]), float(l2[b]), reg, Ob, **extra, **a)
        n_iter = int(out.split("ADMM terminated after ")[1].split()[0])
        singles.append((sol, info, n_iter))
    return res, singles


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("p", [20, 50, 130])
@pytest.mark.parametrize("reg,latent", [("GGL", False), ("FGL", False), ("GGL", True), ("FGL", True)])
def test_batch_matches_single_solves(reg, latent, p, variant):
    if latent and variant != "shared_S_shared_Omega0" and p != 50:
        pytest.skip("latent: every variant at p = 50, the default variant at every p")
    if not latent and variant != "shared_S_shared_Omega0" and p == 20:
        pytest.skip("p = 20 runs the default variant")
    res, singles = _solve_both(reg, latent, p, variant)
    assert len(res) == len(singles)
    for b, ((sol_b, info_b), (sol, info, n_iter)) in enumerate(zip(res, singles)):
        assert set(sol_b) == {"Omega", "Theta", "L", "X"} and set(info_b) == {"status", "residual"}
        assert all(a.shape == sol[k].shape for k, a in sol_b.items())
        _assert_same(sol_b, info_b, sol, info, n_iter, latent, f"problem {b}")


@pytest.mark.parametrize("reg,p", [("GGL", 50), ("FGL", 130)])
def test_mixed_statuses_and_rho_path(reg, p):
    """max_iter between the problems' iteration counts: some problems converge, the others stop at max_iter; each has
    the status, iteration count and rho path of its own run_admm call."""
    from gglasso_b200 import ADMM_MGL_batch
    from gglasso_b200._engine import run_admm
    K, B = 3, 6
    S = _problem_set(K, p, B, 11)
    l1 = np.array([0.3, 0.01, 0.15, 0.005, 0.08, 0.2])
    l2 = np.array([0.1, 0.002, 0.05, 0.001, 0.02, 0.1])
    eye = np.repeat(np.eye(p)[None], K, 0)
    full = ADMM_MGL_batch(S, l1, l2, reg, eye, tol=1e-8, rtol=1e-8)
    n = sorted(len(i["residual"]) for _, i in full)
    assert n[0] < n[-1]
    cap = (n[0] + n[-1]) // 2
    res = ADMM_MGL_batch(S, l1, l2, reg, eye, tol=1e-8, rtol=1e-8, max_iter=cap)
    statuses = {i["status"] for _, i in res}
    assert "max iterations reached" in statuses and len(statuses) > 1
    stb, rb = run_admm("mgl", S.reshape(B * K, p, p), np.tile(eye, (B, 1, 1)), None, None, lambda1=l1, lambda2=l2,
                       reg=reg, tol=1e-8, rtol=1e-8, max_iter=cap, K=K)
    for b in range(B):
        st1, r1 = run_admm("mgl", S[b], eye, None, None, lambda1=float(l1[b]), lambda2=float(l2[b]), reg=reg, tol=1e-8,
                           rtol=1e-8, max_iter=cap)
        nb = int(rb["iters"][b])
        assert nb == int(r1["iters"][0]) == len(res[b][1]["residual"])
        assert rb["status"][b] == r1["status"][0] == res[b][1]["status"]
        assert np.array_equal(rb["hist"][b, :nb, 4], r1["hist"][0, :nb, 4]), f"problem {b}: rho path differs"
        np.testing.assert_allclose(rb["hist"][b, :nb, :4], r1["hist"][0, :nb, :4], rtol=1e-12, atol=0)


@pytest.mark.parametrize("name", ["mgl_ggl_K3_p50", "mgl_fgl_K3_p50"])
def test_batch_reproduces_reference_fixture(golden, name):
    """problem 0 of a batch with other lambdas around it reproduces the reference's fixture to the tolerances of the
    single-problem golden tests"""
    import ast
    from gglasso_b200 import ADMM_MGL_batch
    g = golden(name)
    S = g["S"]
    K, p, _ = S.shape
    kw = dict(ast.literal_eval(str(g["kw"])))
    l1, l2 = float(g["lambda1"]), float(g["lambda2"])
    res = ADMM_MGL_batch(S, [l1, 2 * l1, 0.5 * l1, l1], [l2, l2, 3 * l2, 0.3 * l2], str(g["reg"]),
                         np.repeat(np.eye(p)[None], K, 0), **kw)
    sol, info = res[0]
    n = g["traj"].shape[0]
    assert info["status"] == str(g["status"]) and len(info["residual"]) == n
    np.testing.assert_allclose(info["residual"], g["residual"], rtol=1e-7, atol=1e-12)
    assert _rel(sol["Theta"], g["Theta"]) < 1e-8
    assert np.array_equal(sol["Theta"] != 0, g["Theta"] != 0)
    for k in ("Omega", "X"):
        assert np.linalg.norm(sol[k] - g[k]) <= 1e-8 * max(1.0, np.linalg.norm(g[k])), k


def test_non_finite_problem_is_named():
    from gglasso_b200 import ADMM_MGL_batch, GGLassoB200Error
    K, p, B = 3, 30, 4
    S = _problem_set(K, p, B, 3)
    S[2, 1, 3, 3] = np.nan
    with pytest.raises(GGLassoB200Error, match=r"problem\(s\) \[2\]"):
        ADMM_MGL_batch(S, 0.05, 0.01, "GGL", np.repeat(np.eye(p)[None], K, 0))


def test_verbose_and_warnings_name_problems():
    from gglasso_b200 import ADMM_MGL_batch
    K, p, B = 2, 20, 3
    S = _problem_set(K, p, B, 5)
    eye = np.repeat(np.eye(p)[None], K, 0)
    res, out = _quiet(ADMM_MGL_batch, S, 0.05, 0.01, "FGL", eye)
    assert out == ""
    res, out = _quiet(ADMM_MGL_batch, S, 0.05, 0.01, "FGL", eye, verbose=True)
    lines = out.strip().splitlines()
    assert lines == [f"problem {b}: ADMM terminated after {len(i['residual'])} iterations with status: {i['status']}."
                     for b, (_, i) in enumerate(res)]


@pytest.mark.parametrize("p", [20, 130])
def test_per_problem_smallest_eigenvalue(p):
    """the post-loop PD check of the batch: per problem, a positive Gershgorin bound or the smallest eigenvalue"""
    from gglasso_b200._engine import AdmmState
    K, B = 3, 4
    rng = np.random.default_rng(p)
    A = np.stack([np.eye(p) * 3 + 0.1 * _sym(rng, 1, p)[0] for _ in range(B * K)])
    A[1 * K + 2] = _sym(rng, 1, p)[0]                  # problem 1: an indefinite matrix
    A[3 * K] = -np.eye(p)                               # problem 3: negative definite
    st = AdmmState(A, A, None, None, K, 1.0, 1, False)
    got = st.min_eig_per_problem(torch.from_numpy(A).cuda()).cpu().numpy()
    exact = np.linalg.eigvalsh(A).min(axis=1).reshape(B, K).min(axis=1)
    assert got.shape == (B,)
    assert np.all((got > 0) == (exact > 0))
    for b in range(B):
        if exact[b] <= 0:
            np.testing.assert_allclose(got[b], exact[b], rtol=1e-10, atol=1e-12)
        else:
            assert 0 < got[b] <= exact[b] * (1 + 1e-12)


def test_symmetry_assert():
    from gglasso_b200 import ADMM_MGL_batch
    K, p = 2, 10
    S = _problem_set(K, p, 2, 1)
    eye = np.repeat(np.eye(p)[None], K, 0)
    bad = S.copy()
    bad[1, 0, 0, 1] += 1.0
    with pytest.raises(AssertionError, match="symmetric"):
        ADMM_MGL_batch(bad, 0.1, 0.1, "GGL", eye)


def test_concurrent_threads_are_bitwise_single_thread():
    from gglasso_b200 import ADMM_MGL_batch
    K, p, B = 3, 60, 4
    jobs = [(_problem_set(K, p, B, s), "GGL" if s % 2 else "FGL") for s in (21, 22)]
    eye = np.repeat(np.eye(p)[None], K, 0)
    l1 = np.array([0.03, 0.05, 0.08, 0.1])
    alone = [ADMM_MGL_batch(S, l1, 0.02, reg, eye, tol=1e-7, rtol=1e-7) for S, reg in jobs]
    got, errs = [None, None], []

    def work(i):
        try:
            with torch.cuda.stream(torch.cuda.Stream()):
                S, reg = jobs[i]
                got[i] = ADMM_MGL_batch(S, l1, 0.02, reg, eye, tol=1e-7, rtol=1e-7)
        except Exception as ex:
            errs.append(ex)

    ts = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errs, errs
    for a, g in zip(alone, got):
        for (sa, ia), (sg, ig) in zip(a, g):
            assert ia["status"] == ig["status"] and np.array_equal(ia["residual"], ig["residual"])
            for k in sa:
                assert np.array_equal(sa[k], sg[k]), k
