"""PPDNA on the GPU (gg_ppdna.cu, gglasso_b200/_ppdna.py): the Hessian product and the prox kernel against the numpy
restatement (oracle/ppdna_oracle.py) and gg_prox_mgl, and the public PPDNA / warmPPDNA against ADMM_MGL run to a tight
KKT tolerance."""
import contextlib
import ctypes
import inspect
import io
import os
import threading

import numpy as np
import pytest

torch = pytest.importorskip("torch")
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

from oracle import admm_oracle as orc  # noqa: E402
from oracle import ppdna_oracle as po  # noqa: E402


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _sym(rng, K, p, scale=1.0):
    A = rng.standard_normal((K, p, p)) * scale
    return A + A.transpose(0, 2, 1)


class _Dev:
    """device buffers of one point, filled by the kernels under test from host-given Vt / eigenvalues / V"""

    def __init__(self, Vt, D, V, sigma, l1, l2, reg, Om_t=None, Th_t=None, X=None, S=None):
        from gglasso_b200 import _lib
        self.lib = lib = _lib.load()
        K, p, _ = Vt.shape
        dev = torch.device("cuda")
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
        e = lambda: torch.zeros((K, p, p), dtype=torch.float64, device=dev)  # noqa: E731
        self.K, self.p, self.sigma, self.l1, self.reg = K, p, sigma, l1, reg
        self.regi = 0 if reg == "GGL" else 1
        self.st = torch.cuda.current_stream().cuda_stream
        self.Vt, self.D, self.V = t(Vt), t(D), t(V)
        self.Q, self.Omega, self.Theta, self.G, self.Y, self.Z = e(), e(), e(), e(), e(), e()
        self.phi = torch.zeros((K, p), dtype=torch.float64, device=dev)
        self.logdet = torch.zeros(K, dtype=torch.float64, device=dev)
        self.code = torch.zeros((K, p, p), dtype=torch.uint8, device=dev)
        self.jscale = torch.zeros((p, p), dtype=torch.float64, device=dev)
        self.parts = torch.zeros((lib.gg_ppdna_nparts(p), 6), dtype=torch.float64, device=dev)
        _lib.check(lib.gg_ppdna_spectral(_p(self.Vt), _p(self.D), sigma, K, p, _p(self.Q), _p(self.phi),
                                         _p(self.logdet), _p(self.Omega), None, self.st), "gg_ppdna_spectral")
        Om_t, Th_t, X, S = (e() if a is None else t(a) for a in (Om_t, Th_t, X, S))
        _lib.check(lib.gg_ppdna_prox(_p(self.V), _p(self.Omega), _p(Om_t), _p(Th_t), _p(X), _p(S), l1, l2, sigma,
                                     self.regi, K, p, _p(self.Theta), _p(self.G), _p(self.code), _p(self.jscale),
                                     _p(self.parts), None, self.st), "gg_ppdna_prox")

    def hess(self, Dm):
        from gglasso_b200 import _lib
        Din = torch.from_numpy(np.ascontiguousarray(Dm)).cuda()
        out = torch.empty_like(Din)
        _lib.check(self.lib.gg_ppdna_hess(_p(self.Vt), _p(self.Q), _p(self.phi), _p(Din), _p(self.V), _p(self.code),
                                          _p(self.jscale), self.sigma, self.l1, self.regi, self.K, self.p, _p(self.Y),
                                          _p(self.Z), _p(out), None, None, self.st), "gg_ppdna_hess")
        return out.cpu().numpy()

    def jp(self, Dm):
        from gglasso_b200 import _lib
        Din = torch.from_numpy(np.ascontiguousarray(Dm)).cuda()
        out = torch.empty_like(Din)
        _lib.check(self.lib.gg_ppdna_jp(_p(Din), _p(self.V), _p(self.code), _p(self.jscale), None, self.sigma, self.l1,
                                        self.regi, self.K, self.p, _p(out), None, None, self.st), "gg_ppdna_jp")
        return out.cpu().numpy()


def _oracle_hess(Q, d, V, sigma, l1, l2, reg, Dm):
    phi = po.phi_of(d, sigma)
    G = np.stack([po.gamma_dense(f, sigma) for f in phi])
    Qt = Q.transpose(0, 2, 1)
    jd = po.jac_data(V, sigma * l1, sigma * l2, reg)
    return sigma * (Q @ (G * (Qt @ Dm @ Q)) @ Qt + po.jac_apply(jd, Dm)), jd


def _case(K, p, seed):
    rng = np.random.default_rng(seed)
    W = _sym(rng, K, p)
    V = _sym(rng, K, p, 0.05)
    if K > 2:                                  # ties across k: FGL runs longer than one
        V[1] = V[0]
    Dm = _sym(rng, K, p)
    return W, V, Dm


SHAPES = [(7, 1), (7, 3), (48, 3), (49, 20), (130, 3), (257, 1), (257, 20), (1000, 1), (1000, 20)]


@pytest.mark.gpu
@pytest.mark.parametrize("reg", ["GGL", "FGL"])
@pytest.mark.parametrize("p,K", SHAPES)
def test_hessian_product_from_numpy_eigenvectors(p, K, reg):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    sigma, l1, l2 = 3.0, 0.02, 0.01
    W, V, Dm = _case(K, p, seed=p + K)
    d, Q = np.linalg.eigh(W)
    dv = _Dev(Q.transpose(0, 2, 1), d, V, sigma, l1, l2, reg)
    ref, jd = _oracle_hess(Q, d, V, sigma, l1, l2, reg, Dm)
    out = dv.hess(Dm)
    err = np.abs(out - ref).max() / np.abs(ref).max()
    print(f"hessian p={p} K={K} {reg}: relative error {err:.2e}")
    assert err <= 1e-13
    # the Jacobian of the prox alone, and the spectral map
    jref = sigma * po.jac_apply(jd, Dm)
    assert np.abs(dv.jp(Dm) - jref).max() <= 1e-14 * np.abs(jref).max()
    Om = (Q * po.phi_of(d, sigma)[:, None, :]) @ Q.transpose(0, 2, 1)
    assert np.abs(dv.Omega.cpu().numpy() - Om).max() <= 1e-13 * np.abs(Om).max()
    assert np.abs(dv.logdet.cpu().numpy() - np.log(po.phi_of(d, sigma)).sum(1)).max() <= 1e-12 * p


@pytest.mark.gpu
@pytest.mark.parametrize("reg", ["GGL", "FGL"])
@pytest.mark.parametrize("p,K", [(7, 3), (49, 3), (130, 3), (257, 20)])
def test_hessian_product_through_gg_eigh_is_basis_invariant(p, K, reg):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from gglasso_b200 import _engine
    sigma, l1, l2 = 3.0, 0.02, 0.01
    W, V, Dm = _case(K, p, seed=7 * p + K)
    dev = torch.device("cuda")
    A = torch.from_numpy(W).to(dev)
    eig = _engine.Eigh(K, p, dev)
    Dg = eig.eigh(A, stream=torch.cuda.current_stream().cuda_stream)
    dv = _Dev(A.cpu().numpy(), Dg.cpu().numpy(), V, sigma, l1, l2, reg)
    d, Q = np.linalg.eigh(W)
    ref, _ = _oracle_hess(Q, d, V, sigma, l1, l2, reg, Dm)
    scale = np.abs(ref).max()
    assert np.abs(dv.hess(Dm) - ref).max() <= 1e-11 * scale


@pytest.mark.gpu
@pytest.mark.parametrize("reg", ["GGL", "FGL"])
@pytest.mark.parametrize("p,K", [(49, 3), (130, 20), (300, 5)])
def test_prox_kernel_matches_gg_prox_mgl(p, K, reg):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from gglasso_b200 import _lib
    sigma, l1, l2 = 7.0, 0.01, 0.004
    W, V, _ = _case(K, p, seed=p)
    V = np.round(V, 2) if reg == "FGL" else V         # exact ties: runs of the TV prox
    d, Q = np.linalg.eigh(W)
    rng = np.random.default_rng(p + K)
    Om_t, Th_t, X, S = (_sym(rng, K, p) for _ in range(4))
    dv = _Dev(Q.transpose(0, 2, 1), d, V, sigma, l1, l2, reg, Om_t, Th_t, X, S)
    lib = dv.lib
    Vd = dv.V
    zero = torch.zeros_like(Vd)
    out = torch.empty_like(Vd)
    Cd = torch.empty_like(Vd)
    ctrl = torch.zeros((1, 16), dtype=torch.float64, device=Vd.device)
    ctrl[0, 0] = 1.0
    ctrl[0, 1] = 1.0
    _lib.check(lib.gg_prox_mgl(_p(Vd), _p(Vd), _p(zero), _p(zero), _p(out), _p(Cd), _p(ctrl), sigma * l1, sigma * l2,
                               dv.regi, K, p, None, dv.st), "gg_prox_mgl")
    th, ref = dv.Theta.cpu().numpy(), out.cpu().numpy()
    if reg == "FGL":
        assert np.array_equal(th, ref)
    else:
        assert np.abs(th - ref).max() <= 1e-15 * max(1.0, np.abs(ref).max())
    assert np.abs(th - orc.prox_p(V, sigma * l1, sigma * l2, reg)).max() <= 1e-14
    # the gradient and all six partial sums of Phi
    G, Om = dv.G.cpu().numpy(), dv.Omega.cpu().numpy()
    assert np.array_equal(G, th - Om)
    parts = dv.parts.sum(0).cpu().numpy()
    ref = [np.sum(S * Om), orc.P_val(th, l1, l2, reg), np.sum(X * (Om - th)), np.sum((Om - Om_t) ** 2),
           np.sum((th - Th_t) ** 2), np.sum(G * G)]
    for i, (a, b) in enumerate(zip(parts, ref)):
        assert abs(a - b) <= 1e-12 * max(1.0, abs(b)), (i, a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("reg", ["GGL", "FGL"])
@pytest.mark.parametrize("p,K", [(50, 3), (100, 5)])
def test_engine_phi_and_gradient_match_the_oracle(p, K, reg):
    """Phi and |grad Phi| of one subproblem point, assembled by the engine from gg_eigh, gg_ppdna_spectral and the
    prox kernel's partial sums, against oracle Point at random nonzero Omega_t, Theta_t, X, S"""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from gglasso_b200 import _ppdna
    rng = np.random.default_rng(3 * p + K)
    S = np.stack([np.cov(rng.standard_normal((p, 3 * p)), bias=True) for _ in range(K)])
    Om_t = np.stack([np.eye(p) + 0.05 * (B + B.T) for B in rng.standard_normal((K, p, p))])
    Th_t, X = Om_t + 0.01 * _sym(rng, K, p), 0.05 * _sym(rng, K, p)
    sigma, l1, l2 = 4.0, 0.05, 0.01
    dev = torch.device("cuda", torch.cuda.current_device())
    with torch.cuda.stream(_ppdna._stream(dev)):
        eng = _ppdna.PpdnaEngine(torch.from_numpy(S).to(dev), l1, l2, reg, dev)
        eng.Om_t.copy_(torch.from_numpy(Om_t))
        eng.Th_t.copy_(torch.from_numpy(Th_t))
        pt = eng.evaluate(eng.cur, torch.from_numpy(X).to(dev), None, 0.0, sigma)
        G = pt.G.cpu().numpy()
    ref = po.Point(X, S, Om_t, Th_t, sigma, l1, l2, reg)
    assert abs(pt.Phi - ref.Phi) <= 1e-12 * max(1.0, abs(ref.Phi))
    assert abs(pt.gnorm - ref.gnorm) <= 1e-11 * max(1.0, ref.gnorm)
    assert np.abs(G - ref.grad).max() <= 1e-11 * max(1.0, np.abs(ref.grad).max())


# ---------------------------------------------------------------------------------------------------------------------
def _inputs(name):
    if name.startswith("cfg2"):
        from oracle import ref_inputs
        S = ref_inputs.load(name)
    else:
        S = np.load(os.path.join(GOLDEN, (name[:-2] if name.endswith("K1") else name) + ".npz"))["S"]
        if name.endswith("K1"):
            S = S[:1]
    return S


CASES = [("mgl_ggl_K3_p50", "GGL"), ("mgl_fgl_K3_p50", "FGL"), ("cfg2_ggl", "GGL"), ("cfg2_fgl", "FGL"),
         ("mgl_ggl_K3_p50K1", "GGL")]


@pytest.fixture(scope="module")
def admm_ref():
    cache = {}

    def get(name, reg):
        if name not in cache:
            from gglasso_b200 import ADMM_MGL
            S = _inputs(name)
            K, p, _ = S.shape
            with contextlib.redirect_stdout(io.StringIO()):
                sol, info = ADMM_MGL(S, 0.05, 0.01, reg, np.repeat(np.eye(p)[None], K, 0), tol=1e-10, rtol=1e-10,
                                     stopping_criterion="kkt", max_iter=20000)
            assert info["status"] == "optimal"
            cache[name] = (S, sol)
        return cache[name]
    return get


def _check_solution(S, reg, sol, ref, eps):
    K, p, _ = S.shape
    eta = orc.kkt_residual_mgl(sol["Omega"], sol["Theta"], np.zeros_like(S), sol["X"], S, 0.05, 0.01,
                               np.ones((K, 1, 1)), reg)
    assert eta <= eps, eta
    assert np.abs(sol["Theta"] - ref["Theta"]).max() <= 1e-6
    assert np.array_equal(sol["Theta"] != 0, ref["Theta"] != 0)
    assert np.linalg.eigvalsh(sol["Omega"]).min() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("name,reg", CASES)
def test_ppdna_and_warm_ppdna_reach_the_admm_solution(admm_ref, name, reg):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from gglasso_b200 import PPDNA, warmPPDNA
    S, ref = admm_ref(name, reg)
    K, p, _ = S.shape
    Om0 = np.repeat(np.eye(p)[None], K, 0)
    with contextlib.redirect_stdout(io.StringIO()):
        sol, info = PPDNA(S, 0.05, 0.01, reg, Om0, eps_ppdna=1e-8, measure=True)
    assert info["status"] == "optimal"
    assert set(info) == {"status", "runtime", "residual", "objective"}
    assert info["residual"][-1] <= 1e-8
    _check_solution(S, reg, sol, ref, 1e-8)
    with contextlib.redirect_stdout(io.StringIO()):
        sol, info = warmPPDNA(S, 0.05, 0.01, reg, Om0, eps=1e-8)
    assert info["status"] == "optimal"
    _check_solution(S, reg, sol, ref, 1e-8)


@pytest.mark.gpu
def test_ppdna_max_iter_and_non_finite_input():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from gglasso_b200 import GGLassoB200Error, PPDNA
    S = _inputs("mgl_fgl_K3_p50")
    Om0 = np.repeat(np.eye(50)[None], 3, 0)
    for n in (0, 2):
        with contextlib.redirect_stdout(io.StringIO()):
            sol, info = PPDNA(S, 0.05, 0.01, "FGL", Om0, ppdna_params={"max_iter": n}, eps_ppdna=1e-12, measure=True)
        assert info["status"] == "max iterations reached"
        assert np.all(np.isfinite(sol["Theta"]))
        # one KKT residual per iterate, the last one of the returned iterate
        assert len(info["residual"]) == n + 1
        eta = orc.kkt_residual_mgl(sol["Omega"], sol["Theta"], np.zeros_like(S), sol["X"], S, 0.05, 0.01,
                                   np.ones((3, 1, 1)), "FGL")
        assert abs(info["residual"][-1] - eta) <= 1e-10 * eta
    bad = S.copy()
    bad[1, 3, 4] = bad[1, 4, 3] = np.nan
    with pytest.raises(GGLassoB200Error), contextlib.redirect_stdout(io.StringIO()):
        PPDNA(bad, 0.05, 0.01, "FGL", Om0)


@pytest.mark.gpu
def test_two_threads_solving_at_once_get_their_single_thread_results():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from gglasso_b200 import PPDNA
    jobs = [(_inputs("mgl_ggl_K3_p50"), "GGL"), (_inputs("cfg2_fgl"), "FGL")]

    def solve(S, reg):
        K, p, _ = S.shape
        with contextlib.redirect_stdout(io.StringIO()):
            return PPDNA(S, 0.05, 0.01, reg, np.repeat(np.eye(p)[None], K, 0), eps_ppdna=1e-8)[0]
    single = [solve(*j) for j in jobs]
    out = [None, None]

    def run(i):
        torch.cuda.set_device(0)
        out[i] = solve(*jobs[i])
    ts = [threading.Thread(target=run, args=(i,)) for i in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    for a, b in zip(out, single):
        assert np.array_equal(a["Theta"], b["Theta"]) and np.array_equal(a["X"], b["X"])


def test_signature_and_limits():
    """argument order and defaults of the reference's PPDNA / warmPPDNA; K above the prox kernel's limit is refused"""
    from gglasso_b200 import PPDNA, warmPPDNA
    assert list(inspect.signature(PPDNA).parameters) == ["S", "lambda1", "lambda2", "reg", "Omega_0", "Theta_0", "X_0",
                                                         "ppdna_params", "eps_ppdna", "verbose", "measure"]
    assert list(inspect.signature(warmPPDNA).parameters) == ["S", "lambda1", "lambda2", "reg", "Omega_0", "Theta_0",
                                                             "X_0", "admm_params", "ppdna_params", "eps", "eps_admm",
                                                             "verbose", "measure"]
    assert inspect.signature(PPDNA).parameters["eps_ppdna"].default == 1e-5
    assert inspect.signature(warmPPDNA).parameters["eps_admm"].default == 1e-3
    S = np.repeat(np.eye(3)[None], 91, 0)
    with pytest.raises(NotImplementedError, match="90"):
        PPDNA(S, 0.1, 0.1, "GGL", S)


@pytest.mark.gpu
def test_matches_the_reference_ppdna():
    """signature, info keys and solution of the reference's own PPDNA (skipped without oracle/_ref)"""
    from oracle import ref
    if not ref.available() or not torch.cuda.is_available():
        pytest.skip("oracle/_ref (the reference package) or a CUDA device is missing")
    import importlib
    ref.load()
    rp = importlib.reload(importlib.import_module("gglasso.solver.ppdna_solver"))
    from gglasso_b200 import PPDNA, warmPPDNA
    for mine, theirs in ((PPDNA, rp.PPDNA), (warmPPDNA, rp.warmPPDNA)):
        a, b = inspect.signature(mine).parameters, inspect.signature(theirs).parameters
        assert list(a) == list(b)
        assert all(a[n].default is b[n].default or np.array_equal(a[n].default, b[n].default) for n in a
                   if n not in ("ppdna_params", "admm_params"))
    S = _inputs("mgl_ggl_K3_p50")
    Om0 = np.repeat(np.eye(50)[None], 3, 0)
    with contextlib.redirect_stdout(io.StringIO()):
        rsol, rinfo = rp.PPDNA(S, 0.05, 0.01, "GGL", Om0, eps_ppdna=1e-8, measure=True)
        sol, info = PPDNA(S, 0.05, 0.01, "GGL", Om0, eps_ppdna=1e-8, measure=True)
    assert set(info) == set(rinfo)
    assert np.abs(sol["Theta"] - rsol["Theta"]).max() <= 1e-6
    # the ppdna_params defaults: the reference fills them in inside PPDNA's body
    import ast
    import re
    from gglasso_b200 import _ppdna
    src = inspect.getsource(rp.PPDNA)
    for key, val in _ppdna.PPDNA_DEFAULTS.items():
        m = re.search(r"['\"]%s['\"]\s*:\s*([^,}\n]+)" % key, src)
        assert m is not None, key
        assert ast.literal_eval(m.group(1).strip()) == val, (key, m.group(1))


# ---------------------------------------------------------------------------------------------------------------------
GUARD = 8192          # elements of sentinel before and after every output buffer


def _guarded(shape, dtype, fill):
    n = int(np.prod(shape))
    buf = torch.full((n + 2 * GUARD,), fill, dtype=dtype, device="cuda")
    return buf, buf[GUARD:GUARD + n].view(shape)


def _run_chain(K, p, reg, inputs, Vt, D):
    """every gg_ppdna entry point once (and five CG iterations) with each output in its own guarded buffer; the
    eigendecomposition of W is the given (Vt, D).  Returns {name: (buffer, view, fill)} and W as built."""
    from gglasso_b200 import _lib
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    regi = 0 if reg == "GGL" else 1
    sigma, l1, l2 = 3.0, 0.02, 0.01
    Om_t, Th_t, S, X, dX = (torch.from_numpy(a).cuda() for a in inputs)
    f64, u8 = (torch.float64, 1.5e300), (torch.uint8, 0xA5)
    spec = {"Xs": ((K, p, p), f64), "W": ((K, p, p), f64), "V": ((K, p, p), f64), "Q": ((K, p, p), f64),
            "phi": ((K, p), f64), "logdet": ((K,), f64), "Omega": ((K, p, p), f64), "Theta": ((K, p, p), f64),
            "G": ((K, p, p), f64), "code": ((K, p, p), u8), "jscale": ((p, p), f64),
            "parts": ((lib.gg_ppdna_nparts(p), 6), f64), "Y": ((K, p, p), f64), "Z": ((K, p, p), f64),
            "H": ((K, p, p), f64), "hparts": ((lib.gg_ppdna_jp_nparts(p),), f64), "d": ((K, p, p), f64),
            "r": ((K, p, p), f64), "pv": ((K, p, p), f64), "q": ((K, p, p), f64), "cg": ((8,), f64),
            "cgparts": ((1184,), f64)}
    b = {n: (*_guarded(shape, dt, fill), fill) for n, (shape, (dt, fill)) in spec.items()}
    v = {n: x[1] for n, x in b.items()}
    _lib.check(lib.gg_ppdna_build(_p(Om_t), _p(Th_t), _p(S), _p(X), _p(dX), 0.5, sigma, K, p, _p(v["Xs"]), _p(v["W"]),
                                  _p(v["V"]), None, st), "gg_ppdna_build")
    W_built = v["W"].clone()
    v["W"].copy_(Vt)
    _lib.check(lib.gg_ppdna_spectral(_p(v["W"]), _p(D), sigma, K, p, _p(v["Q"]), _p(v["phi"]), _p(v["logdet"]),
                                     _p(v["Omega"]), None, st), "gg_ppdna_spectral")
    _lib.check(lib.gg_ppdna_prox(_p(v["V"]), _p(v["Omega"]), _p(Om_t), _p(Th_t), _p(v["Xs"]), _p(S), l1, l2, sigma, regi,
                                 K, p, _p(v["Theta"]), _p(v["G"]), _p(v["code"]), _p(v["jscale"]), _p(v["parts"]), None,
                                 st), "gg_ppdna_prox")
    _lib.check(lib.gg_ppdna_hess(_p(v["W"]), _p(v["Q"]), _p(v["phi"]), _p(v["G"]), _p(v["V"]), _p(v["code"]),
                                 _p(v["jscale"]), sigma, l1, regi, K, p, _p(v["Y"]), _p(v["Z"]), _p(v["H"]),
                                 _p(v["hparts"]), None, st), "gg_ppdna_hess")
    _lib.check(lib.gg_ppdna_cg_init(_p(v["G"]), K, p, 0.0, 5, _p(v["d"]), _p(v["r"]), _p(v["pv"]), _p(v["cg"]),
                                    _p(v["cgparts"]), st), "gg_ppdna_cg_init")
    _lib.check(lib.gg_ppdna_cg(7, _p(v["W"]), _p(v["Q"]), _p(v["phi"]), _p(v["V"]), _p(v["code"]), _p(v["jscale"]),
                               sigma, l1, regi, K, p, _p(v["d"]), _p(v["r"]), _p(v["pv"]), _p(v["q"]), _p(v["Y"]),
                               _p(v["Z"]), _p(v["cg"]), _p(v["cgparts"]), st), "gg_ppdna_cg")
    torch.cuda.synchronize()
    return b, W_built


@pytest.mark.gpu
@pytest.mark.parametrize("reg", ["GGL", "FGL"])
@pytest.mark.parametrize("p,K", [(33, 90), (64, 2), (130, 3), (257, 5)])
def test_kernels_write_only_their_outputs_and_repeat_bitwise(p, K, reg):
    """Every output buffer of the chain build -> spectral -> prox -> hess -> CG sits between sentinel
    regions, which must come back untouched (no write outside an output).  A second run of the whole chain must give
    bitwise the same outputs: a race on shared memory or on the device CG state would show up as run-to-run
    differences.  Odd p (8-byte cp.async path), exact tiles, edge tiles, and K = 90 (195 KB of dynamic shared memory
    in the prox kernel).  Both runs take the same eigendecomposition: gg_eigh's eigenvectors are not bitwise
    reproducible from run to run at every size, and it is not under test here."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    rng = np.random.default_rng(p * K)
    inputs = [_sym(rng, K, p) for _ in range(5)]
    inputs[0] = inputs[0] + 4 * p * np.eye(p)        # Omega_t well inside the cone
    from gglasso_b200 import _engine
    A = torch.from_numpy(inputs[0] - 3.0 * (inputs[2] + inputs[3])).cuda()      # W of the chain at s = 0
    eig = _engine.Eigh(K, p, torch.device("cuda", torch.cuda.current_device()))
    D = eig.eigh(A, stream=torch.cuda.current_stream().cuda_stream).clone()
    out = [_run_chain(K, p, reg, inputs, A, D) for _ in range(2)]
    assert torch.equal(out[0][1], out[1][1])
    runs = [o[0] for o in out]
    for name, (_, view, fill) in runs[0].items():
        for r in runs:
            g = r[name][0]
            assert bool((g[:GUARD] == fill).all()) and bool((g[-GUARD:] == fill).all()), name
        a, c = view.cpu().numpy(), runs[1][name][1].cpu().numpy()
        assert np.array_equal(a, c, equal_nan=True), name
    assert float(runs[0]["cg"][1][4]) >= 1          # CG ran
