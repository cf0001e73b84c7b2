"""Device-resident PPDNA (proximal point dual Newton method) for GGL / FGL.

The algorithm, its constants and its stopping rules are stated in DESIGN.md section 9 and restated in numpy by
oracle/ppdna_oracle.py; both follow reference src/gglasso/solver/ppdna_solver.py (PPA_subproblem:65, PPDNA:160).
Every arithmetic step is a CUDA kernel of gg_ppdna.cu / gg_eigh / gg_prox_mgl reached through the C ABI; torch holds
device memory and streams and sums a few hundred partial sums per line-search trial.  The host synchronises once per
line-search trial (Phi and |grad| decide the step) and every ``CG_CHECK`` CG iterations (the device stop flag), never
per CG iteration.
"""
import threading
import time
from types import SimpleNamespace

import numpy as np
import torch

from . import _lib
from ._engine import Eigh, K_TILE_MAX, _kkt_residual, _p, require_cuda, to_dev
from ._lib import CTRL_STRIDE, C_RHO

CG_MAX = 200           # CG iterations per Newton step
NEWTON_MAX = 50        # Newton steps per subproblem
LS_MAX = 40            # Armijo trials per Newton step
ARMIJO_SLACK = 1e-13   # relative slack of the Armijo test: admits steps whose decrease is below the rounding of Phi
CG_CHECK = 8           # CG iterations enqueued between two polls of the device stop flag
PPDNA_DEFAULTS = dict(sigma_0=10.0, max_iter=20, sigma_fix=False, rho=0.5, mu=0.25, eta=0.5, tau=0.5)

_TLS = threading.local()


def _stream(dev):
    """one CUDA stream per host thread and device: concurrent solves from several threads do not share a stream"""
    key = "s%d" % (dev.index if dev.index is not None else torch.cuda.current_device())
    s = getattr(_TLS, key, None)
    if s is None:
        s = torch.cuda.Stream(device=dev)
        setattr(_TLS, key, s)
    return s


class _Point:
    """device buffers of one point X of the subproblem: everything Phi, grad and the Hessian product need"""

    def __init__(self, K, p, dev):
        e = lambda: torch.empty((K, p, p), dtype=torch.float64, device=dev)  # noqa: E731
        self.X, self.W, self.V, self.Q, self.Omega, self.Theta, self.G = e(), e(), e(), e(), e(), e(), e()
        self.D = torch.empty((K, p), dtype=torch.float64, device=dev)
        self.phi = torch.empty((K, p), dtype=torch.float64, device=dev)
        self.logdet = torch.empty(K, dtype=torch.float64, device=dev)
        self.code = torch.empty((K, p, p), dtype=torch.uint8, device=dev)
        self.jscale = torch.empty((p, p), dtype=torch.float64, device=dev)
        self.Phi = self.gnorm = None


class PpdnaEngine:
    """per-call workspace: the subproblem's fixed data (S, Omega_t, Theta_t), two points (current and trial, swapped
    when a trial is accepted) and the CG vectors"""

    def __init__(self, S, lambda1, lambda2, reg, dev):
        self.lib = _lib.load()
        self.dev = dev
        self.S = S
        self.K, self.p = K, p = S.shape[0], S.shape[1]
        self.l1, self.l2 = float(lambda1), float(lambda2)
        self.regi = {"GGL": 0, "FGL": 1}[reg]
        self.stream = torch.cuda.current_stream().cuda_stream
        e = lambda: torch.empty((K, p, p), dtype=torch.float64, device=dev)  # noqa: E731
        self.Om_t, self.Th_t = e(), e()
        self.d, self.r, self.pv, self.q, self.Y, self.Z = e(), e(), e(), e(), e(), e()
        self.cur, self.trial = _Point(K, p, dev), _Point(K, p, dev)
        self.eig = Eigh(K, p, dev)
        self.Dk = torch.empty((K, p), dtype=torch.float64, device=dev)
        self.parts = torch.zeros((self.lib.gg_ppdna_nparts(p), 6), dtype=torch.float64, device=dev)
        self.cg_parts = torch.zeros(2048, dtype=torch.float64, device=dev)
        self.cg = torch.zeros(8, dtype=torch.float64, device=dev)
        self.stats = {"newton": [], "cg": []}

    # -- Phi, grad and the Jacobian data at X + s dX ----------------------------------------------------------------
    def evaluate(self, pt, X, dX, s, sigma):
        lib, st, K, p = self.lib, self.stream, self.K, self.p
        _lib.check(lib.gg_ppdna_build(_p(self.Om_t), _p(self.Th_t), _p(self.S), _p(X), _p(dX), float(s), sigma, K, p,
                                      _p(pt.X), _p(pt.W), _p(pt.V), None, st), "gg_ppdna_build")
        self.eig.D = pt.D
        self.eig.eigh(pt.W, stream=st)                     # pt.W now holds Vt (rows = eigenvectors)
        _lib.check(lib.gg_ppdna_spectral(_p(pt.W), _p(pt.D), sigma, K, p, _p(pt.Q), _p(pt.phi), _p(pt.logdet),
                                         _p(pt.Omega), None, st), "gg_ppdna_spectral")
        _lib.check(lib.gg_ppdna_prox(_p(pt.V), _p(pt.Omega), _p(self.Om_t), _p(self.Th_t), _p(pt.X), _p(self.S),
                                     self.l1, self.l2, sigma, self.regi, K, p, _p(pt.Theta), _p(pt.G), _p(pt.code),
                                     _p(pt.jscale), _p(self.parts), None, st), "gg_ppdna_prox")
        tot = torch.cat([self.parts.sum(0), pt.logdet.sum().reshape(1)]).cpu().numpy()
        s_om, pen, x_om_th, n_om, n_th, g2, logdet = tot
        val = -logdet + s_om + pen + x_om_th + (n_om + n_th) / (2.0 * sigma)
        pt.Phi, pt.gnorm = -float(val), float(np.sqrt(g2))
        if not (np.isfinite(pt.Phi) and np.isfinite(pt.gnorm)):
            raise _lib.GGLassoB200Error("PPDNA: non-finite subproblem value: the input is not finite or an "
                                        "eigendecomposition broke down")
        return pt

    def newton_direction(self, pt, sigma, tol):
        """CG on H d = -grad, on the device; the host polls the stop flag every CG_CHECK iterations"""
        lib, st, K, p = self.lib, self.stream, self.K, self.p
        _lib.check(lib.gg_ppdna_cg_init(_p(pt.G), K, p, float(tol), CG_MAX, _p(self.d), _p(self.r), _p(self.pv),
                                        _p(self.cg), _p(self.cg_parts), st), "gg_ppdna_cg_init")
        done = 0
        while done < CG_MAX:
            n = min(CG_CHECK, CG_MAX - done)
            _lib.check(lib.gg_ppdna_cg(n, _p(pt.W), _p(pt.Q), _p(pt.phi), _p(pt.V), _p(pt.code), _p(pt.jscale), sigma,
                                       self.l1, self.regi, K, p, _p(self.d), _p(self.r), _p(self.pv), _p(self.q),
                                       _p(self.Y), _p(self.Z), _p(self.cg), _p(self.cg_parts), st), "gg_ppdna_cg")
            done += n
            if float(self.cg[3].item()) != 0.0:
                break
        self.stats["cg"].append(int(self.cg[4].item()))
        return self.d

    def subproblem(self, X, sigma, eps_t, prm):
        pt = self.evaluate(self.cur, X, None, 0.0, sigma)
        self.stats["newton"].append(0)
        for _ in range(NEWTON_MAX):
            if pt.gnorm <= eps_t / np.sqrt(sigma):
                break
            d = self.newton_direction(pt, sigma, min(prm["eta"], pt.gnorm ** (1.0 + prm["tau"])))
            gd = float(torch.sum(pt.G * d).item())
            s, new = 1.0, None
            for _m in range(LS_MAX):
                tr = self.evaluate(self.trial, pt.X, d, s, sigma)
                if tr.Phi <= pt.Phi + prm["mu"] * s * gd + ARMIJO_SLACK * (1.0 + abs(pt.Phi)):
                    new = tr
                    break
                s *= prm["rho"]
            self.stats["newton"][-1] += 1
            if new is None:
                break
            self.cur, self.trial = self.trial, self.cur
            pt = self.cur
        return pt

    def kkt(self, Omega, Theta, X):
        """KKT residual of (Omega, Theta, X) with the kernels of ADMM_MGL's 'kkt' criterion"""
        ctrl = torch.zeros((1, CTRL_STRIDE), dtype=torch.float64, device=self.dev)
        ctrl[0, C_RHO] = 1.0
        self.eig.D = self.Dk
        st = SimpleNamespace(lib=self.lib, stream=self.stream, M=self.K, p=self.p, nprob=1, mpp=self.K, dev=self.dev,
                             ctrl=ctrl, X=X, Omega=Omega, Theta=Theta, L=None, nk=None, S=self.S, eig=self.eig,
                             lam_mat=None, mu=None)
        return _kkt_residual("mgl", st, self.l1, self.l2, self.regi, False)


def check_finite(*arrays):
    for a in arrays:
        if a is None:
            continue
        ok = bool(torch.isfinite(a).all().item()) if isinstance(a, torch.Tensor) else bool(np.isfinite(a).all())
        if not ok:
            raise _lib.GGLassoB200Error("PPDNA: the input contains non-finite values")


def run_ppdna(S, lambda1, lambda2, reg, Omega_0, Theta_0=None, X_0=None, ppdna_params=None, eps_ppdna=1e-5,
              verbose=False, measure=False):
    """PPDNA on the device.  S, Omega_0, Theta_0, X_0: numpy arrays or device tensors (K,p,p); X_0 is the unscaled
    dual.  Returns (Omega, Theta, X) as device tensors and an info dict (status; residual, runtime and objective per
    KKT evaluation, the last one belonging to the returned iterate; Newton steps per subproblem; CG iterations per
    Newton step)."""
    K, p, _ = S.shape
    if K > K_TILE_MAX:
        raise NotImplementedError(f"PPDNA supports at most K = {K_TILE_MAX} instances (K_TILE_MAX), got K = {K}")
    prm = dict(PPDNA_DEFAULTS)
    prm.update(ppdna_params or {})
    if int(prm["max_iter"]) < 0:
        raise ValueError(f"ppdna_params['max_iter'] must be >= 0, got {prm['max_iter']}")
    check_finite(S, Omega_0, Theta_0, X_0)
    dev = require_cuda()
    with torch.cuda.stream(_stream(dev)):
        Sd = to_dev(S, dev)
        eng = PpdnaEngine(Sd, lambda1, lambda2, reg, dev)
        Omega = to_dev(Omega_0, dev)
        Theta = Omega.clone() if Theta_0 is None else to_dev(Theta_0, dev)
        X = torch.zeros_like(Sd) if X_0 is None else to_dev(X_0, dev)
        sigma = float(prm["sigma_0"])
        status = "max iterations reached"
        residual, runtime, objective = [], [], []
        if verbose:
            print("------------PPDNA Algorithm for Multiple Graphical Lasso----------------")
            print("%4s\t%10s\t%10s" % ("iter", "kkt residual", "sigma"))
        # max_iter subproblems; the KKT residual is also evaluated for the iterate the last one returns
        for t in range(int(prm["max_iter"]) + 1):
            torch.cuda.current_stream().synchronize()
            t0 = time.time()
            eta_t = eng.kkt(Omega, Theta, X)
            if not np.isfinite(eta_t):
                raise _lib.GGLassoB200Error("PPDNA: non-finite KKT residual: the input is not finite or an "
                                            "eigendecomposition broke down")
            residual.append(eta_t)
            if measure:
                objective.append(_objective(eng, Omega, Theta))
            if verbose:
                print("%4d\t%10.4g\t%10.4g" % (t, eta_t, sigma))
            if eta_t <= eps_ppdna or t == int(prm["max_iter"]):
                status = "optimal" if eta_t <= eps_ppdna else status
                runtime.append(time.time() - t0)
                break
            eps_t = min(0.1 * eta_t, 1.0 / (t + 1) ** 2)
            eng.Om_t.copy_(Omega)
            eng.Th_t.copy_(Theta)
            pt = eng.subproblem(X, sigma, eps_t, prm)
            # the accepted point's buffers are overwritten by later subproblems: keep copies
            Omega, Theta, X = pt.Omega.clone(), pt.Theta.clone(), pt.X.clone()
            if not prm["sigma_fix"]:
                sigma *= 1.3
            torch.cuda.current_stream().synchronize()
            runtime.append(time.time() - t0)
        torch.cuda.current_stream().synchronize()
    info = {"status": status, "residual": np.array(residual), "runtime": np.array(runtime),
            "objective": np.array(objective), "newton": eng.stats["newton"], "cg": eng.stats["cg"]}
    return Omega, Theta, X, info


def _objective(eng, Omega, Theta):
    """f(Omega) + P(Theta) (the objective PPDNA records with measure=True): log det from gg_eigh's eigenvalues"""
    n = eng.lib.gg_objective_nparts(eng.p)
    parts = torch.empty((n, 2), dtype=torch.float64, device=eng.dev)
    _lib.check(eng.lib.gg_objective(_p(Omega), _p(eng.S), _p(Theta), eng.l1, eng.l2, eng.regi, eng.K, eng.p, _p(parts),
                                    eng.stream), "gg_objective")
    eng.eig.D = eng.Dk
    logdet = torch.log(eng.eig.eigh(Omega.clone(), vectors=0, stream=eng.stream)).sum()
    return float((-logdet + parts.sum(0).sum()).item())
