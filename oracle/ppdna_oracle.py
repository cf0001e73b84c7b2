"""
oracle/ppdna_oracle.py -- TEST INFRASTRUCTURE ONLY.

numpy/LAPACK restatement of the proximal point dual Newton method (PPDNA) for the conforming multiple graphical
lasso (GGL / FGL), the algorithm gglasso_b200/_ppdna.py runs on the GPU (reference: src/gglasso/solver/ppdna_solver.py
PPA_subproblem:65, PPDNA:160, warmPPDNA:348; Jacobians and CG in ggl_helper.py:74-159,218-249,323-437).  It is the
checker of the CUDA path and the CPU timing at small sizes.  The product package never imports it.

Notation (DESIGN.md section 9): f(Omega) = sum_k -log det Omega_k + <S_k, Omega_k>, P = prox_p's penalty, X the
UNSCALED dual.  Subproblem at (Omega_t, Theta_t, sigma): minimise over X

    Phi(X) = -[ f(Omega(X)) + P(Theta(X)) + <X, Omega(X) - Theta(X)> + (|Omega(X)-Omega_t|^2 + |Theta(X)-Theta_t|^2)/(2 sigma) ]

    W = Omega_t - sigma (S + X),  Omega(X) = Q diag(phi(d)) Q^T,  phi(d) = (d + sqrt(d^2 + 4 sigma))/2
    V = Theta_t + sigma X,        Theta(X) = prox_p(V, sigma lambda1, sigma lambda2)
    grad Phi = Theta - Omega,     H[D] = sigma (J_phi(W)[D] + J_P(V)[D])
    J_phi(W)[D] = Q (Gamma o (Q^T D Q)) Q^T,  Gamma_ab = phi_a phi_b / (phi_a phi_b + sigma)

Rules shared with the GPU engine (constants below):
  - Newton step: plain CG on H d = -grad to |H d + grad| <= min(eta, |grad|^(1+tau)), at most CG_MAX iterations;
  - Armijo: s = rho^m, accept once Phi(X + s d) <= Phi(X) + mu s <grad, d> + ARMIJO_SLACK (1 + |Phi(X)|), m < LS_MAX;
    the slack admits steps whose decrease is below the rounding of Phi (near the solution);
  - the Newton loop of outer iteration t stops when |grad| <= eps_t / sqrt(sigma_t), eps_t = min(0.1 eta_t, 1/(t+1)^2)
    (summable: criterion (A) of the proximal point method), after NEWTON_MAX steps, or when the line search fails;
  - outer loop: eta_t = KKT residual of (Omega^t, Theta^t, X^t); stop 'optimal' once eta_t <= eps_ppdna, else solve
    the subproblem and set sigma <- 1.3 sigma unless sigma_fix; after max_iter subproblems the returned iterate's
    eta is evaluated once more and the status is 'max iterations reached' unless it is <= eps_ppdna.
"""
import time

import numpy as np

from . import admm_oracle as orc

CG_MAX = 200
NEWTON_MAX = 50
LS_MAX = 40
ARMIJO_SLACK = 1e-13
PPDNA_DEFAULTS = dict(sigma_0=10.0, max_iter=20, sigma_fix=False, rho=0.5, mu=0.25, eta=0.5, tau=0.5)


def phi_of(d, sigma):
    """phi(d) = (d + sqrt(d^2 + 4 sigma))/2, cancellation free for d < 0"""
    d = np.asarray(d, dtype=np.float64)
    r = np.sqrt(d * d + 4.0 * sigma)
    return np.where(d >= 0, 0.5 * (d + r), (2.0 * sigma) / np.where(d >= 0, 1.0, r - d))


def gamma_dense(phi, sigma):
    pp = phi[:, None] * phi[None, :]
    return pp / (pp + sigma)


def gamma_divided(d, sigma):
    """divided differences of phi (phi' on ties): the textbook form of the Jacobian's Loewner matrix"""
    ph = phi_of(d, sigma)
    dd = d[:, None] - d[None, :]
    dphi = 0.5 * (1.0 + d / np.sqrt(d * d + 4.0 * sigma))
    with np.errstate(divide="ignore", invalid="ignore"):
        G = (ph[:, None] - ph[None, :]) / dd
    tie = dd == 0
    G[tie] = np.broadcast_to(dphi[:, None], G.shape)[tie]
    return G


# ---------------------------------------------------------------------------------------------------------------------
# Jacobian data of prox_p and its application
# ---------------------------------------------------------------------------------------------------------------------
def jac_data(V, l1, l2, reg):
    """per strictly-upper entry: ('GGL', mask (K,n), u (K,n), scale (n,) with -1 = zero branch) or
    ('FGL', active (K,n), start (K,n)).  l1, l2 already multiplied by sigma."""
    K, p, _ = V.shape
    iu, ju = np.triu_indices(p, 1)
    v = V[:, iu, ju]
    if reg == "GGL":
        mask = np.abs(v) > l1
        u = np.where(mask, orc.soft_threshold(v, l1), 0.0)
        nrm = np.sqrt((u * u).sum(0))
        scale = np.where(nrm > l2, l2 / np.where(nrm > 0, nrm, 1.0), -1.0)
        return ("GGL", mask, u, scale)
    z = np.empty_like(v)
    for e in range(v.shape[1]):
        z[:, e] = orc.tv1d(v[:, e], l2)
    active = np.abs(z) > l1
    start = np.ones_like(active)
    if K > 1:
        start[1:] = z[1:].view(np.int64) != z[:-1].view(np.int64)
    return ("FGL", active, start)


def jac_apply(jd, Dm):
    """J_P(V)[D] for symmetric D (diagonal: identity)"""
    K, p, _ = Dm.shape
    iu, ju = np.triu_indices(p, 1)
    dv = Dm[:, iu, ju]
    if jd[0] == "GGL":
        _, mask, u, scale = jd
        md = np.where(mask, dv, 0.0)
        uu = (u * u).sum(0)
        ud = (u * dv).sum(0)
        with np.errstate(divide="ignore", invalid="ignore"):
            out = md - scale * (md - u * (ud / uu))
        out = np.where(scale < 0, 0.0, out)
    else:
        _, active, start = jd
        run = np.cumsum(start, axis=0) - 1                 # run index of every (k, entry)
        col = np.broadcast_to(np.arange(dv.shape[1]), dv.shape)
        sums = np.zeros_like(dv)
        cnt = np.zeros_like(dv)
        np.add.at(sums, (run, col), dv)
        np.add.at(cnt, (run, col), 1.0)
        out = np.where(active, sums[run, col] / cnt[run, col], 0.0)
    R = np.zeros_like(Dm)
    R[:, iu, ju] = out
    R[:, ju, iu] = out
    d = np.arange(p)
    R[:, d, d] = Dm[:, d, d]
    return R


# ---------------------------------------------------------------------------------------------------------------------
# the subproblem
# ---------------------------------------------------------------------------------------------------------------------
class Point:
    """everything the Newton loop needs at one X: Phi, grad, and the Hessian operator's data"""

    def __init__(self, X, S, Omega_t, Theta_t, sigma, lambda1, lambda2, reg):
        self.X = X
        self.sigma = sigma
        W = Omega_t - sigma * (S + X)
        d, Q = np.linalg.eigh(W)
        self.Q = Q
        self.phi = phi_of(d, sigma)
        self.Omega = (Q * self.phi[:, None, :]) @ Q.transpose(0, 2, 1)
        V = Theta_t + sigma * X
        self.V = V
        self.Theta = orc.prox_p(V, sigma * lambda1, sigma * lambda2, reg)
        self.jd = jac_data(V, sigma * lambda1, sigma * lambda2, reg)
        self.grad = self.Theta - self.Omega
        f = -np.log(self.phi).sum() + float(np.sum(S * self.Omega))
        val = (f + orc.P_val(self.Theta, lambda1, lambda2, reg) + float(np.sum(X * (self.Omega - self.Theta)))
               + (np.sum((self.Omega - Omega_t) ** 2) + np.sum((self.Theta - Theta_t) ** 2)) / (2.0 * sigma))
        self.Phi = -float(val)
        self.gnorm = float(np.linalg.norm(self.grad))

    def jac_phi(self, Dm):
        G = np.stack([gamma_dense(self.phi[k], self.sigma) for k in range(len(self.phi))])
        Q = self.Q
        Qt = Q.transpose(0, 2, 1)
        return Q @ (G * (Qt @ Dm @ Q)) @ Qt

    def hess(self, Dm):
        return self.sigma * (self.jac_phi(Dm) + jac_apply(self.jd, Dm))


def cg(hess, rhs, tol, maxit):
    """plain CG for hess(d) = rhs from d = 0, |residual| <= tol; returns (d, iterations)"""
    d = np.zeros_like(rhs)
    r = rhs.copy()
    pv = r.copy()
    rr = float(np.sum(r * r))
    it = 0
    while rr > tol * tol and it < maxit:
        q = hess(pv)
        pq = float(np.sum(pv * q))
        if not pq > 0:
            break
        a = rr / pq
        d += a * pv
        r -= a * q
        rrn = float(np.sum(r * r))
        it += 1
        if rrn <= tol * tol:
            break
        pv = r + (rrn / rr) * pv
        rr = rrn
    return d, it


def subproblem(pt, make_point, eps_t, prm, stats):
    """Newton loop with Armijo backtracking from point ``pt``; returns the final point"""
    sigma = pt.sigma
    for _ in range(NEWTON_MAX):
        if pt.gnorm <= eps_t / np.sqrt(sigma):
            break
        tol = min(prm["eta"], pt.gnorm ** (1.0 + prm["tau"]))
        d, ncg = cg(pt.hess, -pt.grad, tol, CG_MAX)
        stats["cg"].append(ncg)
        gd = float(np.sum(pt.grad * d))
        s, new = 1.0, None
        for _m in range(LS_MAX):
            trial = make_point(pt.X + s * d)
            if trial.Phi <= pt.Phi + prm["mu"] * s * gd + ARMIJO_SLACK * (1.0 + abs(pt.Phi)):
                new = trial
                break
            s *= prm["rho"]
        stats["newton"][-1] += 1
        if new is None:
            break
        pt = new
    return pt


def ppdna(S, lambda1, lambda2, reg, Omega_0, Theta_0=None, X_0=None, ppdna_params=None, eps_ppdna=1e-5,
          measure=False):
    """PPDNA for GGL/FGL; returns (sol, info) like the GPU solver, info also has 'newton' and 'cg' counts"""
    assert reg in ("GGL", "FGL") and min(lambda1, lambda2) > 0
    prm = dict(PPDNA_DEFAULTS)
    prm.update(ppdna_params or {})
    K, p, _ = S.shape
    Omega = Omega_0.copy()
    Theta = Omega.copy() if Theta_0 is None or len(Theta_0) == 0 else Theta_0.copy()
    X = np.zeros((K, p, p)) if X_0 is None or len(X_0) == 0 else X_0.copy()
    nk = np.ones((K, 1, 1))
    sigma = float(prm["sigma_0"])
    status = "max iterations reached"
    stats = {"newton": [], "cg": []}
    residual, runtime, objective = [], [], []
    assert int(prm["max_iter"]) >= 0
    for t in range(int(prm["max_iter"]) + 1):     # the returned iterate's KKT residual is evaluated too
        t0 = time.time()
        eta_t = orc.kkt_residual_mgl(Omega, Theta, np.zeros_like(S), X, S, lambda1, lambda2, nk, reg)
        residual.append(eta_t)
        if measure:
            objective.append(orc.objective(Omega, Theta, S, lambda1, lambda2, reg))
        if eta_t <= eps_ppdna or t == int(prm["max_iter"]):
            status = "optimal" if eta_t <= eps_ppdna else status
            runtime.append(time.time() - t0)
            break
        eps_t = min(0.1 * eta_t, 1.0 / (t + 1) ** 2)
        Om_t, Th_t, sg = Omega.copy(), Theta.copy(), sigma

        def make_point(Xn):
            return Point(Xn, S, Om_t, Th_t, sg, lambda1, lambda2, reg)
        stats["newton"].append(0)
        pt = subproblem(make_point(X), make_point, eps_t, prm, stats)
        Omega, Theta, X = pt.Omega, pt.Theta, pt.X
        if not prm["sigma_fix"]:
            sigma *= 1.3
        runtime.append(time.time() - t0)
    sol = {"Omega": Omega, "Theta": Theta, "X": X}
    info = {"status": status, "newton": stats["newton"], "cg": stats["cg"]}
    if measure:
        info.update(residual=np.array(residual), runtime=np.array(runtime), objective=np.array(objective))
    return sol, info
