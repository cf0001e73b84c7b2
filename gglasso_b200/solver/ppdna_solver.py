"""PPDNA and warmPPDNA on B200 -- drop-ins for gglasso.solver.ppdna_solver.PPDNA / warmPPDNA.

Same signatures, asserts and return dicts as the reference (src/gglasso/solver/ppdna_solver.py:160,348); the
proximal point outer loop, the semismooth Newton subproblem and its CG run on the device (gglasso_b200/_ppdna.py).
numpy in, numpy out.  ``ppdna_params`` keys and defaults: sigma_0=10, max_iter=20, sigma_fix=False, rho=0.5 (Armijo
backtracking factor), mu=0.25 (Armijo constant), eta=0.5, tau=0.5 (CG tolerance min(eta, |grad|^(1+tau))).
"""
import time

import numpy as np

from .._engine import K_TILE_MAX, run_admm, to_host_many
from .._ppdna import run_ppdna


def _check(S, lambda1, lambda2, reg, Omega_0):
    assert Omega_0.shape == S.shape
    assert S.shape[1] == S.shape[2]
    assert reg in ['GGL', 'FGL']
    assert min(lambda1, lambda2) > 0
    if S.shape[0] > K_TILE_MAX:
        raise NotImplementedError(f"PPDNA supports at most K = {K_TILE_MAX} instances (K_TILE_MAX), got K = {S.shape[0]}")


def _finish(Omega, Theta, X, res, measure, name, elapsed=None):
    Om, Th, Xh = to_host_many([Omega, Theta, X])
    n_it = len(res["residual"])
    print(f"{name} terminated after {n_it} iterations with accuracy {res['residual'][-1]:.4g} and status: "
          f"{res['status']}.")
    sol = {'Omega': Om, 'Theta': Th, 'X': Xh}
    info = {'status': res['status']}
    if measure:
        info.update(runtime=res['runtime'] if elapsed is None else elapsed, residual=res['residual'],
                    objective=res['objective'])
    return sol, info


def PPDNA(S, lambda1, lambda2, reg, Omega_0, Theta_0=np.array([]), X_0=np.array([]), ppdna_params=dict(),
          eps_ppdna=1e-5, verbose=False, measure=False):
    """Proximal point dual Newton method for GGL/FGL (Zhang, Lin, Toh); see the reference docstring for the model.

    ``X_0`` is the unscaled dual.  Returns ``(sol, info)``: ``sol`` has keys Omega, Theta, X of shape (K,p,p);
    ``info['status']`` is 'optimal' or 'max iterations reached'; with ``measure=True`` also the per-outer-iteration
    'runtime', 'residual' (KKT residual) and 'objective'.
    """
    _check(S, lambda1, lambda2, reg, Omega_0)
    Theta_0 = None if len(Theta_0) == 0 else Theta_0
    X_0 = None if len(X_0) == 0 else X_0
    Omega, Theta, X, res = run_ppdna(S, float(lambda1), float(lambda2), reg, Omega_0, Theta_0, X_0,
                                     ppdna_params=ppdna_params, eps_ppdna=eps_ppdna, verbose=verbose, measure=measure)
    return _finish(Omega, Theta, X, res, measure, "PPDNA")


def warmPPDNA(S, lambda1, lambda2, reg, Omega_0, Theta_0=np.array([]), X_0=np.array([]), admm_params=dict(),
              ppdna_params=dict(), eps=1e-5, eps_admm=1e-3, verbose=False, measure=False):
    """ADMM_MGL (KKT criterion, rho = 1 fixed) to ``eps_admm``, then PPDNA from its Omega, Theta and unscaled dual
    to ``eps``.  The ADMM state stays on the device between the two phases."""
    _check(S, lambda1, lambda2, reg, Omega_0)
    t0 = time.time()
    kw = dict(admm_params)
    st, res = run_admm('mgl', S, Omega_0, None if len(Theta_0) == 0 else Theta_0, None if len(X_0) == 0 else X_0,
                       lambda1=float(lambda1), lambda2=float(lambda2), reg=reg, rho=1.0,
                       max_iter=int(kw.pop('max_iter', 1000)), tol=eps_admm, rtol=eps_admm, stopping_criterion='kkt',
                       update_rho=False, verbose=verbose, check_symmetric=True,
                       header="------------ADMM Algorithm for Multiple Graphical Lasso----------------", **kw)
    print(f"ADMM terminated after {int(res['iters'][0])} iterations with status: {res['status'][0]}.")
    t_admm = time.time() - t0
    # rho = 1 and no rho updates: st.X is the unscaled dual rho X
    Omega, Theta, X, pres = run_ppdna(st.S, float(lambda1), float(lambda2), reg, st.Omega, st.Theta, st.X,
                                      ppdna_params=ppdna_params, eps_ppdna=eps, verbose=verbose, measure=measure)
    elapsed = None
    if measure and len(pres['runtime']):
        elapsed = pres['runtime'].copy()
        elapsed[0] += t_admm
    return _finish(Omega, Theta, X, pres, measure, "PPDNA", elapsed)
