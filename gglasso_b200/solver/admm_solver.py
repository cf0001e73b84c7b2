"""ADMM_MGL on B200 -- drop-in for gglasso.solver.admm_solver.ADMM_MGL.

Same signature, defaults, asserts, printed termination line, return dicts and status strings as
the reference (src/gglasso/solver/admm_solver.py:13-313); the iteration itself runs as CUDA
kernels (see gglasso_b200/_engine.py).  numpy in, numpy out.
"""
import warnings
from typing import Optional, Union

import numpy as np

from .._engine import K_TILE_MAX, require_cuda, run_admm, to_dev, to_host


def ADMM_MGL(S: np.ndarray,
             lambda1: float,
             lambda2: float,
             reg: str,
             Omega_0: np.ndarray,
             Theta_0: np.ndarray = np.array([]),
             X_0: np.ndarray = np.array([]),
             n_samples: Optional[Union[int, np.ndarray]] = None,
             tol: float = 1e-5,
             rtol: float = 1e-4,
             stopping_criterion: str = 'boyd',
             update_rho: bool = True,
             rho: float = 1.,
             max_iter: int = 1000,
             verbose: bool = False,
             measure: bool = False,
             latent: bool = False,
             mu1: Optional[Union[float, np.ndarray]] = None
             ):
    """(Latent variable) Multiple Graphical Lasso by ADMM; see the reference docstring for the model.

    Returns ``(sol, info)``: ``sol`` has keys Omega, Theta, L, X of shape (K,p,p); ``info['status']`` is one of
    'optimal', 'primal optimal', 'dual optimal', 'max iterations reached'; with ``measure=True`` also
    'runtime', 'residual', 'objective' (length = number of iterations).
    """
    assert Omega_0.shape == S.shape
    assert S.shape[1] == S.shape[2]
    assert reg in ['GGL', 'FGL']
    assert min(lambda1, lambda2) > 0
    assert stopping_criterion in ['boyd', 'kkt']

    (K, p, p) = S.shape

    assert rho > 0, "ADMM penalization parameter must be positive."

    mu = None
    if latent:
        if isinstance(mu1, float):
            mu1 = mu1 * np.ones(K)
        assert mu1 is not None
        assert np.all(mu1 > 0)
        mu = np.asarray(mu1, dtype=np.float64).reshape(K)

    # n_samples None -> weights 1; int -> same weight for all k (admm_solver.py:133-139)
    if n_samples is None:
        nk = None
    elif isinstance(n_samples, (int, np.integer)):
        nk = float(n_samples) * np.ones(K)
    else:
        nk = np.asarray(n_samples, dtype=np.float64).reshape(K)
        assert len(nk) == K

    if len(Theta_0) == 0:
        Theta_0 = None          # device-side default: copy of Omega_0
    if len(X_0) == 0:
        X_0 = None              # device-side default: zeros
    # prox_p asserts symmetry of its input (ggl_helper.py:193); with symmetric S and start points the
    # iterates stay symmetric, so the check is done once on the inputs -- on the device, after the upload
    # (run_admm(check_symmetric=True)), not with host-side temporaries.

    st, res = run_admm('mgl', S, Omega_0, Theta_0, X_0, lambda1=float(lambda1), lambda2=float(lambda2), reg=reg,
                       rho=float(rho), max_iter=int(max_iter), tol=tol, rtol=rtol,
                       stopping_criterion=stopping_criterion, update_rho=update_rho, verbose=verbose,
                       measure=measure, latent=latent, mu=mu, nk=nk, check_symmetric=True,
                       header="------------ADMM Algorithm for Multiple Graphical Lasso----------------")
    n_it = int(res["iters"][0])
    status = res["status"][0]
    print(f"ADMM terminated after {n_it} iterations with status: {status}.")

    Omega_d = st.final_omega(res["iters"])
    ### CHECK FOR SYMMETRY
    for name, A in (("Omega", Omega_d), ("Theta", st.Theta), ("L", st.L)):
        if A is None:
            continue
        dev_max = st.asym_max(A)
        if dev_max > 1e-5:
            warnings.warn(f"{name} variable is not symmetric, largest deviation is {dev_max}.")

    ### CHECK FOR POSDEF (eigenvalue computations are enqueued first and overlap the D2H copies of the solution)
    TL = st.Theta - st.L if latent else st.Theta
    loop_done = st.mark()
    pd_min = st.posdef_async(TL, res)
    psd_min = st.posdef_async(st.L) if latent else None
    outs = st.to_host_overlapped([Omega_d, st.Theta, st.X] + ([st.L] if latent else []), after=loop_done)
    if pd_min is not None and float(pd_min.item()) <= 0:
        print("WARNING: Theta (Theta - L resp.) is not positive definite. Solve to higher accuracy!")
    if latent:
        if float(psd_min.item()) < -1e-5:
            print("WARNING: L is not positive semidefinite. Solve to higher accuracy!")

    sol = {'Omega': outs[0], 'Theta': outs[1], 'L': outs[3] if latent else np.zeros((K, p, p)), 'X': outs[2]}
    if measure:
        info = {'status': status,
                'runtime': res["runtime"][:n_it],
                'residual': res["residual"][0],
                'objective': res["objective"][:n_it]}
    else:
        info = {'status': status}
    return sol, info


def _per_problem(a, name, K, p):
    """(K,p,p) shared by every problem -> (None, array); (B,K,p,p) one per problem -> (B, array)"""
    a = np.asarray(a, dtype=np.float64)
    assert a.ndim in (3, 4) and a.shape[-3:] == (K, p, p), f"{name} must have shape (K,p,p) or (B,K,p,p)"
    return (a.shape[0] if a.ndim == 4 else None), a


def ADMM_MGL_batch(S: np.ndarray,
                   lambda1: Union[float, np.ndarray],
                   lambda2: Union[float, np.ndarray],
                   reg: str,
                   Omega_0: np.ndarray,
                   Theta_0: Optional[np.ndarray] = None,
                   X_0: Optional[np.ndarray] = None,
                   n_samples: Optional[Union[int, np.ndarray]] = None,
                   tol: float = 1e-5,
                   rtol: float = 1e-4,
                   update_rho: bool = True,
                   rho: float = 1.,
                   max_iter: int = 1000,
                   verbose: bool = False,
                   latent: bool = False,
                   mu1: Optional[Union[float, np.ndarray]] = None):
    """Solve B independent (latent variable) Multiple Graphical Lasso problems of the same K and p in one device loop:
    lambda paths and grids, stability selection / bootstrap on resampled covariances, cross-validation folds.

    ``S``, ``Omega_0``, ``Theta_0``, ``X_0``: (K,p,p) shared by every problem or (B,K,p,p), one per problem;
    ``Theta_0 = None`` / ``X_0 = None`` mean ADMM_MGL's defaults Theta_0 = Omega_0 and X_0 = 0.  ``lambda1``,
    ``lambda2``: scalars or length-B arrays.  ``mu1`` (latent): scalar, (K,) or (B,K).  The batch size B is the common
    length of all these; a mismatch raises AssertionError.  ``n_samples``, ``reg``, ``latent``, ``tol``, ``rtol``,
    ``rho``, ``update_rho`` and ``max_iter`` are shared.

    Returns a list of B pairs ``(sol, info)``: ``sol`` as returned by ADMM_MGL for that problem alone (Omega, Theta, L,
    X of shape (K,p,p); L is zero when not latent), ``info = {'status', 'residual'}`` with the problem's status string
    and max(r_t, s_t) of each of its iterations.  Each problem runs the iterations ADMM_MGL would run for it, with its
    own rho and stopping test; a problem that has converged is skipped by every kernel while the others continue.

    The Boyd stopping criterion is the only one: ``stopping_criterion='kkt'`` and ``measure=True`` of ADMM_MGL are not
    parameters of the batch.  K > 90 (ADMM_MGL's row-band prox) raises NotImplementedError.  A shared S or start point
    is replicated on the device (B*K*p*p doubles per array).  Symmetry and positive-definiteness warnings are issued
    with ``warnings.warn`` and name the problem; nothing is printed unless ``verbose``, which prints one termination
    line per problem.  A non-finite iterate raises GGLassoB200Error naming the problems.
    """
    S = np.asarray(S, dtype=np.float64)
    assert S.ndim in (3, 4), "S must have shape (K,p,p) or (B,K,p,p)"
    assert S.shape[-2] == S.shape[-1]
    (K, p, p) = S.shape[-3:]
    S_B = S.shape[0] if S.ndim == 4 else None
    assert reg in ['GGL', 'FGL']
    lam1 = np.asarray(lambda1, dtype=np.float64)
    lam2 = np.asarray(lambda2, dtype=np.float64)
    assert lam1.ndim <= 1 and lam2.ndim <= 1, "lambda1 and lambda2 must be scalars or length-B arrays"
    assert min(lam1.min(), lam2.min()) > 0
    assert rho > 0, "ADMM penalization parameter must be positive."
    if K > K_TILE_MAX:
        raise NotImplementedError(f"ADMM_MGL_batch supports K <= {K_TILE_MAX} (tile-pair prox); got K = {K}. "
                                  "Solve such problems one at a time with ADMM_MGL.")

    Om_B, Omega_0 = _per_problem(Omega_0, "Omega_0", K, p)
    Th_B = X_B = None
    if Theta_0 is not None:
        Th_B, Theta_0 = _per_problem(Theta_0, "Theta_0", K, p)
    if X_0 is not None:
        X_B, X_0 = _per_problem(X_0, "X_0", K, p)
    mu = mu_B = None
    if latent:
        if isinstance(mu1, (float, int)) and not isinstance(mu1, bool):
            mu1 = mu1 * np.ones(K)
        assert mu1 is not None
        mu = np.asarray(mu1, dtype=np.float64)
        assert np.all(mu > 0)
        assert mu.shape == (K,) or (mu.ndim == 2 and mu.shape[1] == K), "mu1 must be a scalar, (K,) or (B,K)"
        mu_B = mu.shape[0] if mu.ndim == 2 else None

    sizes = [n for n in (S_B, Om_B, Th_B, X_B, mu_B) + tuple(len(l) for l in (lam1, lam2) if l.ndim == 1)
             if n is not None]
    B = max(sizes, default=1)
    assert all(n in (1, B) for n in sizes), f"batch sizes do not match: {sorted(set(sizes))}"
    assert B >= 1
    lam1 = np.broadcast_to(lam1, (B,)).copy()
    lam2 = np.broadcast_to(lam2, (B,)).copy()

    if n_samples is None:
        nk = None
    elif isinstance(n_samples, (int, np.integer)):
        nk = float(n_samples) * np.ones(K)
    else:
        nk = np.asarray(n_samples, dtype=np.float64).reshape(K)
    if nk is not None:
        nk = np.tile(nk, B)
    if mu is not None:
        mu = np.broadcast_to(mu, (B, K)).reshape(B * K).copy()

    dev = require_cuda()

    def stack(a, n):
        """(B*K,p,p) stack of a per-problem array (uploaded as is) or of a shared one (replicated on the device)"""
        if a is None:
            return None
        if a.ndim == 4 and n == B:
            return a.reshape(B * K, p, p)
        return to_dev(a.reshape(K, p, p), dev).repeat(B, 1, 1)

    st, res = run_admm('mgl', stack(S, S_B), stack(Omega_0, Om_B), stack(Theta_0, Th_B), stack(X_0, X_B),
                       lambda1=lam1, lambda2=lam2, reg=reg, rho=float(rho), max_iter=int(max_iter), tol=tol,
                       rtol=rtol, stopping_criterion='boyd', update_rho=update_rho, latent=latent, mu=mu, nk=nk,
                       check_symmetric=True, K=K)
    iters, statuses = res["iters"], res["status"]
    if verbose:
        for b in range(B):
            print(f"problem {b}: ADMM terminated after {int(iters[b])} iterations with status: {statuses[b]}.")

    Omega_d = st.final_omega(iters)
    ### CHECK FOR SYMMETRY, per problem
    for name, A in (("Omega", Omega_d), ("Theta", st.Theta), ("L", st.L)):
        if A is None:
            continue
        dev_max = st.asym_max(A, per_problem=True)
        for b in np.flatnonzero(dev_max > 1e-5):
            warnings.warn(f"problem {b}: {name} variable is not symmetric, largest deviation is {dev_max[b]}.")

    ### CHECK FOR POSDEF, per problem (eigenvalues enqueued before the D2H copies of the solution)
    loop_done = st.mark()
    pd_min = st.min_eig_per_problem(st.Theta - st.L if latent else st.Theta)
    psd_min = st.min_eig_per_problem(st.L) if latent else None
    outs = st.to_host_overlapped([Omega_d, st.Theta, st.X] + ([st.L] if latent else []), after=loop_done)
    outs = [o.reshape(B, K, p, p) for o in outs]
    for b in np.flatnonzero(pd_min.cpu().numpy() <= 0):
        warnings.warn(f"problem {b}: Theta (Theta - L resp.) is not positive definite. Solve to higher accuracy!")
    if latent:
        for b in np.flatnonzero(psd_min.cpu().numpy() < -1e-5):
            warnings.warn(f"problem {b}: L is not positive semidefinite. Solve to higher accuracy!")

    results = []
    for b in range(B):
        sol = {'Omega': outs[0][b], 'Theta': outs[1][b], 'L': outs[3][b] if latent else np.zeros((K, p, p)),
               'X': outs[2][b]}
        results.append((sol, {'status': statuses[b], 'residual': res["residual"][b]}))
    return results
