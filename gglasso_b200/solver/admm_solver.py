"""ADMM_MGL on B200 -- drop-in for gglasso.solver.admm_solver.ADMM_MGL.

Same signature, defaults, asserts, printed termination line, return dicts and status strings as
the reference (src/gglasso/solver/admm_solver.py:13-313); the iteration itself runs as CUDA
kernels (see gglasso_b200/_engine.py).  numpy in, numpy out.
"""
import warnings
from typing import Optional, Union

import numpy as np
import torch
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components

from .. import _lib
from .._engine import K_TILE_MAX, _p, require_cuda, run_admm, to_dev, to_host
from .single_admm_solver import _BATCH_MAX, _size_buckets


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


#######################################################
## BLOCK-WISE MULTIPLE GRAPHICAL LASSO (exact component screen)
#######################################################

def _class_weights(n_samples, K):
    """n_samples -> (K,) class weights n_k as ADMM_MGL reads them (None: weights 1, returned as None)"""
    if n_samples is None:
        return None
    if isinstance(n_samples, (int, np.integer)):
        return float(n_samples) * np.ones(K)
    nk = np.asarray(n_samples, dtype=np.float64).reshape(K)
    assert len(nk) == K
    return nk


def _mgl_screen(S_dev, nk, lambda1, lambda2, reg):
    """device screen (gg_mgl_screen) of a (K,p,p) device stack: upper-triangle bitmask, (p, ceil(p/32)) uint32 numpy"""
    lib = _lib.load()
    K, p, _ = S_dev.shape
    adj = torch.empty((p, (p + 31) // 32), dtype=torch.int32, device=S_dev.device)
    nk_dev = None if nk is None else to_dev(nk, S_dev.device)
    _lib.check(lib.gg_mgl_screen(_p(S_dev), _p(nk_dev), float(lambda1), float(lambda2), 0 if reg == "GGL" else 1, K,
                                 p, _p(adj), torch.cuda.current_stream().cuda_stream), "gg_mgl_screen")
    return adj.cpu().numpy().view(np.uint32)


def _components_from_bitmask(words, p):
    """connected components of the graph whose upper-triangle adjacency is the bitmask ``words`` (p rows of
    ceil(p/32) words, bit b of word w = column 32 w + b); (numC, allC) as get_connected_components returns them:
    components labelled in order of their smallest node, each an ascending index array."""
    words = np.ascontiguousarray(words, dtype="<u4").reshape(p, -1)
    bits = np.unpackbits(words.view(np.uint8), axis=1, bitorder="little")[:, :p]
    i, j = np.nonzero(bits)
    G = csr_matrix((np.ones(len(i), dtype=np.int8), (i, j)), shape=(p, p))
    numC, labels = connected_components(G, directed=False, return_labels=True)
    order = np.argsort(labels, kind="stable")
    allC = np.split(order, np.cumsum(np.bincount(labels, minlength=numC))[:-1])
    return numC, allC


def mgl_connected_components(S: np.ndarray,
                             lambda1: float,
                             lambda2: float,
                             reg: str,
                             n_samples: Optional[Union[int, np.ndarray]] = None):
    """Connected components of the exact MGL screening graph: (i, j) is an edge iff prox_P(s_ij) != 0, with
    s_ij = (n_k S_k,ij)_k and P the GGL / FGL penalty of one entry (the prox of the ADMM loop at rho = 1).  The MGL
    solution is block diagonal over these components (Danaher, Wang & Witten 2014, section 5).

    The screen runs on the device (gg_mgl_screen), the component search on the host (scipy).  Returns ``(numC, allC)``
    in the order convention of get_connected_components.  K <= 90.
    """
    S = np.asarray(S, dtype=np.float64)
    assert S.ndim == 3 and S.shape[1] == S.shape[2]
    assert reg in ['GGL', 'FGL']
    assert min(lambda1, lambda2) > 0
    (K, p, p) = S.shape
    if K > K_TILE_MAX:
        raise NotImplementedError(f"the MGL screen supports K <= {K_TILE_MAX}; got K = {K}")
    nk = _class_weights(n_samples, K)
    words = _mgl_screen(to_dev(S, require_cuda()), nk, lambda1, lambda2, reg)
    return _components_from_bitmask(words, p)


def block_MGL(S: np.ndarray,
              lambda1: float,
              lambda2: float,
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
              latent: bool = False):
    """Multiple Graphical Lasso (GGL / FGL) solved component by component of the exact screening graph of
    mgl_connected_components, and reassembled; the result is the solution of the full problem.

    Singletons take the closed form Omega_k,ii = Theta_k,ii = 1/S_k,ii (X = 0).  Components of 2..160 nodes are solved
    in ragged device batches (padded to the size bucket of block_SGL, each with its own rho and stopping test); larger
    ones one at a time through ADMM_MGL's device loop.  Each component runs the iterations ADMM_MGL would run on it
    alone, with the Boyd criterion (``stopping_criterion='kkt'`` and ``measure`` are not parameters).  ``latent=True``
    (the latent model does not decompose over components) and K > 90 raise NotImplementedError.  S must be symmetric.

    Returns ``(sol, info)``: ``sol`` has Omega, Theta, L (zeros) and X of shape (K,p,p), zero outside the components;
    X of a component is its scaled dual at its own final rho.  ``info``: 'status' ('optimal' iff every component is,
    otherwise the first other status in component order), 'components' (index arrays), 'component_status',
    'component_iters' (0 for singletons) and 'component_rho'.  Symmetry and positive-definiteness warnings are issued
    with ``warnings.warn`` and name the component; nothing is printed unless ``verbose``, which prints one termination
    line per component of two or more nodes.
    """
    assert Omega_0.shape == S.shape
    assert S.shape[1] == S.shape[2]
    assert reg in ['GGL', 'FGL']
    assert min(lambda1, lambda2) > 0

    (K, p, p) = S.shape

    assert rho > 0, "ADMM penalization parameter must be positive."
    if latent:
        raise NotImplementedError("block_MGL solves the non-latent problem only (the low-rank term couples the "
                                  "components); use ADMM_MGL with latent=True.")
    if K > K_TILE_MAX:
        raise NotImplementedError(f"block_MGL supports K <= {K_TILE_MAX} (tile-pair prox); got K = {K}. "
                                  "Use ADMM_MGL.")

    S = np.asarray(S, dtype=np.float64)
    Omega_0 = np.asarray(Omega_0, dtype=np.float64)
    Theta_0 = Omega_0 if Theta_0 is None else np.asarray(Theta_0, dtype=np.float64)
    X_0 = np.zeros((K, p, p)) if X_0 is None else np.asarray(X_0, dtype=np.float64)
    assert Theta_0.shape == S.shape and X_0.shape == S.shape
    nk = _class_weights(n_samples, K)

    numC, allC = _components_from_bitmask(_mgl_screen(to_dev(S, require_cuda()), nk, lambda1, lambda2, reg), p)
    sol = {'Omega': np.zeros((K, p, p)), 'Theta': np.zeros((K, p, p)), 'L': np.zeros((K, p, p)),
           'X': np.zeros((K, p, p))}
    out = {'status': ['optimal'] * numC, 'iters': np.zeros(numC, dtype=int), 'rho': np.full(numC, float(rho))}
    for C in allC:
        if len(C) == 1:
            i = C[0]
            sol['Omega'][:, i, i] = 1 / S[:, i, i]
            sol['Theta'][:, i, i] = 1 / S[:, i, i]

    kw = dict(lambda1=float(lambda1), lambda2=float(lambda2), reg=reg, rho=float(rho), max_iter=int(max_iter),
              tol=tol, rtol=rtol, stopping_criterion='boyd', update_rho=update_rho, check_symmetric=True)
    small = [ci for ci, C in enumerate(allC) if 1 < len(C) <= _BATCH_MAX]
    large = [ci for ci, C in enumerate(allC) if len(C) > _BATCH_MAX]
    # a batch index travels in gridDim.y (limit 65535 matrices per loop) and every problem keeps a (max_iter, 5)
    # residual history on the device: batches are cut so that both stay bounded
    step = max(1, min(65535 // K, (256 << 20) // (40 * int(max_iter))))
    for bucket in _size_buckets([len(allC[ci]) for ci in small]):
        for lo in range(0, len(bucket), step):
            ids = [small[k] for k in bucket[lo:lo + step]]
            _solve_mgl_batch(S, Omega_0, Theta_0, X_0, nk, [allC[ci] for ci in ids], ids, kw, sol, out)
    for ci in large:
        _solve_mgl_large(S, Omega_0, Theta_0, X_0, nk, allC[ci], ci, kw, sol, out)

    if verbose:
        for ci, C in enumerate(allC):
            if len(C) > 1:
                print(f"component {ci} ({len(C)} nodes): ADMM terminated after {out['iters'][ci]} iterations with "
                      f"status: {out['status'][ci]}.")
    status = next((st for st in out['status'] if st != 'optimal'), 'optimal')
    info = {'status': status, 'components': allC, 'component_status': out['status'],
            'component_iters': out['iters'], 'component_rho': out['rho']}
    return sol, info


def _block(A, C):
    """(K, |C|, |C|) sub-block of a (K,p,p) array on the nodes C"""
    return np.ascontiguousarray(A[:, C[:, None], C[None, :]])


def _solve_mgl_batch(S, Omega_0, Theta_0, X_0, nk, comps, ids, kw, sol, out):
    """one ragged batch of components: each padded to the largest size with decoupled unit diagonal entries
    (S = Omega = Theta = I, X = 0: exact fixed points of the iteration for every rho and weight, left out of the
    residual norms through pvec), as block_SGL does"""
    B, K = len(comps), S.shape[0]
    pm = max(len(C) for C in comps)
    Sb = np.broadcast_to(np.eye(pm), (B, K, pm, pm)).copy()
    Ob, Tb, Xb = Sb.copy(), Sb.copy(), np.zeros((B, K, pm, pm))
    for b, C in enumerate(comps):
        n = len(C)
        Sb[b, :, :n, :n] = _block(S, C)
        Ob[b, :, :n, :n] = _block(Omega_0, C)
        Tb[b, :, :n, :n] = _block(Theta_0, C)
        Xb[b, :, :n, :n] = _block(X_0, C)
    M = B * K
    st, res = run_admm('mgl', Sb.reshape(M, pm, pm), Ob.reshape(M, pm, pm), Tb.reshape(M, pm, pm),
                       Xb.reshape(M, pm, pm), nk=None if nk is None else np.tile(nk, B), K=K,
                       pvec=[len(C) for C in comps], **kw)
    _collect(st, res, comps, ids, sol, out)


def _solve_mgl_large(S, Omega_0, Theta_0, X_0, nk, C, ci, kw, sol, out):
    """one component through the single-problem device loop of ADMM_MGL"""
    st, res = run_admm('mgl', _block(S, C), _block(Omega_0, C), _block(Theta_0, C), _block(X_0, C), nk=nk, **kw)
    _collect(st, res, [C], [ci], sol, out)


def _collect(st, res, comps, ids, sol, out):
    """post-loop checks (per component, as ADMM_MGL_batch does per problem) and scatter of the solutions"""
    K = st.mpp
    iters, statuses = res["iters"], res["status"]
    Omega_d = st.final_omega(iters)
    ### CHECK FOR SYMMETRY, per component
    for name, A in (("Omega", Omega_d), ("Theta", st.Theta)):
        dev_max = st.asym_max(A, per_problem=True)
        for b in np.flatnonzero(dev_max > 1e-5):
            warnings.warn(f"component {ids[b]}: {name} variable is not symmetric, largest deviation is {dev_max[b]}.")
    ### CHECK FOR POSDEF, per component (eigenvalues enqueued before the D2H copies of the solution)
    loop_done = st.mark()
    pd_min = st.min_eig_per_problem(st.Theta)
    Om, Th, Xs = st.to_host_overlapped([Omega_d, st.Theta, st.X], after=loop_done)
    for b in np.flatnonzero(pd_min.cpu().numpy() <= 0):
        warnings.warn(f"component {ids[b]}: Theta variable is not positive definite. Solve to higher accuracy!")
    for b, (C, ci) in enumerate(zip(comps, ids)):
        n = len(C)
        ix = (slice(None), C[:, None], C[None, :])
        sol['Omega'][ix] = Om[b * K:(b + 1) * K, :n, :n]
        sol['Theta'][ix] = Th[b * K:(b + 1) * K, :n, :n]
        sol['X'][ix] = Xs[b * K:(b + 1) * K, :n, :n]
        out['status'][ci] = statuses[b]
        out['iters'][ci] = int(iters[b])
        out['rho'][ci] = float(res["ctrl"][b, _lib.C_RHO])
