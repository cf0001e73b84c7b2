"""ext_ADMM_MGL on B200 -- drop-in for gglasso.solver.ext_admm_solver.ext_ADMM_MGL
(src/gglasso/solver/ext_admm_solver.py:18-327): group graphical lasso for NON-conforming instances (each
instance k has its own dimension p_k; the group penalty couples the entries listed in the bookkeeping array G).

Same signature, asserts, printed lines and return dicts (dicts keyed 0..K-1).  On the device the K matrices are
padded to a common size with decoupled unit diagonal entries (exact fixed points of every update, masked out of
the residual norms), so the batched eigensolver / reconstruction kernels of the conforming path are reused; the
Theta update, the group prox through G and the two dual updates are dedicated kernels (gg_ext_*).
"""
import time
import warnings
from typing import Optional

import numpy as np
import torch

from .. import _lib
from .._engine import AdmmState, _p, boyd_status, control_block, to_dev, to_host
from .._lib import C_DONE, C_ITER, NPART


def check_G(G, p):
    """validation of the bookkeeping array (reference: src/gglasso/helper/ext_admm_helper.py:82-104)."""
    K = G.shape[2]
    assert np.issubdtype(G.dtype, np.integer), "G needs to be an integer array"
    assert np.all(G.sum(axis=2) >= -K), "G has rows with only -1 entries"
    assert np.all(((G == -1).sum(axis=0) == 2) | ((G == -1).sum(axis=0) == 0)), "Only row or column index specified in some group"
    assert np.all((G[0, :, :] + G[1, :, :] == -2) | (G[0, :, :] != G[1, :, :])), "G has entries on the diagonal!"
    assert np.all(G >= -1), "No negative indices allowed (only -1 for indicating a missing feature)"
    assert np.all(G.max(axis=(0, 1)) < p), "indices larger as dimension were found"
    assert np.all(G[0, :, :] <= G[1, :, :]), "Only upper diagonal entries should be contained in G"


def _assert_disjoint_groups(G):
    """The group prox kernel handles all groups in parallel, which is the reference's sequential in-place loop
    (ext_admm_solver.py:394-453) only if no entry (k, i, j) belongs to two groups -- what create_group_array /
    construct_trivial_G produce.  Overlapping groups are rejected instead of being solved differently."""
    Lg, K = G.shape[1], G.shape[2]
    for k in range(K):
        i, j = G[0, :, k], G[1, :, k]
        m = i >= 0
        key = i[m].astype(np.int64) * (int(G.max()) + 2) + j[m]
        assert len(np.unique(key)) == len(key), f"instance {k}: an entry belongs to more than one group (unsupported)"


def _pad(d, K, p, pm, fill_diag):
    out = np.zeros((K, pm, pm))
    for k in range(K):
        out[k, :p[k], :p[k]] = d[k]
        if fill_diag:
            idx = np.arange(p[k], pm)
            out[k, idx, idx] = 1.0
    return out


def ext_ADMM_MGL(S: dict,
                 lambda1: float,
                 lambda2: float,
                 reg: str,
                 Omega_0: dict,
                 G: np.ndarray,
                 X0: Optional[dict] = None,
                 X1: Optional[dict] = None,
                 tol: float = 1e-5,
                 rtol: float = 1e-4,
                 stopping_criterion: str = 'boyd',
                 rho: float = 1.,
                 max_iter: int = 1000,
                 verbose: bool = False,
                 measure: bool = False,
                 latent: bool = False,
                 mu1: Optional[float] = None
                 ):
    """ADMM for the (latent variable) Group Graphical Lasso with non-conforming dimensions; see the reference
    docstring for the model.  Returns ``(sol, info)``; sol has keys Omega, Theta, L, X0, X1, each a dict over k."""
    K = len(S.keys())
    p = np.zeros(K, dtype=int)
    for k in np.arange(K):
        p[k] = S[k].shape[0]

    if isinstance(lambda1, float):
        lambda1 = lambda1 * np.ones(K)
    if latent:
        if isinstance(mu1, float):
            mu1 = mu1 * np.ones(K)
        assert mu1 is not None
        assert np.all(mu1 > 0)

    assert min(lambda1.min(), lambda2) > 0
    assert reg in ['GGL']
    check_G(G, p)
    _assert_disjoint_groups(G)
    assert rho > 0, "ADMM penalization parameter must be positive."
    assert stopping_criterion in ['boyd', 'kkt']

    pm = int(p.max())
    lib = _lib.load()
    Sp = _pad(S, K, p, pm, True)
    Op = _pad(Omega_0, K, p, pm, True)
    X0p = None if X0 is None else _pad(X0, K, p, pm, False)
    st = AdmmState(Sp, Op, None, X0p, K, float(rho), int(max_iter), latent,
                   mu=None if not latent else np.asarray(mu1, dtype=np.float64))
    dev, stream = st.dev, st.stream
    st.pdim.fill_(float(((p ** 2 + p) / 2).sum()))
    pvec = torch.from_numpy(p.astype(np.int32)).to(dev)
    lam1 = to_dev(np.asarray(lambda1, dtype=np.float64), dev)
    Gd = torch.from_numpy(np.ascontiguousarray(G).astype(np.int32)).to(dev)
    Lg = int(G.shape[1])
    X1d = torch.zeros_like(st.S) if X1 is None else to_dev(_pad(X1, K, p, pm, False), dev)
    Lam, Lam_new = st.Omega.clone(), torch.empty_like(st.Omega)       # Lambda_0 = Omega_0
    nparts = lib.gg_sgl_nparts(pm, K) * K
    partials = torch.zeros((nparts, NPART), dtype=torch.float64, device=dev)
    mask = None

    runtime = np.zeros(max_iter)
    kkt_res = np.zeros(max_iter)
    status = ''
    if verbose:
        print("------------ADMM Algorithm for Multiple Graphical Lasso----------------")
        if stopping_criterion == 'boyd':
            print("%4s\t%10s\t%10s\t%10s\t%10s" % ("iter", "r_t", "s_t", "eps_pri", "eps_dual"))
        else:
            print("%4s\t%10s" % ("iter", "kkt residual"))

    it_done = 0
    for it in range(max_iter):
        if measure:
            torch.cuda.synchronize()
            start = time.time()
        st.omega_step()
        C = st.W if latent else None
        _lib.check(lib.gg_ext_theta(_p(st.Omega_new), _p(st.L), _p(st.X), _p(Lam), _p(X1d), _p(lam1), _p(st.ctrl), K, pm,
                                    _p(st.Theta), _p(C), stream), "gg_ext_theta")
        if latent:
            st.l_step()
        _lib.check(lib.gg_ext_lambda(_p(st.Theta), _p(X1d), _p(Gd), Lg, K, pm, float(lambda2), _p(st.ctrl), _p(Lam_new),
                                     stream), "gg_ext_lambda")
        _lib.check(lib.gg_ext_dual(_p(st.X), _p(X1d), _p(st.Omega_new), _p(st.Omega), _p(st.Theta), _p(st.L), _p(Lam_new),
                                   _p(Lam), _p(st.ctrl), _p(pvec), K, pm, _p(partials), stream), "gg_ext_dual")
        if measure:
            torch.cuda.synchronize()
            runtime[it] = time.time() - start
        it_done = it + 1
        if stopping_criterion == 'boyd':
            _lib.check(lib.gg_stop_update(_p(partials), nparts, _p(st.ctrl), _p(st.hist), st.hist_cap, _p(st.pdim),
                                          tol, rtol, 0, 1, stream), "gg_stop_update")
            st.swap()
            Lam, Lam_new = Lam_new, Lam
            ctrl = st.read_ctrl()
            if verbose:
                h = st.hist[0, it].cpu().numpy()
                print("%4d\t%10.4g\t%10.4g\t%10.4g\t%10.4g" % (it, h[0], h[1], h[2], h[3]))
            if ctrl[0, C_DONE] != 0:
                break
        else:
            st.swap()
            Lam, Lam_new = Lam_new, Lam
            if mask is None:
                ar = torch.arange(pm, device=dev)
                mk = (ar[None, :] < pvec[:, None].to(torch.int64))
                mask = (mk[:, :, None] & mk[:, None, :]).to(torch.float64)
            eta = _kkt(st, Lam, X1d, Gd, Lg, lam1, float(lambda2), latent, mask, lib, stream)
            kkt_res[it] = eta
            if verbose:
                print("%4d\t%10.4g" % (it, eta))
            if eta <= tol:
                status = 'optimal'
                break

    ctrl = st.read_ctrl()
    if stopping_criterion == 'boyd':
        n_it = int(ctrl[0, C_ITER])
        status, residual = boyd_status(ctrl[0], st.hist[0, :n_it].cpu().numpy())
    else:
        n_it = it_done
        if status != 'optimal':
            status = 'max iterations reached'
        residual = kkt_res[:n_it]
    print(f"ADMM terminated after {n_it} iterations with status: {status}.")

    Omega_d = st.final_omega([n_it])
    Om, Th, X0h, X1h = to_host(Omega_d), to_host(st.Theta), to_host(st.X), to_host(X1d)
    Lh = to_host(st.L) if latent else np.zeros((K, pm, pm))
    TL = st.Theta - st.L if latent else st.Theta
    D = st.eigvalsh(TL).cpu().numpy()
    DL = st.eigvalsh(st.L).cpu().numpy() if latent else None
    sol = {'Omega': {}, 'Theta': {}, 'L': {}, 'X0': {}, 'X1': {}}
    for k in range(K):
        n = p[k]
        for name, arr in (('Omega', Om), ('Theta', Th), ('L', Lh), ('X0', X0h), ('X1', X1h)):
            sol[name][k] = arr[k, :n, :n].copy()
        for name in ('Omega', 'Theta', 'L'):
            dev_max = abs(sol[name][k].T - sol[name][k]).max()
            if dev_max > 1e-5:
                warnings.warn(f"{name} variable is not symmetric, largest deviation is {dev_max}.")
        # the padded diagonal only adds eigenvalues 1 (0 for L), so the thresholds see the true block
        if D[k].min() <= 1e-5:
            print("WARNING: Theta (Theta-L resp.) may be not positive definite -- increase accuracy!")
        if latent and DL[k].min() <= -1e-5:
            print("WARNING: L may be not positive semidefinite -- increase accuracy!")

    if measure:
        info = {'status': status, 'runtime': runtime[:n_it], 'residual': residual}
    else:
        info = {'status': status}
    return sol, info


def _kkt(st, Lam, X1d, Gd, Lg, lam1, lambda2, latent, mask, lib, stream):
    """KKT residual of the non-conforming problem (ext_admm_solver.py:349-392).  prox / eigendecompositions run
    through the CUDA kernels; norms and differences of resident arrays are torch glue on the device."""
    from .._lib import C_RHO
    K, pm = st.M, st.p
    dev = st.dev
    rho = st.ctrl[0, C_RHO]
    Omega, Theta = st.Omega, st.Theta
    L = st.L if latent else torch.zeros_like(Theta)
    X0u, X1u = rho * st.X, rho * X1d
    ctrl1 = torch.from_numpy(control_block(1, 1.0)).to(dev, non_blocking=True)

    def nrm(A):
        return torch.sqrt(((A * mask) ** 2).sum((1, 2)))

    A = (Omega - st.S - X0u).contiguous()       # padded diagonal: 1 - 1 - 0 = 0 -> phi+(0, 1) = 1 = Omega there
    P = torch.empty_like(Theta)
    st.eig.eigh(A, stream=stream)
    st.eig.recon(A, P, 0, bnum=None, ctrl=None, stream=stream)
    t1 = nrm(Omega - P) / (1 + nrm(Omega))
    # Theta - prox_od_1norm(Theta + X0 - X1, lambda1_k): ext_theta computes prox((Om+L+X0+Lam-X1)/2, lam1/(2 rho));
    # feed Om := 2*(Theta + X0 - X1), everything else zero, rho = 1 and lam1 doubled
    Z = torch.zeros_like(Theta)
    V2 = (2.0 * (Theta + X0u - X1u)).contiguous()
    lam2x = (2.0 * lam1).contiguous()
    _lib.check(lib.gg_ext_theta(_p(V2), None, _p(Z), _p(Z), _p(Z), _p(lam2x), _p(ctrl1), K, pm, _p(P), None, stream),
               "gg_ext_theta")
    t2 = nrm(Theta - P) / (1 + nrm(Theta))
    t3 = torch.zeros(K, dtype=torch.float64, device=dev)
    if latent:
        A = (L - X0u).contiguous()
        st.eig.eigh(A, stream=stream)
        st.eig.recon(A, P, 1, bnum=st.mu, ctrl=None, stream=stream)
        t3 = nrm(L - P) / (1 + nrm(L))
    # V = prox_2norm_G(Lambda + X1, G, lambda2)
    _lib.check(lib.gg_ext_lambda(_p(Lam), _p(X1u.contiguous()), _p(Gd), Lg, K, pm, lambda2, _p(ctrl1), _p(P), stream),
               "gg_ext_lambda")
    t4 = nrm(P - Lam) / (1 + nrm(Lam))
    t5 = nrm(Omega - Theta + L) / (1 + nrm(Theta))
    t6 = nrm(Lam - Theta) / (1 + nrm(Theta))
    return float(torch.stack([torch.linalg.norm(t) for t in (t1, t2, t3, t4, t5, t6)]).max().item())
