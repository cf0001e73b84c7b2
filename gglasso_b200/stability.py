"""Stability selection of lambda1 (StARS: Liu, Roeder & Wasserman, "Stability Approach to Regularization Selection",
NeurIPS 2010) for SGL and MGL from raw samples.

The samples stay on the device.  For each chunk of subsamples the covariances are formed there (gg_subsample_cov),
every one is solved at every lambda1 of the path in one batched ADMM loop (run_admm), and the edges of the solutions are
counted there (gg_edge_count).  Only the instabilities, the mean edge counts and the edge counts at the selected lambda1
come back to the host.
"""
import contextlib
import ctypes
import io
import warnings

import numpy as np
import torch

from . import _lib
from ._engine import K_TILE_MAX, require_cuda, run_admm, to_dev


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def default_subsample_size(n):
    """huge's / pulsar's rule: floor(10 sqrt(n)) if n > 144, else floor(0.8 n)"""
    return int(np.floor(10.0 * np.sqrt(n))) if n > 144 else int(np.floor(0.8 * n))


def draw_indices(n, b, n_subsamples, seed):
    """per class k a (B, b_k) int array of row indices: rng = default_rng(seed), then for s in range(B), for k in
    range(K), rng.choice(n_k, b_k, replace=False)"""
    rng = np.random.default_rng(seed)
    out = [np.empty((n_subsamples, bk), dtype=np.int64) for bk in b]
    for s in range(n_subsamples):
        for k in range(len(n)):
            out[k][s] = rng.choice(n[k], b[k], replace=False)
    return out


def select(instability, beta):
    """StARS rule on a path sorted by decreasing lambda1: Dbar(lambda) = max of D over the path values >= lambda, and the
    selected index is that of the smallest lambda with Dbar <= beta (0, the largest lambda, if there is none).
    Returns (Dbar, index)."""
    dbar = np.maximum.accumulate(np.asarray(instability, dtype=np.float64))
    ok = np.flatnonzero(dbar <= beta)
    return dbar, (int(ok[-1]) if len(ok) else 0)


def sample_covariance(X, scale):
    """np.cov(X, rowvar=False, bias=True), scaled by its diagonal (S_ij / (sqrt(S_ii) sqrt(S_jj))) when ``scale``"""
    S = np.atleast_2d(np.cov(X, rowvar=False, bias=True))
    if scale:
        sq = np.sqrt(np.diag(S))
        S = S / (sq[:, None] * sq[None, :])
    return S


def _check_args(data, lambda1, lambda2, reg, n_subsamples, subsample_size, beta, max_batch):
    """-> (classes as a list of (n_k,p) float64 arrays, sgl flag, sorted lambda1, b per class)"""
    if isinstance(data, (list, tuple)):
        classes = [np.asarray(x, dtype=np.float64) for x in data]
        sgl = False
        if not classes or any(x.ndim != 2 for x in classes):
            raise ValueError("data given as a list must hold K >= 1 arrays of shape (n_k, p)")
    else:
        data = np.asarray(data, dtype=np.float64)
        if data.ndim == 2:
            classes, sgl = [data], True
        elif data.ndim == 3:
            classes, sgl = list(data), False
        else:
            raise ValueError("data must be (n,p) for SGL, or (K,n,p) or a list of K (n_k,p) arrays for MGL")
    p = classes[0].shape[1]
    if any(x.shape[1] != p for x in classes):
        raise ValueError("every class must have the same number of variables p")
    if p < 2:
        raise ValueError("stability selection needs p >= 2 variables")
    if not all(np.all(np.isfinite(x)) for x in classes):
        raise ValueError("data must be finite")
    K = len(classes)
    if sgl:
        if reg is not None or lambda2 is not None:
            raise ValueError("SGL data (n,p): reg and lambda2 must be None")
    else:
        if reg not in ("GGL", "FGL"):
            raise ValueError("MGL data: reg must be 'GGL' or 'FGL'")
        if lambda2 is None or np.ndim(lambda2) != 0 or not float(lambda2) > 0:
            raise ValueError("MGL data: lambda2 must be a scalar > 0")
        if K > K_TILE_MAX:
            raise NotImplementedError(f"stability_selection supports K <= {K_TILE_MAX} (the batched MGL prox); "
                                      f"got K = {K}")
    lam = np.asarray(lambda1, dtype=np.float64)
    if lam.ndim != 1 or lam.size == 0:
        raise ValueError("lambda1 must be a 1-D array of length L > 0")
    if not np.all(np.isfinite(lam)) or not np.all(lam > 0):
        raise ValueError("every lambda1 must be finite and > 0")
    lam = np.sort(lam)[::-1].copy()
    if int(n_subsamples) != n_subsamples or n_subsamples < 1:
        raise ValueError("n_subsamples must be a positive integer")
    if not beta > 0:
        raise ValueError("beta must be > 0")
    n = [x.shape[0] for x in classes]
    if subsample_size is None:
        b = [default_subsample_size(nk) for nk in n]
    elif np.ndim(subsample_size) == 0:
        b = [int(subsample_size)] * K
    else:
        b = [int(v) for v in subsample_size]
        if len(b) != K:
            raise ValueError(f"subsample_size must be an int or one value per class (K = {K})")
    for k in range(K):
        if not 2 <= b[k] < n[k]:
            raise ValueError(f"class {k}: subsample size {b[k]} must satisfy 2 <= b < n = {n[k]}")
    if max_batch is not None and max_batch < len(lam):
        raise ValueError(f"max_batch = {max_batch} must hold the L = {len(lam)} problems of one subsample")
    return classes, sgl, lam, b


class _Resident:
    """the samples of all classes and the drawn row indices on the device"""

    def __init__(self, classes, indices, dev):
        self.K, self.p = len(classes), classes[0].shape[1]
        self.B = indices[0].shape[0]
        self.X = to_dev(np.concatenate(classes, axis=0), dev)
        n = [x.shape[0] for x in classes]
        b = [ix.shape[1] for ix in indices]
        self.rowoff = torch.tensor(np.concatenate([[0], np.cumsum(n)[:-1]]), dtype=torch.int32, device=dev)
        self.boff = torch.tensor(np.concatenate([[0], np.cumsum(b)]), dtype=torch.int32, device=dev)
        self.bsum = int(sum(b))
        self.idx = torch.from_numpy(np.ascontiguousarray(np.concatenate(indices, axis=1), dtype=np.int32)).to(dev)
        self.dev = dev

    def covariances(self, s0, nsub, scale):
        """(nsub*K, p, p) covariances of subsamples s0 .. s0+nsub-1; a zero-variance column with ``scale`` raises"""
        lib = _lib.load()
        K, p = self.K, self.p
        S = torch.empty((nsub * K, p, p), dtype=torch.float64, device=self.dev)
        mean = torch.empty((nsub * K, p), dtype=torch.float64, device=self.dev)
        zero_col = torch.empty(nsub * K, dtype=torch.int32, device=self.dev)
        idx = self.idx[s0:s0 + nsub]
        _lib.check(lib.gg_subsample_cov(_p(self.X), _p(self.rowoff), _p(idx), _p(self.boff), nsub, K, p,
                                        1 if scale else 0, _p(mean), _p(S), _p(zero_col),
                                        torch.cuda.current_stream().cuda_stream), "gg_subsample_cov")
        if scale:
            z = zero_col.cpu().numpy()
            bad = np.flatnonzero(z < p)
            if len(bad):
                s, k = divmod(int(bad[0]), K)
                raise ValueError(f"subsample {s0 + s}, class {k}: column {int(z[bad[0]])} has zero variance, so the "
                                 "covariance cannot be scaled by its diagonal (use scale=False or drop the column)")
        return S


def _device_covariances(classes, indices, scale):
    """(B,K,p,p) device tensor of the subsample covariances the driver forms (``indices`` as in its result)"""
    dev = require_cuda()
    classes = [np.asarray(x, dtype=np.float64) for x in classes]
    res = _Resident(classes, [np.asarray(ix) for ix in indices], dev)
    return res.covariances(0, res.B, scale).reshape(res.B, res.K, res.p, res.p)


def _solve_chunk(S, K, lam, reg, lambda2, tol, rtol, max_iter):
    """S: (nsub*K, p, p) device covariances of nsub subsamples.  Each is replicated once per lambda1 (problem
    q = s*L + l, the layout ADMM_MGL_batch gives a shared S) and the nsub*L problems are solved from Omega_0 = I in one
    device loop: 'mgl' with one lambda1 per problem, or (reg None) 'sgl' with lambda1 of problem q as its lam_mat.
    Returns run_admm's (state, info)."""
    L = len(lam)
    nsub, p = S.shape[0] // K, S.shape[1]
    M = nsub * L * K
    Srep = S.reshape(nsub, 1, K, p, p).expand(nsub, L, K, p, p).reshape(M, p, p)
    Om0 = torch.eye(p, dtype=torch.float64, device=S.device).expand(M, p, p)
    kw = dict(rho=1.0, max_iter=int(max_iter), tol=tol, rtol=rtol, stopping_criterion='boyd', update_rho=True)
    if reg is None:
        lam_mat = torch.from_numpy(np.tile(lam, nsub)).to(S.device)[:, None, None].expand(M, p, p)
        return run_admm('sgl', Srep, Om0, None, None, lambda1=float(lam[0]), lam_mat=lam_mat, **kw)
    return run_admm('mgl', Srep, Om0, None, None, lambda1=np.tile(lam, nsub), lambda2=float(lambda2), reg=reg, K=K,
                    **kw)


def _chunk_subsamples(B, L, K, p, sgl, max_iter, max_batch):
    """subsamples per device loop: max_batch // L, or as many as fit in 60 % of the free device memory (the loop's
    (M,p,p) arrays, the eigensolver workspace, the residual history) -- at most B and at most 65535 matrices"""
    cap = max(1, min(B, 65535 // (L * K)))
    if max_batch is not None:
        return max(1, min(cap, int(max_batch) // L))
    lib = _lib.load()
    free, _ = torch.cuda.mem_get_info()
    # replicated S, the state's S, Omega, Omega_new, Theta, X, W, one array of slack; + warm start (p <= 48), + lam_mat
    arrays = 8 + (p <= 48) + (1 if sgl else 0)
    per_problem = arrays * K * p * p * 8 + int(max_iter) * _lib.HIST_STRIDE * 8 + 4096

    def need(ns):
        return ns * L * per_problem + int(lib.gg_eigh_workspace_bytes(ns * L * K, p)) + 2 * ns * K * p * p * 8

    ns = 1
    while ns < cap and need(min(cap, 2 * ns)) <= 0.6 * free:
        ns = min(cap, 2 * ns)
    lo, hi = ns, min(cap, 2 * ns)
    while lo < hi:                             # largest ns in [lo, hi] that fits
        mid = (lo + hi + 1) // 2
        if need(mid) <= 0.6 * free:
            lo = mid
        else:
            hi = mid - 1
    return lo


def stability_selection(data, lambda1, lambda2=None, reg=None, n_subsamples=20, subsample_size=None, beta=0.05,
                        scale=True, seed=0, refit=True, tol=1e-7, rtol=1e-7, max_iter=1000, max_batch=None,
                        verbose=False):
    """Choose lambda1 by StARS from raw samples, for SGL or MGL (GGL / FGL at a fixed lambda2).

    ``data``: (n,p) for SGL (``reg`` and ``lambda2`` must be None); (K,n,p) or a list of K (n_k,p) arrays for MGL, with
    ``reg`` in {'GGL', 'FGL'} and a scalar ``lambda2`` > 0 (K <= 90).  ``lambda1``: 1-D array of L values > 0, processed
    and reported in decreasing order.

    ``n_subsamples`` (B) subsamples of ``subsample_size`` rows per class are drawn without replacement (default per class
    floor(10 sqrt(n_k)) if n_k > 144, else floor(0.8 n_k); 2 <= b_k < n_k): ``rng = np.random.default_rng(seed)``, then
    for s in range(B), for k in range(K), ``rng.choice(n_k, b_k, replace=False)``.  Each subsample covariance is
    ``np.cov(X_sub, rowvar=False, bias=True)``, scaled to unit diagonal (S_ij / sqrt(S_ii S_jj)) when ``scale``; a
    zero-variance column then raises ValueError naming subsample, class and column.  Every covariance is solved at every
    lambda1 by ADMM from Omega_0 = I (``tol``, ``rtol``, ``max_iter``).

    An edge is an entry Theta_ij != 0 with i < j; theta = (edge count over the subsamples) / B.  The instability of
    class k is D_k = sum_{i<j} 2 theta (1 - theta) / C(p,2), D = mean_k D_k, Dbar(lambda) = max of D over the path values
    >= lambda, and the selected lambda1 is the smallest one with Dbar <= ``beta`` (the largest lambda1 if none is).

    ``max_batch`` caps the problems (subsample x lambda1) of one device loop (at least L); by default it is sized from
    the free device memory.  The samples stay on the device; only per-lambda summaries and the edge counts at the
    selected lambda1 are copied back.

    Returns a dict: ``lambda1`` (sorted), ``lambda2``, ``instability`` (L,), ``instability_bar`` (L,),
    ``instability_per_class`` (L,K), ``mean_edges`` (L,K) (mean edge count per subsample), ``best_index``,
    ``best_lambda1``, ``edge_frequency`` at the selected lambda1 ((K,p,p), or (p,p) for SGL; symmetric, zero diagonal),
    ``indices`` (per class a (B, b_k) int array), ``n_not_optimal`` (L,) (subsample solves that reached ``max_iter``;
    a warning names them), and with ``refit`` also ``sol``, ``info`` of ADMM_MGL / ADMM_SGL on the full-sample
    covariance at the selected lambda1 (same ``scale``, Omega_0 = I).
    """
    classes, sgl, lam, b = _check_args(data, lambda1, lambda2, reg, n_subsamples, subsample_size, beta, max_batch)
    K, p, L, B = len(classes), classes[0].shape[1], len(lam), int(n_subsamples)
    indices = draw_indices([x.shape[0] for x in classes], b, B, seed)
    if refit:                                  # full-sample covariances first: a zero-variance column fails early
        S_full = []
        for k, x in enumerate(classes):
            if scale and np.any(np.ptp(x, axis=0) == 0):
                j = int(np.flatnonzero(np.ptp(x, axis=0) == 0)[0])
                raise ValueError(f"class {k}: column {j} has zero variance in the full sample, so the covariance "
                                 "cannot be scaled by its diagonal (use scale=False or drop the column)")
            S_full.append(sample_covariance(x, scale))
    dev = require_cuda()
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    res = _Resident(classes, indices, dev)
    counts = torch.zeros((L, K, p, p), dtype=torch.int32, device=dev)
    nsub = _chunk_subsamples(B, L, K, p, sgl, max_iter, max_batch)
    not_opt = np.zeros((B, L), dtype=bool)
    for s0 in range(0, B, nsub):
        ns = min(nsub, B - s0)
        S = res.covariances(s0, ns, scale)
        st, info = _solve_chunk(S, K, lam, None if sgl else reg, lambda2, tol, rtol, max_iter)
        not_opt[s0:s0 + ns] = np.asarray(info["status"]).reshape(ns, L) == "max iterations reached"
        _lib.check(lib.gg_edge_count(_p(st.Theta), ns, L, K, p, _p(counts), stream), "gg_edge_count")
        if verbose:
            it = np.asarray(info["iters"]).reshape(ns, L)
            print(f"subsamples {s0}..{s0 + ns - 1}: {ns * L} problems in one device loop, iterations "
                  f"{int(it.min())}..{int(it.max())}")
        del st, S
    out = torch.empty((L, K, 2), dtype=torch.float64, device=dev)
    _lib.check(lib.gg_stars_instability(_p(counts), L, K, p, B, _p(out), stream), "gg_stars_instability")
    out = out.cpu().numpy()
    D_k, mean_edges = out[..., 0], out[..., 1]
    D = D_k.mean(axis=1)
    dbar, best = select(D, beta)
    C = counts[best].cpu().numpy().astype(np.float64)
    freq = (C + C.transpose(0, 2, 1)) / B
    n_not_optimal = not_opt.sum(axis=0)
    if n_not_optimal.any():
        bad = [(int(s), float(lam[l])) for s, l in zip(*np.nonzero(not_opt))]
        warnings.warn(f"stability_selection: {len(bad)} subsample solve(s) reached max_iter = {max_iter} "
                      f"(subsample, lambda1): {bad[:10]}{' ...' if len(bad) > 10 else ''}")
    result = {'lambda1': lam, 'lambda2': None if sgl else float(lambda2), 'instability': D,
              'instability_bar': dbar, 'instability_per_class': D_k, 'mean_edges': mean_edges, 'best_index': best,
              'best_lambda1': float(lam[best]), 'edge_frequency': freq[0] if sgl else freq, 'indices': indices,
              'n_not_optimal': n_not_optimal}
    if refit:
        from .solver.admm_solver import ADMM_MGL
        from .solver.single_admm_solver import ADMM_SGL
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf) if not verbose else contextlib.nullcontext():
            if sgl:
                sol, info = ADMM_SGL(S_full[0], lam[best], np.eye(p), tol=tol, rtol=rtol, max_iter=max_iter)
            else:
                sol, info = ADMM_MGL(np.stack(S_full), lam[best], float(lambda2), reg,
                                     np.repeat(np.eye(p)[None], K, 0), tol=tol, rtol=rtol, max_iter=max_iter)
        result['sol'], result['info'] = sol, info
    return result
