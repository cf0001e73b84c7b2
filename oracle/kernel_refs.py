"""Host references of the ADMM loop's elementwise kernels, reductions and device stopping test, for kernel-level tests.

Elementwise references evaluate each kernel's expression in the kernel's association order (the kernels are compiled
without FMA contraction), so a correct kernel matches them bitwise.  Reductions are compared against exact sums
(math.fsum over the rounded products).  The stopping test and rho update restate admm_solver.py:216-246 of the
reference the way admm_oracle.admm_mgl does (boyd_residuals, _rho_update, the 'optimal' test), over the same five
partial sums the device reduces.
"""
import math
from fractions import Fraction

import numpy as np

NPART = 5


# ---- exact sums ------------------------------------------------------------------------------------------------
def fsum(a):
    """correctly rounded sum of all entries of ``a``"""
    return math.fsum(np.asarray(a, dtype=np.float64).ravel().tolist())


def gershgorin_exact(A):
    """min_i (a_ii - sum_{j != i} |a_ij|) of every matrix of the (M,p,p) stack, exactly (Fraction of the stored
    doubles); returns a list of Fractions"""
    A = np.asarray(A, dtype=np.float64)
    out = []
    for a in A.reshape(-1, A.shape[-1], A.shape[-1]):
        best = None
        for i, row in enumerate(a.tolist()):
            v = Fraction(row[i]) - sum(Fraction(abs(x)) for j, x in enumerate(row) if j != i)
            best = v if best is None or v < best else best
        out.append(best)
    return out


# ---- elementwise kernels in kernel order ------------------------------------------------------------------------
def soft(v, t):
    """gg_soft: sign(v) * max(|v| - t, 0)"""
    a = np.maximum(np.abs(v) - t, 0.0)
    return np.where(v > 0.0, a, np.where(v < 0.0, -a, 0.0))


def _offdiag(p):
    return ~np.eye(p, dtype=bool)


def prox_sgl(Om, Omp, L, X, lam, rho, lam_mat=None, latent=False, pvec=None):
    """gg_prox_sgl for an (M,p,p) stack with per-matrix rho (M,).  Returns Theta, X_new (or C when latent) and the
    five per-matrix partial sums (M,5) as exact sums (non-latent only)."""
    M, p, _ = Om.shape
    inv_rho = (1.0 / np.asarray(rho, dtype=np.float64)).reshape(M, 1, 1)
    a = Om + L if L is not None else Om
    a = a + X
    thr = inv_rho * (lam_mat if lam_mat is not None else lam)
    th = np.where(_offdiag(p), soft(a, thr), a)
    if latent:
        return th, (th - X) - Om, None
    xn = (X + Om) - th
    parts = np.zeros((M, NPART))
    for m in range(M):
        pb = p if pvec is None else int(pvec[m])
        s = (slice(0, pb), slice(0, pb))
        om, t, x, pv = Om[m][s], th[m][s], xn[m][s], Omp[m][s]
        d1, d2 = om - t, om - pv
        parts[m] = [fsum(om * om), fsum(t * t), fsum(x * x), fsum(d1 * d1), fsum(d2 * d2)]
    return th, xn, parts


def block_norms(A, Mblk):
    """fsgl_block_norm_kernel: Frobenius norm of every Mblk x Mblk block of each matrix, summed the way one warp does
    (lane e % 32 adds the squares of block entries e, e + 32, ... in row-major order; then an xor-shuffle tree).
    Returns (M, nb, nb); only the strictly upper blocks are meaningful."""
    M, p, _ = A.shape
    nb = p // Mblk
    B = A.reshape(M, nb, Mblk, nb, Mblk).transpose(0, 1, 3, 2, 4).reshape(M, nb, nb, Mblk * Mblk)
    sq = B * B
    n = Mblk * Mblk
    pad = (-n) % 32
    sq = np.concatenate([sq, np.zeros(sq.shape[:-1] + (pad,))], axis=-1).reshape(M, nb, nb, -1, 32)
    lanes = np.zeros((M, nb, nb, 32))
    for r in range(sq.shape[3]):
        lanes = lanes + sq[:, :, :, r, :]
    idx = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        lanes = lanes + lanes[..., idx ^ o]
    return np.sqrt(lanes[..., 0])


def prox_fsgl(Om, Omp, L, X, lam, rho, Mblk, latent=False):
    """gg_prox_fsgl (prox_sgl_kernel with block norms) in kernel order; returns Theta, X_new or C, partials (M,5)"""
    M, p, _ = Om.shape
    inv_rho = (1.0 / np.asarray(rho, dtype=np.float64)).reshape(M, 1, 1)
    a = Om + L if L is not None else Om
    a = a + X
    thr = inv_rho * lam
    nrm = block_norms(a, Mblk)
    bi = np.arange(p) // Mblk
    nr = nrm[:, np.minimum.outer(bi, bi), np.maximum.outer(bi, bi)]
    aa = np.where(nr > thr, nr, thr)
    with np.errstate(invalid="ignore", divide="ignore"):
        th = np.where((bi[:, None] == bi[None, :])[None], a, (a * (aa - thr)) / aa)
    if latent:
        return th, (th - X) - Om, None
    xn = (X + Om) - th
    d1, d2 = Om - th, Om - Omp
    parts = np.array([[fsum(v[m] * v[m]) for v in (Om, th, xn, d1, d2)] for m in range(M)])
    return th, xn, parts


def prox_sum_frob(A, Mblk, lam):
    """prox_sum_Frob of the reference as admm_oracle.prox_sum_frob states it, for one matrix"""
    pM = A.shape[0]
    nb = pM // Mblk
    Y = np.zeros_like(A)
    for i in range(nb):
        for j in range(i, nb):
            blk = A[i * Mblk:(i + 1) * Mblk, j * Mblk:(j + 1) * Mblk]
            if i == j:
                Y[i * Mblk:(i + 1) * Mblk, j * Mblk:(j + 1) * Mblk] = blk
            else:
                a = max(math.sqrt(fsum(blk * blk)), lam)
                B = blk * (a - lam) / a
                Y[i * Mblk:(i + 1) * Mblk, j * Mblk:(j + 1) * Mblk] = B
                Y[j * Mblk:(j + 1) * Mblk, i * Mblk:(i + 1) * Mblk] = B.T
    return Y


def dual_update(X, Om, Omp, Th, L, sgl_order):
    """gg_dual_update: X_new and the per-matrix partial sums (M,5)"""
    M = X.shape[0]
    res = (Om - Th) + L if L is not None else Om - Th
    if sgl_order:
        xn = ((X + Om) - Th) + L if L is not None else (X + Om) - Th
    else:
        xn = X + res
    tl = Th - L if L is not None else Th
    d2 = Om - Omp
    parts = np.array([[fsum(v[m] * v[m]) for v in (Om, tl, xn, res, d2)] for m in range(M)])
    return xn, parts


def build_w(Th, L, X, S, nk, rho, xs):
    """gg_build_w with per-matrix rho and pending scale xs (M,): returns W and the stored X"""
    M = Th.shape[0]
    rho = np.asarray(rho, dtype=np.float64).reshape(M, 1, 1)
    xs = np.asarray(xs, dtype=np.float64).reshape(M, 1, 1)
    beta = (np.ones((M, 1, 1)) if nk is None else np.asarray(nk, dtype=np.float64).reshape(M, 1, 1)) / rho
    xv = np.where(xs != 1.0, xs * X, X)
    w = Th
    if L is not None:
        w = w - L
    w = w - xv
    w = w - beta * S
    return w, xv


def add3(Om, L, X):
    v = Om + L if L is not None else Om
    return v + X


def ext_theta(Om, L, X0, Lam, X1, lam1, rho):
    """gg_ext_theta on the padded (K,p,p) stack: Theta and C = Theta - X0 - Omega"""
    K, p, _ = Om.shape
    v = Om + L if L is not None else Om
    v = v + X0
    v = v + Lam
    v = (v - X1) * 0.5
    thr = (np.asarray(lam1, dtype=np.float64) / (2.0 * rho)).reshape(K, 1, 1)
    th = np.where(_offdiag(p), soft(v, thr), v)
    return th, (th - X0) - Om


def ext_groups(pvec, rng, hole=0.2):
    """bookkeeping array G (2,Lg,K) of ext_ADMM_MGL for matrices of sizes pvec: one group per pair f < g of global
    features; matrix k holds feature f < p_k at its own local index perm_k[f], and takes part in the group unless a
    random hole (probability ``hole``) drops it; entries (i,j) with i < j, -1 where absent.  Groups of one member
    (pairs only the largest matrices hold) are kept, groups of none dropped."""
    K, P = len(pvec), max(pvec)
    perm = [rng.permutation(pk) for pk in pvec]
    rows = []
    for f in range(P):
        for g in range(f + 1, P):
            e = np.full((2, K), -1, dtype=np.int32)
            for k, pk in enumerate(pvec):
                if g < pk and rng.random() >= hole:
                    a, b = perm[k][f], perm[k][g]
                    e[:, k] = (min(a, b), max(a, b))
            if (e[0] >= 0).any():
                rows.append(e)
    return np.ascontiguousarray(np.stack(rows, axis=1))


def ext_lambda(Th, X1, G, lambda2, rho):
    """gg_ext_lambda: Z = Theta + X1, then every group of G (2,Lg,K) shrunk in Euclidean norm (member order k) and
    written to both triangles"""
    Z = Th + X1
    K = Th.shape[0]
    for l in range(G.shape[1]):
        ks = [k for k in range(K) if G[0, l, k] >= 0]
        ss = 0.0
        for k in ks:
            v = Z[k, G[0, l, k], G[1, l, k]]
            ss += v * v
        lam = (lambda2 / rho) * math.sqrt(float(len(ks)))
        nrm = math.sqrt(ss)
        a = nrm if nrm > lam else lam
        for k in ks:
            i, j = G[0, l, k], G[1, l, k]
            z = ((Th[k, i, j] + X1[k, i, j]) * (a - lam)) / a
            Z[k, i, j] = z
            Z[k, j, i] = z
    return Z


def ext_dual(X0, X1, Om, Omp, Th, L, Lam, Lamp, pvec):
    """gg_ext_dual: X0, X1 and the per-matrix partial sums (K,5) over the leading p_k x p_k block"""
    r0 = (Om - Th) + L if L is not None else Om - Th
    r1 = Th - Lam
    x0, x1 = X0 + r0, X1 + r1
    tl = Th - L if L is not None else Th
    d0, d1 = Om - Omp, Lam - Lamp
    parts = []
    for k, pk in enumerate(pvec):
        s = (k, slice(0, pk), slice(0, pk))
        sq = lambda a, b: np.concatenate([(a[s] * a[s]).ravel(), (b[s] * b[s]).ravel()])  # noqa: E731
        parts.append([fsum(sq(Om, Lam)), fsum(sq(tl, Th)), fsum(sq(x0, x1)), fsum(sq(r0, r1)), fsum(sq(d0, d1))])
    return x0, x1, np.array(parts)


def objective_parts(Om, S, Th, lambda1, lambda2, reg):
    """gg_objective: (<Omega,S>, P(Theta)) exactly, and the sums of absolute terms that bound their rounding error.
    P counts the strict upper triangle twice (ggl_helper.py:162-176); reg -1: P = 0."""
    prod = Om * S
    ip, ip_abs = fsum(prod), fsum(np.abs(prod))
    if reg < 0:
        return ip, ip_abs, 0.0
    K, p, _ = Th.shape
    iu = np.triu_indices(p, 1)
    T = Th[:, iu[0], iu[1]]                                  # (K, n_upper)
    # per-entry norms over k in double (relative error <= K u, K <= 90), their sum exact
    n1 = np.abs(T).sum(axis=0)
    n2 = np.sqrt((T * T).sum(axis=0)) if reg == 0 else np.abs(np.diff(T, axis=0)).sum(axis=0)
    return ip, ip_abs, 2.0 * fsum(lambda1 * n1 + lambda2 * n2)


# ---- stopping test and rho update (stop_update_kernel) ----------------------------------------------------------
def stop_update(sums, ctrl, hist, hist_cap, pdim, tol, rtol, update_rho, C):
    """one gg_stop_update on the host.  sums: (nprob,5) reduced partial sums; ctrl (nprob,16) and hist
    (nprob,hist_cap,5) are updated in place.  C: the ctrl index constants (C_RHO, ...) of gglasso_b200._lib."""
    for q in range(ctrl.shape[0]):
        c = ctrl[q]
        if c[C.C_DONE] != 0.0:
            continue
        a = sums[q]
        rho = c[C.C_RHO]
        nO, nTL, nX = math.sqrt(a[0]), math.sqrt(a[1]), math.sqrt(a[2])
        r = math.sqrt(a[3])
        s = rho * math.sqrt(a[4])
        e_pri = pdim[q] * tol + rtol * max(nO, nTL)
        e_dual = pdim[q] * tol + rtol * rho * nX
        it = int(c[C.C_ITER])
        if it < hist_cap:
            hist[q, it] = [r, s, e_pri, e_dual, rho]
        rho_new = rho
        if update_rho:
            if r >= 10.0 * s:
                rho_new = 2.0 * rho
            elif s >= 10.0 * r:
                rho_new = 0.5 * rho
        c[C.C_XSCALE] = rho / rho_new
        c[C.C_RHO] = rho_new
        c[C.C_R], c[C.C_S], c[C.C_EPRI], c[C.C_EDUAL] = r, s, e_pri, e_dual
        c[C.C_ITER] = it + 1
        if r <= e_pri and s <= e_dual:
            c[C.C_STATUS] = 1.0
            c[C.C_DONE] = 1.0
        if not (math.isfinite(r) and math.isfinite(s)):
            c[C.C_STATUS] = -1.0
            c[C.C_DONE] = 1.0
