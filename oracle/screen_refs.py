"""Host statements of block_MGL's device pieces, for tests (test infrastructure, like the rest of oracle/).

  mgl_screen        the exact component screen: (i, j), i < j, is an edge iff prox_p(n S)[:, i, j] != 0, i.e.
                    admm_oracle.prox_p at rho = 1 (Danaher, Wang & Witten 2014, section 5)
  screen_words      that graph in gg_mgl_screen's layout (p rows of ceil(p/32) uint32 words, bit b of word w =
                    column 32 w + b, upper triangle only)
  components        connected components of the graph (self loops added), as get_connected_components orders them
  prox_mgl_ragged   gg_prox_mgl_ragged in kernel order: Theta, X and each problem's five partial sums over its true
                    p_q x p_q entries (exact sums), next to kernel_refs.prox_sgl's pvec
  block_mgl         screen, admm_oracle.admm_mgl per component, reassembled (numpy restatement of block_MGL)
"""
import numpy as np

from . import admm_oracle as orc
from .kernel_refs import NPART, fsum


def mgl_screen(S, lambda1, lambda2, reg, n_samples=None):
    """(p,p) bool, strictly upper triangle: prox of the weighted K-vector of the entry is nonzero"""
    K, p, _ = S.shape
    nk = np.ones(K) if n_samples is None else np.broadcast_to(np.asarray(n_samples, dtype=np.float64), (K,))
    P = orc.prox_p(nk[:, None, None] * S, lambda1, lambda2, reg)
    return np.triu((P != 0).any(axis=0), 1)


def screen_words(A):
    """upper-triangle bool adjacency (p,p) -> (p, ceil(p/32)) uint32 bitmask"""
    p = A.shape[0]
    nw = (p + 31) // 32
    bits = np.zeros((p, 32 * nw), dtype=np.uint64)
    bits[:, :p] = np.triu(A, 1)
    return (bits.reshape(p, nw, 32) << np.arange(32, dtype=np.uint64)).sum(axis=2).astype(np.uint32)


def components(A):
    """connected components of the symmetric closure of A plus self loops; (numC, allC) in label order"""
    from scipy.sparse.csgraph import connected_components
    G = (A | A.T).astype(int)
    np.fill_diagonal(G, 1)
    n, labels = connected_components(G, directed=False, return_labels=True)
    return n, [np.flatnonzero(labels == i) for i in range(n)]


def prox_mgl_ragged(Om, Omp, X, lambda1, lambda2, reg, rho, K, pvec):
    """Om, Omp, X: (B*K, p, p) padded stacks; rho: (B,).  Returns Theta, X_new (B*K,p,p) and parts (B, 5)."""
    M, p, _ = Om.shape
    B = M // K
    Th = np.empty_like(Om)
    for q in range(B):
        s = slice(q * K, (q + 1) * K)
        inv_rho = 1.0 / float(rho[q])
        Th[s] = orc.prox_p(Om[s] + X[s], inv_rho * lambda1, inv_rho * lambda2, reg)
    d1 = Om - Th
    xn = X + d1
    d2 = Om - Omp
    parts = np.zeros((B, NPART))
    for q in range(B):
        n = int(pvec[q])
        s = (slice(q * K, (q + 1) * K), slice(0, n), slice(0, n))
        parts[q] = [fsum(v[s] * v[s]) for v in (Om, Th, xn, d1, d2)]
    return Th, xn, parts


def block_mgl(S, lambda1, lambda2, reg, Omega_0, n_samples=None, **kw):
    """block_MGL on the host: components of mgl_screen, singletons in closed form, admm_mgl on the others"""
    K, p, _ = S.shape
    numC, allC = components(mgl_screen(S, lambda1, lambda2, reg, n_samples))
    sol = {k: np.zeros((K, p, p)) for k in ("Omega", "Theta", "X")}
    for C in allC:
        ix = (slice(None), C[:, None], C[None, :])
        if len(C) == 1:
            sol["Omega"][ix] = sol["Theta"][ix] = 1 / S[ix]
            continue
        bs, _ = orc.admm_mgl(np.ascontiguousarray(S[ix]), lambda1, lambda2, reg, np.ascontiguousarray(Omega_0[ix]),
                             n_samples=n_samples, **kw)
        for k in sol:
            sol[k][ix] = bs[k]
    return sol, allC
