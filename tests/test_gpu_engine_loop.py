"""The device ADMM loop on a reused AdmmState (``state=``, as the lambda grid runs it) against a fresh state: the same
iterations, status, rho path and Omega / Theta / X, bit for bit.

Sizes: p = 100 (> 48, so the small-matrix eigensolver and its warm start -- which a reused state carries over from
its previous solve -- are not involved) and K <= 5, where two fresh runs are bitwise identical; each case asserts that
first."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

P = 100


def _cov(rng, M, p=P, N=150):
    return np.stack([np.cov(rng.standard_normal((p, N)), bias=True) for _ in range(M)])


def _case(name):
    rng = np.random.default_rng(7)
    kw = dict(tol=1e-7, rtol=1e-7, max_iter=400)
    if name == "sgl":
        return "sgl", _cov(rng, 1), dict(lambda1=0.1, **kw), dict(lambda1=0.3)
    if name == "mgl_upper":
        return "mgl", _cov(rng, 3), dict(lambda1=0.05, lambda2=0.01, reg="GGL", **kw), dict(lambda1=0.2, lambda2=0.05)
    if name == "mgl_latent":
        return ("mgl", _cov(rng, 3), dict(lambda1=0.05, lambda2=0.01, reg="FGL", latent=True, mu=np.full(3, 0.2), **kw),
                dict(lambda1=0.1, lambda2=0.03))
    # ADMM_MGL_batch shape: four problems of K = 3, one (lambda1, lambda2) each, read from the control block
    l1, l2 = np.array([0.3, 0.01, 0.15, 0.05]), np.array([0.1, 0.002, 0.05, 0.01])
    return ("mgl", _cov(rng, 12), dict(lambda1=l1, lambda2=l2, reg="GGL", K=3, **kw),
            dict(lambda1=l1[::-1].copy(), lambda2=2 * l2))


def _solve(kind, S, kw, state=None):
    from gglasso_b200._engine import run_admm
    eye = np.repeat(np.eye(S.shape[1])[None], S.shape[0], 0)
    st, res = run_admm(kind, S, eye, None, None, state=state, **kw)
    n = res["iters"]
    out = dict(iters=n.copy(), status=list(res["status"]),
               hist=[res["hist"][q, :n[q]].copy() for q in range(len(n))],
               Omega=st.final_omega(n).cpu().numpy(), Theta=st.Theta.cpu().numpy(), X=st.X.cpu().numpy())
    return st, out


def _assert_same(a, b):
    np.testing.assert_array_equal(a["iters"], b["iters"])
    assert a["status"] == b["status"]
    for ha, hb in zip(a["hist"], b["hist"]):
        np.testing.assert_array_equal(ha[:, 4], hb[:, 4], err_msg="rho path")
        np.testing.assert_array_equal(ha, hb, err_msg="residual history")
    for k in ("Omega", "Theta", "X"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)


@pytest.mark.parametrize("name", ["sgl", "mgl_upper", "mgl_latent", "mgl_batch"])
def test_reused_state_matches_fresh_state(name):
    from gglasso_b200 import _lib
    assert P > _lib.load().gg_jacobi_max()      # 'mgl_upper' runs on upper triangles, the others on full matrices
    kind, S, kw, other = _case(name)
    _, fresh = _solve(kind, S, kw)
    _, again = _solve(kind, S, kw)
    _assert_same(fresh, again)                  # the size is run-to-run deterministic
    # the state first solves another problem (other lambdas: other iterates, iteration count, Omega buffer parity)
    st, first = _solve(kind, S, dict(kw, **other))
    assert not np.array_equal(first["Theta"], fresh["Theta"])
    _, reused = _solve(kind, S, kw, state=st)
    _assert_same(reused, fresh)
