"""ADMM_MGL_batch argument checks that are decided before any device work (no GPU needed)."""
import numpy as np
import pytest


def _inputs(B, K, p):
    S = np.repeat(np.eye(p)[None, None], B, 0).repeat(K, 1) * 1.0
    return S, np.repeat(np.eye(p)[None], K, 0)


def test_mismatched_batch_sizes():
    from gglasso_b200 import ADMM_MGL_batch
    S, eye = _inputs(2, 3, 4)
    with pytest.raises(AssertionError, match="batch sizes"):
        ADMM_MGL_batch(S, [0.1, 0.2, 0.3], 0.1, "GGL", eye)
    with pytest.raises(AssertionError, match="batch sizes"):
        ADMM_MGL_batch(S[0], [0.1, 0.2], [0.1, 0.2, 0.3], "GGL", eye)
    with pytest.raises(AssertionError, match="batch sizes"):
        ADMM_MGL_batch(S, 0.1, 0.1, "GGL", np.stack([eye] * 3))
    with pytest.raises(AssertionError, match="batch sizes"):
        ADMM_MGL_batch(S, 0.1, 0.1, "GGL", eye, latent=True, mu1=np.ones((3, 3)))


def test_k_above_tile_limit_is_rejected():
    from gglasso_b200 import ADMM_MGL_batch
    S, eye = _inputs(2, 91, 3)
    with pytest.raises(NotImplementedError, match="K <= 90"):
        ADMM_MGL_batch(S, 0.1, 0.1, "GGL", eye)


def test_admm_mgl_asserts():
    from gglasso_b200 import ADMM_MGL_batch
    S, eye = _inputs(2, 2, 5)
    with pytest.raises(AssertionError):
        ADMM_MGL_batch(S, 0.1, 0.1, "LASSO", eye)
    with pytest.raises(AssertionError):
        ADMM_MGL_batch(S, [0.1, 0.0], 0.1, "GGL", eye)
    with pytest.raises(AssertionError):
        ADMM_MGL_batch(S, 0.1, -0.1, "GGL", eye)
    with pytest.raises(AssertionError):
        ADMM_MGL_batch(S, 0.1, 0.1, "GGL", eye, rho=0.0)
    with pytest.raises(AssertionError):
        ADMM_MGL_batch(S, 0.1, 0.1, "GGL", eye, latent=True)
    with pytest.raises(AssertionError):
        ADMM_MGL_batch(S, 0.1, 0.1, "GGL", eye, latent=True, mu1=np.array([1.0, -1.0]))
    with pytest.raises(AssertionError):
        ADMM_MGL_batch(S, 0.1, 0.1, "GGL", eye[:, :4, :4])
    with pytest.raises(AssertionError):
        ADMM_MGL_batch(S[..., :4], 0.1, 0.1, "GGL", eye)


def test_no_kkt_or_measure_parameters():
    import inspect
    from gglasso_b200 import ADMM_MGL_batch
    params = inspect.signature(ADMM_MGL_batch).parameters
    assert "stopping_criterion" not in params and "measure" not in params
    S, eye = _inputs(2, 2, 5)
    with pytest.raises(TypeError):
        ADMM_MGL_batch(S, 0.1, 0.1, "GGL", eye, stopping_criterion="kkt")
    with pytest.raises(TypeError):
        ADMM_MGL_batch(S, 0.1, 0.1, "GGL", eye, measure=True)
