"""stability_selection without a GPU: argument checks, the default subsample size, the index draw and the StARS
selection rule."""
import numpy as np
import pytest

from gglasso_b200 import stability as stars
from gglasso_b200 import stability_selection


def _data(rng, n=60, p=6):
    return rng.standard_normal((n, p))


@pytest.mark.parametrize("kw, exc", [
    (dict(reg="GGL"), ValueError),                        # SGL data with reg
    (dict(lambda2=0.1), ValueError),                      # SGL data with lambda2
    (dict(lambda1=[]), ValueError),
    (dict(lambda1=[0.1, 0.0]), ValueError),
    (dict(lambda1=[0.1, -0.2]), ValueError),
    (dict(lambda1=[[0.1, 0.2]]), ValueError),
    (dict(lambda1=[0.1, np.nan]), ValueError),
    (dict(subsample_size=1), ValueError),                 # b < 2
    (dict(subsample_size=60), ValueError),                # b = n
    (dict(subsample_size=61), ValueError),
    (dict(n_subsamples=0), ValueError),
    (dict(beta=0.0), ValueError),
    (dict(lambda1=[0.1, 0.2, 0.3], max_batch=2), ValueError),   # fewer problems than one subsample's L
])
def test_sgl_argument_checks(kw, exc):
    rng = np.random.default_rng(0)
    args = dict(lambda1=[0.1, 0.2])
    args.update(kw)
    with pytest.raises(exc):
        stability_selection(_data(rng), **args)


@pytest.mark.parametrize("kw, exc", [
    (dict(), ValueError),                                 # reg missing
    (dict(reg="SGL", lambda2=0.1), ValueError),
    (dict(reg="GGL"), ValueError),                        # lambda2 missing
    (dict(reg="FGL", lambda2=0.0), ValueError),
    (dict(reg="GGL", lambda2=[0.1, 0.2]), ValueError),    # lambda2 not a scalar
    (dict(reg="GGL", lambda2=0.1, subsample_size=[10, 10]), ValueError),   # one size per class, K = 3
    (dict(reg="GGL", lambda2=0.1, subsample_size=[10, 10, 40]), ValueError),  # b_k = n_k
])
def test_mgl_argument_checks(kw, exc):
    rng = np.random.default_rng(1)
    data = rng.standard_normal((3, 40, 5))
    with pytest.raises(exc):
        stability_selection(data, [0.1], **kw)


def test_mgl_list_with_different_p_and_k_above_90():
    rng = np.random.default_rng(2)
    with pytest.raises(ValueError):
        stability_selection([rng.standard_normal((30, 5)), rng.standard_normal((30, 6))], [0.1], reg="GGL", lambda2=0.1)
    with pytest.raises(NotImplementedError):
        stability_selection(rng.standard_normal((91, 20, 3)), [0.1], reg="GGL", lambda2=0.1)


def test_dispatch_and_ragged_sizes():
    rng = np.random.default_rng(3)
    c, sgl, lam, b = stars._check_args(_data(rng, 200, 4), [0.2, 0.5, 0.1], None, None, 20, None, 0.05, None)
    assert sgl and len(c) == 1 and list(lam) == [0.5, 0.2, 0.1] and b == [141]
    data = [rng.standard_normal((n, 4)) for n in (30, 145, 144)]
    c, sgl, lam, b = stars._check_args(data, [0.3], 0.1, "FGL", 20, None, 0.05, None)
    assert not sgl and len(c) == 3 and b == [24, 120, 115]
    c, sgl, lam, b = stars._check_args(rng.standard_normal((2, 50, 4)), [0.3], 0.1, "GGL", 5, 7, 0.05, 1)
    assert not sgl and b == [7, 7]


def test_default_subsample_size_rule():
    for n in (3, 10, 100, 143, 144):
        assert stars.default_subsample_size(n) == int(np.floor(0.8 * n))
    for n in (145, 200, 1000, 10 ** 6):
        assert stars.default_subsample_size(n) == int(np.floor(10 * np.sqrt(n)))
    assert stars.default_subsample_size(144) == 115 and stars.default_subsample_size(145) == 120


def test_index_draw_reproduced_from_seed():
    n, b, B = [30, 50, 40], [10, 17, 2], 6
    idx = stars.draw_indices(n, b, B, seed=11)
    rng = np.random.default_rng(11)
    for s in range(B):
        for k in range(3):
            ref = rng.choice(n[k], b[k], replace=False)
            assert np.array_equal(idx[k][s], ref)
            assert len(set(idx[k][s])) == b[k] and idx[k][s].max() < n[k]
    again = stars.draw_indices(n, b, B, seed=11)
    assert all(np.array_equal(x, y) for x, y in zip(idx, again))
    assert not np.array_equal(stars.draw_indices(n, b, B, seed=12)[1], idx[1])


def test_selection_rule_on_hand_made_curves():
    beta = 0.05
    # non-monotone: D dips back below beta after exceeding it; Dbar keeps the maximum so the dip is not selected
    D = np.array([0.0, 0.01, 0.06, 0.02, 0.04, 0.08])
    dbar, best = stars.select(D, beta)
    assert np.array_equal(dbar, [0.0, 0.01, 0.06, 0.06, 0.06, 0.08])
    assert best == 1
    # all above beta: the largest lambda
    assert stars.select(np.array([0.1, 0.2, 0.3]), beta)[1] == 0
    # all below beta: the smallest lambda
    assert stars.select(np.array([0.0, 0.01, 0.049]), beta)[1] == 2
    # ties at beta qualify (Dbar <= beta)
    assert stars.select(np.array([0.0, 0.05, 0.05, 0.0500001]), beta)[1] == 2
    assert stars.select(np.array([0.05]), beta)[1] == 0


def test_sample_covariance_matches_numpy_and_scaling():
    rng = np.random.default_rng(4)
    X = rng.standard_normal((40, 6)) * np.arange(1, 7)
    S = stars.sample_covariance(X, False)
    assert np.array_equal(S, np.cov(X, rowvar=False, bias=True))
    Ss = stars.sample_covariance(X, True)
    d = np.sqrt(np.diag(S))
    assert np.allclose(Ss, S / np.outer(d, d), rtol=1e-15, atol=0)
    assert np.max(np.abs(np.diag(Ss) - 1)) <= 1e-15
