"""The path-independent C-SVC checks of oracle/pysvm.py on sklearn's own fits: they must accept libsvm's fits and their
decision values, and reject a fit that is off by a small amount -- so the checker is neither empty nor too tight before
it judges the GPU solver (tests/test_gpu_svm.py, tests/test_gpu_resident_scale.py)."""
import warnings

import numpy as np
import pytest

import pysvm

SVC = pytest.importorskip("sklearn.svm").SVC


@pytest.fixture(scope="module")
def rbf():
    """a seeded PSD matrix: an RBF kernel of random features, two classes shifted apart, 400 points"""
    rng = np.random.default_rng(17)
    n = 400
    X = rng.standard_normal((n, 20))
    y = (np.arange(n) % 3 == 0).astype(int)   # 134 : 266
    X[y == 1, :4] += 0.7
    sq = (X * X).sum(1)
    K = np.exp(-0.05 * np.maximum(sq[:, None] + sq[None] - 2 * X @ X.T, 0.0))
    np.fill_diagonal(K, 1.0)
    perm = rng.permutation(n)
    return K, y, perm[:320], perm[320:]


def sklearn_fit(K, y, train, test, C, eps, max_iter=-1):
    sv = SVC(kernel="precomputed", C=C, tol=eps, shrinking=False, cache_size=200, max_iter=max_iter)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")   # ConvergenceWarning of a truncated run
        sv.fit(K[np.ix_(train, train)], y[train])
    order, y_pm = pysvm.grouped(train, y)
    alpha = pysvm.alpha_from_sklearn(order, train, sv.support_, sv.dual_coef_[0])
    return sv, order, y_pm, alpha


@pytest.mark.parametrize("C,eps", [(1.0, 1e-3), (0.05, 1e-3), (10.0, 1e-4), (100.0, 1e-3)])
def test_sklearn_fits_pass(rbf, C, eps):
    K, y, train, test = rbf
    sv, order, y_pm, alpha = sklearn_fit(K, y, train, test, C, eps)
    assert np.count_nonzero(alpha) == len(sv.support_)
    pysvm.check_fit(K, order, y_pm, alpha, sv.intercept_[0], C, eps)
    sv_ids = order[alpha > 0]
    coef = (alpha * y_pm)[alpha > 0]
    exact, bound = pysvm.exact_scores(K, test, sv_ids, coef, sv.intercept_[0])
    ref = sv.decision_function(K[np.ix_(test, train)])
    assert np.all(np.abs(ref - exact) <= bound)


def test_small_errors_fail(rbf):
    K, y, train, test = rbf
    C, eps = 1.0, 1e-3
    sv, order, y_pm, alpha = sklearn_fit(K, y, train, test, C, eps)
    rho = sv.intercept_[0]
    free = np.flatnonzero((alpha > 0) & (alpha < C))
    assert len(free) > 0
    bad = alpha.copy()
    bad[free[0]] += 1e-7 * C
    with pytest.raises(AssertionError):
        pysvm.check_fit(K, order, y_pm, bad, rho, C, eps)
    with pytest.raises(AssertionError):
        pysvm.check_fit(K, order, y_pm, bad, rho, C, eps, truncated=True)
    # an alpha above C by one ulp, a shifted rho, a run stopped long before eps
    bad = alpha.copy()
    bad[np.argmax(alpha)] = np.nextafter(C, np.inf)
    with pytest.raises(AssertionError):
        pysvm.check_fit(K, order, y_pm, bad, rho, C, eps, truncated=True)
    with pytest.raises(AssertionError):
        pysvm.check_fit(K, order, y_pm, alpha, rho + 2 * eps, C, eps)
    sv5, order5, y5, alpha5 = sklearn_fit(K, y, train, test, C, eps, max_iter=5)
    assert sv5.n_iter_[0] == 5
    pysvm.check_fit(K, order5, y5, alpha5, sv5.intercept_[0], C, eps, truncated=True)
    with pytest.raises(AssertionError):
        pysvm.check_fit(K, order5, y5, alpha5, sv5.intercept_[0], C, eps)
    # scores: one coefficient off by a relative 1e-9 moves some decision value outside the bound
    sv_ids = order[alpha > 0]
    coef = (alpha * y_pm)[alpha > 0]
    _, bound = pysvm.exact_scores(K, test, sv_ids, coef, rho)
    ref = sv.decision_function(K[np.ix_(test, train)])
    coef2 = coef.copy()
    coef2[np.argmax(np.abs(coef))] *= 1 + 1e-9
    exact2, _ = pysvm.exact_scores(K, test, sv_ids, coef2, rho)
    assert np.any(np.abs(ref - exact2) > bound)
