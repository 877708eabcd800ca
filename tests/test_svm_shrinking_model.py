"""The numpy restatement of libsvm's shrinking solver (tests/pysvm_shrink.py, the data-parallel form gkm_svm.cu uses)
against sklearn's SVC(kernel="precomputed", shrinking=True): same iterations, support set, dual_coef_ and intercept_, on
the matrix test_svm_checks.py builds, converged and truncated.  And the prefix-count partition against libsvm's own
sequential swap loop.  This checks the algorithm of the GPU's shrinking solver without a GPU."""
import warnings

import numpy as np
import pytest

import pysvm
import pysvm_shrink
from test_svm_checks import rbf  # noqa: F401  (the fixture)

SVC = pytest.importorskip("sklearn.svm").SVC
hypothesis = pytest.importorskip("hypothesis")
from hypothesis import given, settings  # noqa: E402
from hypothesis import strategies as st  # noqa: E402


def sklearn_shrinking_fit(K, y, train, C, eps, max_iter=-1):
    sv = SVC(kernel="precomputed", C=C, tol=eps, shrinking=True, cache_size=200, max_iter=max_iter)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")   # ConvergenceWarning of a truncated run
        sv.fit(K[np.ix_(train, train)], y[train])
    return sv


def assert_model_equals_sklearn(K, y, train, C, eps, max_iter=-1):
    order, y_pm = pysvm.grouped(train, y)
    m = pysvm_shrink.solve(K, order, y_pm, C, eps, max_iter)
    sv = sklearn_shrinking_fit(K, y, train, C, eps, max_iter)
    assert m["n_iter"] == sv.n_iter_[0], (m["n_iter"], sv.n_iter_[0])
    a = m["alpha"]
    assert np.array_equal(np.sort(order[a > 0]), np.sort(np.asarray(train)[sv.support_]))
    ref = pysvm.alpha_from_sklearn(order, train, sv.support_, sv.dual_coef_[0])
    assert np.array_equal(a, ref), np.max(np.abs(a - ref))
    assert m["rho"] == sv.intercept_[0], (m["rho"], sv.intercept_[0])
    pysvm.check_fit(K, order, y_pm, a, m["rho"], C, eps, truncated=max_iter >= 0)
    return m


STATS = []


@pytest.mark.parametrize("C,eps", [(1.0, 1e-3), (0.05, 1e-3), (10.0, 1e-4), (100.0, 1e-3)])
def test_model_follows_sklearn_shrinking(rbf, C, eps):  # noqa: F811
    K, y, train, test = rbf
    m = assert_model_equals_sklearn(K, y, train, C, eps)
    STATS.append(m)


@pytest.mark.parametrize("extra", [0, 1, 2, "2l+1", "unshrink+1"])
def test_truncated_model_follows_sklearn_shrinking(rbf, extra):  # noqa: F811
    """max_iter around the shrink counter (l, l + 1, l + 2, 2l + 1) and one iteration past the unshrink"""
    K, y, train, test = rbf
    C, eps = 10.0, 1e-4
    l = len(train)
    if extra == "unshrink+1":
        order, y_pm = pysvm.grouped(train, y)
        u = pysvm_shrink.solve(K, order, y_pm, C, eps)["unshrink_iter"]
        assert u > 0
        max_iter = u + 1
    elif extra == "2l+1":
        max_iter = 2 * l + 1
    else:
        max_iter = l + extra
    m = assert_model_equals_sklearn(K, y, train, C, eps, max_iter)
    assert m["n_iter"] == max_iter
    STATS.append(m)


def test_model_covers_every_path(rbf):  # noqa: F811
    """shrink passes that leave a smaller active set, the unshrink, and both reconstruction orders all ran above"""
    K, y, train, test = rbf
    l = len(train)
    assert len(STATS) == 9, "run the whole module"
    assert any(m["shrink_passes"] >= 2 and m["min_active"] < l for m in STATS)
    assert any(m["unshrink_iter"] >= 0 for m in STATS)
    assert any(m["recon_a"] > 0 for m in STATS)
    assert any(m["recon_b"] > 0 for m in STATS)


@settings(derandomize=True, max_examples=400, deadline=None)
@given(st.lists(st.booleans(), min_size=0, max_size=80), st.integers(0, 3))
def test_prefix_partition_is_libsvms_swap_loop(flags, bias):
    """shrink_pairs' pairing (block prefix counts) leaves the same active size and the same permutation as libsvm's
    two-pointer loop; `bias` thins the shrunk flags so long runs of either kind are drawn too"""
    flags = [f and (i % (bias + 1) == 0) for i, f in enumerate(flags)]
    n_ref, perm_ref = pysvm_shrink.shrink_sequential(flags)
    n_keep, low, high = pysvm_shrink.shrink_pairs(flags)
    perm = list(range(len(flags)))
    for p, q in zip(low, high):
        perm[p], perm[q] = perm[q], perm[p]
    assert n_keep == n_ref
    assert perm == perm_ref
