"""float64 checks of a C-SVC fit on a precomputed kernel matrix that do not depend on the solver's path (TEST
INFRASTRUCTURE ONLY; plain numpy, no product code).

Where the GPU solver and sklearn's libsvm follow the same iterates, the tests compare them value for value.  These
checks hold for any correct fit, so they also judge a fit where the two paths might part, and they judge sklearn itself:

* ``check_fit``     -- the box and equality constraints of the dual, and libsvm's stopping rule recomputed from the
                       matrix (not from the solver's incrementally updated gradient);
* ``exact_scores``  -- decision values from a correctly rounded sum, with the error bound of a sequential double sum.

Conventions are libsvm's sub-problem: the training points of a fit in grouped order (``order``: label 0 first, the
order libsvm's svm_group_classes gives them), ``y_pm`` = +1 for that first class and -1 for the other, ``alpha`` in the
same order, ``coef = alpha * y_pm`` of the support vectors (= minus sklearn's ``dual_coef_``), and ``rho`` (= sklearn's
``intercept_``).  A decision value is sklearn's: -(sum_k coef_k K(x, sv_k) - rho), positive for label 1.
"""
import math

import numpy as np


def grouped(train, y01):
    """(order, y_pm) of a fit on the training ids `train` with 0/1 labels `y01` (indexed by id)"""
    train = np.asarray(train)
    lab = np.asarray(y01)[train]
    order = np.concatenate((train[lab == 0], train[lab == 1]))
    return order, np.where(np.asarray(y01)[order] == 0, 1, -1)


def alpha_from_sklearn(order, train, support, dual_coef):
    """alpha in grouped order from a fitted sklearn SVC: `support` indexes `train`, |dual_coef_| = alpha"""
    a = dict(zip(np.asarray(train)[support].tolist(), np.abs(np.asarray(dual_coef)).tolist()))
    return np.array([a.get(int(i), 0.0) for i in order])


def q_tilde(K, rows, cols, y_rows, y_cols):
    """the Q libsvm iterates with: float32(y_i y_k K_ik) (its kernel-row cache holds floats), promoted to double"""
    return ((np.multiply.outer(y_rows, y_cols).astype(np.float64) * K[np.ix_(rows, cols)]).astype(np.float32)
            .astype(np.float64))


def check_fit(K, order, y_pm, alpha, rho, C, eps, truncated=False):
    """raise AssertionError unless (alpha, rho) is a fit libsvm could have stopped at (any path, same C and eps)"""
    order = np.asarray(order)
    y = np.asarray(y_pm, np.float64)
    a = np.asarray(alpha, np.float64)
    l = len(order)
    assert a.shape == (l,) and y.shape == (l,)
    assert np.all(a >= 0.0) and np.all(a <= C), "alpha outside [0, C]: min %r max %r" % (a.min(), a.max())
    s = math.fsum((y * a).tolist())
    assert abs(s) <= 1e-12 * C * l, "sum y alpha = %r" % s
    if truncated:
        return
    # G = Q~ alpha - 1 over the support vectors, in bands of rows to bound the memory
    sv = np.flatnonzero(a > 0)
    G = np.empty(l)
    for b in range(0, l, 2048):
        rows = slice(b, min(l, b + 2048))
        G[rows] = q_tilde(K, order[rows], order[sv], y[rows], y[sv]) @ a[sv] - 1.0
    up = np.where(y > 0, a < C, a > 0)
    low = np.where(y > 0, a > 0, a < C)
    m_up = np.max(-y[up] * G[up]) if up.any() else -np.inf
    m_low = np.min(-y[low] * G[low]) if low.any() else np.inf
    # The solver updates G incrementally, so its G differs from this one by rounding only: the slack is relative to the
    # size of G (|G| grows with C), 1e-9 of it is far above the rounding of any run here and far below eps.
    slack = 1e-9 * max(1.0, float(np.max(np.abs(G))))
    assert m_up - m_low < eps + slack, "stopping rule: max_up(-yG) - min_low(-yG) = %r >= eps = %r" % (m_up - m_low, eps)
    # rho: libsvm takes the mean of y G over the free vectors, or the midpoint of the bounds set by the others; with the
    # stopping rule, either lies within eps of every bound [lb, ub] those vectors give
    yG = y * G
    at_ub = ((a >= C) & (y < 0)) | ((a <= 0) & (y > 0))
    at_lb = ((a >= C) & (y > 0)) | ((a <= 0) & (y < 0))
    ub = np.min(yG[at_ub]) if at_ub.any() else np.inf
    lb = np.max(yG[at_lb]) if at_lb.any() else -np.inf
    assert lb - eps - slack <= rho <= ub + eps + slack, "rho = %r outside [%r, %r] +- eps" % (rho, lb, ub)
    free = (a > 0) & (a < C)   # in I_up and I_low both: y G of each is within eps of rho
    if free.any():
        dev = float(np.max(np.abs(yG[free] - rho)))
        assert dev < eps + slack, "free vectors: max |yG - rho| = %r" % dev


def assert_follows_sklearn(K, y01, train, test, scores, fit, alpha, sv, ref, C, eps, truncated=False):
    """a solver's fit of one split -- decision values `scores` of `test`, `fit` (rho, nu, n_iter, n_sv), `alpha` in
    grouped order -- against sklearn's SVC `sv` fitted on the same split with the same C, tol and max_iter, and its
    decision values `ref`: the same path (iterations, support set, dual_coef_, intercept_, decision values to 1e-9),
    then the path-independent checks above"""
    train = np.asarray(train)
    order, y_pm = grouped(train, y01)
    alpha = np.asarray(alpha)
    assert fit["n_iter"] == sv.n_iter_[0], (fit["n_iter"], sv.n_iter_[0])
    assert fit["n_sv"] == len(sv.support_)
    sv_ids = order[alpha > 0]
    assert np.array_equal(np.sort(sv_ids), np.sort(train[sv.support_]))
    coef = (alpha * y_pm)[alpha > 0]
    by_id = dict(zip(train[sv.support_].tolist(), (-sv.dual_coef_[0]).tolist()))
    np.testing.assert_allclose(coef, [by_id[int(i)] for i in sv_ids], rtol=1e-9, atol=1e-12)
    assert abs(fit["rho"] - sv.intercept_[0]) <= 1e-9 * abs(sv.intercept_[0]) + 1e-12, (fit["rho"], sv.intercept_[0])
    np.testing.assert_allclose(scores, ref, rtol=1e-9, atol=1e-11)
    assert abs(fit["nu"] - np.sum(np.abs(sv.dual_coef_[0])) / len(train)) <= 1e-9 * fit["nu"]
    check_fit(K, order, y_pm, alpha, fit["rho"], C, eps, truncated)
    exact, bound = exact_scores(K, test, sv_ids, coef, fit["rho"])
    assert np.all(np.abs(np.asarray(scores) - exact) <= bound), np.max(np.abs(np.asarray(scores) - exact) - bound)


def exact_scores(K, test, sv_ids, coef, rho):
    """(decision values of the rows `test` from a correctly rounded sum of the rounded products coef_k K[r, sv_k],
    error bound of a sequential double sum of the same terms) -- a solver's scores must lie within the bound"""
    sv_ids = np.asarray(sv_ids)
    coef = np.asarray(coef, np.float64)
    test = np.asarray(test)
    out = np.empty(len(test))
    bound = np.empty(len(test))
    for r, t in enumerate(test):
        terms = coef * K[t, sv_ids]
        out[r] = -(math.fsum(terms.tolist()) - rho)
        # the bound needs no exact sum: 1e-12 relative covers numpy's own rounding of sum |terms|
        bound[r] = (len(sv_ids) + 2) * 2.0 ** -53 * (float(np.sum(np.abs(terms))) * (1 + 1e-12) + abs(rho))
    return out, bound
