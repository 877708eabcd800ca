"""GPU tier of the shrinking solver (gkmb200_svm_cv_ex with shrinking = 1) against sklearn's
SVC(kernel="precomputed", shrinking=True): the same path as libsvm's Solver::Solve with shrinking -- iterations,
support vectors, dual_coef_, intercept_ and decision values to 1e-9 through pysvm.assert_follows_sklearn -- and the same
shrink passes, unshrink and gradient reconstructions as the numpy restatement in tests/pysvm_shrink.py.  The per-fit
statistics the entry point reports show that the shrink passes, the unshrink and both reconstruction orders ran."""
import warnings

import numpy as np
import pytest

import pysvm
import pysvm_shrink
from gkmqc_b200 import capi, driver
from test_gpu_svm import hard_seqs, planted_seqs
from test_svm_checks import rbf  # noqa: F401  (the fixture)

pytestmark = pytest.mark.gpu

SVC = pytest.importorskip("sklearn.svm").SVC
from sklearn.exceptions import ConvergenceWarning
from sklearn.metrics import roc_auc_score
from sklearn.model_selection import StratifiedKFold

PLANTED = [(1.0, 1e-3), (0.1, 1e-3), (10.0, 1e-4)]
HARD_C = [1e-4, 1.0, 100.0]
RBF = [(1.0, 1e-3), (0.05, 1e-3), (10.0, 1e-4), (100.0, 1e-3)]


def shrinking_fit(K, y, train, test, C, eps, max_iter=-1):
    sv = SVC(kernel="precomputed", C=C, tol=eps, shrinking=True, gamma=1.0, cache_size=500, max_iter=max_iter)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", ConvergenceWarning)
        sv.fit(K[np.ix_(train, train)], y[train])
    return sv, sv.decision_function(K[np.ix_(test, train)])


def kernel_of(seqs):
    with capi.Problem(4, 10, 6, 3, 50, 50.0, 1.0) as P:
        P.add_many(seqs)
        K = P.kernel_lower()
    return np.maximum(K, K.T)


@pytest.fixture(scope="module")
def planted():
    """the 600-sequence planted problem of test_gpu_svm.py, 5 folds; the device problem stays open for the resident runs"""
    capi.load()
    seqs = planted_seqs(300, 300, 200)
    P = capi.Problem(4, 10, 6, 3, 50, 50.0, 1.0)
    P.add_many(seqs)
    K = P.kernel_lower()
    K = np.maximum(K, K.T)
    y = np.concatenate((np.ones(300, int), np.zeros(300, int)))
    splits = list(StratifiedKFold(n_splits=5, shuffle=True, random_state=3).split(np.zeros(len(y)), y))
    runs = {ce: capi.svm_cv(y, splits, kmat=K, C=ce[0], eps=ce[1], shrinking=1, stats=True) for ce in PLANTED}
    yield P, K, y, splits, runs
    P.close()


@pytest.fixture(scope="module")
def hard():
    """313 : 32 classes with exact duplicates (test_gpu_svm.py's hard problem), 5 folds"""
    capi.load()
    seqs, npos = hard_seqs()
    K = kernel_of(seqs)
    y = np.concatenate((np.ones(npos, int), np.zeros(len(seqs) - npos, int)))
    splits = list(StratifiedKFold(n_splits=5, shuffle=True, random_state=4).split(np.zeros(len(y)), y))
    runs = {C: capi.svm_cv(y, splits, kmat=K, C=C, eps=1e-3, shrinking=1, stats=True) for C in HARD_C}
    return K, y, splits, runs


@pytest.fixture(scope="module")
def rbf_runs(rbf):  # noqa: F811
    """the 400-point RBF matrix of test_svm_checks.py as a host matrix, at the (C, eps) of the CPU tier: at C = 1 libsvm
    rebuilds the gradient with few free vectors, i.e. in its second loop order"""
    K, y, train, test = rbf
    splits = [(train, test)]
    return K, y, splits, {ce: capi.svm_cv(y, splits, kmat=K, C=ce[0], eps=ce[1], shrinking=1, stats=True) for ce in RBF}


def follows(K, y, splits, run, C, eps, max_iter=-1):
    """every fit of `run` against sklearn with shrinking and against the numpy restatement (stats included)"""
    for (train, test), s, f, a, st in zip(splits, *run):
        sv, ref = shrinking_fit(K, y, train, test, C, eps, max_iter)
        truncated = max_iter >= 0 and f["n_iter"] == max_iter
        pysvm.assert_follows_sklearn(K, y, train, test, s, f, a, sv, ref, C, eps, truncated=truncated)
        order, y_pm = pysvm.grouped(train, y)
        m = pysvm_shrink.solve(K, order, y_pm, C, eps, max_iter)
        assert {k: m[k] for k in st} == st, (m, st)
        assert np.array_equal(m["alpha"], a) and m["rho"] == f["rho"]


@pytest.mark.parametrize("C,eps", PLANTED)
def test_shrinking_fits_follow_libsvm(planted, C, eps):
    P, K, y, splits, runs = planted
    follows(K, y, splits, runs[(C, eps)], C, eps)


@pytest.mark.parametrize("at", ["l", "l+1", "l+2", "2l+1", "unshrink+1"])
def test_truncated_shrinking_runs_follow_libsvm(planted, at):
    """max_iter around the shrink counter (the first pass comes after l iterations) and one iteration past the unshrink
    the untruncated run reports; a fit that converges before max_iter is compared as it is"""
    P, K, y, splits, runs = planted
    C, eps = 10.0, 1e-4
    full = runs[(C, eps)]
    stopped = 0
    for t, (train, test) in enumerate(splits[:3]):
        l = len(train)
        if at == "unshrink+1":
            u = full[3][t]["unshrink_iter"]
            if u < 0:
                continue
            max_iter = u + 1
        else:
            max_iter = {"l": l, "l+1": l + 1, "l+2": l + 2, "2l+1": 2 * l + 1}[at]
        run = capi.svm_cv(y, [(train, test)], kmat=K, C=C, eps=eps, max_iter=max_iter, shrinking=1, stats=True)
        assert run[1][0]["n_iter"] == min(max_iter, full[1][t]["n_iter"])
        stopped += run[1][0]["n_iter"] == max_iter
        follows(K, y, [(train, test)], run, C, eps, max_iter)
    assert stopped > 0, "no fit ran long enough to be cut at %s" % at


@pytest.mark.parametrize("C", HARD_C)
def test_hard_problems_follow_libsvm_with_shrinking(hard, C):
    K, y, splits, runs = hard
    follows(K, y, splits, runs[C], C, 1e-3)


@pytest.mark.parametrize("C,eps", RBF)
def test_rbf_matrix_follows_libsvm_with_shrinking(rbf_runs, C, eps):
    K, y, splits, runs = rbf_runs
    follows(K, y, splits, runs[(C, eps)], C, eps)


def test_the_stats_cover_every_path(planted, hard, rbf_runs):
    """across the fits above: two or more shrink passes with a smaller active set, an unshrink, and a gradient
    reconstruction in each of libsvm's two loop orders -- a solver that never shrinks cannot pass"""
    P, K, y, splits, runs = planted
    stats = [(len(tr), st) for r in runs.values() for (tr, _), st in zip(splits, r[3])]
    K, y, splits, runs = hard
    stats += [(len(tr), st) for r in runs.values() for (tr, _), st in zip(splits, r[3])]
    K, y, splits, runs = rbf_runs
    stats += [(len(tr), st) for r in runs.values() for (tr, _), st in zip(splits, r[3])]
    assert any(st["shrink_passes"] >= 2 and st["min_active"] < l for l, st in stats)
    assert any(st["unshrink_iter"] >= 0 for _, st in stats)
    assert any(st["recon_a"] > 0 for _, st in stats)
    assert any(st["recon_b"] > 0 for _, st in stats)


def test_resident_matrix_equals_host_matrix_with_shrinking(planted):
    P, K, y, splits, runs = planted
    host = runs[(1.0, 1e-3)]
    dev = capi.svm_cv(y, splits, problem=P, C=1.0, eps=1e-3, shrinking=1, stats=True)
    for a, b in zip(host[0] + host[2], dev[0] + dev[2]):
        assert np.array_equal(a, b)
    assert host[1] == dev[1] and host[3] == dev[3]


def test_shrinking_off_is_svm_cv(planted):
    """gkmb200_svm_cv_ex with shrinking = 0 is gkmb200_svm_cv, bit for bit, and reports that nothing shrank"""
    P, K, y, splits, runs = planted
    s0, f0, a0 = capi.svm_cv(y, splits, kmat=K, C=1.0, eps=1e-3)
    s1, f1, a1, st = capi.svm_cv(y, splits, kmat=K, C=1.0, eps=1e-3, shrinking=0, stats=True)
    for a, b in zip(s0 + a0, s1 + a1):
        assert np.array_equal(a, b)
    assert f0 == f1
    assert st == [dict(shrink_passes=0, min_active=len(tr), unshrink_iter=-1, recon_a=0, recon_b=0) for tr, _ in splits]


def test_bad_shrinking_value_is_rejected(planted):
    P, K, y, splits, runs = planted
    for bad in (2, -1):
        with pytest.raises(capi.GkmError, match="shrinking must be 0 or 1"):
            capi.svm_cv(y, splits[:1], kmat=K, shrinking=bad)


def test_global_state_fit_with_shrinking():
    """one fit of 10 800 points, above the 10 724 whose state fits shared memory: the permuted gather index and labels
    are the solver's own copies, so the caller's train_idx is untouched and the decision values read the grouped order"""
    capi.load()
    npos = nneg = 5500
    K = kernel_of(planted_seqs(npos, nneg, 200, seed=81, motif_seed=82))
    y = np.concatenate((np.ones(npos, int), np.zeros(nneg, int)))
    perm = np.random.default_rng(5).permutation(len(y))
    train, test = np.sort(perm[:10800]), np.sort(perm[10800:])
    assert 21 * len(train) + 64 > 220 * 1024
    tasks, tr, ty, te = capi.svm_prepare_tasks(y, [(train, test)])
    tr0, ty0 = tr.copy(), ty.copy()
    scores, alpha = np.zeros(len(te)), np.zeros(len(tr))
    fits = (capi.gkmb200_svm_fit * 1)()
    st = (capi.gkmb200_svm_shrink_stats * 1)()
    opt = capi.gkmb200_svm_options(1.0, 1e-3, -1, 1, 0)
    lib = capi.load()
    rc = lib.gkmb200_svm_cv_ex(None, K.ctypes.data, len(y), len(y), 1, tasks, tr.ctypes.data_as(capi.c_int_p),
                               ty.ctypes.data_as(capi.ctypes.POINTER(capi.ctypes.c_byte)), te.ctypes.data_as(capi.c_int_p),
                               capi.ctypes.byref(opt), scores.ctypes.data_as(capi.c_dbl_p), fits, alpha.ctypes.data_as(capi.c_dbl_p), st)
    assert rc == 0, capi.last_error()
    assert np.array_equal(tr, tr0) and np.array_equal(ty, ty0)
    assert st[0].shrink_passes >= 1 and st[0].min_active < len(train), st[0].as_dict()
    f = fits[0]
    sv, ref = shrinking_fit(K, y, train, test, 1.0, 1e-3)
    pysvm.assert_follows_sklearn(K, y, train, test, scores, dict(rho=f.rho, nu=f.nu, n_iter=f.n_iter, n_sv=f.n_sv), alpha,
                                 sv, ref, 1.0, 1e-3)


def test_driver_crossValidate_honours_shrinking(planted):
    """-u 1: gkmsvm.crossValidate restated with SVC(shrinking=True), against the driver mirror"""
    P, K, y, splits, runs = planted
    npos = int(y.sum())
    mean_gpu, std_gpu = driver.crossValidate([1.0, 0.001, 1, 100, 5, 2, 0, 7, 4], K, npos, len(y) - npos)
    aucs = []
    for _ in range(2):
        for train, test in StratifiedKFold(n_splits=5, shuffle=True, random_state=7).split(np.zeros(len(y)), y):
            _, ref = shrinking_fit(K, y, train, test, 1.0, 0.001)
            aucs.append(roc_auc_score(y[test], ref))
    assert mean_gpu == pytest.approx(np.mean(aucs), abs=1e-9)
    assert std_gpu == pytest.approx(np.std(aucs), abs=1e-9)


def test_peer_written_resident_matrix_with_shrinking_if_available(planted):
    """the resident matrix every GPU of the process wrote a share of: the same shrinking fits as on the host matrix"""
    ndev = capi.device_count()
    if ndev < 2:
        pytest.skip("single GPU box")
    P0, K, y, splits, runs = planted
    lib = capi.load()
    try:
        arr = (capi.ctypes.c_int * ndev)(*range(ndev))
        assert lib.gkmb200_set_devices(arr, ndev) == 0, capi.last_error()
        with capi.Problem(4, 10, 6, 3, 50, 50.0, 1.0) as P:
            P.add_many(planted_seqs(300, 300, 200))
            dev = capi.svm_cv(y, splits, problem=P, C=1.0, eps=1e-3, shrinking=1, stats=True)
            assert P.stats()["devices"] == ndev
        host = runs[(1.0, 1e-3)]
        for a, b in zip(host[0] + host[2], dev[0] + dev[2]):
            assert np.array_equal(a, b)
        assert host[1] == dev[1] and host[3] == dev[3]
    finally:
        ids = (capi.ctypes.c_int * 1)(0)
        lib.gkmb200_set_devices(ids, 1)
