"""GPU tier for the consumer of the kernel matrix (SURVEY.md 8f/f4): the C-SVC cross-validation of
scripts/gkmsvm.py:104-160 on the GPU against sklearn's SVC(kernel="precomputed") -- sklearn's bundled libsvm is the
reference implementation of this piece (third-party; scikit-learn 1.9.0 in this image and on the GPU box).

Bar: the GPU solver restates libsvm's SMO arithmetic (float-cached Q rows, tie rules, unfused updates), so the
iterates coincide: same iteration count and support vectors, alpha and decision values to 1e-9 relative.  Should the
paths ever part (they stop within eps = 1e-3 of the same optimum), the looser tier still holds: AUC within 2e-3."""
import warnings

import numpy as np
import pytest

import pysvm
from conftest import random_seqs
from gkmqc_b200 import capi, driver

pytestmark = pytest.mark.gpu

SVC = pytest.importorskip("sklearn.svm").SVC
from sklearn.exceptions import ConvergenceWarning
from sklearn.metrics import roc_auc_score
from sklearn.model_selection import StratifiedKFold


def planted_seqs(npos, nneg, length, seed=21, motif_seed=5):
    """npos + nneg random sequences; the first npos carry one to three planted 10-bp motifs (one base mutated half the
    time), so that the SVM has something to learn"""
    rng = np.random.default_rng(motif_seed)
    seqs = random_seqs(npos + nneg, length, seed=seed)
    motifs = ["GATAAGGCAT", "TTGACGTCAA", "CCCGCCCCTA"]
    for i in range(npos):
        s = list(seqs[i])
        for m in motifs[: 1 + i % 3]:
            p = int(rng.integers(0, length - 10))
            mm = list(m)
            if rng.random() < 0.5:
                mm[int(rng.integers(0, 10))] = "ACGT"[int(rng.integers(0, 4))]
            s[p:p + 10] = mm
        seqs[i] = "".join(s)
    return seqs


@pytest.fixture(scope="module")
def problem():
    """two classes that differ by planted motifs"""
    capi.load()
    npos = nneg = 300
    seqs = planted_seqs(npos, nneg, 200)
    P = capi.Problem(4, 10, 6, 3, 50, 50.0, 1.0)
    P.add_many(seqs)
    K = P.kernel_lower()
    K = np.maximum(K, K.T)
    y = np.concatenate((np.ones(npos, int), np.zeros(nneg, int)))
    yield P, K, y
    P.close()


def hard_seqs():
    """313 positives : 32 negatives with exact duplicates -- 10 positives and 3 negatives repeated in their own class,
    3 negatives repeated as positives and 4 positives as negatives (identical rows of K: exact ties in G)"""
    base = planted_seqs(300, 25, 200, seed=33, motif_seed=9)
    pos = base[:300] + base[:10] + base[300:303]
    neg = base[300:325] + base[303:306] + base[10:14]
    return pos + neg, len(pos)


@pytest.fixture(scope="module")
def hard():
    capi.load()
    seqs, npos = hard_seqs()
    with capi.Problem(4, 10, 6, 3, 50, 50.0, 1.0) as P:
        P.add_many(seqs)
        K = P.kernel_lower()
    K = np.maximum(K, K.T)
    y = np.concatenate((np.ones(npos, int), np.zeros(len(seqs) - npos, int)))
    return K, y


def sklearn_fit(K, y, train, test, C, eps, max_iter=-1):
    sv = SVC(kernel="precomputed", C=C, tol=eps, shrinking=False, gamma=1.0, cache_size=500, max_iter=max_iter)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", ConvergenceWarning)   # a truncated run (max_iter) says so
        sv.fit(K[np.ix_(train, train)], y[train])
    return sv, sv.decision_function(K[np.ix_(test, train)])


@pytest.mark.parametrize("C,eps", [(1.0, 1e-3), (0.1, 1e-3), (10.0, 1e-4)])
def test_fits_follow_libsvm(problem, C, eps):
    P, K, y = problem
    kf = StratifiedKFold(n_splits=5, shuffle=True, random_state=3)
    splits = list(kf.split(np.zeros(len(y)), y))
    scores, fits, alphas = capi.svm_cv(y, splits, kmat=K, C=C, eps=eps)
    for (train, test), s, f, a in zip(splits, scores, fits, alphas):
        sv, ref = sklearn_fit(K, y, train, test, C, eps)
        # loose tier first: whatever the path, the optimum is the same within the stopping tolerance
        assert abs(roc_auc_score(y[test], s) - roc_auc_score(y[test], ref)) < 2e-3
        np.testing.assert_allclose(s, ref, atol=5 * eps * max(1.0, C))
        # strict tier: same path (iterations, support vectors, dual_coef_, intercept_, nu, decision values to 1e-9),
        # then the path-independent checks
        pysvm.assert_follows_sklearn(K, y, train, test, s, f, a, sv, ref, C, eps)


def test_resident_matrix_equals_host_matrix(problem):
    """kmat = NULL: the kernel matrix is computed on the device, mirrored there and consumed there"""
    P, K, y = problem
    kf = StratifiedKFold(n_splits=4, shuffle=True, random_state=11)
    splits = list(kf.split(np.zeros(len(y)), y))
    s_host, f_host, _ = capi.svm_cv(y, splits, kmat=K, C=1.0, eps=1e-3)
    s_dev, f_dev, _ = capi.svm_cv(y, splits, problem=P, C=1.0, eps=1e-3)
    for a, b in zip(s_host, s_dev):
        assert np.array_equal(a, b)
    assert [f["n_iter"] for f in f_host] == [f["n_iter"] for f in f_dev]


def test_driver_crossValidate_matches_the_reference_flow(problem):
    """gkmsvm.crossValidate (gkmsvm.py:126-176) restated with sklearn fits, against the driver mirror"""
    P, K, y = problem
    npos = int(y.sum())
    args_svm = [1.0, 0.001, 0, 100, 5, 2, 0, 7, 4]
    mean_gpu, std_gpu = driver.crossValidate(args_svm, K, npos, len(y) - npos)
    aucs = []
    for _ in range(2):
        kf = StratifiedKFold(n_splits=5, shuffle=True, random_state=7)
        for train, test in kf.split(np.zeros(len(y)), y):
            _, ref = sklearn_fit(K, y, train, test, 1.0, 0.001)
            aucs.append(roc_auc_score(y[test], ref))
    assert mean_gpu == pytest.approx(np.mean(aucs), abs=1e-9)
    assert std_gpu == pytest.approx(np.std(aucs), abs=1e-9)
    assert 0.6 < mean_gpu <= 1.0


def test_bad_arguments(problem):
    P, K, y = problem
    with pytest.raises(ValueError):
        capi.svm_cv(y, [(np.arange(10), np.arange(10, 20))], kmat=K)   # one class only
    with pytest.raises(capi.GkmError):
        capi.svm_cv(y, [(np.arange(len(y)), np.arange(5))], kmat=K, C=-1.0)


@pytest.mark.parametrize("max_iter", [1, 2, 17, 200])
def test_truncated_runs_follow_libsvm(problem, max_iter):
    """max_iter stops both solvers after exactly that many updates: comparing them before convergence shows that the
    iterates themselves coincide, not only the optimum they approach"""
    P, K, y = problem
    splits = list(StratifiedKFold(n_splits=5, shuffle=True, random_state=3).split(np.zeros(len(y)), y))[:3]
    scores, fits, alphas = capi.svm_cv(y, splits, kmat=K, C=1.0, eps=1e-3, max_iter=max_iter)
    for (train, test), s, f, a in zip(splits, scores, fits, alphas):
        sv, ref = sklearn_fit(K, y, train, test, 1.0, 1e-3, max_iter=max_iter)
        assert f["n_iter"] == max_iter
        pysvm.assert_follows_sklearn(K, y, train, test, s, f, a, sv, ref, 1.0, 1e-3, truncated=True)


@pytest.mark.parametrize("C", [1e-4, 1.0, 100.0])
def test_hard_problems_follow_libsvm(hard, C):
    """313 : 32 classes with exact duplicates in a class and across the classes; C = 1e-4 leaves every alpha at a bound
    (no free vector: rho is the midpoint of the bounds), C = 100 leaves most of them free"""
    K, y = hard
    splits = list(StratifiedKFold(n_splits=5, shuffle=True, random_state=4).split(np.zeros(len(y)), y))
    scores, fits, alphas = capi.svm_cv(y, splits, kmat=K, C=C, eps=1e-3)
    for (train, test), s, f, a in zip(splits, scores, fits, alphas):
        sv, ref = sklearn_fit(K, y, train, test, C, 1e-3)
        pysvm.assert_follows_sklearn(K, y, train, test, s, f, a, sv, ref, C, 1e-3)
        nr_free = np.count_nonzero((a > 0) & (a < C))
        if C == 1e-4:
            assert nr_free == 0
        else:
            assert nr_free > 0
    # the duplicates are there: identical rows of K, apart from the pair's own entries
    for i, j in [(0, 300), (9, 309), (310, 313), (316, 338), (13, 344)]:
        keep = np.ones(len(y), bool)
        keep[[i, j]] = False
        assert np.array_equal(K[i, keep], K[j, keep])


def test_host_matrix_with_ld_greater_than_n(problem):
    """kmat = a view of the top-left n x n corner of a larger buffer: passed in place with ld = its row stride; the
    rest of the buffer is NaN, so any read outside the corner would show"""
    P, K, y = problem
    n = len(y)
    buf = np.full((n + 37, n + 61), np.nan)
    buf[:n, :n] = K
    view = buf[:n, :n]
    assert view.strides == ((n + 61) * 8, 8) and not view.flags.c_contiguous
    splits = list(StratifiedKFold(n_splits=5, shuffle=True, random_state=8).split(np.zeros(n), y))
    s_pad, f_pad, a_pad = capi.svm_cv(y, splits, kmat=view, C=1.0, eps=1e-3)
    s_ref, f_ref, a_ref = capi.svm_cv(y, splits, kmat=np.ascontiguousarray(K), C=1.0, eps=1e-3)
    for a, b in zip(s_pad + a_pad, s_ref + a_ref):
        assert np.array_equal(a, b)
    assert f_pad == f_ref


def test_single_class_task_is_rejected(problem):
    """the C entry point itself refuses a fit whose training labels are all +1 or all -1 (libsvm's rho would be infinite)
    and names the task; capi.svm_cv's own check is bypassed here"""
    P, K, y = problem
    lib = capi.load()
    kmat = np.ascontiguousarray(K)

    def call(fits_spec):
        """fits_spec: [(training ids, their +1/-1 labels, test ids), ...] -> (rc, scores)"""
        tasks = (capi.gkmb200_svm_task * len(fits_spec))()
        toff = eoff = 0
        for t, (tr, ty, te) in enumerate(fits_spec):
            tasks[t].train_off, tasks[t].test_off, tasks[t].ntrain, tasks[t].ntest = toff, eoff, len(tr), len(te)
            toff += len(tr)
            eoff += len(te)
        tr = np.ascontiguousarray(np.concatenate([f[0] for f in fits_spec]), np.int32)
        ty = np.ascontiguousarray(np.concatenate([f[1] for f in fits_spec]), np.int8)
        te = np.ascontiguousarray(np.concatenate([f[2] for f in fits_spec]), np.int32)
        scores = np.full(eoff, 7.0)
        rc = lib.gkmb200_svm_cv(None, kmat.ctypes.data, len(y), len(y), len(fits_spec), tasks, tr.ctypes.data_as(capi.c_int_p),
                                ty.ctypes.data_as(capi.ctypes.POINTER(capi.ctypes.c_byte)), te.ctypes.data_as(capi.c_int_p),
                                1.0, 1e-3, -1, scores.ctypes.data_as(capi.c_dbl_p), None, None)
        return rc, scores

    good = (np.r_[300:310, 0:10], np.r_[[1] * 10, [-1] * 10], np.r_[100:105])
    for one in (1, -1):
        bad = (np.r_[310:330], np.full(20, one), np.r_[105:110])
        for spec, t in (([bad], 0), ([good, bad], 1)):
            rc, scores = call(spec)
            assert rc != 0
            assert "svm task %d" % t in capi.last_error() and "+1 and -1" in capi.last_error(), capi.last_error()
            assert np.all(scores == 7.0)
    rc, scores = call([good])
    assert rc == 0, capi.last_error()
    assert np.all(np.isfinite(scores))


def test_init_mirrors_one_bin_of_evaluate(tmp_path):
    """driver.init = gkmsvm.init (gkmsvm.py:182-222): kernel matrix + 2 x 3 cross-validation + the line in <name>.gkmqc.eval.out;
    the AUCs are those of sklearn's SVC on the same splits (what the reference's pool computes), host matrix or resident"""
    import types
    from sklearn.metrics import roc_auc_score
    from sklearn.model_selection import StratifiedKFold
    from sklearn.svm import SVC
    from gkmqc_b200 import driver
    rng = np.random.default_rng(11)
    n, npos = 240, 120
    acgt = np.frombuffer(b"ACGT", np.uint8)
    arr = acgt[rng.integers(0, 4, (n, 200))]
    for i in range(npos):   # a motif the positives share
        at = int(rng.integers(0, 190))
        arr[i, at:at + 10] = np.frombuffer(b"GATAAGGCAT", np.uint8)
    pos, neg = tmp_path / "p.fa", tmp_path / "n.fa"
    pos.write_text("".join(">p%d\n%s\n" % (i, arr[i].tobytes().decode()) for i in range(npos)))
    neg.write_text("".join(">n%d\n%s\n" % (i, arr[i].tobytes().decode()) for i in range(npos, n)))
    args = types.SimpleNamespace(kernel_type=4, full_word_length=10, non_gap_length=6, max_num_gaps=3, init_decay=50, half_life_decay=50.0,
                                 rbf_gamma=1.0, n_processes=1, verbosity=0, regularization=1.0, precision=1e-3, shrinking=0, cache_size=100,
                                 ncv=3, repeats=2, fast_estimation=0, random_seeds=5, name=str(tmp_path / "bin0"))
    auc, std = driver.init(str(pos), str(neg), args)
    auc_r, std_r = driver.init(str(pos), str(neg), args, resident=True)
    assert abs(auc - auc_r) < 1e-12 and abs(std - std_r) < 1e-12
    lines = open(args.name + ".gkmqc.eval.out").read().splitlines()
    assert len(lines) == 2 and lines[0].split("\t")[:3] == [str(pos), str(neg), str(npos)]
    assert abs(float(lines[0].split("\t")[3]) - auc) < 1e-15
    # the reference's own flow on the same matrix and splits (gkmsvm.py:104-160)
    kmat, _, _ = driver.computeGkmKernel([4, 10, 6, 3, 50, 50.0, 1.0, str(pos), str(neg), 1, 0], max_seqs=n)
    y = np.concatenate((np.repeat(1, npos), np.repeat(0, n - npos)))
    aucs = []
    for _ in range(2):
        for tr, te in StratifiedKFold(n_splits=3, shuffle=True, random_state=5).split(np.zeros(n), y):
            sv = SVC(kernel="precomputed", C=1.0, tol=1e-3, shrinking=False, gamma=1.0, cache_size=100)
            aucs.append(roc_auc_score(y[te], sv.fit(kmat[tr][:, tr], y[tr]).decision_function(kmat[te][:, tr])))
    assert abs(np.mean(aucs) - auc) < 1e-9 and abs(np.std(aucs) - std) < 1e-9 and auc > 0.7


def test_command_line_of_gkmsvm_on_the_engine(tmp_path):
    """python -m gkmqc_b200.driver: the option set and defaults of scripts/gkmsvm.py (gkmsvm.py:236-320) -- wgkm L=10 k=6 d=3 M=50
    H=50, C=1, eps=1e-3, 5-fold x 1 repeat -- and its output line"""
    from gkmqc_b200 import driver
    rng = np.random.default_rng(2)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    arr = acgt[rng.integers(0, 4, (160, 150))]
    for i in range(80):
        at = int(rng.integers(0, 140))
        arr[i, at:at + 10] = np.frombuffer(b"TTGACGTCAA", np.uint8)
    pos, neg = tmp_path / "p.fa", tmp_path / "n.fa"
    pos.write_text("".join(">p%d\n%s\n" % (i, arr[i].tobytes().decode()) for i in range(80)))
    neg.write_text("".join(">n%d\n%s\n" % (i, arr[i].tobytes().decode()) for i in range(80, 160)))
    name = str(tmp_path / "run")
    auc, std = driver.main(["-p", str(pos), "-n", str(neg), "-w", name, "-s", "3", "-v", "0"])
    auc2, std2 = driver.main(["-p", str(pos), "-n", str(neg), "-w", name, "-s", "3", "-v", "0", "--resident"])
    assert auc == auc2 and std == std2 and 0.5 < auc <= 1.0
    lines = [l.split("\t") for l in open(name + ".gkmqc.eval.out").read().splitlines()]
    assert len(lines) == 2 and lines[0][2] == "80" and float(lines[1][3]) == auc
    # the defaults are gkmQC's: the same call spelled out
    auc3, _ = driver.main(["-p", str(pos), "-n", str(neg), "-w", name, "-s", "3", "-v", "0", "-t", "4", "-L", "10", "-k", "6", "-d", "3",
                           "-M", "50", "-H", "50", "-C", "1.0", "-e", "0.001", "-x", "5", "-r", "1"])
    assert auc3 == auc


def _resident_against_host_matrix(ids):
    """the matrix kept on the device (gkmb200_resident_rows) = the caller-side matrix of the same problem, symmetrised like
    gkmsvm.py:96-97 -- on the GPUs `ids` of this process: with several, every GPU stores its chunks into the first one's
    memory (peer access), so the comparison covers rows written by each of them"""
    lib = capi.load()
    arr = (capi.ctypes.c_int * len(ids))(*ids)
    assert lib.gkmb200_set_devices(arr, len(ids)) == 0, capi.last_error()
    seqs = random_seqs(1300, 260, seed=41, ragged=True)
    # (variant, kernel type, L, k, d, index_cols (0: what fits), sequences): index_cols = 256 makes several column blocks
    # write the matrix; 20 and 33 sequences give gkm_svm_symmetrize_kernel one partial tile, and one tile plus one row
    cases = [("diag", 2, 11, 7, 3, 0, 1300), ("index", 2, 11, 7, 3, 0, 1300), ("index", 4, 10, 6, 3, 0, 1300),
             ("mma", 4, 10, 6, 3, 0, 1300), ("index", 2, 11, 7, 3, 256, 1300), ("index", 4, 10, 6, 3, 256, 1300),
             ("index", 2, 11, 7, 3, 0, 20), ("diag", 4, 10, 6, 3, 0, 33), ("index", 4, 10, 6, 3, 0, 33)]
    try:
        for variant, kt, L, k, d, cols, nseq in cases:
            capi.set_option("kernel", variant)
            capi.set_option("index_cols", cols)
            with capi.Problem(kt, L, k, d, 50, 50.0, 1.0) as P:
                P.add_many(seqs[:nseq])
                R = P.resident_matrix()
                st = P.stats()
                nblk = P.index_layout()[0]
                assert st["devices"] == len(ids), (variant, st)
                low = np.tril(P.kernel_lower(), -1)
                K = low + low.T + np.eye(P.n)
                assert np.array_equal(R, K), (variant, kt, cols, nseq, len(ids))
                assert np.array_equal(P.resident_matrix(5, 7), K[5:12])          # a band of the matrix that is already there
                with pytest.raises(capi.GkmError):
                    P.resident_matrix(P.n - 3, 4)
            if variant == "index":
                assert st["kernel_variant"] == 4
                assert (nblk >= 5) if cols else (nblk == 1), (kt, cols, nseq, nblk)
    finally:
        capi.set_option("kernel", "auto")
        capi.set_option("index_cols", 0)


def test_resident_matrix_read_back():
    _resident_against_host_matrix([0])


def test_resident_matrix_shared_by_the_gpus_of_one_process_if_available(problem):
    ndev = capi.device_count()
    if ndev < 2:
        pytest.skip("single GPU box")
    try:
        _resident_against_host_matrix(list(range(ndev)))
        # the consumer on a matrix every GPU wrote a share of: the same fits, bit for bit, as on the host matrix
        P0, K, y = problem
        splits = list(StratifiedKFold(n_splits=4, shuffle=True, random_state=11).split(np.zeros(len(y)), y))
        s_host, f_host, _ = capi.svm_cv(y, splits, kmat=K, C=1.0, eps=1e-3)
        with capi.Problem(4, 10, 6, 3, 50, 50.0, 1.0) as P:
            for i in range(P0.n):
                f, _ = P0.codes(i)
                P.add(bytes(b"ACGT"[c - 1] for c in f))
            s_dev, f_dev, _ = capi.svm_cv(y, splits, problem=P, C=1.0, eps=1e-3)
            assert P.stats()["devices"] == ndev
        for a, b in zip(s_host, s_dev):
            assert np.array_equal(a, b)
        assert [f["n_iter"] for f in f_host] == [f["n_iter"] for f in f_dev]
    finally:
        ids = (capi.ctypes.c_int * 1)(0)
        capi.load().gkmb200_set_devices(ids, 1)
