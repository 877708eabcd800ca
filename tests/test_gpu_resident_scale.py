"""The resident kernel matrix and its C-SVC consumer at the sizes gkmQC and the benchmark run them.

* A gkmQC-size bin: 15 000 sequences (driver.MAX_SEQS), 5-fold: 12 000 training points per fit keep the solver state
  in global memory (gkm_svm.cu keeps it in shared memory up to 10 724 points) and 3 000 test points per fit take 12
  blocks of the decision kernel.  Every fit against sklearn (same path) and the path-independent checks of
  oracle/pysvm.py; the resident matrix gives the same fits bit for bit.
* gkmQC's own call: driver.crossValidate with 5 folds x 10 repeats, the 50 fits in one call.
* The benchmark's matrix: 50 000 x 50 000 (bench.py's headline problem), made resident by the index kernel and by
  the bit-sliced kernel, read back in bands and compared through position-dependent digests and stored rows.  Past
  row 42 949, row * ld exceeds 2^31: an int offset anywhere in the store or mirror path would show there.
"""
import time

import numpy as np
import pytest

import pysvm
from gkmqc_b200 import capi, driver
from test_gpu_svm import planted_seqs, sklearn_fit

pytestmark = pytest.mark.gpu

from sklearn.metrics import roc_auc_score
from sklearn.model_selection import StratifiedKFold

SMEM_LIMIT = 220 * 1024      # gkm_svm_run: in_smem = (smem_need = 21 * lmax + 64) <= 220 KiB


@pytest.fixture(scope="module")
def bin15k():
    """7 500 + 7 500 sequences of 300 bp with planted motifs, wgkm L=10 k=6 d=3 (gkmQC's kernel)"""
    capi.load()
    npos = nneg = 7500
    seqs = planted_seqs(npos, nneg, 300, seed=61, motif_seed=62)
    P = capi.Problem(4, 10, 6, 3, 50, 50.0, 1.0)
    P.add_many(seqs)
    K = P.kernel_lower()
    K = np.maximum(K, K.T)
    y = np.concatenate((np.ones(npos, int), np.zeros(nneg, int)))
    yield P, K, y
    P.close()


def _against_sklearn(K, y, splits, scores, fits, alphas, C=1.0, eps=1e-3):
    for (train, test), s, f, a in zip(splits, scores, fits, alphas):
        sv, ref = sklearn_fit(K, y, train, test, C, eps)
        pysvm.assert_follows_sklearn(K, y, train, test, s, f, a, sv, ref, C, eps)


def test_gkmqc_size_bin_five_folds(bin15k):
    P, K, y = bin15k
    splits = list(StratifiedKFold(n_splits=5, shuffle=True, random_state=13).split(np.zeros(len(y)), y))
    assert all(len(tr) == 12000 and len(te) == 3000 for tr, te in splits)
    assert 21 * 12000 + 64 > SMEM_LIMIT and (3000 + 255) // 256 == 12
    t0 = time.time()
    s_host, f_host, a_host = capi.svm_cv(y, splits, kmat=K, C=1.0, eps=1e-3)
    t_host = time.time() - t0
    _against_sklearn(K, y, splits, s_host, f_host, a_host)
    s_dev, f_dev, a_dev = capi.svm_cv(y, splits, problem=P, C=1.0, eps=1e-3)
    for a, b in zip(s_host + a_host, s_dev + a_dev):
        assert np.array_equal(a, b)
    assert [f["n_iter"] for f in f_host] == [f["n_iter"] for f in f_dev]
    print("15k bin: 5 fits of 12 000 points in %.2f s on the host matrix, iterations %s"
          % (t_host, [f["n_iter"] for f in f_host]))


@pytest.mark.parametrize("ntrain", [10724, 10725])
def test_shared_memory_boundary(bin15k, ntrain):
    """the largest fit whose solver state fits shared memory, and one point more (global memory)"""
    # gkm_svm_run (gkm_svm.cu): smem_need = 21 * lmax + 64 bytes (G, alpha: 8 + 8, gather index: 4, y: 1 per point)
    assert (21 * ntrain + 64 <= SMEM_LIMIT) == (ntrain == 10724)
    P, K, y = bin15k
    perm = np.random.default_rng(ntrain).permutation(len(y))
    splits = [(np.sort(perm[:ntrain]), np.sort(perm[ntrain:ntrain + 1000]))]
    scores, fits, alphas = capi.svm_cv(y, splits, kmat=K, C=1.0, eps=1e-3)
    _against_sklearn(K, y, splits, scores, fits, alphas)


def test_mixed_fit_sizes_in_one_call(bin15k):
    """the largest fit of a call decides where the solver state lives: a fit of 3 000 points next to one of 12 000 runs
    from global memory too"""
    P, K, y = bin15k
    big_tr, big_te = next(StratifiedKFold(n_splits=5, shuffle=True, random_state=17).split(np.zeros(len(y)), y))
    small_tr = big_te
    small_te = np.sort(np.random.default_rng(3).choice(big_tr, 2000, replace=False))
    splits = [(big_tr, big_te), (small_tr, small_te)]
    scores, fits, alphas = capi.svm_cv(y, splits, kmat=K, C=1.0, eps=1e-3)
    _against_sklearn(K, y, splits, scores, fits, alphas)
    # the small fit alone (shared-memory state) follows the same path
    s1, f1, a1 = capi.svm_cv(y, splits[1:], kmat=K, C=1.0, eps=1e-3)
    assert np.array_equal(s1[0], scores[1]) and np.array_equal(a1[0], alphas[1]) and f1[0] == fits[1]


def test_crossValidate_fifty_fits(monkeypatch):
    """gkmQC's evaluate on one bin: 5 folds x 10 repeats in one call (driver.crossValidate); every fit against sklearn
    on the same splits, and the mean and std of the AUCs"""
    capi.load()
    npos = nneg = 1000
    with capi.Problem(4, 10, 6, 3, 50, 50.0, 1.0) as P:
        P.add_many(planted_seqs(npos, nneg, 300, seed=71, motif_seed=72))
        K = P.kernel_lower()
    K = np.maximum(K, K.T)
    y = np.concatenate((np.ones(npos, int), np.zeros(nneg, int)))
    calls = []
    svm_cv = capi.svm_cv

    def recording(yy, splits, **kw):
        out = svm_cv(yy, splits, **kw)
        calls.append((list(splits), out))
        return out

    monkeypatch.setattr(capi, "svm_cv", recording)
    state = np.random.get_state()
    np.random.seed(12)   # random_seeds = -1: StratifiedKFold draws from numpy's global generator, so every repeat differs
    try:
        mean, std = driver.crossValidate([1.0, 1e-3, 0, 100, 5, 10, 0, -1, 1], K, npos, nneg)
    finally:
        np.random.set_state(state)
    assert len(calls) == 1
    splits, (scores, fits, alphas) = calls[0]
    assert len(splits) == 50 and len({tuple(te[:8]) for _, te in splits}) == 50
    _against_sklearn(K, y, splits, scores, fits, alphas)
    aucs = []
    for train, test in splits:
        _, ref = sklearn_fit(K, y, train, test, 1.0, 1e-3)
        aucs.append(roc_auc_score(y[test], ref))
    assert abs(mean - np.mean(aucs)) <= 1e-12 and abs(std - np.std(aucs)) <= 1e-12
    assert 0.6 < mean <= 1.0


N50K = 50000
BAND = 1000
# rows on both sides of the index kernel's column-block edges (22 528-column blocks), where row * ld passes 2^31, the last
KEEP = (0, 22527, 22528, 45055, 45056, 42949, 42950, N50K - 1)


def _digest(u, w):
    """sum of bits_i * (2i + 1) mod 2^64 over the uint64 view: any changed, moved or swapped entry changes it"""
    return int(np.sum(u * w[:len(u)], dtype=np.uint64))


def _resident_50k(variant, ids):
    lib = capi.load()
    arr = (capi.ctypes.c_int * len(ids))(*ids)
    assert lib.gkmb200_set_devices(arr, len(ids)) == 0, capi.last_error()
    import bench
    capi.set_option("kernel", variant)
    w = np.arange(BAND * N50K, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    try:
        with capi.Problem(2, 11, 7, 3) as P:
            P.add_block(bench.synth(N50K))
            t0 = time.time()
            P.resident_matrix(0, 0)
            t_pass = time.time() - t0
            st, layout = P.stats(), P.index_layout()
            assert st["devices"] == len(ids)
            digests, kept = [], {}
            for r0 in range(0, N50K, BAND):
                R = P.resident_matrix(r0, min(BAND, N50K - r0))
                digests.append(_digest(R.view(np.uint64).ravel(), w))
                for r in KEEP:
                    if r0 <= r < r0 + len(R):
                        kept[r] = R[r - r0].copy()
            print("50k resident, %s on %d GPU(s): %.2f s for the pass, %.2f s in all" % (variant, len(ids), t_pass, time.time() - t0))
        return st, layout, digests, kept
    finally:
        capi.set_option("kernel", "auto")
        ids0 = (capi.ctypes.c_int * 1)(0)
        lib.gkmb200_set_devices(ids0, 1)


@pytest.fixture(scope="module")
def index50k():
    return _resident_50k("index", [0])


def test_benchmark_matrix_resident_index_equals_bitsliced(index50k):
    """the 20 GB resident matrix of bench.py's headline problem (50 000 x 300 bp, type 2, L=11 k=7 d=3), index kernel
    against bit-sliced kernel, every entry through the band digests; one problem at a time on the device"""
    st_i, layout, dig_i, kept_i = index50k
    assert st_i["kernel_variant"] == 4 and layout[:2] == (3, 22528), layout
    st_d, _, dig_d, kept_d = _resident_50k("diag", [0])
    assert st_d["kernel_variant"] == 2
    for r in KEEP:
        assert np.array_equal(kept_i[r], kept_d[r]), "row %d" % r
        assert kept_i[r][r] == 1.0
        assert np.all(np.isfinite(kept_i[r])) and np.all(kept_i[r] >= 0.0)
        for s in KEEP:
            assert kept_i[r][s] == kept_i[s][r], (r, s)
    bad = [b * BAND for b, (x, z) in enumerate(zip(dig_i, dig_d)) if x != z]
    assert not bad, "bands starting at rows %s differ" % bad[:10]


def test_benchmark_matrix_shared_by_the_gpus_if_available(index50k):
    """every GPU of the process stores its chunks into the first one's matrix: the same digests as on one GPU"""
    ndev = capi.device_count()
    if ndev < 2:
        pytest.skip("single GPU box")
    st_m, _, dig_m, kept_m = _resident_50k("index", list(range(ndev)))
    assert st_m["devices"] == ndev
    assert dig_m == index50k[2]
    for r in KEEP:
        assert np.array_equal(kept_m[r], index50k[3][r])
