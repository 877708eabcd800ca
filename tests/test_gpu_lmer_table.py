"""GPU tier of the L-mer table (gkmb200_lmer_table_*, DESIGN.md 4.5): the exported table and the scores equal the numpy
restatement (tests/lmer_table_model.py) bit for bit, the scores lie within the rounding bound eps(r) of
gkmb200_decision_values (derived in tests/test_lmer_table_model.py), and every refusal says why."""
import contextlib
import ctypes

import numpy as np
import pytest

from gkmqc_b200 import capi
import lmer_table_model as ltm

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    capi.load()
    if capi.device_count() < 1:
        pytest.skip("no B200: " + capi.last_error())
    ids = (ctypes.c_int * 1)(0)
    assert capi.load().gkmb200_set_devices(ids, 1) == 0


@contextlib.contextmanager
def max_L16():
    capi.set_option("max_L", 16)
    try:
        yield
    finally:
        capi.set_option("max_L", 12)


def sv_seqs(L, n, seed, length=120):
    """ragged random SVs plus the awkward ones: exactly L bases, N and lower case, a duplicate, a reverse complement and
    a homopolymer (a long run in S)"""
    rng = np.random.default_rng(seed)
    acgt = np.array(list("ACGT"))
    seqs = ["".join(acgt[rng.integers(0, 4, int(rng.integers(max(L, length // 3), length + 1)))]) for _ in range(n)]
    s = seqs[1]
    seqs += [seqs[0][:L], s[:5].lower() + "N" + s[6:len(s) // 2] + "n" + s[len(s) // 2 + 1:], seqs[2],
             s[::-1].translate(str.maketrans("ACGT", "TGCA")), "A" * (L + 200)]
    return seqs


def alphas(n, seed):
    rng = np.random.default_rng(seed)
    a = rng.standard_normal(n)
    a[rng.random(n) < 0.2] = 0.0
    return a


def bound(P, model, row0, nrows, col0, alpha, w, norm, chunk=2048):
    """eps(r) for the rows [row0, row0 + nrows) against the columns [col0, col0 + len(alpha)), B from gkmb200_hist_block"""
    ncols = len(alpha)
    run = model.longest_run(col0, ncols)
    out = np.zeros(nrows)
    for r0 in range(0, nrows, chunk):
        nr = min(chunk, nrows - r0)
        H = P.hist_block(row0 + r0, nr, col0, ncols).astype(np.float64)
        rows = np.arange(row0 + r0, row0 + r0 + nr)
        B = (H @ np.abs(w)) @ (np.abs(alpha) / norm[col0:col0 + ncols]) / norm[rows]
        win = np.array([P.seqlen(r) - model.L + 1 for r in rows])
        out[r0:r0 + nr] = (ncols + run + 4 * model.L + win + 16) * 2.0 ** -52 * B
    return out


CASES = [  # (type, L, k, d, M, H)
    (0, 2, 1, 1, 50, 50.0), (1, 6, 3, 3, 50, 50.0), (2, 6, 3, 3, 50, 50.0), (4, 10, 6, 3, 50, 50.0),
    (2, 11, 7, 3, 50, 50.0), (1, 11, 7, 3, 50, 50.0), (4, 11, 7, 3, 50, 50.0), (0, 12, 8, 4, 50, 50.0),
    (2, 13, 12, 1, 50, 50.0), (0, 5, 0, 5, 50, 50.0), (4, 5, 0, 5, 50, 50.0),
]


@pytest.mark.parametrize("kt,L,k,d,M,H", CASES)
def test_table_and_scores_equal_the_restatement(kt, L, k, d, M, H):
    params = dict(kernel_type=kt, L=L, k=k, d=d, M=M, H=H)
    with (max_L16() if L > 12 else contextlib.nullcontext()), capi.Problem(**params) as P:
        seqs = sv_seqs(L, 40, seed=L * 10 + kt)
        P.add_many(seqs)
        n = P.n
        norm = P.sqnorm()
        model = ltm.Model(P, kt, L, d, M, H)
        col0, ncols = 3, n - 3
        alpha = alphas(ncols, L)
        T = model.table(col0, alpha, norm)
        with P.lmer_table(col0, ncols, alpha) as t:
            assert np.array_equal(t.weights(), ltm.export(T, L)), "table"
            got = t.scores(P, 1, n - 1, bias=0.125)
            assert np.array_equal(got, model.scores(T, norm, range(1, n), bias=0.125)), "scores"
            dv = P.decision_values(1, n - 1, col0, ncols, alpha, 0.125)
            eps = bound(P, model, 1, n - 1, col0, alpha, model.w, norm)
            assert np.all(np.abs(got - dv) <= eps), float(np.max(np.abs(got - dv) / eps))
            # a second problem with the same parameters: rows that are not SVs
            with capi.Problem(**params) as Q:
                Q.add_many(sv_seqs(L, 25, seed=999 + L)[:25])
                qn = Q.sqnorm()
                qm = ltm.Model(Q, kt, L, d, M, H)
                assert np.array_equal(t.scores(Q, 2, Q.n - 2, bias=-1.0), qm.scores(T, qn, range(2, Q.n), bias=-1.0))


@pytest.mark.parametrize("kt", [0, 1, 2])
def test_every_lmer_scores_its_own_table_entry(kt):
    """L = 6: the 4 096 L-mers as sequences, in lexicographic order; for unit weights the score of u is T_lex[u] / |u| + bias
    exactly.  This pins the export order."""
    L, k, d = 6, 4, 2
    with capi.Problem(kernel_type=kt, L=L, k=k, d=d) as P, capi.Problem(kernel_type=kt, L=L, k=k, d=d) as Q:
        P.add_many(sv_seqs(L, 30, seed=60 + kt))
        alpha = alphas(P.n, 5)
        lex = np.arange(4 ** L)
        letters = np.array([[b"ACGT"[(x >> (2 * (L - 1 - t))) & 3] for t in range(L)] for x in lex], np.uint8)
        Q.add_block(letters)
        with P.lmer_table(0, P.n, alpha) as t:
            Tl = t.weights()
            got = t.scores(Q, 0, Q.n, bias=0.5)
        assert np.array_equal(got, Tl / Q.sqnorm() + 0.5)


def scale_problem(params, nsv, nrows, length, seed):
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    P = capi.Problem(**params)
    P.add_block(acgt[rng.integers(0, 4, (nsv + nrows, length))])
    return P


@pytest.mark.parametrize("params,length", [(dict(kernel_type=2, L=11, k=7, d=3), 300),
                                           (dict(kernel_type=4, L=10, k=6, d=3, M=50, H=50.0), 600)])
def test_scale(params, length):
    """2 000 SVs (the columns [0, 2 000)) and 20 000 further rows: the bound on every row, numpy bit for bit on a sample"""
    nsv, nrows = 2000, 20000
    with scale_problem(params, nsv, nrows, length, seed=length) as P:
        norm = P.sqnorm()
        kt, L, d = params["kernel_type"], params["L"], params["d"]
        model = ltm.Model(P, kt, L, d, params.get("M", 50), params.get("H", 50.0))
        alpha = alphas(nsv, 3)
        with P.lmer_table(0, nsv, alpha) as t:
            got = t.scores(P, 0, nsv + nrows, bias=0.3)
        dv = P.decision_values(0, nsv + nrows, 0, nsv, alpha, 0.3)
        eps = bound(P, model, 0, nsv + nrows, 0, alpha, model.w, norm, chunk=4000)
        assert np.all(np.abs(got - dv) <= eps), float(np.max(np.abs(got - dv) / eps))
        T = model.table(0, alpha, norm)
        sample = np.random.default_rng(1).choice(nsv + nrows, 200, replace=False)
        assert np.array_equal(got[sample], model.scores(T, norm, sample, bias=0.3))


def test_refusals():
    lib = capi.load()
    for kt in (3, 5):
        with capi.Problem(kernel_type=kt, L=6, k=3, d=2) as P:
            P.add_many(sv_seqs(6, 5, 1))
            with pytest.raises(capi.GkmError, match="RBF"):
                P.lmer_table(0, P.n, np.ones(P.n))
    with max_L16():
        for L, d in ((16, 0), (16, 3), (15, 1)):
            with capi.Problem(kernel_type=0, L=L, k=L - d, d=d) as P:
                P.add("ACGT" * 8)
                with pytest.raises(capi.GkmError, match="more than 17179869184"):
                    P.lmer_table(0, 1, [1.0])
    with capi.Problem(kernel_type=2, L=6, k=3, d=2) as P:
        P.add_many(sv_seqs(6, 5, 2))
        for col0, ncols in ((-1, 2), (0, P.n + 1), (P.n, 1), (0, 0)):
            with pytest.raises(capi.GkmError, match="outside the problem"):
                P.lmer_table(col0, ncols, np.ones(ncols))
        assert not lib.gkmb200_lmer_table_new(P.h, 0, 1, None)
        assert "null" in capi.last_error()
        with P.lmer_table(0, P.n, np.ones(P.n)) as t:
            for row0, nrows in ((-1, 1), (0, P.n + 1), (P.n, 1)):
                with pytest.raises(capi.GkmError, match="outside the problem"):
                    t.scores(P, row0, nrows)
            assert lib.gkmb200_lmer_table_scores(t.h, None, 0, 1, 0.0, None) == 1
            assert "null" in capi.last_error()
            for other in (dict(kernel_type=1, L=6, k=3, d=2), dict(kernel_type=2, L=6, k=4, d=2), dict(kernel_type=2, L=7, k=3, d=2),
                          dict(kernel_type=2, L=6, k=3, d=1), dict(kernel_type=2, L=6, k=3, d=2, M=40),
                          dict(kernel_type=2, L=6, k=3, d=2, H=20.0)):
                with capi.Problem(**other) as Q:
                    Q.add_many(sv_seqs(7, 3, 3))
                    with pytest.raises(capi.GkmError, match="does not match the L-mer table"):
                        t.scores(Q, 0, 1)
    # more columns than the keys' 24-bit column field: refused before anything is uploaded
    with capi.Problem(kernel_type=2, L=3, k=2, d=1) as P:
        n = (1 << 24) + 1
        P.add_block(np.full((n, 3), ord("A"), np.uint8))
        with pytest.raises(capi.GkmError, match="at most 16777216"):
            P.lmer_table(0, n, np.zeros(n))


def test_multi_gpu_if_available():
    """rows sliced over two GPUs score what one GPU scores, bit for bit; a problem on other GPUs is refused"""
    lib = capi.load()
    if capi.device_count() < 2:
        pytest.skip("needs two GPUs")
    params = dict(kernel_type=4, L=10, k=6, d=3, M=50, H=50.0)
    seqs = sv_seqs(10, 300, seed=42, length=300)
    alpha = alphas(len(seqs), 9)
    try:
        res = {}
        for ids in ((0,), (0, 1)):
            arr = (ctypes.c_int * len(ids))(*ids)
            assert lib.gkmb200_set_devices(arr, len(ids)) == 0
            with capi.Problem(**params) as P:
                P.add_many(seqs)
                with P.lmer_table(0, P.n, alpha) as t:
                    res[ids] = (t.weights(), t.scores(P, 0, P.n, bias=0.1))
                    if len(ids) == 2:
                        one = (ctypes.c_int * 1)(0)
                        assert lib.gkmb200_set_devices(one, 1) == 0
                        with capi.Problem(**params) as Q:
                            Q.add_many(seqs[:4])
                            with pytest.raises(capi.GkmError, match="other GPUs"):
                                t.scores(Q, 0, 1)
        assert np.array_equal(res[(0,)][0], res[(0, 1)][0])
        assert np.array_equal(res[(0,)][1], res[(0, 1)][1])
    finally:
        one = (ctypes.c_int * 1)(0)
        lib.gkmb200_set_devices(one, 1)
