"""GPU tier of the single-base substitutions (gkmb200_lmer_table_substitutions, DESIGN.md 4.6): every entry equals, bit for
bit, LmerTable.scores of a second problem that holds the materialised mutants (its norms computed by its own upload), and
the site list, the split over GPUs and every refusal behave as documented."""
import contextlib
import ctypes

import numpy as np
import pytest

from gkmqc_b200 import capi

pytestmark = pytest.mark.gpu

ACGT = np.frombuffer(b"ACGT", np.uint8)


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


def ragged(L, n, seed, length=120):
    """ragged random rows plus the awkward ones: exactly L bases, N and lower case, a palindrome, a homopolymer, a tandem
    repeat"""
    rng = np.random.default_rng(seed)
    seqs = ["".join(rng.choice(list("ACGT"), int(rng.integers(L, length + 1)))) for _ in range(n)]
    half = seqs[0][:max(L // 2 + 1, 3)]
    seqs += [seqs[1][:L], seqs[2][:5].lower() + "N" + seqs[2][6:-4] + "nN" + seqs[2][-2:],
             half + half[::-1].translate(str.maketrans("ACGT", "TGCA")), "A" * (L + 30), ("ACG" * 40)[:L + 40]]
    return [s for s in seqs if len(s) >= L]


def mutants(seqs, rows, pos):
    out = []
    for r, p in zip(rows, pos):
        s = seqs[r]
        out += [s[:p] + c + s[p + 1:] for c in "ACGT"]
    return out


def materialised(t, params, seqs, rows, pos, bias):
    """LmerTable.scores of a problem that holds the mutants, as (nsites, 4)"""
    with capi.Problem(**params) as Q:
        m = mutants(seqs, rows, pos)
        if len({len(s) for s in m}) == 1:
            Q.add_block(np.frombuffer("".join(m).encode(), np.uint8).reshape(len(m), -1))
        else:
            Q.add_many(m)
        return t.scores(Q, 0, Q.n, bias=bias).reshape(-1, 4)


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint64), np.ascontiguousarray(b).view(np.uint64))


def alphas(n, seed):
    rng = np.random.default_rng(seed)
    a = rng.standard_normal(n)
    a[rng.random(n) < 0.2] = 0.0
    return a


CASES = [  # (type, L, k, d, M, H)
    (0, 2, 1, 1, 50, 50.0), (1, 6, 3, 3, 50, 50.0), (2, 6, 3, 3, 50, 50.0), (4, 10, 6, 3, 50, 50.0),
    (2, 11, 7, 3, 50, 50.0), (4, 11, 7, 3, 50, 50.0), (0, 12, 8, 4, 50, 50.0), (2, 13, 12, 1, 50, 50.0),
    (0, 5, 0, 5, 50, 50.0), (4, 5, 0, 5, 50, 50.0), (4, 6, 3, 3, 255, 50.0),
]


@pytest.mark.parametrize("kt,L,k,d,M,H", CASES)
def test_every_site_equals_the_materialised_mutant(kt, L, k, d, M, H):
    params = dict(kernel_type=kt, L=L, k=k, d=d, M=M, H=H)
    rng = np.random.default_rng(L * 7 + kt)
    seqs = ragged(L, 12, seed=L * 10 + kt)
    long_row = L in (10, 11)
    if long_row:
        seqs.append("".join(rng.choice(list("ACGT"), 2047)))
    with (max_L16() if L > 12 else contextlib.nullcontext()), capi.Problem(**params) as P:
        P.add_many(seqs)
        with P.lmer_table(0, P.n, alphas(P.n, L)) as t:
            rows = np.concatenate([np.full(len(s), r) for r, s in enumerate(seqs[:len(seqs) - long_row])]).astype(np.int32)
            pos = np.concatenate([np.arange(len(s)) for s in seqs[:len(seqs) - long_row]]).astype(np.int32)
            if long_row:
                lp = np.concatenate([[0, L - 2, 2046], rng.integers(0, 2047, 300)]).astype(np.int32)
                rows = np.concatenate([rows, np.full(len(lp), len(seqs) - 1, np.int32)])
                pos = np.concatenate([pos, lp])
            got = t.substitutions(P, rows, pos, bias=-0.25)
            want = materialised(t, params, seqs, rows, pos, bias=-0.25)
            assert same_bits(got, want), (params, int(np.sum(got.view(np.uint64) != want.view(np.uint64))))
            own = np.array([P.codes(r)[0][p] - 1 for r, p in zip(rows, pos)])
            sc = t.scores(P, 0, P.n, bias=-0.25)
            assert same_bits(got[np.arange(len(rows)), own], sc[rows])
            if M == 255:
                assert np.isnan(got[rows == seqs.index(seqs[1][:L])]).all()  # a row of L bases: centre weight 0, norm 0


def test_site_list_handling():
    params = dict(kernel_type=4, L=8, k=5, d=3)
    seqs = ragged(8, 20, seed=3, length=90)
    rng = np.random.default_rng(4)
    with capi.Problem(**params) as P, capi.Problem(**params) as R:
        P.add_many(seqs)
        R.add_many(seqs[5:])  # a problem other than the table's
        with P.lmer_table(0, 10, alphas(10, 2)) as t:
            rows = np.concatenate([np.full(len(s), r) for r, s in enumerate(seqs)]).astype(np.int32)
            pos = np.concatenate([np.arange(len(s)) for s in seqs]).astype(np.int32)
            ref = t.substitutions(P, rows, pos, bias=0.5)
            order = np.concatenate([rng.permutation(len(rows)), rng.integers(0, len(rows), 500)])
            assert same_bits(t.substitutions(P, rows[order], pos[order], bias=0.5), ref[order])
            # ism: row0 > 0, one (len, 4) array per row, through the other problem
            ism = t.ism(R, 2, 6, bias=0.5)
            assert [a.shape for a in ism] == [(len(seqs[5 + r]), 4) for r in range(2, 8)]
            at = np.searchsorted(rows, 7)
            for r in range(2, 8):
                n = len(seqs[5 + r])
                assert same_bits(ism[r - 2], ref[at:at + n])
                at += n
            assert t.substitutions(P, [], [], bias=0.5).shape == (0, 4)
            assert t.ism(P, 3, 0) == []
            lib = P.lib
            out = np.zeros(4)
            one = (ctypes.c_int * 1)(0)
            for r, p, msg in ((-1, 0, "outside the problem"), (P.n, 0, "outside the problem"), (0, -1, "outside row"),
                              (0, len(seqs[0]), "outside row")):
                with pytest.raises(capi.GkmError, match=msg):
                    t.substitutions(P, [r], [p])
            with pytest.raises(capi.GkmError, match="sites"):
                capi._check(lib.gkmb200_lmer_table_substitutions(t.h, P.h, -1, one, one, 0.0, out.ctypes.data_as(capi.c_dbl_p)), lib)
            for args in ((None, P.h), (t.h, None)):
                with pytest.raises(capi.GkmError, match="null"):
                    capi._check(lib.gkmb200_lmer_table_substitutions(*args, 1, one, one, 0.0, out.ctypes.data_as(capi.c_dbl_p)), lib)
            for a, b, c in ((None, one, out.ctypes.data_as(capi.c_dbl_p)), (one, None, out.ctypes.data_as(capi.c_dbl_p)), (one, one, None)):
                with pytest.raises(capi.GkmError, match="null"):
                    capi._check(lib.gkmb200_lmer_table_substitutions(t.h, P.h, 1, a, b, 0.0, c), lib)
            assert lib.gkmb200_lmer_table_substitutions(t.h, P.h, 0, None, None, 0.0, None) == 0
            with capi.Problem(kernel_type=4, L=8, k=5, d=2) as X:
                X.add_many(seqs[:3])
                with pytest.raises(capi.GkmError, match="does not match"):
                    t.substitutions(X, [0], [0])


DEFAULT = dict(kernel_type=4, L=10, k=6, d=3, M=50, H=50.0)  # gkmQC's default model


def block(rng, n, length):
    return ACGT[rng.integers(0, 4, (n, length))]


def test_full_ism_at_scale():
    """2 000 x 600-bp rows: 20 rows materialised, every own-base entry against scores"""
    rng = np.random.default_rng(11)
    B = block(rng, 2000, 600)
    seqs = [bytes(r).decode() for r in B]
    with capi.Problem(**DEFAULT) as P:
        P.add_block(B)
        with P.lmer_table(0, 500, alphas(500, 12)) as t:
            ism = np.stack(t.ism(P, 0, 2000, bias=0.1))  # (2000, 600, 4)
            sc = t.scores(P, 0, 2000, bias=0.1)
            own = (np.searchsorted(ACGT, B)).astype(np.int64)
            assert same_bits(np.take_along_axis(ism, own[:, :, None], 2)[:, :, 0], np.repeat(sc[:, None], 600, 1))
            pick = rng.choice(2000, 20, replace=False)
            rows = np.repeat(pick, 600).astype(np.int32)
            pos = np.tile(np.arange(600), 20).astype(np.int32)
            assert same_bits(ism[pick].reshape(-1, 4), materialised(t, DEFAULT, seqs, rows, pos, bias=0.1))


def test_variant_effect_shape_at_scale():
    """100 000 one-site 600-bp rows (one window per SNP); 300 sampled rows materialised"""
    rng = np.random.default_rng(13)
    B = block(rng, 100000, 600)
    with capi.Problem(**DEFAULT) as P:
        P.add_block(B)
        pos = rng.integers(0, 600, 100000).astype(np.int32)
        with P.lmer_table(0, 1000, alphas(1000, 14)) as t:
            got = t.substitutions(P, np.arange(100000, dtype=np.int32), pos, bias=-1.0)
            pick = np.sort(rng.choice(100000, 300, replace=False))
            seqs = {int(r): bytes(B[r]).decode() for r in pick}
            want = materialised(t, DEFAULT, seqs, pick, pos[pick], bias=-1.0)
            assert same_bits(got[pick], want)
            own = np.searchsorted(ACGT, B[np.arange(100000), pos])
            assert same_bits(got[np.arange(100000), own], t.scores(P, 0, 100000, bias=-1.0))


def test_two_gpus_equal_one():
    lib = capi.load()
    if capi.device_count() < 2:
        pytest.skip("needs two GPUs")
    rng = np.random.default_rng(21)
    B = block(rng, 300, 300)
    rows = np.concatenate([np.repeat(np.arange(300), 50), rng.integers(0, 300, 777)]).astype(np.int32)
    pos = rng.integers(0, 300, len(rows)).astype(np.int32)
    try:
        res = {}
        for ids in ((0,), (0, 1)):
            arr = (ctypes.c_int * len(ids))(*ids)
            assert lib.gkmb200_set_devices(arr, len(ids)) == 0
            with capi.Problem(**DEFAULT) as P:
                P.add_block(B)
                with P.lmer_table(0, 100, alphas(100, 3)) as t:
                    res[ids] = t.substitutions(P, rows, pos, bias=0.2)
                    if len(ids) == 2:
                        one = (ctypes.c_int * 1)(0)
                        assert lib.gkmb200_set_devices(one, 1) == 0
                        with capi.Problem(**DEFAULT) as Q:
                            Q.add_block(B[:4])
                            with pytest.raises(capi.GkmError, match="other GPUs"):
                                t.substitutions(Q, [0], [0])
        assert same_bits(res[(0,)], res[(0, 1)])
    finally:
        one = (ctypes.c_int * 1)(0)
        lib.gkmb200_set_devices(one, 1)
