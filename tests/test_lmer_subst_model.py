"""CPU tier of the single-base substitutions (gkm_lmer_subst.h, DESIGN.md 4.6): the emulator, which runs the header with
one lane, against the materialised mutants.

- H' of every mutant equals the oracle's self histogram of that mutant, exactly as integers.
- Every substitution score equals, bit for bit, the emulated table score (gkm_emu_lmer_scores) of a problem that holds the
  mutant, with the mutant's norm sqrt(sum_m w[m] H'_m) taken in gkm_kraw's order from the oracle's histogram.

T is any table: random doubles exercise the numerator as well as a trained model would.
"""
import ctypes
import math
import os
import sys

import numpy as np
import pytest

from gkmqc_b200 import capi

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import pyoracle  # noqa: E402

c_i32_p = ctypes.POINTER(ctypes.c_int32)
c_int_p = ctypes.POINTER(ctypes.c_int)


@pytest.fixture(scope="module")
def emu(emu_lib):
    emu_lib.gkm_emu_lmer_scores.argtypes = [ctypes.c_void_p, capi.c_dbl_p, capi.c_dbl_p, ctypes.c_int, ctypes.c_int, ctypes.c_double, capi.c_dbl_p]
    emu_lib.gkm_emu_lmer_subst.argtypes = [ctypes.c_void_p, capi.c_dbl_p, c_i32_p, ctypes.c_longlong, c_int_p, c_int_p, ctypes.c_double,
                                           capi.c_dbl_p, c_i32_p]
    return emu_lib


def random_seq(rng, n, alphabet="ACGT"):
    return "".join(rng.choice(list(alphabet), n))


def kraw_norm(w, h):
    """gkm_kraw + __dsqrt_rn: ascending m from 0.0, one rounding per operation"""
    s = 0.0
    for m in range(len(h)):
        s = s + float(w[m]) * float(int(h[m]))
    return math.sqrt(s)


def mutate(seq, p, v):
    return seq[:p] + "ACGT"[v] + seq[p + 1:]


def check(emu, cfg, seqs, sites, seed=0, bias=0.125):
    """sites: (row, pos) pairs; every check of the module on one set of sequences"""
    kt, L, k, d, M = cfg
    rng = np.random.default_rng(seed)
    T = rng.standard_normal(4 ** L)
    rows = np.array([s[0] for s in sites], np.int32)
    pos = np.array([s[1] for s in sites], np.int32)
    o = pyoracle.Oracle(kt, L, k, d, M=M)
    for s in seqs:
        o.add(s)
    H = np.ascontiguousarray([o.hist(i, i) for i in range(len(seqs))], np.int32)
    mutants = [mutate(seqs[r], p, v) for r, p in zip(rows, pos) for v in range(4)]
    for s in mutants:
        o.add(s)
    Hm = np.array([o.hist(len(seqs) + j, len(seqs) + j) for j in range(len(mutants))], np.int32)
    with capi.Problem(kt, L, k, d, M=M, lib=emu) as P:
        P.add_many(seqs)
        w = P.weights()
        out = np.zeros(4 * len(sites))
        Hout = np.zeros((len(sites), 4, d + 1), np.int32)
        assert emu.gkm_emu_lmer_subst(P.h, T.ctypes.data_as(capi.c_dbl_p), H.ctypes.data_as(c_i32_p), len(sites),
                                      rows.ctypes.data_as(c_int_p), pos.ctypes.data_as(c_int_p), bias,
                                      out.ctypes.data_as(capi.c_dbl_p), Hout.ctypes.data_as(c_i32_p)) == 0
    assert np.array_equal(Hout.reshape(-1, d + 1), Hm), (cfg, "H' differs from the oracle's histogram of the mutant")
    norm = np.array([kraw_norm(w, h) for h in Hm])
    want = np.zeros(len(mutants))
    with capi.Problem(kt, L, k, d, M=M, lib=emu) as Q:
        Q.add_many(mutants)
        assert emu.gkm_emu_lmer_scores(Q.h, T.ctypes.data_as(capi.c_dbl_p), norm.ctypes.data_as(capi.c_dbl_p), 0, len(mutants), bias,
                                       want.ctypes.data_as(capi.c_dbl_p)) == 0
    assert np.array_equal(out.view(np.uint64), want.view(np.uint64)), (cfg, "scores differ from the materialised mutants")
    return out.reshape(-1, 4)


def all_sites(seqs):
    return [(r, p) for r, s in enumerate(seqs) for p in range(len(s))]


GRID = [(kt, L, L - d, d) for L in range(2, 9) for d in range(L + 1) for kt in (2, 4)]


@pytest.mark.parametrize("kt,L,k,d", GRID)
def test_every_site_of_short_rows(emu, kt, L, k, d):
    """lengths L, L + 1, 2 L + 3 and 3 L, every position and base; a palindrome, a homopolymer, a tandem repeat, N and
    lower case among them"""
    rng = np.random.default_rng(100 * L + 10 * d + kt)
    half = random_seq(rng, L)
    pal = half + half[::-1].translate(str.maketrans("ACGT", "TGCA"))     # its own reverse complement
    seqs = [random_seq(rng, L), random_seq(rng, L + 1), random_seq(rng, 2 * L + 3), pal, "A" * (2 * L + 1),
            ("ACG" * L)[:3 * L], random_seq(rng, 2 * L, "ACGTNacgt")]
    check(emu, (kt, L, k, d, 50), seqs, all_sites(seqs), seed=L * 31 + d)


@pytest.mark.parametrize("L,d", [(2, 1), (5, 2), (8, 3), (8, 8)])
def test_long_rows_sampled_sites(emu, L, d):
    """rows up to 300 bp, positions 0, L - 2, len - 1 and random ones, both weighted and unit weights"""
    rng = np.random.default_rng(L + d)
    seqs = [random_seq(rng, n) for n in (300, 151, 64, 33)] + [random_seq(rng, 120, "ACGTNacgtn")]
    sites = []
    for r, s in enumerate(seqs):
        sites += [(r, 0), (r, max(L - 2, 0)), (r, len(s) - 1)] + [(r, int(p)) for p in rng.integers(0, len(s), 6)]
    for kt in (2, 4):
        check(emu, (kt, L, L - d, d, 50), seqs, sites, seed=d)


@pytest.mark.parametrize("L,d", [(3, 1), (6, 2), (8, 4)])
def test_m255_and_zero_norms(emu, L, d):
    """M = 255 gives the centre window weight 0: a row of length L has norm 0 and its scores are the same inf / NaN"""
    rng = np.random.default_rng(L)
    seqs = [random_seq(rng, L), random_seq(rng, L + 2), random_seq(rng, 40), "C" * 30]
    out = check(emu, (4, L, L - d, d, 255), seqs, all_sites(seqs), seed=L)
    assert np.all(np.isnan(out[:L]))


def test_sites_in_any_order(emu):
    """shuffled sites with repeats give the sorted run's results, row for row"""
    rng = np.random.default_rng(5)
    seqs = [random_seq(rng, n) for n in (40, 23, 57)]
    sites = all_sites(seqs)
    ref = check(emu, (4, 6, 3, 3, 50), seqs, sites)
    order = np.concatenate([rng.permutation(len(sites)), rng.integers(0, len(sites), 50)])
    got = check(emu, (4, 6, 3, 3, 50), seqs, [sites[i] for i in order])
    assert np.array_equal(got.view(np.uint64), ref[order].view(np.uint64))


def test_own_base_is_the_unmutated_score(emu):
    """the entry of the row's own base (N counts as A) equals the row's table score"""
    rng = np.random.default_rng(9)
    seqs = [random_seq(rng, 50, "ACGTNacgt") for _ in range(4)]
    cfg = (2, 7, 4, 3, 50)
    out = check(emu, cfg, seqs, all_sites(seqs))
    o = pyoracle.Oracle(2, 7, 4, 3)
    for s in seqs:
        o.add(s)
    T = np.random.default_rng(0).standard_normal(4 ** 7)
    with capi.Problem(2, 7, 4, 3, lib=emu) as P:
        P.add_many(seqs)
        w = P.weights()
        norm = np.array([kraw_norm(w, o.hist(i, i)) for i in range(len(seqs))])
        sc = np.zeros(len(seqs))
        assert emu.gkm_emu_lmer_scores(P.h, T.ctypes.data_as(capi.c_dbl_p), norm.ctypes.data_as(capi.c_dbl_p), 0, len(seqs), 0.125,
                                       sc.ctypes.data_as(capi.c_dbl_p)) == 0
        at = 0
        for r, s in enumerate(seqs):
            own = P.codes(r)[0].astype(int) - 1
            for p in range(len(s)):
                assert out[at + p, own[p]] == sc[r]
            at += len(s)
