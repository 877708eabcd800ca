"""CPU tier of the index row kernel's launch space (tests/index_grid.py): the grid's restatement of the host rules equals the
library's own functions, the grid covers exactly the reachable gkm_index_rows_kernel instances, and every case reaches the
instance it is built for by the library's rules.  The GPU tier (test_gpu_index_space.py) runs the same cases and reads
back, through gkmb200_problem_index_blocks, what actually ran."""
import ctypes
import itertools

import numpy as np
import pytest

import index_grid as ig


@pytest.fixture(scope="module")
def lib(product_lib):
    L = product_lib
    L.gkm_idx_row_smem.restype = ctypes.c_uint
    L.gkm_idx_row_smem.argtypes = [ctypes.c_int] * 5
    L.gkm_idx_max_cols.argtypes = [ctypes.c_int] * 3
    L.gkm_idx_two_cta.argtypes = [ctypes.c_int] * 6 + [ctypes.c_double]
    L.gkm_idx_block_fmt.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_size_t, ctypes.c_int]
    L.gkm_plan_index_blocks.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
    return L


MAXQS = (32, 64, 96, 320, 640, 1024, 2048)


def test_row_smem_and_max_cols_match_the_library(lib):
    for nbins, maxq, w, c16 in itertools.product(range(1, 17), MAXQS, (0, 1), (0, 1)):
        assert lib.gkm_idx_max_cols(nbins, maxq, w) == ig.max_cols(nbins, maxq, w), (nbins, maxq, w)
        for ldh in (32, 64, 4096, 10784, 10816, 12768, 12800, 24800, 32736):
            assert lib.gkm_idx_row_smem(nbins, ldh, maxq, w, c16) == ig.row_smem(nbins, ldh, maxq, w, c16), (nbins, ldh, maxq, w, c16)


def test_two_cta_rule_matches_the_library(lib):
    """every format, one block and several, skew on both sides of 10, block widths across both shared-memory limits"""
    for nbins, maxq, fmt, nblk, skew in itertools.product((1, 2, 3, 9), MAXQS, (ig.P32, ig.C16, ig.W20), (1, 2, 5),
                                                          (1.0, 10.0, 10.000001, 500.0)):
        for w in ((0,) if fmt == ig.C16 else (1,) if fmt == ig.W20 else (0, 1)):
            for cols in range(32, 26000, 352):
                for c in (cols, cols + 1, cols + 31):
                    assert lib.gkm_idx_two_cta(nbins, c, maxq, w, fmt, nblk, skew) == ig.two_cta(nbins, c, maxq, w, fmt, nblk, skew), \
                        (nbins, c, maxq, w, fmt, nblk, skew)


def test_block_plan_and_format_match_the_library(lib):
    cols = ctypes.c_int()
    for span, cap, greedy in itertools.product((1, 31, 32, 150, 10784, 10912, 20000, 32736, 50000), (0, 32, 128, 10784, 16352, 22528, 32736),
                                               (0, 1)):
        nblk = lib.gkm_plan_index_blocks(span, cap, greedy, ctypes.byref(cols))
        assert (nblk, cols.value) == ig.plan_index_blocks(span, cap, greedy), (span, cap, greedy)
    for w, M, ncols, P, wide in itertools.product((0, 1), (50, 63, 64, 255), (100, 16352, 16353, 0x7FFF, 0x8000),
                                                  (1000, 3 * (4 << 22) // 4 - 48, 3 * (4 << 22) // 4), (0, 1)):
        assert lib.gkm_idx_block_fmt(w, M, ncols, P, wide) == ig.block_fmt(w, M, ncols, P, wide), (w, M, ncols, P, wide)


def test_limits_the_limit_and_boundary_cases_stand_on():
    """the numbers the limit and boundary cases stand on: two-CTA limits at 40-bp rows, the widest block at a 2 047-bp row
    and the shared memory of its launch in each format (out of 232 448 bytes, 256 of them taken by the static `red`)"""
    assert ig.last_two_cta_cols(2, 64, False, ig.C16, False) == 12768
    assert ig.last_two_cta_cols(2, 64, False, ig.C16, True) == 10784
    assert ig.max_cols(2, 2048, False) == 24800
    assert ig.row_smem(2, 24800, 2048, False, False) == 231296 and 231296 + 256 <= ig.SMEM_LIMIT
    assert ig.row_smem(2, 24800, 2048, False, True) == 219008
    assert ig.index_block_cap(1, 64, False, 32736) == 32736 == (ig.C16_MAX_COLS & ~31)


def test_grid_covers_exactly_the_reachable_instances():
    """12 reachable instances, each with and without cold bins; the 4 left out are P32 at two CTAs per SM"""
    compiled, reach = ig.compiled_instances(), ig.reachable_instances()
    assert len(compiled) == 16 and len(reach) == 12
    assert compiled - reach == {(ig.P32, w, r, 2) for w in (False, True) for r in (0, 1)}
    got = [(c.target, c.cold) for c in ig.INSTANCE_CASES]
    assert len(got) == len(set(got)) == 24
    assert set(got) == {(i, cold) for i in reach for cold in (False, True)}
    assert all(c.target in reach for c in ig.CASES)


def test_decision_values_span_three_launches_per_format():
    """for every slot format a case with cold bins whose decision values take >= 3 launches (both streams' cold scratch)"""
    fmts = {c.target[0] for c in ig.CASES if c.cold and c.decision_rows > 2 * ig.DECISION_ROWS}
    assert fmts == {ig.P32, ig.C16, ig.W20}


def test_boundary_cases_straddle_the_two_cta_limit():
    """each boundary pair: the last column count that runs two CTAs per SM, and one warp more that runs one"""
    by = {}
    for c in ig.BOUNDARY_CASES:
        cb, ce = c.blocks()[0]
        by.setdefault((c.target[0], len(c.blocks()) > 1), []).append((ce - cb, c.stats()[0][4]))
    assert len(by) == 4
    for (fmt, several), pair in by.items():
        (c0, m0), (c1, m1) = sorted(pair)
        assert c1 == c0 + 32 and (m0, m1) == (2, 1), (fmt, several, pair)


@pytest.mark.parametrize("case", ig.CASES, ids=repr)
def test_case_reaches_its_instance_by_the_library_rule(case, lib):
    """the block plan, the slot format and the CTAs per SM of the case's target block, from the library's own functions on
    the case's sequences (skew from numpy), and a call of the case that asks for RANGE as the target says"""
    seqs = case.seqs()
    maxlen = max(map(len, seqs))
    assert case.maxq == 32 * ((maxlen + 31) // 32)
    cols = ctypes.c_int()
    nblk = lib.gkm_plan_index_blocks(case.n, case.cap, 1, ctypes.byref(cols))
    bl = case.blocks()
    assert nblk == len(bl) and all(cb == k * cols.value for k, (cb, _) in enumerate(bl))
    cb, ce = bl[case.block]
    P, sumsq = ig.block_stats(seqs, case.L, cb, ce)
    assert P == sum(2 * (len(s) - case.L + 1) for s in seqs[cb:ce])
    fmt = lib.gkm_idx_block_fmt(int(case.weighted), case.M, ce - cb, P, case.wide)
    two = lib.gkm_idx_two_cta(case.nbins, ce - cb, case.maxq, int(case.weighted), fmt, nblk, sumsq / P)
    f, w, r, m = case.target
    assert (fmt, 2 if two else 1) == (f, m)
    want = ig.inst_bit(r, m)
    assert any(case.predict(c).get(case.block, (0, 0))[0] == want for c in case.calls()), "no call runs the target instance"
    # every shared-memory request of the case fits the opt-in limit
    assert max(s for c in case.calls() for _, s in case.predict(c).values()) + 256 <= ig.SMEM_LIMIT


def test_numpy_run_lengths_count_both_strands():
    """block_stats on a hand-checked block: AAAA (L = 2) has AA x3 forward and TT x3 reverse; ACGT is its own reverse complement"""
    assert ig.block_stats(["AAAA"], 2, 0, 1) == (6, 18)
    P, sq = ig.block_stats(["ACGT"], 2, 0, 1)
    assert (P, sq) == (6, 12)  # AC, CG, GT twice each


def test_emulator_build_refuses_the_index_record():
    import __graft_entry__ as ge
    from gkmqc_b200 import capi
    lib = ctypes.CDLL(ge.build_abi_emulator())
    capi._declare(lib)
    with capi.Problem(lib=lib) as P:
        P.add("ACGT" * 10)
        with pytest.raises(capi.GkmError, match="needs the device"):
            P.index_blocks()
