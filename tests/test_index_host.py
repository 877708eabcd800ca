"""CPU tier for the "index" kernel variant (gkmqc_b200/csrc/gkm_index.h): the list of XOR masks a query
L-mer is probed with, the table address of an L-mer, the cost model behind kernel = auto, and -- through
tests/emu/index_emu.cc -- the slot encoding and walk rules against the reference's histograms."""
import ctypes
from math import comb

import numpy as np
import pytest

import pyoracle
from conftest import golden_names, load_golden, random_seqs
from gkmqc_b200 import capi


@pytest.fixture(scope="module")
def lib(product_lib):
    product_lib.gkm_idx_delta_count.restype = ctypes.c_longlong
    product_lib.gkm_idx_delta_count.argtypes = [ctypes.c_int, ctypes.c_int]
    product_lib.gkm_idx_deltas.restype = ctypes.c_longlong
    product_lib.gkm_idx_deltas.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_longlong]
    product_lib.gkm_idx_supported.argtypes = [ctypes.c_int] * 3
    product_lib.gkm_idx_cold_count.restype = ctypes.c_longlong
    product_lib.gkm_idx_cold_count.argtypes = [ctypes.c_int, ctypes.c_int]
    product_lib.gkm_idx_cost_ms.restype = ctypes.c_double
    product_lib.gkm_idx_cost_ms.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_longlong, ctypes.c_double, ctypes.c_double,
                                            ctypes.c_longlong, ctypes.c_double]
    product_lib.gkm_diag_cost_ms.restype = ctypes.c_double
    product_lib.gkm_diag_cost_ms.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_longlong, ctypes.c_double]
    return product_lib


def code_of(bases, L):
    """gkm_idx_code restated: the first two bases interleaved in the low four bits, the rest planar"""
    lb = min(2, L)
    c = 0
    for t, b in enumerate(bases):
        if t < lb:
            c |= b << (2 * t)
        else:
            c |= (b & 1) << (lb + t)
            c |= (b >> 1) << (L + t)
    return c


@pytest.mark.parametrize("L,d", [(11, 3), (10, 2), (12, 4), (14, 4), (2, 1), (2, 2), (3, 3), (5, 0), (6, 6), (13, 1)])
def test_mask_list_is_the_hamming_ball(L, d, lib):
    n = lib.gkm_idx_delta_count(L, d)
    assert n == sum(comb(L, m) * 3 ** m for m in range(min(d, L) + 1))
    a = np.zeros(n, dtype=np.uint32)
    assert lib.gkm_idx_deltas(L, d, a.ctypes.data, n) == n
    masks, ms = a & 0x0FFFFFFF, a >> 28
    assert len(np.unique(masks)) == n, "every mask once"
    assert np.array_equal(np.bincount(ms, minlength=d + 1)[: min(d, L) + 1],
                          [comb(L, m) * 3 ** m for m in range(min(d, L) + 1)])
    # a mask is the XOR of the codes of two L-mers; its label is their Hamming distance
    rng = np.random.default_rng(L * 31 + d)
    x = rng.integers(0, 4, L)
    seen = set()
    for mk, m in zip(masks.tolist()[:: max(1, n // 3000)], ms.tolist()[:: max(1, n // 3000)]):
        y_code = code_of(x, L) ^ mk
        # decode y and count the substituted bases
        lb = min(2, L)
        y = [((y_code >> (2 * t)) & 3) if t < lb else (((y_code >> (lb + t)) & 1) | (((y_code >> (L + t)) & 1) << 1)) for t in range(L)]
        assert sum(int(u != v) for u, v in zip(x, y)) == m
        assert code_of(y, L) == y_code
        seen.add(y_code)
    # the masks of the cold bins (m <= d - 2) come first; inside each part masks that differ only in the low
    # bases are adjacent: at most one group per upper mask
    ncold = lib.gkm_idx_cold_count(L, d)
    assert ncold == sum(comb(L, m) * 3 ** m for m in range(min(d, L) - 1))
    assert np.all(ms[:ncold] <= d - 2) and np.all(ms[ncold:] >= max(0, min(d, L) - 1))
    for part in (masks[:ncold], masks[ncold:]):
        if len(part) == 0:
            continue
        upper = part >> 4
        changes = int(np.count_nonzero(np.diff(upper.astype(np.int64)))) + 1
        assert changes == len(np.unique(upper))


def test_supported_and_cost_model(lib):
    assert lib.gkm_idx_supported(11, 3, 4) == 1
    assert lib.gkm_idx_supported(14, 4, 5) == 1
    assert lib.gkm_idx_supported(15, 3, 4) == 0 and lib.gkm_idx_supported(16, 4, 5) == 0
    assert lib.gkm_idx_supported(11, 3, 5) == 0
    assert lib.gkm_idx_supported(14, 12, 13) == 0, "mask list beyond 64 Mi entries"
    nq, pairs = 290.0, 2.0 * 290 * 290
    # BASELINE configs[1]: the index wins by a wide margin; configs[0] (1 000 sequences): the bit-sliced kernel does
    big = 10000 * 9999 // 2
    assert lib.gkm_idx_cost_ms(11, 3, 0, 10000, nq, 1, big, pairs) < 0.25 * lib.gkm_diag_cost_ms(3, 0, big, pairs)
    assert 35 < lib.gkm_idx_cost_ms(11, 3, 0, 10000, nq, 1, big, pairs) < 50, "calibrated on the 41 ms of configs[1]"
    small = 1000 * 999 // 2
    assert lib.gkm_idx_cost_ms(11, 3, 0, 1000, nq, 1, small, pairs) > lib.gkm_diag_cost_ms(3, 0, small, pairs)
    # L = 14, d = 4 on 20 000 sequences (the top of configs[2]): 91 771 masks per L-mer, the table leaves L2
    n20 = 20000 * 19999 // 2
    assert lib.gkm_idx_cost_ms(14, 4, 0, 20000, 287.0, 2, n20, 2.0 * 287 * 287) > lib.gkm_diag_cost_ms(4, 0, n20, 2.0 * 287 * 287)


def test_block_format_choice(lib):
    P32, C16, W20 = 0, 1, 2
    lib.gkm_idx_block_fmt.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_size_t, ctypes.c_int]
    fmt = lib.gkm_idx_block_fmt
    # unit weights: 16-bit columns below 0x8000
    assert fmt(0, 50, 0x7FFF, 10 ** 6, 0) == C16 and fmt(0, 50, 0x8000, 10 ** 6, 0) == P32
    # weights: <= 63, <= 16 352 columns, overflow offsets below 2^22 units (worst case 4/3 entries per posting + 64)
    assert fmt(1, 63, 16352, 10 ** 6, 0) == W20
    assert fmt(1, 64, 16352, 10 ** 6, 0) == P32
    assert fmt(1, 50, 16353, 10 ** 6, 0) == P32
    p_max = (3 * (4 << 22) - 3 * 64 - 1) // 4  # the most postings with (4 P) / 3 + 64 < 4 * 2^22
    assert (4 * p_max) // 3 + 64 < 4 << 22 <= (4 * (p_max + 1)) // 3 + 64
    assert fmt(1, 50, 16352, p_max, 0) == W20 and fmt(1, 50, 16352, p_max + 1, 0) == P32
    # index_wide: the 16-byte slots whatever fits
    assert fmt(0, 50, 100, 1000, 1) == P32 and fmt(1, 50, 100, 1000, 1) == P32


@pytest.fixture(scope="module")
def emu(emu_lib):
    emu_lib.gkm_emu_index_cost.restype = ctypes.c_longlong
    emu_lib.gkm_emu_index_cost.argtypes = [ctypes.c_void_p]
    emu_lib.gkm_emu_index_hist_lower.argtypes = [ctypes.c_void_p, ctypes.c_int, capi.c_i32_p]
    emu_lib.gkm_emu_index_hist_rect.argtypes = [ctypes.c_void_p] + [ctypes.c_int] * 4 + [capi.c_i32_p]
    return emu_lib


@pytest.mark.parametrize("name", golden_names())
def test_emulated_index_matches_reference_histograms(name, emu):
    g, cfg, pos, neg = load_golden(name)
    P = capi.Problem(lib=emu, **cfg)
    assert P.read(pos, neg) == int(g["npos"])
    if cfg["L"] > 14:
        pytest.skip("the index variant stops at L = 14")
    if emu.gkm_emu_index_cost(P.h) > 3e8:
        pytest.skip("too many probes for a CPU emulation (%d)" % emu.gkm_emu_index_cost(P.h))
    n = P.n
    cheap = emu.gkm_emu_index_cost(P.h) < 5e7
    for block_cols in ((0, 7) if cheap else (7,)):  # one column block, and several (a row that does not fit shared memory)
        H = np.zeros((n, n, cfg["d"] + 1), np.int32)
        assert emu.gkm_emu_index_hist_lower(P.h, block_cols, H.ctypes.data_as(capi.c_i32_p)) == 0
        w = P.weights()
        sq = np.array([np.sqrt(sum(w[m] * H[a, a, m] for m in range(len(w)))) for a in range(n)])
        assert np.array_equal(sq, g["sqnorm"]), "diagonal histograms (sqnorm)"
        for a in range(n):
            H[a, a:, :] = 0
        assert np.array_equal(H, g["hist"])
    P.close()


@pytest.fixture
def wide(request, emu):
    """the emulator library's own index_wide option: 16-byte slots (1) instead of the compact ones (C16 / W20)"""
    assert emu.gkmb200_set_option(b"index_wide", b"1" if request.param else b"0") == 0
    yield request.param
    emu.gkmb200_set_option(b"index_wide", b"0")


@pytest.mark.parametrize("wide", [False, True], indirect=True)
@pytest.mark.parametrize("kernel_type,L,d", [(2, 8, 2), (4, 9, 3), (2, 6, 4), (4, 5, 1)])
def test_emulated_index_long_lists_and_ranges(kernel_type, L, d, wide, emu):
    """few distinct L-mers (short L, repeats): posting lists far beyond the four inline slots, so the overflow
    walk, its end markers and the column-range cut are exercised; plus a rectangular block with col0 > 0"""
    seqs = random_seqs(40, 90, seed=17 * L + d, ragged=True)
    seqs = [s if len(s) >= L else s + "ACGT" * 4 for s in seqs]
    seqs[7] = seqs[6]
    seqs[9] = "A" * 60
    seqs[11] = "ACAC" * 20
    k = L - d
    o = pyoracle.Oracle(kernel_type, L, k, d)
    P = capi.Problem(kernel_type, L, k, d, lib=emu)
    for s in seqs:
        o.add(s)
        P.add(s)
    n = len(seqs)
    _, Ho = o.matrix_lower()
    for block_cols in (0, 16):
        H = np.zeros((n, n, d + 1), np.int32)
        assert emu.gkm_emu_index_hist_lower(P.h, block_cols, H.ctypes.data_as(capi.c_i32_p)) == 0
        for a in range(n):
            H[a, a:, :] = 0
        assert np.array_equal(H, Ho)
    rows = np.arange(20, 40)
    _, Hr = o.rect(rows, 20)
    Hq = np.zeros((len(rows), 15, d + 1), np.int32)
    assert emu.gkm_emu_index_hist_rect(P.h, 20, len(rows), 5, 15, Hq.ctypes.data_as(capi.c_i32_p)) == 0
    assert np.array_equal(Hq, Hr[:, 5:20])
    P.close()
