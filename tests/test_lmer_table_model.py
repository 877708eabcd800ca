"""CPU tier of the L-mer table (gkm_lmer_table.h, DESIGN.md 4.5): the numpy restatement (tests/lmer_table_model.py) against
brute force and against the reference's kernel values, and the CPU emulator, which runs the header itself, against the
restatement bit for bit.

The rounding bound.  Every score is a sum of signed terms alpha_c wt_c(y) w[m] wt_r(x) / (|r| |c|), one per L-mer pair
(x, y) within d mismatches; B(r) is the sum of their magnitudes:
    B(r) = sum_c |alpha_c| sum_m |w[m]| H_m(r, c) / (|r| |c|).
Each partial sum on the way, in either evaluation, is at most B(r) in magnitude, and each rounding of fp64 errs by at most
2^-53 of its result.  The table's path to one score chains: one division (beta_c), one product (beta_c wt), the additions
of S (at most the longest run of one code), 3 additions per base of the transform for each level of m (at most 4 L in all
along one path, counting the level above), d + 1 products and additions of the combine, one product and one addition per
window of r, one division.  The sum over the columns (Sigma_c alpha_c K(r, c)) takes at most ncols additions after one
product per term, and each K(r, c) carries a few roundings of its own.  So both results lie within
    eps(r) = (ncols + longest run of S + 4 L + windows of r + 16) 2^-52 B(r)
of the exact value, and within eps(r) of each other.  A misplaced L-mer pair (wrong strand, weight or mask) moves a
score by about B(r) / (pairs within d), near 1e-6 B(r), far above eps(r) ~ 1e-13 B(r).
"""
import ctypes

import numpy as np
import pytest

from conftest import golden_names, load_golden
from gkmqc_b200 import capi
import lmer_table_model as ltm

LINEAR = [n for n in golden_names() if int(n.split("_t")[1][0]) in (0, 1, 2, 4) and int(n.split("_L")[1].split("k")[0]) <= 12]


def alphas(n, seed):
    """mixed signs, with zeros"""
    rng = np.random.default_rng(seed)
    a = rng.standard_normal(n)
    a[rng.random(n) < 0.2] = 0.0
    return a


def eps_bound(model, alpha, col0, B, rows):
    ncols = len(alpha)
    run = model.longest_run(col0, ncols)
    win = np.array([len(model.fwd[r]) - model.L + 1 for r in rows])
    return (ncols + run + 4 * model.L + win + 16) * 2.0 ** -52 * B


@pytest.mark.parametrize("L", range(1, 7))
def test_transform_equals_brute_force_neighbours(L):
    """A_m[u] = sum over the v at Hamming distance m of S[v], for every d <= L; integer S, so both sides are exact"""
    rng = np.random.default_rng(L)
    S = rng.integers(-1000, 1000, 4 ** L).astype(np.float64)
    bases = ltm.code_bases(L)
    ham = np.zeros((4 ** L, 4 ** L), np.int8)
    for t in range(L):
        ham += (bases[:, None, t] != bases[None, :, t])
    for d in range(L + 1):
        A = ltm.transform(S, L, d)
        for m in range(d + 1):
            assert np.array_equal(A[m], (ham == m).astype(np.float64) @ S), (L, d, m)


def test_code_layout_is_the_index_variants():
    """the restatement's codes are gkm_idx_code's: a substitution at base t flips exactly the bits of the index
    variant's masks (gkm_idx_deltas lists them at d = 1)"""
    lib = capi.load()
    lib.gkm_idx_deltas.restype = ctypes.c_longlong
    lib.gkm_idx_deltas.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_uint32), ctypes.c_longlong]
    for L in (1, 2, 3, 6, 11, 14):
        out = np.zeros(1 + 3 * L, np.uint32)
        assert lib.gkm_idx_deltas(L, 1, out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), len(out)) == len(out)
        masks = {int(x) & 0x0FFFFFFF for x in out if x >> 28 == 1}
        mine = {((v & 1) << ltm.base_bit(t, L, 0)) | ((v >> 1) << ltm.base_bit(t, L, 1)) for t in range(L) for v in (1, 2, 3)}
        assert masks == mine, L


@pytest.fixture(scope="module")
def golden_models():
    cache = {}

    def get(name):
        if name not in cache:
            g, cfg, pos, neg = load_golden(name)
            P = capi.Problem(**cfg)
            P.read(pos, neg)
            cache[name] = (g, cfg, P, ltm.Model(P, cfg["kernel_type"], cfg["L"], cfg["d"], cfg["M"], cfg["H"]))
        return cache[name]
    yield get
    for v in cache.values():
        v[2].close()


def full_matrices(g):
    """the golden files hold the lower triangle and a unit diagonal of K, and the strict lower triangle of H"""
    K, H = g["kmat"], g["hist"].astype(np.float64)
    K = np.tril(K, -1) + np.tril(K, -1).T + np.eye(len(K))
    H = H + H.transpose(1, 0, 2)
    return K, H


@pytest.mark.parametrize("name", LINEAR)
def test_table_scores_match_the_reference_kernel_values(golden_models, name):
    g, cfg, P, model = golden_models(name)
    n, L = P.n, cfg["L"]
    K, H = full_matrices(g)
    norm, w = g["sqnorm"], model.w
    Hd = [model.hist(r, r) for r in range(n)]  # the diagonal, which the golden files leave out
    for col0, ncols, seed in ((0, n, 1), (3, n - 5, 2)):
        alpha = alphas(ncols, seed)
        T = model.table(col0, alpha, norm)
        rows = np.arange(n)
        got = model.scores(T, norm, rows, bias=0.25)
        cols = np.arange(col0, col0 + ncols)
        want = np.array([np.float64(0.25) + np.sum(alpha * K[r, cols]) for r in rows])
        B = np.array([np.sum(np.abs(alpha) * (np.abs(w) @ H[r, cols].T) / (norm[r] * norm[cols])) +
                      (abs(alpha[r - col0]) * (np.abs(w) @ Hd[r]) / norm[r] ** 2 if col0 <= r < col0 + ncols else 0.0) for r in rows])
        eps = eps_bound(model, alpha, col0, B, rows)
        dev = np.abs(got - want)
        assert np.all(dev <= eps), (name, col0, float(np.max(dev / np.maximum(eps, 1e-300))))
        assert np.max(B) > 0


@pytest.fixture(scope="module")
def emu(emu_lib):
    emu_lib.gkm_emu_lmer_table.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, capi.c_dbl_p, capi.c_dbl_p, capi.c_dbl_p, capi.c_dbl_p]
    emu_lib.gkm_emu_lmer_scores.argtypes = [ctypes.c_void_p, capi.c_dbl_p, capi.c_dbl_p, ctypes.c_int, ctypes.c_int, ctypes.c_double, capi.c_dbl_p]
    return emu_lib


@pytest.mark.parametrize("name", LINEAR)
def test_emulator_runs_the_header_like_the_restatement(emu, golden_models, name):
    g, cfg, _, model = golden_models(name)
    L = cfg["L"]
    g, cfg, pos, neg = load_golden(name)
    with capi.Problem(lib=emu, **cfg) as P:
        P.read(pos, neg)
        n = P.n
        norm = np.ascontiguousarray(g["sqnorm"])
        col0, ncols = 2, n - 4
        alpha = alphas(ncols, 7)
        T = np.zeros(4 ** L)
        lex = np.zeros(4 ** L)
        assert emu.gkm_emu_lmer_table(P.h, col0, ncols, alpha.ctypes.data_as(capi.c_dbl_p), norm.ctypes.data_as(capi.c_dbl_p),
                                      T.ctypes.data_as(capi.c_dbl_p), lex.ctypes.data_as(capi.c_dbl_p)) == 0
        Tn = model.table(col0, alpha, norm)
        assert np.array_equal(T, Tn), name
        assert np.array_equal(lex, ltm.export(Tn, L)), name
        out = np.zeros(n - 1)
        assert emu.gkm_emu_lmer_scores(P.h, T.ctypes.data_as(capi.c_dbl_p), norm.ctypes.data_as(capi.c_dbl_p), 1, n - 1, -0.5,
                                       out.ctypes.data_as(capi.c_dbl_p)) == 0
        assert np.array_equal(out, model.scores(Tn, norm, range(1, n), bias=-0.5)), name


def test_refusals_before_any_device_work():
    """the host-side refusals of gkmb200_lmer_table_new come before the device is touched (GPU tier: all of them)"""
    with capi.Problem(kernel_type=5, L=6, k=3, d=2) as P:
        P.add("ACGTACGTAC")
        with pytest.raises(capi.GkmError, match="RBF"):
            P.lmer_table(0, 1, [1.0])
    with capi.Problem(kernel_type=2, L=6, k=3, d=2) as P:
        P.add("ACGTACGTAC")
        with pytest.raises(capi.GkmError, match="outside"):
            P.lmer_table(0, 2, [1.0, 1.0])
