"""GPU tier (-m gpu): the launch space of the all-pairs kernels against the oracle.

tests/launch_grid.py names the cases: one per bit-sliced kernel instance a caller can reach, and one per tile-shape class
of the bit-sliced, lmer and tcgen05 (mma) kernels.  Every case is compared with the oracle in each launch mode the library
has (the sqnorm diagonal, the lower triangle, a rectangle across the diagonal, a lower block off the origin, fused
decision values), and
gkmb200_problem_launch_shape confirms that the case ran the instance and the tile shape it was built for.  Each test
records the shape it saw as the junit property "launch_shape" ((variant, TA, TB, shared bytes); mma: TA = queries per CTA).

Bars: integer histograms and non-RBF kernel values bit-exact; RBF kernel values within 1e-9 relative (device exp());
decision values within the rounding bound of a sum of the same products in any order (oracle/pysvm.exact_scores)."""
import contextlib

import numpy as np
import pytest

import launch_grid
import pyoracle
import pysvm
from conftest import write_fasta
from gkmqc_b200 import capi

pytestmark = pytest.mark.gpu

RTOL_RBF = 1e-9
CODE = launch_grid.VARIANT_CODE


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    capi.load()
    if capi.device_count() < 1:
        pytest.fail("no B200 visible; the product has no CPU fallback")


@contextlib.contextmanager
def forced(variant):
    capi.set_option("kernel", variant)
    try:
        yield
    finally:
        capi.set_option("kernel", "auto")


def check_kmat(K, Kref, kernel_type, what=""):
    if kernel_type in launch_grid.RBF_TYPES:
        np.testing.assert_allclose(K, Kref, rtol=RTOL_RBF, atol=0, err_msg=what)
    else:
        assert np.array_equal(K, Kref), "%s: max abs diff %g" % (what, np.max(np.abs(K - Kref)))


def oracle_full(params, seqs):
    """(sqnorm, K, H) of every ordered pair, from the oracle"""
    o = pyoracle.Oracle(**params)
    for s in seqs:
        o.add(s)
    n = len(seqs)
    K, H = o.rect(np.arange(n), n)
    return o.sqnorm(), K, H


def run_against_oracle(params, seqs, variant, ran, shape=None, diag_shape=None, record=None):
    """every launch mode of the forced variant against the oracle.  ran: the kernel_variant code that must have run;
    shape / diag_shape: the launch_shape() the all-pairs calls / the sqnorm diagonal must report (mma: no byte count)"""
    n, kt = len(seqs), params["kernel_type"]
    sq, K, H = oracle_full(params, seqs)
    low = np.tril(np.ones((n, n), bool), -1)
    r0, c0, c1 = 5, 3, n - 4                                    # off-tile start, crosses the diagonal
    alpha = np.random.default_rng(n).standard_normal(c1 - c0)
    seen = []

    def expect(want, what):
        got = P.launch_shape()
        seen.append(got)
        if want is not None:
            assert got[:3] == tuple(want[:3]) and want[3] in (None, got[3]), (what, got, want)

    with forced(variant), capi.Problem(**params) as P:
        P.add_many(seqs)
        assert np.array_equal(P.sqnorm(), sq), "sqnorm"
        expect(diag_shape, "sqnorm")
        assert np.array_equal(P.hist_block(0, n, 0, n, lower=True), np.where(low[..., None], H, 0)), "lower histograms"
        assert P.stats()["kernel_variant"] == ran
        expect(shape, "hist_block lower")
        check_kmat(P.kernel_lower(), np.where(low, K, 0.0) + np.eye(n), kt, "kernel_lower")
        assert P.stats()["kernel_variant"] == ran
        expect(shape, "kernel_lower")
        assert np.array_equal(P.hist_block(r0, n - r0, c0, c1 - c0), H[r0:, c0:c1]), "rectangle histograms"
        expect(shape, "hist_block rectangle")
        Kb = P.kernel_block(r0, n - r0, c0, c1 - c0)
        check_kmat(Kb, K[r0:, c0:c1], kt, "kernel_block")
        assert P.stats()["kernel_variant"] == ran
        # a lower block off the origin (row0 > col0 > 0) through the raw ABI, into a NaN-filled buffer with ld > ncols: the
        # entries below the diagonal and the unit diagonal are written, the cells above it and the padding stay NaN
        lr0, lc0, lnc, ld = r0 + 4, c0 + 2, c1 - c0 - 2, c1 - c0 + 3
        buf = np.full((n - lr0, ld), np.nan)
        capi._check(P.lib.gkmb200_kernel_block(P.h, lr0, n - lr0, lc0, lnc, 1, buf.ctypes.data_as(capi.c_dbl_p), ld), P.lib)
        rr, cc = np.arange(lr0, n)[:, None], np.arange(lc0, lc0 + lnc)[None, :]
        want = np.full_like(buf, np.nan)
        want[:, :lnc] = np.where(cc < rr, K[lr0:, lc0:lc0 + lnc], np.where(cc == rr, 1.0, np.nan))
        if kt in launch_grid.RBF_TYPES:
            np.testing.assert_allclose(buf, want, rtol=RTOL_RBF, atol=0, equal_nan=True, err_msg="lower block off the origin")
        else:
            assert np.array_equal(buf, want, equal_nan=True), "lower block off the origin"
        assert P.stats()["kernel_variant"] == ran
        expect(shape, "kernel_block lower off the origin")
        dv = P.decision_values(r0, n - r0, c0, c1 - c0, alpha, bias=0.25)
        # the device's own kernel values (RBF: within 1e-9 of the oracle's, checked above), summed exactly
        want, bound = pysvm.exact_scores(Kb, np.arange(n - r0), np.arange(c1 - c0), alpha, -0.25)
        err = np.abs(dv + want)
        assert np.all(err <= bound), "decision values: worst excess %g" % np.max(err - bound)
    if record is not None:
        record("launch_shape", sorted(set(seen)))
    return seen


@pytest.mark.parametrize("case", launch_grid.INSTANCE_CASES, ids=repr)
def test_every_bitsliced_instance(case, record_property):
    """each reachable gkm_diag_kernel<L, NB, WEIGHTED, D4>, forced, on the grid's edge-case sequences"""
    seqs = case.seqs()
    shape = launch_grid.expected_shape("diag", max(map(len, seqs)), case.L, case.d, case.weighted)
    run_against_oracle(case.params, seqs, "diag", CODE["diag"], shape=shape, diag_shape=shape, record=record_property)


@pytest.mark.parametrize("case", launch_grid.SHAPE_CASES, ids=repr)
def test_every_tile_shape(case, record_property):
    """each tile-shape class of the bit-sliced, lmer and mma kernels, its longest sequence at the largest length of the
    class; the sqnorm diagonal runs the bit-sliced kernel under mma and the lmer kernel under lmer"""
    seqs = case.seqs()
    assert max(map(len, seqs)) == case.maxlen
    diag_variant = "lmer" if case.variant == "lmer" else "diag"
    diag_shape = launch_grid.expected_shape(diag_variant, case.maxlen, case.L, case.d, case.weighted)
    run_against_oracle(case.params, seqs, case.variant, CODE[case.variant], shape=case.shape, diag_shape=diag_shape,
                       record=record_property)


@pytest.mark.parametrize("variant", ["lmer", "mma"])
@pytest.mark.parametrize("weighted", [False, True], ids=["u", "w"])
@pytest.mark.parametrize("L", range(2, 17))
def test_lmer_and_mma_across_L(L, weighted, variant, record_property):
    """d = L - 1: one matching base per hit, the smallest threshold the mma kernel takes; L = 16 leaves its L-mer word no
    spare byte"""
    params = dict(kernel_type=4 if weighted else 2, L=L, k=1, d=L - 1, M=50, H=50.0, gamma=0.7)
    seqs = launch_grid.case_seqs(L, 45, 130, seed=1000 + 2 * L + weighted)
    maxlen = max(map(len, seqs))
    shape = launch_grid.expected_shape(variant, maxlen, L, L - 1, weighted)
    diag_shape = launch_grid.expected_shape("lmer" if variant == "lmer" else "diag", maxlen, L, L - 1, weighted)
    run_against_oracle(params, seqs, variant, CODE[variant], shape=shape, diag_shape=diag_shape, record=record_property)


@pytest.mark.parametrize("variant", ["diag", "lmer", "mma", "index"])
@pytest.mark.parametrize("L,kernel_type", [(2, 0), (5, 4), (8, 3)])
def test_every_lmer_pair_is_a_hit(L, kernel_type, variant, record_property):
    """k = 0, d = L: the gate admits it and every L-mer pair counts.  The mma kernel needs a matching base per hit, so
    the bit-sliced kernel runs instead"""
    params = dict(kernel_type=kernel_type, L=L, k=0, d=L, M=50, H=50.0, gamma=0.7)
    seqs = launch_grid.case_seqs(L, 45, 130, seed=2000 + L)
    ran = {"diag": "diag", "lmer": "lmer", "mma": "diag", "index": "index"}[variant]
    maxlen, w = max(map(len, seqs)), kernel_type in launch_grid.WEIGHTED_TYPES
    shape = None if ran == "index" else launch_grid.expected_shape(ran, maxlen, L, L, w)
    diag_shape = launch_grid.expected_shape("lmer" if ran == "lmer" else "diag", maxlen, L, L, w)
    run_against_oracle(params, seqs, variant, CODE[ran], shape=shape, diag_shape=diag_shape, record=record_property)


def test_gkmqc_default_bin(tmp_path, record_property):
    """gkmQC's default bin: wgkm (type 4, M = 50, H = 50), L = 10, k = 6, d = 3, 1 200 windows of 590 .. 600 bp.  Its
    sqnorm runs the weighted bit-sliced kernel on the (4, 16) tile.  kernel = auto, index and diag: every sqnorm and 48
    rows against the oracle, the whole lower triangle of index against diag, and the same problem through computeGkmKernel"""
    import bench
    from gkmqc_b200 import driver
    n, L, k, d = 1200, 10, 6, 3
    params = dict(kernel_type=4, L=L, k=k, d=d, M=50, H=50.0, gamma=1.0)
    rng = np.random.default_rng(600)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    lens = rng.integers(590, 601, n)
    lens[::7] = 600
    seqs = [acgt[rng.integers(0, 4, int(ln))].tobytes().decode() for ln in lens]
    o = pyoracle.Oracle(**params)
    for s in seqs:
        o.add(s)
    sq = o.sqnorm()
    got, ran, rows = {}, {}, None
    for v in ("index", "diag", "auto"):
        with forced(v), capi.Problem(**params) as P:
            P.add_many(seqs)
            assert np.array_equal(P.sqnorm(), sq), "sqnorm (%s)" % v
            assert P.launch_shape() == launch_grid.expected_shape("diag", 600, L, d, True)
            assert P.launch_shape()[1:3] == (4, 16)
            got[v] = P.kernel_lower()
            ran[v] = P.stats()["kernel_variant"]
            if v == "index":
                nblk, cols, _ = P.index_layout()
                rows = bench.parity_rows(n, cols or n, nblk, want=48)[:48]
                hist = P.hist_block(0, n, 0, n, lower=True)[rows]
    record_property("kernel_variant", ran)
    assert ran["index"] == 4 and ran["diag"] == 2
    assert np.array_equal(got["index"], got["diag"]), "index and bit-sliced kernels differ in the lower triangle"
    assert np.array_equal(got["auto"], got["diag"])
    Ko, Ho = o.rect(rows, int(rows.max()))
    for i, r in enumerate(rows):
        assert np.array_equal(got["index"][r, :r], Ko[i, :r]), "row %d" % r
        assert np.array_equal(hist[i, :r], Ho[i, :r]), "histograms of row %d" % r
    pos, neg = str(tmp_path / "pos.fa"), str(tmp_path / "neg.fa")
    write_fasta(pos, seqs[: n // 2], "p")
    write_fasta(neg, seqs[n // 2:], "n")
    kmat, npos, nneg = driver.computeGkmKernel([4, L, k, d, 50, 50.0, 1.0, pos, neg, 4, 0], max_seqs=n)
    assert (npos, nneg) == (n // 2, n - n // 2)
    assert np.array_equal(kmat, np.maximum(got["diag"], got["diag"].T))
