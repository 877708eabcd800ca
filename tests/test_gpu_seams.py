"""GPU tier (-m gpu): every cut the device layer makes in a call, one step past it, against the oracle.

tests/seam_grid.py names the cases and predicts each call's pieces, the rows or sites on both sides of every cut and the
kernel launches.  For every case:

* the rows (or sites) on both sides of each cut, the first, the last, any 2 047-bp row and a seeded sample are checked
  against the oracle (integer histograms and non-RBF kernel values bit for bit, RBF within 1e-9 relative), decision values
  within oracle/pysvm.exact_scores' bound, substitutions bit for bit against table scores of the materialised mutants;
* the whole result equals, bit for bit (decision values: within the bound), the same work done in calls below the cut;
* gkmb200_stats.launches equals the prediction on both sides, so a case that stops crossing its cut fails.

Each case records its pieces and launches as the junit property "seam".  The GPU-share case needs two or more GPUs; the
buffers that grow between calls (band, staging, cold-bin scratch, the mma image) are run small -> large -> small."""
import contextlib
import ctypes

import numpy as np
import pytest

import pyoracle
import pysvm
import seam_grid as sg
from conftest import write_fasta
from gkmqc_b200 import capi

pytestmark = pytest.mark.gpu

RTOL_RBF = 1e-9
RBF_TYPES = (3, 5)
DEFAULTS = dict(kernel="auto", chunk_mb=sg.CHUNK_MB_DEFAULT)


@pytest.fixture(scope="module", autouse=True)
def _one_gpu():
    capi.load()
    if capi.device_count() < 1:
        pytest.fail("no B200 visible; the product has no CPU fallback")
    ids = (ctypes.c_int * 1)(0)
    assert capi.load().gkmb200_set_devices(ids, 1) == 0


@contextlib.contextmanager
def options(**kw):
    try:
        for k, v in kw.items():
            capi.set_option(k, v)
        yield
    finally:
        for k, v in DEFAULTS.items():
            capi.set_option(k, v)


def load(P, seqs):
    if len({len(s) for s in seqs}) == 1:
        P.add_block(np.frombuffer("".join(seqs).encode(), np.uint8).reshape(len(seqs), -1))
    else:
        P.add_many(seqs)


def oracle_at(params, seqs, rows, cols):
    """(K, H) of rows x cols from an oracle over those sequences only: an entry depends on its two sequences alone"""
    o = pyoracle.Oracle(**params)
    for c in cols:
        o.add(seqs[c])
    for r in rows:
        o.add(seqs[r])
    return o.rect(np.arange(len(cols), len(cols) + len(rows)), len(cols))


def check_vals(got, want, kt, what):
    if kt in RBF_TYPES:
        np.testing.assert_allclose(got, want, rtol=RTOL_RBF, atol=0, err_msg=what)
    else:
        assert np.array_equal(got, want), "%s: max abs diff %g" % (what, np.max(np.abs(got - want)))


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint64), np.ascontiguousarray(b).view(np.uint64))


def sample(case, call, pred, seqs, k=5):
    """rows of a call to hold against the oracle: both sides of each cut, first, last, 2 047-bp rows, k seeded ones"""
    lo, hi = call.row0, call.row0 + call.nrows
    rng = np.random.default_rng(sg.launch_grid._seed(case.name))
    rows = {lo, hi - 1} | {r for s in pred["seams"] for r in s} | set(rng.integers(lo, hi, k).tolist())
    rows |= {r for r in range(lo, hi) if len(seqs[r]) == sg.launch_grid.MAX_LEN}
    return sorted(r for r in rows if lo <= r < hi)


def launches_of(P, case, call, what):
    pred = sg.predict(case, call, lib=P.lib)
    got = P.stats()["launches"]
    assert got == pred["launches"], (what, call, got, pred["launches"])
    return pred


def scores_in_bound(dv, Kb, alpha, bias, what):
    want, bound = pysvm.exact_scores(Kb, np.arange(Kb.shape[0]), np.arange(Kb.shape[1]), alpha, -bias)
    err = np.abs(dv + want)
    assert np.all(err <= bound), "%s: worst excess %g" % (what, np.max(err - bound))


UPLOAD = [c for c in sg.CASES if c.call.kind == "upload"]
COMPUTE = [c for c in sg.CASES if c.call.kind in ("block", "lower", "decision")]
SUBST = [c for c in sg.CASES if c.call.kind == "subst"]


@pytest.mark.parametrize("case", UPLOAD, ids=repr)
def test_sqnorm_across_the_diagonal_step(case, record_property):
    """copies of 45 rows on both sides of both 1 024-row cuts; every copy's norm is the oracle's norm of its original"""
    seqs = case.seqs()
    o = pyoracle.Oracle(**case.params)
    for s in seqs[:45]:
        o.add(s)
    base = o.sqnorm()
    seen = []
    for call in [case.call] + case.below:
        with options(kernel=case.variant), capi.Problem(**case.params) as P:
            load(P, seqs[:call.nrows])
            sq = P.sqnorm()
            pred = launches_of(P, case, call, "sqnorm")
            seen.append((len(pred["pieces"]), pred["launches"]))
            want = base[np.arange(call.nrows) % 45]
            assert np.array_equal(sq, want), "%s: %d norms differ" % (call, int(np.sum(sq != want)))
    record_property("seam", seen)


@pytest.mark.parametrize("case", COMPUTE, ids=repr)
def test_compute_call_across_its_cut(case, record_property, tmp_path):
    seqs, kt, call = case.seqs(), case.kernel_type, case.call
    rng = np.random.default_rng(3)
    alpha = rng.standard_normal(call.ncols)
    seen = []
    with options(kernel=case.variant), capi.Problem(**case.params) as P:
        load(P, seqs)
        P.sqnorm()

        def run(c, what):
            with options(kernel=case.variant, **c.options):
                if c.kind == "decision":
                    if case.variant == "index":     # build the column blocks first: the count below is of the call alone
                        P.decision_values(c.row0, 1, c.col0, c.ncols, alpha)
                    out = P.decision_values(c.row0, c.nrows, c.col0, c.ncols, alpha, bias=0.25)
                elif c.kind == "lower" and c.row0 == 0 and c.nrows == P.n:
                    out = P.kernel_lower()
                else:
                    out = P.kernel_block(c.row0, c.nrows, c.col0, c.ncols, lower=c.kind == "lower")
                pred = launches_of(P, case, c, what)
                seen.append((what, len(pred["pieces"]), pred["launches"]))
                hist = P.hist_block(c.row0, c.nrows, c.col0, c.ncols) if c.kind == "block" else None
                if hist is not None:            # the histogram path: one chunk at a time, the same cuts
                    assert P.stats()["launches"] == pred["launches"], (what, "hist_block")
            return out, hist, pred

        out, hist, pred = run(call, "across")
        below = [run(c, "below %d" % i) for i, c in enumerate(case.below)]
        rows = sample(case, call, pred, seqs)
        cols = list(range(call.col0, call.col0 + call.ncols))
        Ko, Ho = oracle_at(case.params, seqs, rows, cols)
        if call.kind == "decision":
            Kb = P.kernel_block(call.row0, call.nrows, call.col0, call.ncols)
            for i, r in enumerate(rows):
                check_vals(Kb[r - call.row0], Ko[i], kt, "row %d" % r)
            scores_in_bound(out, Kb, alpha, 0.25, "across")
            scores_in_bound(np.concatenate([b[0] for b in below]), Kb, alpha, 0.25, "below")
        elif call.kind == "block":
            for i, r in enumerate(rows):
                check_vals(out[r - call.row0], Ko[i], kt, "row %d" % r)
                assert np.array_equal(hist[r - call.row0], Ho[i]), "histograms of row %d" % r
            assert same_bits(out, np.concatenate([b[0] for b in below])), "kernel values differ from the calls below the cut"
            assert np.array_equal(hist, np.concatenate([b[1] for b in below])), "histograms differ from the calls below the cut"
        else:
            n = P.n
            for i, r in enumerate(rows):
                check_vals(out[r, :r], Ko[i, :r], kt, "row %d" % r)
            parts = np.zeros((n, n))
            for c, (b, _, _) in zip(case.below, below):
                parts[c.row0:c.row0 + c.nrows, c.col0:c.col0 + c.ncols] = b
            assert same_bits(out, parts), "the triangle differs from the calls below the cut"
            with options(kernel="diag"):
                assert same_bits(out, P.kernel_lower()), "the triangle differs from the bit-sliced kernel's"
            if case.variant == "lmer":          # gkm_main_pywrapper's row-pointer scatter, chunk by chunk
                pos, neg = str(tmp_path / "pos.fa"), str(tmp_path / "neg.fa")
                write_fasta(pos, seqs[:n // 2], "p")
                write_fasta(neg, seqs[n // 2:], "n")
                p = case.params
                with options(kernel="lmer", **call.options):
                    ret, kmat, npos, nneg = capi.main_pywrapper(pos, neg, p["kernel_type"], p["L"], p["k"], p["d"], p["M"],
                                                                p["H"], p["gamma"], nmax=n)
                assert ret == 0 and (npos, nneg) == (n // 2, n - n // 2)
                assert same_bits(kmat, out), "gkm_main_pywrapper differs from kernel_lower"
    record_property("seam", seen)


def materialised(t, params, seqs, rows, pos, bias):
    """LmerTable.scores of a problem that holds the mutants, as (nsites, 4)"""
    m = []
    for r, p in zip(rows, pos):
        s = seqs[r]
        m += [s[:p] + c + s[p + 1:] for c in "ACGT"]
    with capi.Problem(**params) as Q:
        load(Q, m)
        return t.scores(Q, 0, Q.n, bias=bias).reshape(-1, 4)


@pytest.mark.parametrize("case", SUBST, ids=repr)
def test_substitutions_across_their_cuts(case, record_property):
    seqs = case.seqs()
    lens = [len(s) for s in seqs]
    rows, pos = case.sites(lens)
    ns = len(rows)
    alpha = np.random.default_rng(9).standard_normal(case.table_cols)
    seen = []
    with options(kernel=case.variant), capi.Problem(**case.params) as P:
        load(P, seqs)
        P.sqnorm()
        with P.lmer_table(0, case.table_cols, alpha) as t:
            def run(c, what):
                a, b = c.sites
                out = t.substitutions(P, rows[a:b], pos[a:b], bias=-0.5)
                pred = sg.predict(case, c, lens=lens)
                got = P.stats()["launches"]
                assert got == pred["launches"], (what, c, got, pred["launches"])
                seen.append((what, len(pred["pieces"]), pred["launches"]))
                return out, pred

            got, pred = run(case.call, "across")
            below = [run(c, "below %d" % i)[0] for i, c in enumerate(case.below)]
            assert same_bits(got, np.concatenate(below)), "substitutions differ from the calls below the cut"
            rng = np.random.default_rng(sg.launch_grid._seed(case.name))
            pick = {0, ns - 1} | set(range(max(0, sg.SUBST_BATCH - 2), min(ns, sg.SUBST_BATCH + 3)))
            pick |= set(rng.integers(0, ns, 20).tolist())
            for before, after in sg.diag_seams(case, lens):  # a site on each row next to a diagonal step
                for r in (before, after):
                    hit = np.flatnonzero(rows == r)
                    if len(hit):
                        pick.add(int(hit[0]))
            pick = np.array(sorted(pick))
            want = materialised(t, case.params, seqs, rows[pick], pos[pick], bias=-0.5)
            assert same_bits(got[pick], want), "sites %s" % pick[np.any(got[pick].view(np.uint64) != want.view(np.uint64), 1)]
    record_property("seam", seen)


def test_gpu_shares(record_property):
    """decision values and table scores at nrows 1, 7, 8 ndev - 1, 8 ndev + 1, and substitutions whose GPU shares each cross
    2^21 sites, on every GPU against one"""
    lib = capi.load()
    ndev = capi.device_count()
    if ndev < 2:
        pytest.skip("GPU shares need two or more GPUs; %d visible" % ndev)
    case = sg.Case("shares", None, sg.DEFAULT, "auto", ("ism", 3500), None, [], sites=sg._ism(3500), table_cols=60)
    seqs = case.seqs()
    rows, pos = case.sites([600] * 3500)
    rows, pos = np.resize(rows, ndev * sg.SUBST_BATCH + 2 * ndev), np.resize(pos, ndev * sg.SUBST_BATCH + 2 * ndev)
    alpha = np.random.default_rng(4).standard_normal(60)
    counts = (1, 7, 8 * ndev - 1, 8 * ndev + 1)
    res, seen = {}, []
    try:
        capi.set_option("kernel", "diag")     # decision values: 8 192 rows per launch, no index build in the count
        for ids in (tuple(range(ndev)), (0,)):
            arr = (ctypes.c_int * len(ids))(*ids)
            assert lib.gkmb200_set_devices(arr, len(ids)) == 0
            with capi.Problem(**sg.DEFAULT) as P:
                load(P, seqs)
                P.sqnorm()
                with P.lmer_table(0, 60, alpha) as t:
                    for nr in counts:
                        r0 = 100
                        dv = P.decision_values(r0, nr, 0, 60, alpha, bias=0.5)
                        want = sg.predict(case, sg.Call("decision", r0, nr, 0, 60, options=dict(kernel="diag")), ndev=len(ids))
                        assert P.stats()["launches"] == want["launches"], ("decision", ids, nr)
                        sc = t.scores(P, r0, nr, bias=0.5)
                        assert P.stats()["launches"] == sg.predict(case, sg.Call("scores", r0, nr), ndev=len(ids))["launches"]
                        Kb = P.kernel_block(r0, nr, 0, 60)
                        scores_in_bound(dv, Kb, alpha, 0.5, "decision values on %d GPUs, %d rows" % (len(ids), nr))
                        res[ids, nr] = sc
                        seen.append((len(ids), nr, len(want["pieces"])))
                    res[ids, "subst"] = t.substitutions(P, rows, pos, bias=0.5)
        for nr in counts:
            assert same_bits(res[tuple(range(ndev)), nr], res[(0,), nr]), "table scores of %d rows" % nr
        assert same_bits(res[tuple(range(ndev)), "subst"], res[(0,), "subst"]), "substitutions"
    finally:
        capi.set_option("kernel", "auto")
        one = (ctypes.c_int * 1)(0)
        lib.gkmb200_set_devices(one, 1)
    record_property("seam", seen)


@pytest.mark.parametrize("variant", ["diag", "lmer", "mma", "index"])
def test_buffers_grow_between_calls(variant):
    """small -> large -> small kernel blocks and decision values on one problem: the band and staging buffers, the mma
    image (made by the first mma launch) and, for the index with d = 3, the cold-bin scratch of both streams grow between
    calls; every call holds against the oracle"""
    params = sg._p(2)
    rng = np.random.default_rng(17)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    seqs = [acgt[rng.integers(0, 4, int(ln))].tobytes().decode() for ln in rng.integers(10, 120, 6000)]
    calls = [(0, 40, 0, 30), (0, 6000, 0, 1200), (5, 40, 3, 30)]
    with options(kernel=variant), capi.Problem(**params) as P:
        load(P, seqs)
        for r0, nr, c0, nc in calls:
            alpha = rng.standard_normal(nc)
            Kb = P.kernel_block(r0, nr, c0, nc)
            dv = P.decision_values(r0, nr, c0, nc, alpha, bias=0.1)
            rows = sorted({r0, r0 + nr - 1, r0 + nr // 2} | set(rng.integers(r0, r0 + nr, 3).tolist()))
            Ko, _ = oracle_at(params, seqs, rows, list(range(c0, c0 + nc)))
            for i, r in enumerate(rows):
                assert np.array_equal(Kb[r - r0], Ko[i]), (variant, (r0, nr, c0, nc), r)
            scores_in_bound(dv, Kb, alpha, 0.1, "%s %s" % (variant, (r0, nr, c0, nc)))
