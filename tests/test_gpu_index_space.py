"""GPU tier (-m gpu): the launch space of the index variant's row kernel against the oracle.

tests/index_grid.py names the cases: each reachable gkm_index_rows_kernel<WEIGHTED, RANGE, FMT, MINB> with and without
cold bins, the limits of the slot formats and of shared memory, and each two-CTA boundary.  Every case runs its calls with
kernel = index -- the lower triangle (sampled bands when n is large), rectangles across the diagonal with col0 inside a
block and at a block edge, a lower block off the origin written through the raw ABI into a NaN-filled buffer with
ld > ncols, and decision values -- and each is checked:

* against the oracle on sampled rows (integer histograms and non-RBF kernel values bit-exact, RBF within 1e-9 relative);
* against the bit-sliced kernel over the whole call (histograms and kernel values bit-exact);
* decision values within the rounding bound of oracle/pysvm.exact_scores over the call's own kernel values;
* through gkmb200_problem_index_blocks: every block ran exactly the instances and the shared memory the grid predicts, its
  slot format is the grid's, and its postings and sum of squared posting-list lengths equal numpy's.

The instance each case ran on its target block is recorded as the junit property "index_instance".  The tests at the end
carry state from call to call: reuse of a partition, a rebuild outside it, a rebuild that a named index_split forces, and
two problems with different (L, d) taking turns on one GPU's mask list."""
import contextlib
import ctypes
import math

import numpy as np
import pytest

import index_grid as ig
import pyoracle
import pysvm
from gkmqc_b200 import capi

pytestmark = pytest.mark.gpu

RTOL_RBF = 1e-9
DEFAULTS = dict(kernel="auto", index_cols=0, index_wide=0, index_split="auto")


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    capi.load()
    if capi.device_count() < 1:
        pytest.fail("no B200 visible; the product has no CPU fallback")
    ids = (ctypes.c_int * 1)(0)
    assert capi.load().gkmb200_set_devices(ids, 1) == 0  # the record covers the first GPU: give each call all of its rows


@contextlib.contextmanager
def options(**kw):
    try:
        for k, v in kw.items():
            capi.set_option(k, v)
        yield
    finally:
        for k, v in DEFAULTS.items():
            capi.set_option(k, v)


def same(got, want, kernel_type, what, exact=False):
    if kernel_type in ig.RBF_TYPES and not exact:
        np.testing.assert_allclose(got, want, rtol=RTOL_RBF, atol=0, equal_nan=True, err_msg=what)
    else:
        assert np.array_equal(got, want, equal_nan=True), "%s: %d entries differ" % (what, int(np.sum(~((got == want) | (np.isnan(got) & np.isnan(want))))))


def sample_rows(call, extra=()):
    r0, r1 = call.row0, call.row0 + call.nrows
    return sorted({r0, r1 - 1, (r0 + r1) // 2} | {r for r in extra if r0 <= r < r1})


def run_call(P, call, alpha=None):
    """the outputs of one call of the forced variant: {name: array}; the record is read after each compute call"""
    out, rec = {}, {}
    r0, nr, c0, nc = call.row0, call.nrows, call.col0, call.ncols
    if call.kind in ("lower", "rect"):
        lower = call.kind == "lower"
        out["hist"] = P.hist_block(r0, nr, c0, nc, lower=lower)
        rec["hist"] = P.index_blocks()
        out["kernel"] = P.kernel_block(r0, nr, c0, nc, lower=lower)
        rec["kernel"] = P.index_blocks()
    elif call.kind == "lower_raw":
        ld = nc + 5
        buf = np.full((nr, ld), np.nan)
        capi._check(P.lib.gkmb200_kernel_block(P.h, r0, nr, c0, nc, 1, buf.ctypes.data_as(capi.c_dbl_p), ld), P.lib)
        out["raw"] = buf
        rec["raw"] = P.index_blocks()
    else:
        out["dv"] = P.decision_values(r0, nr, c0, nc, alpha, bias=0.25)
        rec["dv"] = P.index_blocks()
        out["kernel"] = P.kernel_block(r0, nr, c0, nc)
        rec["kernel"] = P.index_blocks()
    return out, rec


def check_record(case, call, rec, what):
    """each block ran exactly the predicted instances with the predicted shared memory; returns {block: mask}"""
    pred, st, bl = case.predict(call), case.stats(), case.blocks()
    assert [(b["cb"], b["ce"]) for b in rec] == bl, (what, rec)
    seen = {}
    for k, b in enumerate(rec):
        P, sq, _, fmt, _ = st[k]
        assert (b["fmt"], b["postings"], b["sumsq"]) == (fmt, P, sq), (what, k, b, st[k])
        want, smem = pred.get(k, (0, 0))
        assert (b["inst"], b["smem"]) == (want, smem), (what, k, b, pred)
        assert (b["launches"] > 0) == (want != 0), (what, k, b)
        if what.endswith(" dv") and want:   # decision values: 16 waves of rows per launch
            assert b["launches"] == math.ceil(call.nrows / ig.DECISION_ROWS), (what, k, b)
        seen[k] = b["inst"]
    return seen


def oracle_checks(case, o, call, out, alpha):
    """sampled rows of the call against the oracle"""
    kt, r0, c0, c1 = case.kernel_type, call.row0, call.col0, call.col0 + call.ncols
    rows = sample_rows(call, extra=[i for i, s in enumerate(case.seqs()) if len(s) > 1000])
    Ko, Ho = o.rect(np.array(rows), c1)
    Ko, Ho = Ko[:, c0:], Ho[:, c0:]
    cols = np.arange(c0, c1)
    for i, r in enumerate(rows):
        below = cols < r
        if call.kind in ("rect", "decision"):
            if "hist" in out:
                assert np.array_equal(out["hist"][r - r0], Ho[i]), "%r row %d histograms" % (call, r)
            same(out["kernel"][r - r0], Ko[i], kt, "%r row %d" % (call, r))
        elif call.kind == "lower":
            assert np.array_equal(out["hist"][r - r0], np.where(below[:, None], Ho[i], 0)), "%r row %d histograms" % (call, r)
            same(out["kernel"][r - r0], np.where(below, Ko[i], np.where(cols == r, 1.0, 0.0)), kt, "%r row %d" % (call, r))
        else:
            want = np.full(call.ncols + 5, np.nan)
            want[: call.ncols] = np.where(below, Ko[i], np.where(cols == r, 1.0, np.nan))
            same(out["raw"][r - r0], want, kt, "%r row %d" % (call, r))
    if call.kind == "lower_raw":
        # cells on or above the diagonal are never written, nor is the padding behind ncols
        rr = np.arange(r0, r0 + call.nrows)[:, None]
        assert np.all(np.isnan(out["raw"][:, call.ncols:]))
        assert np.all(np.isnan(out["raw"][:, : call.ncols][cols[None, :] > rr]))
        assert np.all(out["raw"][:, : call.ncols][cols[None, :] == rr] == 1.0)
    if call.kind == "decision":
        want, bound = pysvm.exact_scores(out["kernel"], np.arange(call.nrows), np.arange(call.ncols), alpha, -0.25)
        # a row of zero norm (a weighted row of exactly L bases) is NaN in the oracle, the kernel and its decision value
        nan = np.isnan(want)
        assert np.array_equal(np.isnan(out["dv"]), nan), "decision values: NaN rows"
        err = np.abs(out["dv"][~nan] + want[~nan])
        assert np.all(err <= bound[~nan]), "decision values: worst excess %g" % np.max(err - bound[~nan])


@pytest.mark.parametrize("case", ig.CASES, ids=repr)
def test_every_index_instance(case, record_property):
    seqs = case.seqs()
    o = pyoracle.Oracle(**case.params)
    for s in seqs:
        o.add(s)
    calls = case.calls()
    alphas = {i: np.random.default_rng(i).standard_normal(c.ncols) for i, c in enumerate(calls)}
    got, seen = [], {}
    with options(**case.options), capi.Problem(**case.params) as P:
        P.add_many(seqs)
        for i, call in enumerate(calls):
            out, rec = run_call(P, call, alphas[i])
            for what, r in rec.items():
                for k, m in check_record(case, call, r, "%r %s" % (call, what)).items():
                    seen[k] = seen.get(k, 0) | m
            assert P.stats()["kernel_variant"] == 4
            got.append(out)
        if case.n <= 600:   # the whole triangle through the reference's entry point as well
            K = P.kernel_lower()
            check_record(case, ig.Call("lower", 0, case.n, 0, case.n), P.index_blocks(), "kernel_lower")
            Kl, Hl = o.matrix_lower()
            same(K, np.where(np.tri(case.n, k=-1, dtype=bool), Kl, 0.0) + np.eye(case.n), case.kernel_type, "kernel_lower")
            assert np.array_equal(got[0]["hist"], Hl), "lower histograms"
        capi.set_option("kernel", "diag")
        for i, call in enumerate(calls):   # the bit-sliced kernel over the whole of every call
            ref, _ = run_call(P, call, alphas[i])
            assert P.stats()["kernel_variant"] == 2
            for name in ref:
                if name != "dv":
                    same(got[i][name], ref[name], case.kernel_type, "%r %s: index vs bit-sliced" % (call, name), exact=True)
    for i, call in enumerate(calls):
        oracle_checks(case, o, call, got[i], alphas[i])
    f, w, r, m = case.target
    ran = {k: [ig.inst_name(case.stats()[k][3], case.weighted, bit >= 2, bit % 2 + 1) for bit in range(4) if mask >> bit & 1]
           for k, mask in seen.items()}
    record_property("index_instance", {"target": ig.inst_name(f, w, r, m), "cold_bins": case.cold, "ran": ran,
                                       "smem": max(s for c in calls for _, s in case.predict(c).values())})
    assert seen.get(case.block, 0) & ig.inst_bit(r, m), "the target instance never ran: %s" % ran


# ---- state carried between calls ----
def _problem(params, seqs):
    o = pyoracle.Oracle(**params)
    for s in seqs:
        o.add(s)
    return o


def _rect_vs_oracle(P, o, r0, nr, c0, nc, kt):
    K = P.kernel_block(r0, nr, c0, nc)
    rows = np.array([r0, r0 + nr // 2, r0 + nr - 1])
    Ko, _ = o.rect(rows, c0 + nc, with_hist=False)
    for i, r in enumerate(rows):
        same(K[r - r0], Ko[i, c0:], kt, "row %d" % r)
    return K


def test_later_calls_reuse_the_partition_and_range_inside_it():
    """after the lower triangle over [0, 300) cut blocks of 128, 128 and 44 columns, a rectangle from column 150 reuses
    them: the layout stays, only the blocks it touches launch, the one it starts inside with RANGE"""
    params = dict(kernel_type=2, L=9, k=7, d=2, M=50, H=50.0, gamma=0.7)
    seqs = ig.make_seqs(9, 300, 40, 31)
    o = _problem(params, seqs)
    with options(kernel="index", index_cols=128), capi.Problem(**params) as P:
        P.add_many(seqs)
        _, Hl = o.matrix_lower()
        assert np.array_equal(P.hist_block(0, 300, 0, 300, lower=True), Hl)
        assert P.index_layout() == (3, 128, 0)
        _rect_vs_oracle(P, o, 100, 100, 150, 120, 2)
        assert P.index_layout() == (3, 128, 0)
        assert [b["inst"] for b in P.index_blocks()] == [0, ig.inst_bit(1, 2), ig.inst_bit(0, 2)]


def test_a_call_outside_the_partition_rebuilds():
    """decision values over the columns [0, 100) cut the partition [0, 100); a rectangle over [50, 250) lies outside it and
    starts over from column 50 (no RANGE there), and a later one from column 120 ranges inside the new block"""
    params = dict(kernel_type=4, L=10, k=7, d=3, M=50, H=50.0, gamma=0.7)
    seqs = ig.make_seqs(10, 260, 40, 37)
    o = _problem(params, seqs)
    alpha = np.random.default_rng(5).standard_normal(100)
    with options(kernel="index"), capi.Problem(**params) as P:
        P.add_many(seqs)
        dv = P.decision_values(0, 260, 0, 100, alpha)
        assert P.index_layout() == (1, 128, 0)
        Kb = P.kernel_block(0, 260, 0, 100)
        want, bound = pysvm.exact_scores(Kb, np.arange(260), np.arange(100), alpha, 0.0)
        assert np.all(np.abs(dv + want) <= bound)
        _rect_vs_oracle(P, o, 40, 200, 50, 200, 4)
        assert P.index_layout() == (1, 224, 50)
        assert [(b["cb"], b["ce"], b["inst"]) for b in P.index_blocks()] == [(50, 250, ig.inst_bit(0, 2))]
        _rect_vs_oracle(P, o, 100, 60, 120, 60, 4)
        assert P.index_layout() == (1, 224, 50)
        assert [b["inst"] for b in P.index_blocks()] == [ig.inst_bit(1, 2)]


def test_a_named_split_forces_a_rebuild():
    """150 columns at cap 128: equal shares are blocks of 96, greedy ones of 128.  Naming greedy after an equal split
    rebuilds even for a call inside the partition; back on auto a rectangle keeps what is there"""
    params = dict(kernel_type=0, L=8, k=6, d=2, M=50, H=50.0, gamma=0.7)
    seqs = ig.make_seqs(8, 150, 40, 41)
    o = _problem(params, seqs)
    _, Hl = o.matrix_lower()
    with options(kernel="index", index_cols=128), capi.Problem(**params) as P:
        P.add_many(seqs)
        capi.set_option("index_split", "equal")
        assert np.array_equal(P.hist_block(0, 150, 0, 150, lower=True), Hl)
        assert P.index_layout() == (2, 96, 0)
        capi.set_option("index_split", "greedy")
        assert np.array_equal(P.hist_block(0, 150, 0, 150, lower=True), Hl)
        assert P.index_layout() == (2, 128, 0)
        assert [(b["cb"], b["ce"]) for b in P.index_blocks()] == [(0, 128), (128, 150)]
        capi.set_option("index_split", "auto")
        _rect_vs_oracle(P, o, 10, 140, 0, 150, 0)
        assert P.index_layout() == (2, 128, 0)


def test_two_problems_take_turns_on_one_mask_list():
    """the GPU keeps the XOR masks of the last (L, d) it served: two problems with different (L, d) alternating must each
    get their own, every time"""
    pa = dict(kernel_type=2, L=8, k=6, d=2, M=50, H=50.0, gamma=0.7)
    pb = dict(kernel_type=4, L=10, k=7, d=3, M=50, H=50.0, gamma=0.7)
    sa, sb = ig.make_seqs(8, 120, 40, 43), ig.make_seqs(10, 130, 40, 47)
    Ha = _problem(pa, sa).matrix_lower()[1]
    Hb = _problem(pb, sb).matrix_lower()[1]
    with options(kernel="index"), capi.Problem(**pa) as A, capi.Problem(**pb) as B:
        A.add_many(sa)
        B.add_many(sb)
        for _ in range(2):
            assert np.array_equal(A.hist_block(0, 120, 0, 120, lower=True), Ha), "problem A (L = 8, d = 2)"
            assert np.array_equal(B.hist_block(0, 130, 0, 130, lower=True), Hb), "problem B (L = 10, d = 3)"
            assert np.array_equal(A.hist_block(60, 60, 0, 120), _problem(pa, sa).rect(np.arange(60, 120), 120)[1])
