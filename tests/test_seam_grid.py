"""CPU tier: the cuts of tests/seam_grid.py against the library's host code, and the grid's coverage of them -- every cut,
for every variant it applies to, has a case one step past it whose first call below sits exactly at it (one piece), and
the launch counts the GPU tier asserts differ on the two sides."""
import pytest

import seam_grid as sg
from gkmqc_b200 import capi


@pytest.fixture(scope="module")
def lib():
    return capi.load()


@pytest.mark.parametrize("lower", [0, 1])
@pytest.mark.parametrize("variant", ["diag", "index"])
def test_restated_budget_reproduces_the_planner(lib, variant, lower):
    """plan_budget and the caps, restated, give the chunk lists the product's plan_chunks makes: tiled rows, the row cap,
    the byte budget per GPU count and chunk_mb"""
    for nrows in (1, 15, 16, 17, 147, 593, 1000, 5000, sg.ROW_CAP - 1, sg.ROW_CAP, sg.ROW_CAP + 1, sg.ROW_CAP + 100, 140000):
        for ncols in (1, 8, 9, 300, 3000):
            for ndev, mb in ((1, 128), (2, 128), (8, 1), (1, 1), (3, 7)):
                ch = sg.plan_chunks(lib, variant, 5, nrows, 3, ncols, lower, ndev, mb)
                assert ch[0][0] == 5 and ch[-1][1] == 5 + nrows
                budget = sg.plan_budget(nrows * ncols // (2 if lower else 1), ndev, mb)
                tile, cap = (sg.WAVE_ROWS, sg.WAVE_CAP) if variant == "index" else (sg.TILE_ROWS, sg.ROW_CAP)
                for rb, re_, cb, ce in ch:
                    if re_ - rb > tile:
                        assert re_ - rb <= cap and (re_ - rb) * (ce - cb) * 8 <= budget
                for (rb, re_, cb, ce), nxt in zip(ch, ch[1:]):
                    # a chunk stops only when one more tile would break the row cap or the byte budget
                    ne = min(re_ + tile, 5 + nrows)
                    wide = (min(3 + ncols, ne) if lower else 3 + ncols) - 3
                    assert ne - rb > cap or (ne - rb) * max(wide, 0) * 8 > budget, (nrows, ncols, ndev, mb, rb, re_)


def test_budget_floor_and_cap():
    assert sg.plan_budget(0, 1) == 4 << 20
    assert sg.plan_budget(10 ** 10, 1) == 128 << 20
    assert sg.plan_budget(10 ** 10, 1, chunk_mb=1) == 1 << 20
    assert sg.plan_budget(50000 * 50000 // 2, 8) == 50000 * 50000 // 2 * 8 // 128


def test_shares():
    assert sg.shares(1, 2, 8) == [(0, 1), (1, 1)]
    assert sg.shares(17, 2, 8) == [(0, 16), (16, 17)]
    assert sg.shares(15, 2, 8) == [(0, 8), (8, 15)]
    assert sg.shares(7, 3, 1) == [(0, 3), (3, 6), (6, 7)]


def _lens(case, cache={}):
    if case.name not in cache:
        cache[case.name] = case.lens()
    return cache[case.name]


@pytest.mark.parametrize("case", sg.CASES, ids=repr)
def test_case_crosses_its_cut_and_its_twin_does_not(lib, case):
    lens = _lens(case)
    pred = sg.predict(case, case.call, lib=lib, lens=lens)
    twin = sg.predict(case, case.below[0], lib=lib, lens=lens)
    if case.cut == "diag-step" and sg.diag_step(case.variant) == sg.DIAG_STEP_BITSLICED and case.call.kind == "upload":
        # mma and index hand the diagonal to the bit-sliced kernel: one launch where lmer takes three
        assert len(pred["pieces"]) == 1 and pred["launches"] == 2
        return
    if case.call.kind == "subst" and case.cut == "diag-step":
        assert len(sg.diag_seams(case, lens)) == 1
    else:
        assert len(pred["pieces"]) >= 2 and len(pred["seams"]) == len(pred["pieces"]) - 1
    assert len(twin["pieces"]) == 1, twin
    assert pred["launches"] != twin["launches"], (pred["launches"], twin["launches"])
    if case.cut == "chunk-bytes":
        assert len(pred["pieces"]) >= 5
    if case.cut == "chunk-rows":
        assert pred["seams"][0] == (sg.ROW_CAP - 1, sg.ROW_CAP)
        assert twin["pieces"] == [(0, sg.ROW_CAP)]
    # the calls below the cut cover the crossing call's rows or sites exactly
    if case.call.kind == "subst":
        assert [c.sites for c in case.below][0][0] == case.call.sites[0]
        assert [c.sites for c in case.below][-1][1] == case.call.sites[1]
    elif case.call.kind != "upload":
        assert case.below[0].row0 == case.call.row0
        assert sum(c.nrows for c in case.below) == case.call.nrows


def test_every_cut_has_cases_on_both_sides_for_every_variant():
    have = {}
    for case in sg.CASES:
        if case.cut == "diag-step" and case.call.kind == "upload" and case.variant != "lmer":
            continue
        have.setdefault(case.cut, set()).add(case.variant)
    assert {cut: set(v) for cut, v in sg.CUTS.items()} == have


def test_smallest_row_tile_where_the_row_cap_matters(lib):
    """the 2 047-bp row of the 65 620-row rectangles: mma takes one query per CTA (65 520 row tiles, the cap itself),
    the bit-sliced kernel a row tile of two, weighted lmer (2, 2); a 65 536-row chunk would be refused on the host with a
    one-row tile only"""
    for case in sg.CASES:
        if case.cut != "chunk-rows":
            continue
        ta = launch_grid_shape(case)[1]
        assert sg.ROW_CAP // ta <= 65535
        assert (65536 // ta > 65535) == (case.variant == "mma")


def launch_grid_shape(case):
    import launch_grid
    return launch_grid.expected_shape(case.variant, case.maxlen(), case.L, case.d, case.weighted)
