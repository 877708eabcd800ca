"""CPU tier: gkm_bitslice.h -- the arithmetic the sm_100a kernel runs per lane -- executed serially by the
lane emulator (tests/emu/diag_emu.cc) over the product's own packed image, against the golden histograms."""
import numpy as np
import pytest

import launch_grid
import pyoracle
from conftest import golden_names, load_golden
from gkmqc_b200 import capi


@pytest.mark.parametrize("name", golden_names())
def test_emulated_lanes_match_reference_histograms(name, emu_lib):
    g, cfg, pos, neg = load_golden(name)
    P = capi.Problem(lib=emu_lib, **cfg)
    assert P.read(pos, neg) == int(g["npos"])
    n = P.n
    H = np.zeros((n, n, cfg["d"] + 1), np.int32)
    assert emu_lib.gkm_emu_hist_lower(P.h, H.ctypes.data_as(capi.c_i32_p)) == 0
    w = P.weights()
    sq = np.array([np.sqrt(sum(w[m] * H[a, a, m] for m in range(len(w)))) for a in range(n)])
    assert np.array_equal(sq, g["sqnorm"]), "diagonal histograms (sqnorm)"
    for a in range(n):
        H[a, a:, :] = 0
    assert np.array_equal(H, g["hist"])
    P.close()


@pytest.mark.parametrize("case", launch_grid.INSTANCE_CASES, ids=repr)
def test_emulated_lanes_random_ragged(case, emu_lib):
    """every bit-sliced instance a caller can reach (tests/launch_grid.py), on the grid's edge-case sequences: query pairs
    as the kernel takes them (lower triangle and diagonal), and single queries against targets above the diagonal"""
    seqs = case.seqs()
    n, d = len(seqs), case.d
    o = pyoracle.Oracle(**case.params)
    P = capi.Problem(lib=emu_lib, **case.params)
    for s in seqs:
        o.add(s)
        P.add(s)
    H = np.zeros((n, n, d + 1), np.int32)
    assert emu_lib.gkm_emu_hist_lower(P.h, H.ctypes.data_as(capi.c_i32_p)) == 0
    for a in range(n):
        for b in range(a + 1):
            assert np.array_equal(H[a, b], o.hist(a, b)), (a, b)
    h = np.zeros(d + 1, np.int32)
    for a in range(n):
        for b in range(a + 1, n):
            assert emu_lib.gkm_emu_hist(P.h, a, b, h.ctypes.data_as(capi.c_i32_p)) == 0
            assert np.array_equal(h, o.hist(a, b)), (a, b)
    P.close()


def test_instance_grid_covers_the_reachable_instances(emu_lib):
    """the grid holds one case per instance the parameter gate lets a caller reach, and the compiled instances it leaves
    out are exactly the unreachable ones"""
    reach = launch_grid.reachable_instances()
    grid = [c.inst for c in launch_grid.INSTANCE_CASES]
    assert len(grid) == len(set(grid)) == len(reach) == 86 and set(grid) == reach
    # the restated gate is the library's (which admits L <= 12 through this entry point)
    for L in range(2, 13):
        for k in range(-1, L + 2):
            for d in range(-1, L + 2):
                assert launch_grid.gate_ok(L, k, d) == (capi.check_parameter(lib=emu_lib, kernel_type=2, L=L, k=k, d=d) is None), (L, k, d)
    left = launch_grid.compiled_instances() - reach
    want = {(L, 8, w, d4) for L in (2, 3) for w, d4 in ((False, False), (False, True), (True, False))}
    want |= {(4, 8, False, False)}
    want |= {(L, 16, w, False) for L in range(2, 8) for w in (False, True)}
    assert len(launch_grid.compiled_instances()) == 105 and left == want and len(left) == 19
    # d = L - 1, d = L (k = 0) and d = 15 at L = 15 and 16 all occur; so does every kernel type
    assert any(c.d == c.L - 1 for c in launch_grid.INSTANCE_CASES)
    assert any(c.d == c.L and c.k == 0 for c in launch_grid.INSTANCE_CASES)
    assert {(c.L, c.d) for c in launch_grid.INSTANCE_CASES} >= {(15, 15), (16, 15)}
    assert {c.kernel_type for c in launch_grid.INSTANCE_CASES} == set(range(6))
    # the sequence recipe: n a multiple of neither 8 nor 32, one of exactly L bases, 16m - 1, 16m, 16m + 1
    for c in launch_grid.INSTANCE_CASES[:3] + launch_grid.SHAPE_CASES:
        lens = [len(s) for s in c.seqs()]
        assert len(lens) % 8 and min(lens) == c.L and max(lens) == c.maxlen
        assert any(ln - 1 in lens and ln in lens and ln + 1 in lens for ln in range(16, c.maxlen, 16))
