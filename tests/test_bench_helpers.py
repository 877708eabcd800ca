"""CPU tier: the pieces of bench.py that decide whether a bench line may be trusted -- the synthetic FASTA it writes,
the rows it picks for the in-line parity check, the check itself (it must pass on the reference's own numbers and
fail on a single flipped bit) and the output sample --dump-outputs writes."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from conftest import load_golden  # noqa: E402
from gkmqc_b200 import capi  # noqa: E402


def test_written_fasta_is_what_the_reader_reads(tmp_path):
    pos, neg = bench.write_problem(str(tmp_path), 37, seed=5)
    arr = bench.synth(37, seed=5)
    with capi.Problem(2, 11, 7, 3) as P:
        assert P.read(pos, neg) == 18 and P.n == 37
        for i in (0, 17, 18, 36):
            assert P.sid(i) == b"s%d" % i and P.seqlen(i) == 300
            assert np.array_equal(P.codes(i)[0], np.searchsorted(np.frombuffer(b"ACGT", np.uint8), arr[i]) + 1)


def test_parity_rows_cover_both_sides_of_every_boundary():
    n, cols, nblk = 50000, 12512, 4
    rows = bench.parity_rows(n, cols, nblk)
    assert len(rows) >= 64 and rows.min() >= 1 and rows.max() == n - 1 and len(set(rows)) == len(rows)
    for k in (1, 2, 3):
        assert {k * cols - 1, k * cols, k * cols + 1} <= set(rows)
    assert any(r % 148 == 0 for r in rows) and any(r % 148 == 147 for r in rows) and any(r % 592 == 0 for r in rows)
    small = bench.parity_rows(40, 40, 1)
    assert len(small) == 39 and small.min() == 1 and small.max() == 39


def test_dumped_outputs_are_a_fixed_sample_within_64_mb(tmp_path):
    n = bench.BASE_N
    rows = bench.dump_rows(np.arange(n), n)
    assert np.array_equal(rows, bench.dump_rows(np.arange(n), n)) and len(set(rows)) == len(rows) > 64
    assert len(rows) * n * 8 + (len(rows) + 2) * 8 < 64 << 20
    assert np.array_equal(bench.dump_rows(np.arange(7), 7), np.arange(7))
    kmat = np.tril(np.random.default_rng(1).random((300, 300)), -1) + np.eye(300)
    bench.dump_outputs(str(tmp_path / "out"), kmat, 150, 150)
    got = {f: np.load(tmp_path / "out" / (f + ".npy")) for f in ("kmat_rows", "kmat_row_ids", "kmat_size")}
    assert all(a.dtype == np.float64 for a in got.values())
    ids = got["kmat_row_ids"].astype(int)
    assert np.array_equal(ids, bench.dump_rows(np.arange(300), 300)) and np.array_equal(got["kmat_rows"], kmat[ids])
    assert list(got["kmat_size"]) == [150, 150]
    # a sharded call: rows of other ranks' chunks stay zero in this rank's matrix and are not sampled
    kmat[::2] = 0.0
    bench.dump_outputs(str(tmp_path / "shard"), kmat, 150, 150)
    ids = np.load(tmp_path / "shard" / "kmat_row_ids.npy").astype(int)
    assert len(ids) == 150 and np.all(ids % 2 == 1)


class StoredReference:
    """the reference's own rows and mismatch histograms of a stored problem (tests/golden, written from the unmodified
    reference by oracle/gen_golden.py), answered through the one pyoracle.RefHook call check_parity makes"""

    def __init__(self, g):
        self.K, self.H = g["kmat"], g["hist"]

    def rows_values(self, rows, nthreads):
        ld = int(max(rows.max(), 1))
        K = np.zeros((len(rows), ld))
        H = np.zeros((len(rows), self.H.shape[2], ld), np.int32)
        for i, r in enumerate(rows):
            K[i, :r] = self.K[r, :r]
            H[i, :, :r] = self.H[r, :r].T
        return K, H, 0.0


def test_parity_check_passes_on_the_reference_and_catches_one_bit():
    g, cfg, _, _ = load_golden("uni_t2_L11k7d3")      # bench.py's kernel type and (L, k, d)
    assert (cfg["kernel_type"], cfg["L"], cfg["k"], cfg["d"]) == (bench.KTYPE, bench.L, bench.K, bench.D)
    h = StoredReference(g)
    n = len(g["lens"])
    rows = np.arange(1, n, dtype=np.int32)
    K, H, _ = h.rows_values(rows, 2)
    kmat = np.zeros((n, n))
    hist = {}
    for i, r in enumerate(rows):
        kmat[r, :r] = K[i, :r]
        hist[int(r)] = H[i, :, :r].T.copy()
    np.fill_diagonal(kmat, 1.0)
    par, _ = bench.check_parity(h, kmat, lambda r: hist[r], n, (1, n, 0), 2, owned_only=False)
    assert par["ok"] and par["hist_bit_exact"] and par["kmat_max_rel"] == 0.0 and par["rows"] == n - 1
    bad = kmat.copy()
    bad[17, 5] = np.nextafter(bad[17, 5], 2.0)          # one ulp
    par, _ = bench.check_parity(h, bad, lambda r: hist[r], n, (1, n, 0), 2, owned_only=False)
    assert not par["kmat_bit_identical"] and 17 in par["mismatching_rows"]
    hist[12][3, 2] += 1                                   # one count
    par, _ = bench.check_parity(h, kmat, lambda r: hist[r], n, (1, n, 0), 2, owned_only=False)
    assert not par["ok"] and not par["hist_bit_exact"]
    touched = kmat.copy()
    touched[10, 15] = 0.5                                 # the upper triangle belongs to the caller
    par, _ = bench.check_parity(h, touched, lambda r: hist[r], n, (1, n, 0), 2, owned_only=False)
    assert 10 in par["mismatching_rows"]
