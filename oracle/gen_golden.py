#!/usr/bin/env python
"""Generate tests/golden/* from the UNMODIFIED reference (oracle/_ref, built by
`make -C oracle ref` from /root/reference/src).  Run in the build container only:

    python oracle/gen_golden.py

Writes the FASTA fixtures and one .npz per parameter set holding what the
reference itself produced: w[m], sqnorm, positional weights, the integer
mismatch profiles (through the DFS probe in oracle/ref_hook.cc) and the
normalised kernel rows.  The committed fixtures are what pins the oracle
(tests/test_oracle_golden.py) and the CUDA path (tests/test_gpu_parity.py) on
machines where /root/reference does not exist.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import pyoracle  # noqa: E402

GOLD = os.path.join(os.path.dirname(HERE), "tests", "golden")

# (name, fixture, kernel_type, L, k, d, M, H, gamma)
CONFIGS = [
    ("uni_t0_L11k7d3", "uni", 0, 11, 7, 3, 50, 50.0, 1.0),
    ("uni_t1_L11k7d3", "uni", 1, 11, 7, 3, 50, 50.0, 1.0),
    ("uni_t2_L11k7d3", "uni", 2, 11, 7, 3, 50, 50.0, 1.0),
    ("uni_t3_L11k7d3", "uni", 3, 11, 7, 3, 50, 50.0, 2.0),
    ("uni_t4_L11k7d3", "uni", 4, 11, 7, 3, 50, 50.0, 1.0),
    ("uni_t5_L11k7d3", "uni", 5, 11, 7, 3, 50, 50.0, 0.5),
    ("uni_t4_L10k6d3", "uni", 4, 10, 6, 3, 50, 50.0, 1.0),   # gkmQC defaults, bin/gkmqc.py:169-199
    ("mix_t2_L11k7d3", "mix", 2, 11, 7, 3, 50, 50.0, 1.0),
    ("mix_t4_L11k7d3", "mix", 4, 11, 7, 3, 50, 50.0, 1.0),
    ("mix_t4_L10k6d3_M255", "mix", 4, 10, 6, 3, 255, 20.0, 1.0),
    ("mix_t2_L10k6d4", "mix", 2, 10, 6, 4, 50, 50.0, 1.0),
    ("mix_t2_L10k6d2", "mix", 2, 10, 6, 2, 50, 50.0, 1.0),
    ("mix_t2_L11k7d4", "mix", 2, 11, 7, 4, 50, 50.0, 1.0),
    ("mix_t2_L12k8d4", "mix", 2, 12, 8, 4, 50, 50.0, 1.0),
    ("mix_t0_L12k6d6", "mix", 0, 12, 6, 6, 50, 50.0, 1.0),
    ("mix_t2_L12k4d8", "mix", 2, 12, 4, 8, 50, 50.0, 1.0),
    ("mix_t2_L13k7d4", "mix", 2, 13, 7, 4, 50, 50.0, 1.0),   # needs the MAX_MM=16 probe build
    ("mix_t4_L14k8d4", "mix", 4, 14, 8, 4, 50, 50.0, 1.0),
    ("mix_t2_L8k4d4", "mix", 2, 8, 4, 4, 50, 50.0, 1.0),
    ("mix_t2_L6k4d2", "mix", 2, 6, 4, 2, 50, 50.0, 1.0),
    ("mix_t2_L3k2d1", "mix", 2, 3, 2, 1, 50, 50.0, 1.0),
    ("mix_t0_L2k1d1", "mix", 0, 2, 1, 1, 50, 50.0, 1.0),
    ("mix_t2_L9k9d0", "mix", 2, 9, 9, 0, 50, 50.0, 1.0),
]

WEIGHT_GRID = [(t, L, k) for t in (0, 1, 2) for L in range(2, 17) for k in range(1, L + 1)]


def wrap(s, w):
    return [s[i:i + w] for i in range(0, len(s), w)] or [""]


def write_fixtures():
    os.makedirs(GOLD, exist_ok=True)
    rng = np.random.default_rng(20261018)
    acgt = np.array(list("ACGT"))

    def rnd(n):
        return "".join(rng.choice(acgt, n))

    # uniform: 10 + 10 sequences of 300 bp, one record per two lines
    for name, n in (("uni_pos.fa", 10), ("uni_neg.fa", 10)):
        with open(os.path.join(GOLD, name), "w") as f:
            for i in range(n):
                f.write(">%s_%d some description\n%s\n" % (name[:-3], i, rnd(300)))

    # mixed: ragged lengths, quirks of read_fasta_file (libgkm.c:1251-1314)
    base = rnd(220)
    pal = rnd(40)
    comp = {"A": "T", "C": "G", "G": "C", "T": "A"}
    pal = pal + "".join(comp[c] for c in reversed(pal))          # reverse-palindrome, 80 bp
    pos = [
        ("m0", rnd(300), 60, "\n"),
        ("m1", base, 50, "\n"),
        ("m2\textra", base[:100].lower() + base[100:], 70, "\r\n"),  # lower case + CRLF; same bases as m1
        ("m3", base[:110] + "N" + base[111:200] + "nRY", 80, "\n"),  # non-ACGT -> 'A'
        ("m4", "A" * 64, 64, "\n"),                                  # homopolymer: every pair hits
        ("m5", "ACGT" * 30, 33, "\n"),                               # tandem repeat
        ("m6", pal, 1000, "\n"),
        ("m7", rnd(14), 1000, "\n"),                                 # exactly one 14-mer
    ]
    neg = [
        ("n0", rnd(2500), 100, "\n"),                                # > 2047: truncated
        ("n1", rnd(451), 60, "\n"),
        ("n2", base[30:190], 60, "\n"),                              # substring of m1
        ("n3", "".join(comp[c] for c in reversed(base)), 60, "\n"),  # reverse complement of m1
        ("n4", rnd(33), 10, "\n"),
        ("n5", rnd(32), 32, "\n"),
        ("n6", rnd(97) + "A" * 20 + rnd(64), 61, "\n"),
    ]
    for name, recs in (("mix_pos.fa", pos), ("mix_neg.fa", neg)):
        with open(os.path.join(GOLD, name), "w", newline="") as f:
            for j, (sid, s, w, nl) in enumerate(recs):
                f.write(">" + sid + nl)
                for piece in wrap(s, w):
                    f.write(piece + nl)
                if j % 3 == 1:
                    f.write(nl)                                     # blank line between records
            # NB: the last line keeps its newline -- without one the reference's readline()
            # reallocs a by-value buffer and double-frees it (libgkm.c:1207-1225, :1312)


# gkmb200_problem_index_layout() of the full-size problem below on a B200, per kernel type: (column blocks, columns per
# block).  10 000 columns fit one block for both types (full blocks of 22 528 and 16 352 columns); a layout with more
# blocks puts the stored rows and columns on both sides of every block boundary, like the rows the full-size GPU test
# checks live.
FULL10K_INDEX_LAYOUT = {2: (1, 22528), 4: (1, 16352)}


def full_size_rows(nrows=32, ncols=256, seed=20261020):
    """tests/golden/full10k_rows_kt{2,4}.npz: BASELINE configs[1] at full size (bench.synth(10000), 300 bp, L=11 k=7 d=3) --
    kernel values and mismatch histograms of the rows tests/test_gpu_parity.py's full-size test checks (bench.parity_rows on
    the index layout: both sides of every column block and chunk boundary), at ncols seeded columns below each row plus the
    block boundary columns.  Where oracle/_ref is built the numbers are the unmodified reference's (RefHook.rows_values) and
    the C restatement must give the same; elsewhere they are the C restatement's, which is bit-identical to the reference
    on every golden set above.
        python oracle/gen_golden.py --full-size"""
    import tempfile
    sys.path.insert(0, os.path.dirname(HERE))
    import bench
    n = 10000
    arr = bench.synth(n)
    tmp = tempfile.mkdtemp(prefix="gkmgold_")
    pos, neg = os.path.join(tmp, "p.fa"), os.path.join(tmp, "n.fa")
    bench.write_fasta(pos, arr[: n // 2], 0)
    bench.write_fasta(neg, arr[n // 2:], n // 2)
    for kt in (2, 4):
        nblk, blk_cols = FULL10K_INDEX_LAYOUT[kt]
        rows = bench.parity_rows(n, blk_cols, nblk, want=nrows)[:40]
        edges = np.array([k * blk_cols + e for k in range(1, nblk) for e in (-1, 0, 1)], np.int64)
        rng = np.random.default_rng(seed + kt)
        pairs = [(int(r), int(c)) for r in rows
                 for c in np.union1d(rng.choice(r, size=min(r, ncols), replace=False), edges[edges < r])]
        row, col = (np.array(x, np.int32) for x in zip(*pairs))
        o = pyoracle.Oracle(kt, 11, 7, 3)
        assert o.read_problem(pos, neg) == n
        K = np.array([o.kernel(a, b) for a, b in pairs])
        Hm = np.array([o.hist(a, b) for a, b in pairs], np.int32)
        o.close()
        source = "C restatement"
        if pyoracle.have_ref():
            h = pyoracle.RefHook(pos, neg, kt, 11, 7, 3)
            try:
                Kr, Hr, _ = h.rows_values(rows, os.cpu_count() or 1)
            finally:
                h.close()
            at = {int(r): i for i, r in enumerate(rows)}
            Kref = np.array([Kr[at[a], b] for a, b in pairs])
            Href = np.array([Hr[at[a], :, b] for a, b in pairs], np.int32)
            assert np.array_equal(Kref, K) and np.array_equal(Href, Hm), "C restatement differs from the reference"
            K, Hm, source = Kref, Href, "reference (C restatement identical)"
        np.savez_compressed(os.path.join(GOLD, "full10k_rows_kt%d.npz" % kt), row=row, col=col, kmat=K, hist=Hm)
        print("full10k_rows_kt%d: %d entries of %d rows, from the %s" % (kt, len(pairs), len(rows), source))
    for f in (pos, neg):
        os.remove(f)
    os.rmdir(tmp)


def main():
    pyoracle.build_oracle()
    if sys.argv[1:] == ["--full-size"]:
        return full_size_rows()
    if not pyoracle.build_ref():
        raise SystemExit("reference sources not present; cannot generate golden vectors")
    write_fixtures()

    # 1. weight table from the reference for a grid of (type, L, k)
    wt = {}
    for (t, L, k) in WEIGHT_GRID:
        if L < 2:
            continue
        w = pyoracle.ref_weights(t, L, k)
        if t == 0:
            w[L - k + 1:] = 0.0  # slots the reference leaves uninitialised (libgkm.c:212-216)
        wt["t%d_L%d_k%d" % (t, L, k)] = w
        wo = pyoracle.oracle_weights(t, L, k)
        assert np.array_equal(w, wo), ("oracle weights differ", t, L, k, w, wo)
    np.savez_compressed(os.path.join(GOLD, "weights.npz"), **wt)
    print("weights: %d parameter sets, oracle bit-identical" % len(wt))

    # 2. per-config problems
    for (name, fx, t, L, k, d, M, H, gamma) in CONFIGS:
        pos = os.path.join(GOLD, fx + "_pos.fa")
        neg = os.path.join(GOLD, fx + "_neg.fa")
        h = pyoracle.RefHook(pos, neg, t, L, k, d, M, H, gamma)
        n = h.n
        K = np.zeros((n, n))
        Hm = np.zeros((n, n, d + 1), np.int32)
        for a in range(n):
            K[a, :a] = h.row(a, 0, a)
            K[a, a] = 1.0
            Hm[a, :a, :] = h.mmprofile(a, a).T
        sq = h.sqnorm()
        w = h.weights(d + 1)
        lens = np.array([h.seqlen(i) for i in range(n)], np.int32)
        pw = np.zeros((n, 2, int(lens.max())), np.uint8)
        for i in range(n):
            a, b = h.poswt(i)
            pw[i, 0, :len(a)] = a
            pw[i, 1, :len(b)] = b
        # the diagonal profile: sqnorm^2 = sum w*H(a,a); take it from row(a) of a doubled problem? no --
        # the reference never runs the DFS on (a,a); sqnorm above is its own dense loop (libgkm.c:723-759).
        npos = h.npos
        h.close()

        out = dict(kernel_type=t, L=L, k=k, d=d, M=M, H=H, gamma=gamma, npos=npos, lens=lens,
                   weights=w, sqnorm=sq, poswt=pw, kmat=K, hist=Hm)

        # stock pywrapper (only inside its own parameter gate), 3 threads to exercise the remainder rows
        if L <= 12:
            ret, kw, np_, nn_ = pyoracle.call_pywrapper(pyoracle.ref_pywrapper(), pos, neg, t, L, k, d, M, H, gamma,
                                                         nthreads=3, verbosity=0, nmax=n + 3)
            assert ret == 0 and np_ == npos and np_ + nn_ == n
            assert np.array_equal(kw[:n, :n], K), "pywrapper and probe rows differ"
            assert not kw[n:].any() and not np.triu(kw[:n, :n], 1).any()

        # cross-check the C restatement while we are here
        o = pyoracle.Oracle(t, L, k, d, M, H, gamma)
        assert o.read_problem(pos, neg) == n and o.npos == npos
        Ko, Ho = o.matrix_lower()
        assert np.array_equal(Ho, Hm), (name, "histograms differ")
        assert np.array_equal(o.weights()[:d + 1], w), (name, "weights differ")
        assert np.array_equal(o.sqnorm(), sq), (name, "sqnorm differs")
        if t in (3, 5):
            err = np.max(np.abs(Ko - K) / np.maximum(np.abs(K), 1e-300))
            assert err < 1e-12, (name, err)
        else:
            assert np.array_equal(Ko, K), (name, "kernel values differ", np.max(np.abs(Ko - K)))
        for i in range(n):
            a, b = o.poswt(i)
            assert np.array_equal(a, pw[i, 0, :len(a)]) and np.array_equal(b, pw[i, 1, :len(b)])
        o.close()
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
        print("%-24s n=%d  hits=%d  oracle == reference" % (name, n, int(Hm.sum())))


if __name__ == "__main__":
    main()
