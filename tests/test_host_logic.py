"""CPU tier: everything in gkmkern_pylib.so that runs on the host -- parameter gate, w[m], positional
weights, FASTA reader, base coding, chunk planning -- plus the C-ABI surface itself.  No compute calls."""
import ctypes
import os
import re

import numpy as np
import pytest

import pyoracle
from conftest import GOLD, ROOT, golden_names, load_golden, random_seqs
from gkmqc_b200 import capi


def test_library_exports_every_declared_symbol(product_lib):
    declared = set()
    for hdr in ("gkm_abi.h", "gkm_b200.h"):
        text = open(os.path.join(ROOT, "include", hdr)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        declared |= set(re.findall(r"\b(gkm[a-z0-9_]*)\s*\(", text))
    declared -= {"gkm_abi"}
    assert {"gkm_main_pywrapper", "gkmkernel_init", "gkmkernel_kernelfunc_batch_all", "gkmb200_kernel_lower"} <= declared
    missing = [s for s in sorted(declared) if not hasattr(product_lib, s)]
    assert not missing, "declared in include/*.h but not exported: %s" % missing


def test_struct_layouts_match_the_reference_abi():
    # SURVEY.md 8b: gkmOpt offsets probed from the reference build
    assert ctypes.sizeof(capi.gkmOpt) == 64
    assert capi.gkmOpt.M.offset == 16 and capi.gkmOpt.H.offset == 24 and capi.gkmOpt.gamma.offset == 32
    assert capi.gkmOpt.posfile.offset == 40 and capi.gkmOpt.negfile.offset == 48
    assert capi.gkmOpt.nthreads.offset == 56 and capi.gkmOpt.verbosity.offset == 60
    assert ctypes.sizeof(capi.gkm_parameter) == 48


def test_parameter_gate_messages(product_lib):
    # gkmkern_pylib.c:38-64
    ok = dict(kernel_type=2, L=11, k=7, d=3)
    assert capi.check_parameter(**ok) is None
    assert capi.check_parameter(**dict(ok, kernel_type=6)) == "unknown kernel type"
    assert capi.check_parameter(**dict(ok, kernel_type=-1)) == "unknown kernel type"
    assert capi.check_parameter(**dict(ok, L=1, k=1, d=0)) == "L < 2"
    assert capi.check_parameter(**dict(ok, L=13)) == "L > 12"
    assert capi.check_parameter(**dict(ok, k=12)) == "k > L"
    assert capi.check_parameter(**dict(ok, d=5)) == "d > L - k"
    for L in range(2, 13):
        assert capi.check_parameter(kernel_type=4, L=L, k=max(1, L - 3), d=min(3, L - max(1, L - 3))) is None


def test_weights_bit_identical_to_reference(product_lib):
    W = np.load(GOLD + "/weights.npz")
    for key in W.files:
        t, L, k = [int(x[1:]) for x in key.split("_")]
        assert np.array_equal(capi.weights(t, L, k), W[key]), key
    for t in (3, 4, 5):  # same table as type 2 (dispatch libgkm.c:997-1019)
        assert np.array_equal(capi.weights(t, 11, 7), W["t2_L11_k7"])


@pytest.mark.parametrize("M,H", [(50, 50.0), (255, 20.0), (1, 3.0), (200, 1000.0)])
def test_positional_weights_match_oracle(M, H, product_lib):
    for nk in (1, 2, 7, 290, 291, 2037):
        a, b = capi.posweights(nk, 4, M, H)
        o = pyoracle.Oracle(4, 11, 7, 3, M, H)
        o.add("A" * (nk + 10))
        oa, ob = o.poswt(0)
        assert np.array_equal(a, oa) and np.array_equal(b, ob)
    a, b = capi.posweights(9, 2, 50, 50.0)
    assert np.all(a == 1) and np.all(b == 1)


@pytest.mark.parametrize("name", ["mix_t2_L11k7d3", "uni_t4_L10k6d3", "mix_t4_L14k8d4"])
def test_fasta_reader_and_coding_match_reference(name, product_lib):
    g, cfg, pos, neg = load_golden(name)
    with capi.Problem(**cfg) as P:
        assert P.read(pos, neg) == int(g["npos"])
        assert [P.seqlen(i) for i in range(P.n)] == list(g["lens"])
        assert np.array_equal(P.weights(), g["weights"])
        o = pyoracle.Oracle(**cfg)
        o.read_problem(pos, neg)
        for i in range(P.n):
            f, r = P.codes(i)
            of, orc = o.codes(i)
            assert np.array_equal(f, of) and np.array_equal(r, orc)


def test_fasta_quirks(tmp_path, product_lib):
    p = tmp_path / "q.fa"
    p.write_bytes(b"ignored text before the first record\n>id1 desc\r\nACGTACGTAC\r\nGTACGT\n\n>id2\nacgtnnacgtacgtac\n>id3\n" + b"A" * 3000 + b"\n>id4\nACGTACGTACGTA")
    with capi.Problem(2, 11, 7, 3) as P:
        assert P.read_fasta(str(p)) == 4
        assert [P.seqlen(i) for i in range(4)] == [16, 16, 2047, 13]
        assert [P.sid(i) for i in range(4)] == [b"id1", b"id2", b"id3", b"id4"]  # first token behind '>' (libgkm.c:1287-1292)
        assert P.add("ACGTACGTACGTACGT") == 4 and P.sid(4) is None
        assert list(P.codes(1)[0]) == [1, 2, 3, 4, 1, 1, 1, 2, 3, 4, 1, 2, 3, 4, 1, 2]  # n -> A
        with pytest.raises(capi.GkmError):
            P.read_fasta(str(tmp_path / "nope.fa"))
    ids = tmp_path / "ids.fa"
    ids.write_bytes(b">\tchr1:5-20 extra\nACGTACGTACGTAC\n> spaced\nACGTACGTACGTAC\n>tab\there\r\nACGTACGTACGTAC\n")
    with capi.Problem(2, 11, 7, 3) as P:
        assert P.read_fasta(str(ids)) == 3
        assert [P.sid(i) for i in range(3)] == [b"", b"", b"tab"]
    short = tmp_path / "s.fa"
    short.write_text(">x\nACGT\n")
    with capi.Problem(2, 11, 7, 3) as P:
        with pytest.raises(capi.GkmError):
            P.read_fasta(str(short))


def _plan(lib, row0, nrows, col0, ncols, lower, tile_rows, max_bytes):
    class Chunk(ctypes.Structure):
        _fields_ = [("row_begin", ctypes.c_int), ("row_end", ctypes.c_int), ("col_begin", ctypes.c_int),
                    ("col_end", ctypes.c_int), ("entries", ctypes.c_longlong)]
    buf = (Chunk * 4096)()
    lib.gkm_plan_chunks.argtypes = [ctypes.c_int] * 6 + [ctypes.c_longlong, ctypes.POINTER(Chunk), ctypes.c_int]
    n = lib.gkm_plan_chunks(row0, nrows, col0, ncols, lower, tile_rows, max_bytes, buf, 4096)
    assert n >= 0
    return [(c.row_begin, c.row_end, c.col_begin, c.col_end, c.entries) for c in buf[:n]]


@pytest.mark.parametrize("n,lower,budget", [(1000, 1, 1 << 20), (1000, 0, 1 << 20), (17, 1, 1 << 30), (1, 1, 64), (10000, 1, 25 << 20), (5, 0, 8)])
def test_chunk_plan_covers_exactly_once(n, lower, budget, product_lib):
    chunks = _plan(product_lib, 0, n, 0, n, lower, 16, budget)
    rows = []
    total = 0
    for rb, re_, cb, ce, ent in chunks:
        assert rb < re_ and cb == 0
        assert ce == (min(n, re_) if lower else n)
        assert (re_ - rb) % 16 == 0 or re_ == n
        rows += list(range(rb, re_))
        total += ent
    assert rows == list(range(n)), "row ranges must tile [0,n) without gaps or overlap"
    assert total == (n * (n - 1) // 2 if lower else n * n)
    if len(chunks) > 1:
        assert all((re_ - rb) * (ce - cb) * 8 <= max(budget, 16 * (ce - cb) * 8) for rb, re_, cb, ce, _ in chunks)


def test_chunk_plan_offsets(product_lib):
    chunks = _plan(product_lib, 100, 50, 20, 30, 0, 16, 1 << 12)
    assert chunks[0][0] == 100 and chunks[-1][1] == 150 and all(c[2] == 20 and c[3] == 50 for c in chunks)
    assert sum(c[4] for c in chunks) == 50 * 30


def test_set_option_keys_refuses_retired_switches(product_lib):
    """A/B switches whose measurements are settled are no longer options; the ones tests and callers use are still taken"""
    for key, value in (("diag_flavor", "2"), ("tile_rows", "4"), ("pack", "host")):
        with pytest.raises(capi.GkmError, match="unknown option " + key):
            capi.set_option(key, value)
    try:
        for key, value in (("kernel", "diag"), ("index_cols", "128"), ("index_split", "greedy"), ("index_wide", "1")):
            capi.set_option(key, value)
    finally:
        for key, value in (("kernel", "auto"), ("index_cols", "0"), ("index_split", "auto"), ("index_wide", "0")):
            capi.set_option(key, value)


def test_compute_fails_loudly_without_gpu(product_lib):
    if capi.device_count() > 0:
        pytest.skip("a GPU is visible")
    with capi.Problem(2, 11, 7, 3) as P:
        P.add_many(random_seqs(4, 50, 1))
        with pytest.raises(capi.GkmError, match="no CPU fallback"):
            P.kernel_lower()
        with pytest.raises(capi.GkmError):
            P.sqnorm()
    ret, kmat, _, _ = capi.main_pywrapper(GOLD + "/uni_pos.fa", GOLD + "/uni_neg.fa", nmax=20)
    assert ret == 1 and not kmat.any()


def test_product_never_touches_the_oracle():
    """the oracle is test infrastructure: nothing under gkmqc_b200/ may import, link or open it"""
    bad = []
    for dirpath, _, files in os.walk(os.path.join(ROOT, "gkmqc_b200")):
        for f in files:
            if f.endswith((".py", ".c", ".cu", ".cuh", ".h")) or f == "Makefile":
                text = open(os.path.join(dirpath, f), errors="replace").read()
                if re.search(r"pyoracle|gkm_oracle|oracle/|gkmo_|gkmref_", text):
                    bad.append(os.path.join(dirpath, f))
    assert not bad, bad


def test_svm_task_preparation_follows_libsvm_grouping():
    """host logic of the f4 consumer: per fit the training ids are grouped label 0 first (libsvm's svm_group_classes
    with sklearn's label sort) and that class is the sub-problem's +1"""
    import numpy as np
    import pytest
    from gkmqc_b200 import capi
    y = np.array([1, 0, 1, 0, 0, 1, 1, 0])
    splits = [(np.array([6, 1, 0, 3, 5]), np.array([2, 4, 7])), (np.array([7, 2, 4, 5]), np.array([0]))]
    tasks, tr, ty, te = capi.svm_prepare_tasks(y, splits)
    assert (tasks[0].train_off, tasks[0].test_off, tasks[0].ntrain, tasks[0].ntest) == (0, 0, 5, 3)
    assert (tasks[1].train_off, tasks[1].test_off, tasks[1].ntrain, tasks[1].ntest) == (5, 3, 4, 1)
    assert tr.tolist() == [1, 3, 6, 0, 5, 7, 4, 2, 5] and ty.tolist() == [1, 1, -1, -1, -1, 1, 1, -1, -1]
    assert te.tolist() == [2, 4, 7, 0]
    with pytest.raises(ValueError):
        capi.svm_prepare_tasks(y, [(np.array([0, 2]), np.array([1]))])


def test_copy_threads_policy(monkeypatch):
    """the reference's nthreads (default 1 in bin/gkmqc.py) is only a lower bound on the copy-out threads: the library
    takes the cores of its affinity mask (no fixed cap: the 8-GPU box has 32), shared among the ranks of a
    one-process-per-GPU run; GKM_COPY_THREADS overrides (gkm_compute.cu:gkm_copy_threads_shared)"""
    import ctypes
    lib = capi.load()
    for f in (lib.gkm_copy_threads, lib.gkm_copy_threads_shared):
        f.restype = ctypes.c_int
    lib.gkm_copy_threads.argtypes = [ctypes.c_int]
    lib.gkm_copy_threads_shared.argtypes = [ctypes.c_int, ctypes.c_int]
    monkeypatch.delenv("GKM_COPY_THREADS", raising=False)
    avail = min(64, len(os.sched_getaffinity(0)))
    assert lib.gkm_copy_threads(1) == avail
    assert lib.gkm_copy_threads(avail + 3) == min(64, avail + 3)
    assert lib.gkm_copy_threads(1000) == 64
    assert lib.gkm_copy_threads_shared(1, 2) == max(1, avail // 2)
    assert lib.gkm_copy_threads_shared(1, 8) == max(1, avail // 8)
    assert lib.gkm_copy_threads_shared(3, 10 ** 6) == 3          # never below what the caller asked for
    monkeypatch.setenv("GKM_COPY_THREADS", "5")
    assert lib.gkm_copy_threads(1) == 5 and lib.gkm_copy_threads_shared(32, 8) == 5
    # under taskset -c 0 the affinity mask is what counts, not the machine
    import subprocess, sys
    code = ("import ctypes,sys; sys.path.insert(0, %r); from gkmqc_b200 import capi; l = capi.load(); "
            "l.gkm_copy_threads.restype = ctypes.c_int; print(l.gkm_copy_threads(1))" % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    env = {k: v for k, v in os.environ.items() if k != "GKM_COPY_THREADS"}
    cpu = sorted(os.sched_getaffinity(0))[0]
    out = subprocess.run(["taskset", "-c", str(cpu), sys.executable, "-c", code], capture_output=True, text=True, env=env)
    if out.returncode == 0:   # taskset may be missing in a minimal image
        assert out.stdout.strip() == "1"


def test_two_file_read_equals_two_sequential_reads(tmp_path):
    """gkmb200_problem_read parses the negatives on a helper thread and appends them: ids, order and codes must be
    those of two sequential reads (positives 0..n_pos-1, negatives behind: libgkm.c:1316-1333)"""
    seqs = random_seqs(301, 90, seed=5, ragged=True)
    seqs = [s if len(s) >= 11 else s + "ACGTACGTACG" for s in seqs]
    pos, neg = tmp_path / "p.fa", tmp_path / "n.fa"
    pos.write_text("".join(">p%d\n%s\n" % (i, s) for i, s in enumerate(seqs[:120])))
    neg.write_text("".join(">n%d\r\n%s\r\n" % (i, s.lower()) for i, s in enumerate(seqs[120:])))
    a = capi.Problem(2, 11, 7, 3)
    b = capi.Problem(2, 11, 7, 3)
    try:
        assert a.read(str(pos), str(neg)) == 120
        assert b.read_fasta(str(pos)) == 120 and b.read_fasta(str(neg)) == 181
        assert a.n == b.n == 301
        for i in (0, 1, 119, 120, 121, 200, 300):
            assert a.seqlen(i) == b.seqlen(i) == len(seqs[i])
            fa, ra = a.codes(i)
            fb, rb = b.codes(i)
            assert np.array_equal(fa, fb) and np.array_equal(ra, rb)
        with pytest.raises(capi.GkmError):
            capi.Problem(2, 11, 7, 3).read(str(pos), str(tmp_path / "missing.fa"))
    finally:
        a.close()
        b.close()


def test_base_coding_of_every_byte_value():
    """A,C,G,T in either case -> 1..4 (gkm_data.seq codes); every other byte counts as A like the reference does
    (libgkm.c:864-875).  All 256 byte values, at every position of the 16-byte vector path and of the scalar tail."""
    lib = capi.load()
    lib.gkmb200_set_verbosity(0)   # the warnings about the 248 other bytes are not the point here
    want = {ord("A"): 1, ord("a"): 1, ord("C"): 2, ord("c"): 2, ord("G"): 3, ord("g"): 3, ord("T"): 4, ord("t"): 4}
    P = capi.Problem(2, 11, 7, 3)
    try:
        for shift in (0, 5, 16):
            raw = bytes((b + shift) & 0xFF for b in range(256)) + bytes(range(37))   # 293 bytes: 18 vectors + 5 tail bytes
            i = P.add(raw)
            fwd, rc = P.codes(i)
            exp = np.array([want.get(b, 1) for b in raw], np.uint8)
            assert np.array_equal(fwd, exp)
            assert np.array_equal(rc, (5 - exp)[::-1])
    finally:
        P.close()
        lib.gkmb200_set_verbosity(2)
