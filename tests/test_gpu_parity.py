"""GPU tier (-m gpu): the CUDA path, called through the C-ABI of gkmkern_pylib.so, against
(1) golden vectors from the unmodified reference, (2) the oracle on seeded inputs, and
(3) size-independent properties at BASELINE.json sizes.

Bars: integer mismatch histograms bit-exact; kernel values bit-identical for the non-RBF
kernel types and within 1e-9 relative (north_star) for the RBF types (device exp())."""
import os

import numpy as np
import pytest

import pyoracle
from conftest import GOLD, golden_names, load_golden, random_seqs, write_fasta
from gkmqc_b200 import capi

pytestmark = pytest.mark.gpu

RTOL_RBF = 1e-9


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    capi.load()
    if capi.device_count() < 1:
        pytest.fail("no B200 visible; the product has no CPU fallback")


@pytest.fixture(params=["diag", "lmer", "mma", "index"])
def variant(request):
    capi.set_option("kernel", request.param)
    yield request.param
    capi.set_option("kernel", "auto")


def check_kmat(K, Kref, kernel_type):
    if kernel_type in (3, 5):
        np.testing.assert_allclose(K, Kref, rtol=RTOL_RBF, atol=0)
    else:
        assert np.array_equal(K, Kref), "max abs diff %g" % np.max(np.abs(K - Kref))


@pytest.mark.parametrize("name", golden_names())
def test_golden_histograms_and_kernel(name, variant):
    g, cfg, pos, neg = load_golden(name)
    with capi.Problem(**cfg) as P:
        assert P.read(pos, neg) == int(g["npos"])
        n = P.n
        assert np.array_equal(P.weights(), g["weights"])
        assert np.array_equal(P.sqnorm(), g["sqnorm"]), "sqnorm (device diagonal)"
        H = P.hist_block(0, n, 0, n, lower=True)
        assert np.array_equal(H, g["hist"]), "integer mismatch histograms"
        K = P.kernel_lower()
        check_kmat(K, g["kmat"], cfg["kernel_type"])
        st = P.stats()
        assert st["launches"] > 0 and st["kernel_variant"] == {"lmer": 1, "diag": 2, "mma": 3, "index": 4}[variant]


@pytest.mark.parametrize("name", [n for n in golden_names() if int(n.split("_L")[1].split("k")[0]) <= 12])
def test_pywrapper_is_drop_in(name):
    """gkm_main_pywrapper exactly as scripts/gkmsvm.py:75-88 calls it: padded kmat, row pointers, int[2]"""
    g, cfg, pos, neg = load_golden(name)
    n = len(g["lens"])
    ret, kmat, npos, nneg = capi.main_pywrapper(pos, neg, nthreads=3, verbosity=0, nmax=n + 5, **cfg)
    assert ret == 0, capi.last_error()
    assert (npos, nneg) == (int(g["npos"]), n - int(g["npos"]))
    check_kmat(kmat[:n, :n], g["kmat"], cfg["kernel_type"])
    assert not kmat[n:].any() and not kmat[:, n:].any(), "wrote outside rows/cols 0..N-1"
    assert not np.triu(kmat[:n, :n], 1).any(), "upper triangle must stay untouched"


def test_pywrapper_parameter_gate_and_errors(tmp_path):
    g, cfg, pos, neg = load_golden("uni_t2_L11k7d3")
    for bad in (dict(L=13, k=7, d=3), dict(L=1, k=1, d=0), dict(L=10, k=11, d=0), dict(L=10, k=8, d=3), dict(kernel_type=6)):
        c = dict(cfg)
        c.update(bad)
        ret, kmat, _, _ = capi.main_pywrapper(pos, neg, nmax=24, **c)
        assert ret == 1 and not kmat.any()
    ret, kmat, _, _ = capi.main_pywrapper(str(tmp_path / "missing.fa"), neg, nmax=24, **cfg)
    assert ret == 1 and not kmat.any()


def test_long_L_opt_in():
    g, cfg, pos, neg = load_golden("mix_t2_L13k7d4")
    n = len(g["lens"])
    ret, _, _, _ = capi.main_pywrapper(pos, neg, nmax=n, **cfg)
    assert ret == 1  # reference gate: L <= 12 (gkmkern_pylib.c:54)
    capi.set_option("max_L", 16)
    try:
        ret, kmat, _, _ = capi.main_pywrapper(pos, neg, nmax=n, **cfg)
        assert ret == 0
        assert np.array_equal(kmat, g["kmat"])
    finally:
        capi.set_option("max_L", 12)


@pytest.mark.parametrize("kernel_type,L,k,d,length,ragged", [
    (2, 11, 7, 3, 300, False), (4, 10, 6, 3, 300, False), (2, 11, 7, 3, 600, True), (4, 12, 8, 4, 257, True),
    (0, 8, 4, 4, 64, True), (5, 14, 8, 4, 320, False), (2, 16, 12, 4, 200, True), (1, 6, 3, 3, 96, False),
])
def test_seeded_against_oracle(kernel_type, L, k, d, length, ragged, variant):
    n = 96 if length <= 320 else 40
    seqs = random_seqs(n, length, seed=7 * L + d + kernel_type, ragged=ragged)
    seqs[3] = seqs[2]                       # duplicate
    seqs[5] = seqs[4][: max(L, length // 2)]  # prefix
    o = pyoracle.Oracle(kernel_type, L, k, d, 50, 50.0, 0.7)
    with capi.Problem(kernel_type, L, k, d, 50, 50.0, 0.7) as P:
        for s in seqs:
            o.add(s)
            P.add(s)
        Ko, Ho = o.matrix_lower()
        assert np.array_equal(P.sqnorm(), o.sqnorm())
        assert np.array_equal(P.hist_block(0, n, 0, n, lower=True), Ho)
        check_kmat(P.kernel_lower(), Ko, kernel_type)
        # rectangular "test x SV" shape: SVs at ids [0,nsv), tests after them (SURVEY.md 3.4)
        nsv = n // 3
        Kr, Hr = o.rect(np.arange(nsv, n), nsv)
        assert np.array_equal(P.hist_block(nsv, n - nsv, 0, nsv), Hr)
        check_kmat(P.kernel_block(nsv, n - nsv, 0, nsv), Kr, kernel_type)
        # fused decision values against the dense block
        alpha = np.random.default_rng(1).standard_normal(nsv)
        dv = P.decision_values(nsv, n - nsv, 0, nsv, alpha, bias=0.25)
        np.testing.assert_allclose(dv, Kr @ alpha + 0.25, rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("kernel_type,L,k,d,cols,wide", [(2, 11, 7, 3, 32, 0), (4, 10, 6, 3, 64, 0), (2, 8, 4, 4, 32, 0), (4, 6, 5, 1, 32, 0),
                                                          (0, 9, 9, 0, 32, 0), (2, 8, 4, 4, 32, 1), (2, 11, 7, 3, 0, 1), (1, 7, 4, 3, 0, 0),
                                                          # nearly every slot holds a LONG list (whole-warp walks, and more than 32 of
                                                          # them per probe iteration: the long queue overflows into per-lane walks)
                                                          (4, 5, 4, 1, 0, 0), (2, 4, 3, 1, 0, 0), (2, 4, 3, 1, 64, 0), (2, 5, 3, 2, 0, 1),
                                                          # weighted types: compact 20-bit postings (wide = 0) and the 16-byte slots (1)
                                                          (4, 5, 4, 1, 0, 1), (4, 10, 6, 3, 64, 1), (5, 11, 7, 3, 0, 0), (5, 11, 7, 3, 0, 1), (4, 7, 5, 2, 32, 0)])
def test_index_column_blocks(kernel_type, L, k, d, cols, wide):
    """index variant with the columns cut into several index blocks (what a problem larger than one
    shared-memory histogram row gets), long posting lists (short L, repeats) and a column window that
    starts inside a block"""
    n = 150
    seqs = random_seqs(n, 120, seed=11 * L + d + kernel_type, ragged=True)
    seqs = [s if len(s) >= L else s + "ACGT" * 4 for s in seqs]
    seqs[3] = seqs[2]
    seqs[70] = "A" * 100
    seqs[71] = "ACAC" * 25
    seqs[140] = seqs[2]
    o = pyoracle.Oracle(kernel_type, L, k, d, 50, 50.0, 0.7)
    capi.set_option("kernel", "index")
    capi.set_option("index_cols", str(cols))
    capi.set_option("index_wide", str(wide))  # compact 8-byte slots (0: C16 / W20 by kernel type) or the 16-byte ones (1)
    try:
        with capi.Problem(kernel_type, L, k, d, 50, 50.0, 0.7) as P:
            for s in seqs:
                o.add(s)
                P.add(s)
            Ko, Ho = o.matrix_lower()
            assert np.array_equal(P.hist_block(0, n, 0, n, lower=True), Ho)
            assert P.stats()["kernel_variant"] == 4
            check_kmat(P.kernel_lower(), Ko, kernel_type)
            Kr, Hr = o.rect(np.arange(100, n), 100)
            assert np.array_equal(P.hist_block(100, n - 100, 40, 60), Hr[:, 40:100])
            check_kmat(P.kernel_block(100, n - 100, 40, 60), Kr[:, 40:100], kernel_type)
            alpha = np.random.default_rng(2).standard_normal(60)
            dv = P.decision_values(100, n - 100, 40, 60, alpha, bias=-0.5)
            np.testing.assert_allclose(dv, Kr[:, 40:100] @ alpha - 0.5, rtol=1e-9, atol=1e-12)
    finally:
        capi.set_option("index_cols", "0")
        capi.set_option("index_wide", "0")
        capi.set_option("kernel", "auto")


@pytest.mark.parametrize("kernel_type", [2, 4])
def test_nonuniform_index_vs_bitsliced(kernel_type):
    """SURVEY.md 8(d): genome-like inputs (poly-A tracts, dinucleotide repeats, a repeat family, exact duplicates,
    AT-rich composition) put thousands of postings into a few slots.  The index kernel (neighbour enumeration, long
    lists walked by whole warps) and the bit-sliced kernel (dense diagonals) are independent constructions: their
    integer histograms and kernel doubles must agree bit for bit."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("nonuniform", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "nonuniform.py"))
    nu = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(nu)
    n, L, k, d = 1500, 11, 7, 3
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    try:
        for name, x in nu.workloads(n, seed=99).items():
            if name in ("uniform", "at_rich"):
                continue
            seqs = [acgt[r].tobytes().decode() for r in x]
            out = {}
            for v in ("index", "diag"):
                capi.set_option("kernel", v)
                with capi.Problem(kernel_type, L, k, d, 50, 50.0, 1.0) as P:
                    P.add_many(seqs)
                    out[v] = (P.hist_block(n - 200, 200, 0, n - 200), P.kernel_block(n - 200, 200, 0, n - 200), P.stats()["kernel_variant"])
            assert out["index"][2] == 4 and out["diag"][2] == 2
            assert np.array_equal(out["index"][0], out["diag"][0]), name
            assert np.array_equal(out["index"][1], out["diag"][1]), name
    finally:
        capi.set_option("kernel", "auto")


def test_auto_leaves_the_index_on_low_complexity_input():
    """kernel = auto looks at the posting lists the index build produced: half of the sequences being poly-A makes the
    exact-match term of the index kernel larger than the whole bit-sliced pass, so auto runs the bit-sliced kernel --
    and both give the same integers"""
    n, L, k, d = 3000, 11, 7, 3
    rng = np.random.default_rng(8)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    seqs = [acgt[r].tobytes().decode() for r in rng.integers(0, 4, size=(n, 300))]
    for i in range(0, n, 2):
        seqs[i] = "A" * 300 if (i // 2) % 2 == 0 else "T" * 150 + "A" * 150
    out = {}
    try:
        for v in ("auto", "index"):
            capi.set_option("kernel", v)
            with capi.Problem(2, L, k, d) as P:
                P.add_many(seqs)
                K = P.kernel_lower()
                out[v] = (K[n - 40:, :], P.stats()["kernel_variant"])
    finally:
        capi.set_option("kernel", "auto")
    assert out["index"][1] == 4 and out["auto"][1] == 2
    assert np.array_equal(out["auto"][0], out["index"][0])


def test_sqnorm_beyond_one_launch():
    """sqnorm is the diagonal of the kernel, computed by one column of CTAs per launch of at most 131 070 rows: more
    rows than that take several launches.  Copies of the same sequences on both sides of the boundary must get the
    same value, and the values must be the oracle's."""
    base = random_seqs(300, 60, seed=77, ragged=True)
    base = [s if len(s) >= 11 else s + "ACGTACGTACG" for s in base]
    reps = 131070 // len(base) + 2
    seqs = (base * reps)[:131070 + 450]
    o = pyoracle.Oracle(4, 11, 7, 3)
    for s in base:
        o.add(s)
    want = o.sqnorm() if hasattr(o, "sqnorm") else None
    with capi.Problem(4, 11, 7, 3) as P:
        P.add_many(seqs)
        sq = P.sqnorm()
    assert len(sq) == len(seqs)
    per = np.asarray(sq[:len(base)])
    for start in range(0, len(seqs), len(base)):
        part = np.asarray(sq[start:start + len(base)])
        assert np.array_equal(part, per[:len(part)]), start
    if want is not None:
        assert np.array_equal(per, np.asarray(want))


def test_edge_cases(variant):
    L, k, d = 11, 7, 3
    seqs = ["ACGTACGTACG",               # exactly one L-mer
            "A" * 40, "T" * 40,           # homopolymers, reverse complements of each other
            "ACGTTGCAACGTTGCAACGT",       # short
            random_seqs(1, 2047, 5)[0],   # maximum length (2047 bases, libgkm.c:1294-1299)
            random_seqs(1, 33, 6)[0], random_seqs(1, 32, 7)[0], random_seqs(1, 31, 8)[0], random_seqs(1, 65, 9)[0]]
    o = pyoracle.Oracle(4, L, k, d)
    with capi.Problem(4, L, k, d) as P:
        for s in seqs:
            o.add(s)
            P.add(s)
        n = len(seqs)
        Ko, Ho = o.matrix_lower()
        assert np.array_equal(P.hist_block(0, n, 0, n, lower=True), Ho)
        assert np.array_equal(P.kernel_lower(), Ko)
        # single sequence problem and empty blocks
        assert P.kernel_block(0, 0, 0, 0).shape == (0, 0)
    with capi.Problem(2, L, k, d) as P1:
        P1.add(seqs[4])
        assert np.array_equal(P1.kernel_lower(), [[1.0]])
    with capi.Problem(2, L, k, d) as P2:
        with pytest.raises(capi.GkmError):
            P2.add("ACGT")  # shorter than L


def test_fasta_without_trailing_newline(tmp_path):
    seqs = random_seqs(5, 80, 11)
    p = tmp_path / "p.fa"
    p.write_text("".join(">s%d x\n%s\n" % (i, s) for i, s in enumerate(seqs[:3])))
    q = tmp_path / "q.fa"
    q.write_text(">a\n" + seqs[3] + "\n>b\n" + seqs[4])  # the reference double-frees on this (libgkm.c:1207-1225)
    ret, kmat, npos, nneg = capi.main_pywrapper(str(p), str(q), nmax=5)
    assert ret == 0 and (npos, nneg) == (3, 2)
    o = pyoracle.Oracle()
    for s in seqs:
        o.add(s)
    assert np.array_equal(kmat, o.matrix_lower(False)[0])


def test_reference_abi_functions(tmp_path):
    """the lower-level libgkm.h surface: init / read_problems / build_tree / batch_all / swap / destroy"""
    import ctypes
    lib = capi.load()
    g, cfg, pos, neg = load_golden("mix_t4_L11k7d3")
    n = len(g["lens"])

    class svm_problem(ctypes.Structure):
        _fields_ = [("l", ctypes.c_int), ("y", capi.c_dbl_p), ("x", ctypes.POINTER(ctypes.c_void_p))]

    lib.gkmkernel_init.restype = ctypes.c_void_p
    lib.gkmkernel_init.argtypes = [ctypes.POINTER(capi.gkm_parameter)]
    lib.gkmkernel_read_problems.argtypes = [ctypes.c_void_p, ctypes.POINTER(svm_problem), ctypes.c_char_p, ctypes.c_char_p]
    lib.gkmkernel_build_tree.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_int]
    lib.gkmkernel_kernelfunc_batch_all.restype = capi.c_dbl_p
    lib.gkmkernel_kernelfunc_batch_all.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, capi.c_dbl_p]
    lib.gkmkernel_swap_index.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    lib.gkmkernel_update_index.argtypes = [ctypes.c_void_p]
    lib.gkmkernel_delete_object.argtypes = [ctypes.c_void_p]
    lib.gkmkernel_destroy.argtypes = [ctypes.c_void_p]
    lib.gkmkernel_new_object.restype = ctypes.c_void_p
    lib.gkmkernel_new_object.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int]

    param = capi.make_param(**cfg)
    kern = lib.gkmkernel_init(ctypes.byref(param))
    assert kern
    prob = svm_problem()
    assert lib.gkmkernel_read_problems(kern, ctypes.byref(prob), os.fsencode(pos), os.fsencode(neg)) == int(g["npos"])
    assert prob.l == n
    sq = np.array([ctypes.cast(prob.x[i] + 80, capi.c_dbl_p)[0] for i in range(n)])  # gkm_data.sqnorm @80
    assert np.array_equal(sq, g["sqnorm"])
    lib.gkmkernel_build_tree(kern, prob.x, n)
    res = np.zeros(n)
    for a in (1, 7, n - 1):
        lib.gkmkernel_kernelfunc_batch_all(kern, a, 0, a, res.ctypes.data_as(capi.c_dbl_p))
        assert np.array_equal(res[:a], g["kmat"][a, :a])
    lib.gkmkernel_kernelfunc_batch_all(kern, n - 1, 3, 9, res.ctypes.data_as(capi.c_dbl_p))
    assert np.array_equal(res[:6], g["kmat"][n - 1, 3:9])
    # permutation bookkeeping (libgkm.c:1071-1109): after swap+update id 2 and id 5 trade places
    lib.gkmkernel_swap_index(kern, 2, 5)
    lib.gkmkernel_update_index(kern)
    lib.gkmkernel_kernelfunc_batch_all(kern, 7, 0, 7, res.ctypes.data_as(capi.c_dbl_p))
    perm = list(range(n))
    perm[2], perm[5] = perm[5], perm[2]
    full = np.maximum(g["kmat"], g["kmat"].T)
    assert np.array_equal(res[:7], full[7, perm[:7]])
    # new_object fills sqnorm from the device
    obj = lib.gkmkernel_new_object(kern, b"ACGTTGCAACGTTGCAACGTAAA", b"x", 99)
    assert obj
    o = pyoracle.Oracle(**cfg)
    o.add("ACGTTGCAACGTTGCAACGTAAA")
    assert ctypes.cast(obj + 80, capi.c_dbl_p)[0] == o.sqnorm()[0]
    lib.gkmkernel_delete_object(obj)
    for i in range(n):
        lib.gkmkernel_delete_object(prob.x[i])
    lib.gkmkernel_destroy(kern)


def test_properties_at_scale():
    """config-1 size (1 000 x 300 bp): things that must hold whatever the inputs are"""
    n, L, k, d = 1000, 11, 7, 3
    seqs = random_seqs(n, 300, seed=1234)
    comp = str.maketrans("ACGT", "TGCA")
    seqs[10] = seqs[9].translate(comp)[::-1]  # reverse complement of seq 9
    with capi.Problem(2, L, k, d) as P:
        P.add_many(seqs)
        K = P.kernel_lower()
        assert np.all(np.diag(K) == 1.0) and not np.triu(K, 1).any()
        low = K[np.tril_indices(n, -1)]
        assert np.all(np.isfinite(low)) and low.min() >= 0 and low.max() <= 1.0 + 1e-12
        assert K[10, 9] == 1.0  # K(x, revcomp(x)) = 1: both strands of the target are scanned
        # symmetry: the block above the diagonal computed the other way round
        U = P.kernel_block(0, 200, 200, 300)
        assert np.array_equal(U, K[200:500, 0:200].T)
        H = P.hist_block(500, 40, 0, 500)
        Hd4 = None
        with capi.Problem(2, L, 7, 4) as P4:  # H for d=3 is a prefix of H for d=4; k never touches H
            P4.add_many(seqs[:540])
            Hd4 = P4.hist_block(500, 40, 0, 500)
        assert np.array_equal(H, Hd4[..., :4])
        # checksum against the oracle on a stated subsample of rows
        o = pyoracle.Oracle(2, L, k, d)
        for s in seqs:
            o.add(s)
        rows = np.array([1, 17, 333, 999])
        for r in rows:
            Kr, Hr = o.rect(np.array([r]), int(r))
            assert np.array_equal(Kr[0], K[r, :r])


def test_multi_gpu_in_one_process_if_available():
    """all GPUs of the box in one process against one GPU: the kernel matrix (index forced: every GPU builds its own
    index) and fused decision values (one slice of the test rows per GPU)"""
    ndev = capi.device_count()
    if ndev < 2:
        pytest.skip("single GPU box")
    lib = capi.load()
    ids = (capi.ctypes.c_int * ndev)(*range(ndev))
    seqs = random_seqs(700, 300, seed=77)
    alpha = np.random.default_rng(3).standard_normal(500)
    try:
        for kernel in ("auto", "index"):
            capi.set_option("kernel", kernel)
            assert lib.gkmb200_set_devices(ids, ndev) == 0
            with capi.Problem(2, 11, 7, 3) as P:
                P.add_many(seqs)
                K = P.kernel_lower()
                st = P.stats()
                dv = P.decision_values(500, 200, 0, 500, alpha, bias=0.25)
            assert st["devices"] == ndev
            assert kernel == "auto" or st["kernel_variant"] == 4
            np.testing.assert_allclose(dv, K[500:, :500] @ alpha + 0.25, rtol=1e-9, atol=1e-12)
            assert lib.gkmb200_set_devices(ids, 1) == 0
            with capi.Problem(2, 11, 7, 3) as P:
                P.add_many(seqs)
                assert np.array_equal(P.kernel_lower(), K)
                np.testing.assert_allclose(P.decision_values(500, 200, 0, 500, alpha, bias=0.25), dv, rtol=1e-9, atol=1e-12)
    finally:
        capi.set_option("kernel", "auto")
        lib.gkmb200_set_devices(ids, 1)


def test_sharded_ranks_cover_the_matrix():
    """two 'ranks' in one process: each computes only the chunks it owns; together = the full triangle"""
    seqs = random_seqs(900, 300, seed=5)
    parts = []
    for rank in range(2):
        with capi.Problem(2, 11, 7, 3) as P:
            P.add_many(seqs)
            P.set_shard(rank, 2)
            parts.append(P.kernel_lower())
    with capi.Problem(2, 11, 7, 3) as P:
        P.add_many(seqs)
        full = P.kernel_lower()
    low = np.tril_indices(900, -1)
    a, b = parts[0][low], parts[1][low]
    assert not np.any((a != 0) & (b != 0)), "shards overlap"
    assert np.array_equal(a + b, full[low])


def test_driver_mirror_returns_what_gkmsvm_would():
    """computeGkmKernel(args_gkm) with gkmQC's default parameters (bin/gkmqc.py:169-199): wgkm, L=10 k=6 d=3"""
    from gkmqc_b200 import driver
    g, cfg, pos, neg = load_golden("uni_t4_L10k6d3")
    kmat, npos, nneg = driver.computeGkmKernel([4, 10, 6, 3, 50, 50.0, 1.0, pos, neg, 4, 0], max_seqs=64)
    n = len(g["lens"])
    assert (npos, nneg) == (int(g["npos"]), n - int(g["npos"])) and kmat.shape == (n, n)
    assert np.array_equal(kmat, np.maximum(g["kmat"], g["kmat"].T))


@pytest.mark.parametrize("kernel_type", [2, 4])
def test_full_size_index_against_bitsliced_and_reference(kernel_type, tmp_path):
    """BASELINE configs[1] at full size (5k + 5k x 300 bp): the build that produces the headline number (compact slots,
    two CTAs per SM) against the bit-sliced kernel on the WHOLE matrix, and against the unmodified reference on 32 rows
    (doubles and integer histograms) where oracle/_ref exists"""
    import bench
    n = 10000
    arr = bench.synth(n)
    pos, neg = str(tmp_path / "p.fa"), str(tmp_path / "n.fa")
    bench.write_fasta(pos, arr[: n // 2], 0)
    bench.write_fasta(neg, arr[n // 2:], n // 2)
    mats = {}
    for v in ("index", "diag"):
        capi.set_option("kernel", v)
        try:
            with capi.Problem(kernel_type, 11, 7, 3) as P:
                P.read(pos, neg)
                mats[v] = P.kernel_lower()
                assert P.stats()["kernel_variant"] == {"diag": 2, "index": 4}[v]
                if v == "index":
                    rows = bench.parity_rows(n, P.index_layout()[1] or n, P.index_layout()[0], want=32)[:40]
                    hist = {int(r): P.hist_block(int(r), 1, 0, int(r))[0] for r in rows}
        finally:
            capi.set_option("kernel", "auto")
    assert np.array_equal(mats["index"], mats["diag"]), "index and bit-sliced kernels differ somewhere in the 10k x 10k matrix"
    K = mats["index"]
    assert np.all(np.diag(K) == 1.0) and not np.triu(K, 1).any()
    if not pyoracle.have_ref():
        pytest.skip("oracle/_ref not built here: the cross-variant half of the test ran")
    h = pyoracle.RefHook(pos, neg, kernel_type, 11, 7, 3)
    try:
        Kr, Hr, _ = h.rows_values(rows, os.cpu_count() or 1)
        for i, r in enumerate(rows):
            assert np.array_equal(K[r, :r], Kr[i, :r]), "row %d differs from the reference" % r
            assert np.array_equal(hist[int(r)], Hr[i, :, :r].T), "histograms of row %d differ from the reference" % r
    finally:
        h.close()


@pytest.mark.parametrize("kernel_type", [2, 4])
def test_full_size_index_against_stored_rows(kernel_type, tmp_path):
    """the problem of test_full_size_index_against_bitsliced_and_reference, without a reference build: the index kernel's
    matrix and integer histograms at the stored sample of tests/golden/full10k_rows_kt*.npz (oracle/gen_golden.py
    --full-size: rows on both sides of the index column blocks and of the chunk boundaries, seeded columns below them)"""
    import bench
    stored = np.load(os.path.join(GOLD, "full10k_rows_kt%d.npz" % kernel_type))
    n = 10000
    arr = bench.synth(n)
    pos, neg = str(tmp_path / "p.fa"), str(tmp_path / "n.fa")
    bench.write_fasta(pos, arr[: n // 2], 0)
    bench.write_fasta(neg, arr[n // 2:], n // 2)
    capi.set_option("kernel", "index")
    try:
        with capi.Problem(kernel_type, 11, 7, 3) as P:
            P.read(pos, neg)
            K = P.kernel_lower()
            assert P.stats()["kernel_variant"] == 4
            hist = {int(r): P.hist_block(int(r), 1, 0, int(r))[0] for r in np.unique(stored["row"])}
    finally:
        capi.set_option("kernel", "auto")
    rows, cols = stored["row"], stored["col"]
    assert np.array_equal(K[rows, cols], stored["kmat"]), "kernel values differ from the stored ones"
    assert np.array_equal(np.stack([hist[int(r)][c] for r, c in zip(rows, cols)]), stored["hist"]), "histograms differ from the stored ones"


def test_one_core_affinity_still_correct(tmp_path):
    """a caller pinned to one core (slurm job that asked for one): the copy-out runs on that core alone and the
    matrix is the same"""
    import subprocess
    import sys
    g, cfg, pos, neg = load_golden("uni_t2_L11k7d3")
    out = tmp_path / "k.npy"
    code = ("import sys, numpy as np; sys.path.insert(0, %r); from gkmqc_b200 import capi; "
            "ret, k, a, b = capi.main_pywrapper(%r, %r, kernel_type=2, L=11, k=7, d=3, nthreads=1, nmax=64); "
            "st = capi.gkmb200_stats(); capi.load().gkmb200_get_stats(None, capi.ctypes.byref(st)); "
            "assert ret == 0 and st.copy_threads == 1, (ret, st.copy_threads); np.save(%r, k)"
            % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), pos, neg, str(out)))
    env = {k: v for k, v in os.environ.items() if k != "GKM_COPY_THREADS"}
    cpu = sorted(os.sched_getaffinity(0))[0]
    r = subprocess.run(["taskset", "-c", str(cpu), sys.executable, "-c", code], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    n = len(g["lens"])
    assert np.array_equal(np.load(out)[:n, :n], g["kmat"])


@pytest.mark.parametrize("kernel_type,L,k,d", [(2, 11, 7, 3), (4, 10, 6, 3), (2, 6, 4, 2)])
def test_index_split_layouts(kernel_type, L, k, d):
    """the two ways of cutting a lower triangle's columns into index blocks (option index_split: equal shares / full blocks
    first, which is what a lower triangle gets by default) give the oracle's integers and doubles, from different layouts"""
    n = 150
    seqs = random_seqs(n, 120, seed=5 * L + d + kernel_type, ragged=True)
    seqs = [s if len(s) >= L else s + "ACGT" * 4 for s in seqs]
    seqs[127] = seqs[2]
    seqs[128] = seqs[3]
    o = pyoracle.Oracle(kernel_type, L, k, d, 50, 50.0, 0.7)
    for s in seqs:
        o.add(s)
    Ko, Ho = o.matrix_lower()
    capi.set_option("kernel", "index")
    capi.set_option("index_cols", "128")
    layouts = {}
    try:
        for split in ("equal", "greedy", "auto"):
            capi.set_option("index_split", split)
            with capi.Problem(kernel_type, L, k, d, 50, 50.0, 0.7) as P:
                P.add_many(seqs)
                assert np.array_equal(P.hist_block(0, n, 0, n, lower=True), Ho), split
                layouts[split] = P.index_layout()
                check_kmat(P.kernel_lower(), Ko, kernel_type)
                assert P.stats()["kernel_variant"] == 4
    finally:
        capi.set_option("index_cols", "0")
        capi.set_option("index_split", "auto")
        capi.set_option("kernel", "auto")
    assert layouts["equal"][:2] == (2, 96) and layouts["greedy"][:2] == (2, 128) and layouts["auto"] == layouts["greedy"]


@pytest.mark.parametrize("kernel_type,split", [(2, "equal"), (4, "equal"), (2, "greedy"), (4, "greedy")])
def test_two_column_blocks_at_20k_index_against_bitsliced(kernel_type, split):
    """20 000 x 300 bp with at most 16 384 columns per index block: two column blocks, cut into equal shares or full block
    first (rows of the second block probe both); rows on both sides of the block boundary, the first and the last rows:
    integers and doubles against the bit-sliced kernel"""
    import bench
    n = 20000
    arr = bench.synth(n, seed=77)
    got = {}
    for v in ("index", "diag"):
        capi.set_option("kernel", v)
        capi.set_option("index_cols", "16384")
        capi.set_option("index_split", split)
        try:
            with capi.Problem(kernel_type, 11, 7, 3) as P:
                P.add_block(arr)
                P.upload()
                if v == "index":
                    K0 = P.kernel_block(n - 1, 1, 0, n - 1)     # creates the partition over all columns
                    nblk, cols, _ = P.index_layout()
                    assert nblk == 2
                    assert cols == (10016 if split == "equal" else 16384 if kernel_type == 2 else 16352)
                    rows = sorted({1, 2, cols - 1, cols, cols + 1, cols + 147, cols + 148, n - 149, n - 148, n - 2, n - 1, 12345})
                got[v] = [(P.hist_block(r, 1, 0, r)[0], P.kernel_block(r, 1, 0, r)[0]) for r in rows]
                assert P.stats()["kernel_variant"] == {"diag": 2, "index": 4}[v]
        finally:
            capi.set_option("kernel", "auto")
            capi.set_option("index_cols", "0")
            capi.set_option("index_split", "auto")
    for r, (hi, ki), (hd, kd) in zip(rows, got["index"], got["diag"]):
        assert np.array_equal(hi, hd), "histograms of row %d" % r
        assert np.array_equal(ki, kd), "kernel values of row %d" % r


def test_ragged_lengths_at_scale_index_against_bitsliced():
    """4 000 sequences of 40 .. 1 200 bp (weighted kernel type, gkmQC's default L=10 k=6 d=3): the whole matrix of the index
    kernel against the bit-sliced kernel's"""
    rng = np.random.default_rng(21)
    letters = np.frombuffer(b"ACGT", np.uint8)
    seqs = [letters[rng.integers(0, 4, int(rng.integers(40, 1201)))].tobytes().decode() for _ in range(4000)]
    mats = {}
    for v in ("index", "diag"):
        capi.set_option("kernel", v)
        try:
            with capi.Problem(4, 10, 6, 3, 50, 50.0, 1.0) as P:
                P.add_many(seqs)
                mats[v] = P.kernel_lower()
        finally:
            capi.set_option("kernel", "auto")
    assert np.array_equal(mats["index"], mats["diag"])
    K = mats["index"]
    low = K[np.tril_indices(4000, -1)]
    assert np.all(np.diag(K) == 1.0) and low.min() >= 0 and low.max() <= 1.0 + 1e-12 and np.count_nonzero(low) > 0.9 * low.size  # 40-bp pairs may share nothing
