"""GPU tier: the rest of the libgkm.h surface (SURVEY.md 8 a13) on the engine -- the objects gkmkernel_read_problems
and gkmkernel_new_object hand out (libgkm.c:841-938), gkmkernel_kernelfunc_batch (libgkm.c:1115-1153, its intended
meaning: SURVEY.md 3.4), the image hand-over from read_problems to build_tree, and the scope of GKM_SHARD."""
import ctypes
import os

import numpy as np
import pytest

import pack_model
import pyoracle
from conftest import load_golden, random_seqs
from gkmqc_b200 import capi

pytestmark = pytest.mark.gpu


class gkm_data(ctypes.Structure):
    """struct _gkm_data, libgkm.h:66-79 (88 bytes)"""
    _fields_ = [("sid", ctypes.c_char_p), ("seqid", ctypes.c_int), ("label", ctypes.c_int), ("seqlen", ctypes.c_int),
                ("seq", capi.c_u8_p), ("seq_rc", capi.c_u8_p), ("wt", capi.c_u8_p), ("wt_rc", capi.c_u8_p),
                ("kmerids", capi.c_int_p), ("kmerids_rc", capi.c_int_p), ("seq_string", ctypes.c_char_p), ("sqnorm", ctypes.c_double)]


class svm_problem(ctypes.Structure):
    _fields_ = [("l", ctypes.c_int), ("y", capi.c_dbl_p), ("x", ctypes.POINTER(ctypes.POINTER(gkm_data)))]


@pytest.fixture(scope="module")
def lib():
    lib = capi.load()
    if capi.device_count() < 1:
        pytest.fail("no B200 visible; the product has no CPU fallback")
    assert ctypes.sizeof(gkm_data) == 88
    lib.gkmkernel_init.restype = ctypes.c_void_p
    lib.gkmkernel_init.argtypes = [ctypes.POINTER(capi.gkm_parameter)]
    lib.gkmkernel_read_problems.argtypes = [ctypes.c_void_p, ctypes.POINTER(svm_problem), ctypes.c_char_p, ctypes.c_char_p]
    lib.gkmkernel_build_tree.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.POINTER(gkm_data)), ctypes.c_int]
    lib.gkmkernel_kernelfunc_batch_all.restype = capi.c_dbl_p
    lib.gkmkernel_kernelfunc_batch_all.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, capi.c_dbl_p]
    lib.gkmkernel_kernelfunc_batch.restype = capi.c_dbl_p
    lib.gkmkernel_kernelfunc_batch.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.POINTER(gkm_data)), ctypes.c_int, capi.c_dbl_p]
    lib.gkmkernel_delete_object.argtypes = [ctypes.POINTER(gkm_data)]
    lib.gkmkernel_destroy.argtypes = [ctypes.c_void_p]
    lib.gkmkernel_new_object.restype = ctypes.POINTER(gkm_data)
    lib.gkmkernel_new_object.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int]
    return lib


def read_fasta_like_the_reference(path):
    """(id, bases) per record: id = first whitespace token behind '>' (libgkm.c:1287-1292), lines concatenated"""
    out = []
    for line in open(path, "rb").read().split(b"\n"):
        line = line.split(b"\r")[0]
        if line.startswith(b">"):
            tok = line.split()
            out.append([tok[0][1:] if tok else b"", b""])
        elif out:
            out[-1][1] = (out[-1][1] + line)[:2047]
    return out


def expected_arrays(bases, L):
    """seq / seq_rc (codes 1..4, non-ACGT -> 1: libgkm.c:864-888) and the base-4 L-mer ids (libgkm.c:891-908)"""
    code = {ord("A"): 1, ord("C"): 2, ord("G"): 3, ord("T"): 4}
    seq = np.array([code.get(c, 1) for c in bases.upper()], np.int64)
    rc = 5 - seq[::-1]
    ids = []
    for s in (seq, rc):
        v = np.zeros(len(s) - L + 1, np.int64)
        for i in range(L):
            v = v * 4 + (s[i:i + len(v)] - 1)
        ids.append(v)
    return seq, rc, ids[0], ids[1]


@pytest.mark.parametrize("name", ["mix_t4_L11k7d3", "uni_t2_L11k7d3"])
def test_read_problems_fills_what_the_reference_fills(name, lib):
    g, cfg, pos, neg = load_golden(name)
    param = capi.make_param(**cfg)
    kern = lib.gkmkernel_init(ctypes.byref(param))
    prob = svm_problem()
    npos = lib.gkmkernel_read_problems(kern, ctypes.byref(prob), os.fsencode(pos), os.fsencode(neg))
    assert npos == int(g["npos"])
    recs = read_fasta_like_the_reference(pos) + read_fasta_like_the_reference(neg)
    assert prob.l == len(recs)
    o = pyoracle.Oracle(**cfg)
    o.read_problem(pos, neg)
    for i, (sid, bases) in enumerate(recs):
        d = prob.x[i].contents
        L = cfg["L"]
        seq, rc, ids, ids_rc = expected_arrays(bases, L)
        nk = len(seq) - L + 1
        assert d.sid == sid and d.seqid == i and d.seqlen == len(seq) and d.label == (1 if i < npos else -1)
        assert prob.y[i] == d.label
        assert np.array_equal(np.ctypeslib.as_array(d.seq, (len(seq),)), seq)
        assert np.array_equal(np.ctypeslib.as_array(d.seq_rc, (len(seq),)), rc)
        assert np.array_equal(np.ctypeslib.as_array(d.kmerids, (nk,)), ids)
        assert np.array_equal(np.ctypeslib.as_array(d.kmerids_rc, (nk,)), ids_rc)
        wt, wt_rc = o.poswt(i)
        assert np.array_equal(np.ctypeslib.as_array(d.wt, (nk,)), wt) and np.array_equal(np.ctypeslib.as_array(d.wt_rc, (nk,)), wt_rc)
        assert d.seq_string == bases                      # the file's own spelling (lower case, N ...), like strcpy in libgkm.c:859-860
        assert d.sqnorm == g["sqnorm"][i]
    # build_tree over exactly these objects adopts the image read_problems uploaded: no second upload
    st0 = capi.gkmb200_stats()
    lib.gkmkernel_build_tree(kern, prob.x, prob.l)
    res = np.zeros(prob.l)
    a = prob.l - 1
    lib.gkmkernel_kernelfunc_batch_all(kern, a, 0, a, res.ctypes.data_as(capi.c_dbl_p))
    assert np.array_equal(res[:a], g["kmat"][a, :a])
    for i in range(prob.l):
        lib.gkmkernel_delete_object(prob.x[i])
    lib.gkmkernel_destroy(kern)
    del st0


@pytest.mark.parametrize("kernel_type", [2, 4, 5])
def test_kernelfunc_batch_against_oracle(kernel_type, lib, tmp_path):
    """res[i] = K(prob[a], db_array[i]), normalised (+RBF), for objects that need not belong to the problem"""
    seqs = random_seqs(24, 120, seed=31, ragged=True)
    seqs = [s if len(s) >= 12 else s + "ACGTACGTACGT" for s in seqs]
    cfg = dict(kernel_type=kernel_type, L=10, k=6, d=3, M=50, H=50.0, gamma=1.0)
    param = capi.make_param(**cfg)
    kern = lib.gkmkernel_init(ctypes.byref(param))
    objs = [lib.gkmkernel_new_object(kern, s.encode(), b"s%d" % i, i) for i, s in enumerate(seqs)]
    assert all(objs)
    nprob = 16
    arr = (ctypes.POINTER(gkm_data) * nprob)(*objs[:nprob])
    lib.gkmkernel_build_tree(kern, arr, nprob)
    o = pyoracle.Oracle(**cfg)
    for s in seqs:
        o.add(s)
    db_ids = [20, 3, 23, 16, 9]            # outsiders and members of the problem, in any order
    db = (ctypes.POINTER(gkm_data) * len(db_ids))(*[objs[i] for i in db_ids])
    res = np.full(len(db_ids), -7.0)
    for a in (0, 5, nprob - 1):
        lib.gkmkernel_kernelfunc_batch(kern, a, db, len(db_ids), res.ctypes.data_as(capi.c_dbl_p))
        want = np.array([o.kernel(a, j) for j in db_ids])
        if kernel_type == 5:
            np.testing.assert_allclose(res, want, rtol=1e-9, atol=0)
        else:
            assert np.array_equal(res, want)
    # n = 0 and an out-of-range query leave nothing behind but zeros
    res[:] = -7.0
    lib.gkmkernel_kernelfunc_batch(kern, nprob + 3, db, len(db_ids), res.ctypes.data_as(capi.c_dbl_p))
    assert not res.any()
    for ob in objs:
        lib.gkmkernel_delete_object(ob)
    lib.gkmkernel_destroy(kern)


def test_new_object_cuts_what_the_engine_cannot_hold(lib):
    """the reference bounds the length only in read_fasta_file (libgkm.c:1294-1299); a longer string handed to
    gkmkernel_new_object directly is cut to 2047 bases and every field describes the cut sequence (ADVICE r1)"""
    rng = np.random.default_rng(3)
    long_seq = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 5000)].tobytes()
    cfg = dict(kernel_type=4, L=11, k=7, d=3, M=50, H=50.0, gamma=1.0)
    param = capi.make_param(**cfg)
    kern = lib.gkmkernel_init(ctypes.byref(param))
    ob = lib.gkmkernel_new_object(kern, long_seq, b"long", 0)
    short = lib.gkmkernel_new_object(kern, long_seq[:2047], b"cut", 1)
    assert ob and short
    d, e = ob.contents, short.contents
    assert d.seqlen == 2047 and len(d.seq_string) == 2047 and d.sqnorm == e.sqnorm
    nk = 2047 - 11 + 1
    assert np.array_equal(np.ctypeslib.as_array(d.kmerids, (nk,)), np.ctypeslib.as_array(e.kmerids, (nk,)))
    assert np.array_equal(np.ctypeslib.as_array(d.wt_rc, (nk,)), np.ctypeslib.as_array(e.wt_rc, (nk,)))
    arr = (ctypes.POINTER(gkm_data) * 2)(ob, short)
    lib.gkmkernel_build_tree(kern, arr, 2)
    res = np.zeros(1)
    lib.gkmkernel_kernelfunc_batch_all(kern, 1, 0, 1, res.ctypes.data_as(capi.c_dbl_p))
    assert abs(res[0] - 1.0) < 1e-12
    # a hand-made object that claims more bases than the engine holds is refused, not copied
    d.seqlen = 4000
    res[0] = -1.0
    lib.gkmkernel_kernelfunc_batch(kern, 0, arr, 1, res.ctypes.data_as(capi.c_dbl_p))
    assert res[0] == 0.0 and b"engine holds" in capi.load().gkmb200_last_error()
    d.seqlen = 2047
    lib.gkmkernel_delete_object(ob)
    lib.gkmkernel_delete_object(short)
    lib.gkmkernel_destroy(kern)


def test_gkm_shard_reaches_the_pywrapper_only(lib, tmp_path, monkeypatch):
    """GKM_SHARD (one process per GPU) shards gkm_main_pywrapper's matrix; every other entry point computes all of
    its chunks whatever the environment says, and the stats name the shard (ADVICE r1)"""
    g, cfg, pos, neg = load_golden("uni_t2_L11k7d3")
    n = len(g["lens"])
    monkeypatch.setenv("GKM_SHARD", "1/2")
    with capi.Problem(**cfg) as P:
        P.read(pos, neg)
        assert np.array_equal(P.kernel_lower(), g["kmat"])
        assert P.stats()["shard_world"] == 1
    param = capi.make_param(**cfg)
    kern = lib.gkmkernel_init(ctypes.byref(param))
    prob = svm_problem()
    lib.gkmkernel_read_problems(kern, ctypes.byref(prob), os.fsencode(pos), os.fsencode(neg))
    lib.gkmkernel_build_tree(kern, prob.x, prob.l)
    res = np.zeros(n)
    lib.gkmkernel_kernelfunc_batch_all(kern, n - 1, 0, n - 1, res.ctypes.data_as(capi.c_dbl_p))
    assert np.array_equal(res[:n - 1], g["kmat"][n - 1, :n - 1])
    for i in range(prob.l):
        lib.gkmkernel_delete_object(prob.x[i])
    lib.gkmkernel_destroy(kern)
    parts = []
    for rank in range(2):
        monkeypatch.setenv("GKM_SHARD", "%d/2" % rank)
        ret, kmat, _, _ = capi.main_pywrapper(pos, neg, nmax=n + 3, **{k: v for k, v in cfg.items()})
        assert ret == 0
        st = capi.gkmb200_stats()
        lib.gkmb200_get_stats(None, ctypes.byref(st))
        assert (st.shard_rank, st.shard_world) == (rank, 2)
        parts.append(kmat[:n, :n])
    low = np.tril_indices(n, -1)
    assert np.array_equal(parts[0][low] + parts[1][low], g["kmat"][low])


@pytest.mark.parametrize("kernel_type,L,M,H", pack_model.PARAMS)
def test_device_packing_equals_model(kernel_type, L, M, H, lib):
    """SURVEY.md 8f/f2: the GPU builds the 2-bit plane image (both strands, window-end plane, positional weights by end
    position) from one byte per base, by the rule of gkm_pack.h.  It must equal the numpy model of the image; the CPU tier
    holds the host packer of the emulators to the same model (test_pack_model.py), so the two packers agree."""
    seqs = pack_model.sequences(L)
    with capi.Problem(*pack_model.problem_args(kernel_type, L, M, H)) as P:
        P.add_many(seqs)
        planes, wend = P.image()
    want_planes, want_wend = pack_model.image(seqs, L, kernel_type, M, H)
    assert np.array_equal(planes, want_planes), "bit planes"
    if kernel_type in (4, 5):
        assert np.array_equal(wend, want_wend), "positional weights by window end"
        assert wend.max() == (M if M < 255 else 247)  # M = 255: the centre weight 256 wraps to 0 in the reference's u_int8_t
    else:
        assert wend is None
