"""ctypes binding of gkmkern_pylib.so -- both the reference's C-ABI (include/gkm_abi.h,
i.e. src/libgkm.h of Dongwon-Lee/gkmQC) and the extended entry points (include/gkm_b200.h).

The library is plain C + CUDA (no torch); this module only marshals pointers.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
BIN_DIR = os.path.join(HERE, "bin")
LIB_NAME = "gkmkern_pylib.so"  # artefact name of the reference, src/Makefile:6,13-14

c_int_p = ctypes.POINTER(ctypes.c_int)
c_i32_p = ctypes.POINTER(ctypes.c_int32)
c_dbl_p = ctypes.POINTER(ctypes.c_double)
c_u8_p = ctypes.POINTER(ctypes.c_uint8)


class gkm_parameter(ctypes.Structure):
    """struct _gkm_parameter, libgkm.h:53-64"""
    _fields_ = (
        ("kernel_type", ctypes.c_int), ("L", ctypes.c_int), ("k", ctypes.c_int), ("d", ctypes.c_int),
        ("M", ctypes.c_uint8), ("H", ctypes.c_double), ("gamma", ctypes.c_double), ("nthreads", ctypes.c_int),
    )


class gkmOpt(ctypes.Structure):
    """struct _gkmOpt, libgkm.h:149-161; identical to scripts/gkmsvm.py:48-61"""
    _fields_ = (
        ("kernel_type", ctypes.c_int), ("L", ctypes.c_int), ("k", ctypes.c_int), ("d", ctypes.c_int),
        ("M", ctypes.c_uint8), ("H", ctypes.c_double), ("gamma", ctypes.c_double),
        ("posfile", ctypes.c_char_p), ("negfile", ctypes.c_char_p),
        ("nthreads", ctypes.c_int), ("verbosity", ctypes.c_int),
    )


class gkmb200_stats(ctypes.Structure):
    _fields_ = (
        ("kernel_ms", ctypes.c_double), ("wall_ms", ctypes.c_double), ("upload_ms", ctypes.c_double),
        ("launches", ctypes.c_longlong), ("entries", ctypes.c_longlong), ("lmer_pairs", ctypes.c_longlong),
        ("h2d_bytes", ctypes.c_longlong), ("d2h_bytes", ctypes.c_longlong),
        ("devices", ctypes.c_int), ("kernel_variant", ctypes.c_int), ("shard_rank", ctypes.c_int), ("shard_world", ctypes.c_int),
        ("copy_threads", ctypes.c_int), ("thp_chunks", ctypes.c_int), ("scatter_ms", ctypes.c_float), ("wait_ms", ctypes.c_float),
    )

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class gkmb200_svm_task(ctypes.Structure):
    _fields_ = [("train_off", ctypes.c_longlong), ("test_off", ctypes.c_longlong), ("ntrain", ctypes.c_int), ("ntest", ctypes.c_int)]


class gkmb200_svm_fit(ctypes.Structure):
    _fields_ = [("rho", ctypes.c_double), ("obj", ctypes.c_double), ("nu", ctypes.c_double),
                ("n_iter", ctypes.c_int), ("n_sv", ctypes.c_int), ("reserved", ctypes.c_longlong)]


class gkmb200_svm_options(ctypes.Structure):
    _fields_ = [("C", ctypes.c_double), ("eps", ctypes.c_double), ("max_iter", ctypes.c_int), ("shrinking", ctypes.c_int),
                ("reserved", ctypes.c_longlong)]


class gkmb200_svm_shrink_stats(ctypes.Structure):
    _fields_ = [("shrink_passes", ctypes.c_int), ("min_active", ctypes.c_int), ("unshrink_iter", ctypes.c_int),
                ("recon_a", ctypes.c_int), ("recon_b", ctypes.c_int), ("reserved", ctypes.c_int)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class GkmError(RuntimeError):
    pass


_lib = None


def lib_path():
    # GKM_PYLIB: another build of the same library (the sanitised host build of tools/asan_host.sh, or a build that
    # tools/mma_time.py and tools/wgkm_time.py time); the product path is bin/
    return os.environ.get("GKM_PYLIB") or os.path.join(BIN_DIR, LIB_NAME)


def load(path=None):
    """load gkmkern_pylib.so (built by __graft_entry__.build / gkmqc_b200/csrc/Makefile); fails loudly if absent"""
    global _lib
    if path is None:
        if _lib is not None:
            return _lib
        path = lib_path()
    if not os.path.exists(path):
        raise GkmError("%s not built: run `python -c 'import __graft_entry__ as g; g.build()'` or `make -C gkmqc_b200/csrc`" % path)
    lib = ctypes.CDLL(path)
    _declare(lib)
    if path == lib_path():
        _lib = lib
    return lib


def _declare(lib):
    P = ctypes.c_void_p
    I = ctypes.c_int
    lib.gkmb200_last_error.restype = ctypes.c_char_p
    lib.gkmb200_check_parameter.restype = ctypes.c_char_p
    lib.gkmb200_check_parameter.argtypes = [ctypes.POINTER(gkm_parameter)]
    lib.gkmb200_weights.argtypes = [I, I, I, c_dbl_p]
    lib.gkmb200_posweights.argtypes = [I, I, I, ctypes.c_double, c_u8_p, c_u8_p]
    lib.gkmb200_problem_new.restype = P
    lib.gkmb200_problem_new.argtypes = [ctypes.POINTER(gkm_parameter)]
    lib.gkmb200_problem_free.argtypes = [P]
    lib.gkmb200_problem_add.argtypes = [P, ctypes.c_char_p, I]
    lib.gkmb200_problem_add_block.argtypes = [P, ctypes.c_void_p, ctypes.c_long, I, I]
    lib.gkmb200_problem_read_fasta.argtypes = [P, ctypes.c_char_p]
    lib.gkmb200_problem_read.argtypes = [P, ctypes.c_char_p, ctypes.c_char_p]
    lib.gkmb200_problem_size.argtypes = [P]
    lib.gkmb200_problem_seqlen.argtypes = [P, I]
    lib.gkmb200_problem_sid.argtypes = [P, I]
    lib.gkmb200_problem_sid.restype = ctypes.c_char_p
    lib.gkmb200_problem_codes.argtypes = [P, I, c_u8_p, c_u8_p]
    lib.gkmb200_problem_get_weights.argtypes = [P, c_dbl_p]
    lib.gkmb200_problem_set_shard.argtypes = [P, I, I]
    # entry points below exist only in the full library (not in the CPU emulator build)
    for name, args in (
        ("gkmb200_problem_upload", [P]),
        ("gkmb200_problem_sqnorm", [P, c_dbl_p]),
        ("gkmb200_kernel_lower", [P, ctypes.c_void_p, I]),
        ("gkmb200_kernel_block", [P, I, I, I, I, I, c_dbl_p, ctypes.c_long]),
        ("gkmb200_hist_block", [P, I, I, I, I, I, c_i32_p]),
        ("gkmb200_decision_values", [P, I, I, I, I, c_dbl_p, ctypes.c_double, c_dbl_p]),
        ("gkmb200_get_stats", [P, ctypes.POINTER(gkmb200_stats)]),
        ("gkmb200_problem_index_layout", [P, c_int_p]),
        ("gkmb200_problem_launch_shape", [P, c_int_p]),
        ("gkmb200_problem_index_blocks", [P, ctypes.POINTER(ctypes.c_longlong), I]),
        ("gkmb200_problem_image", [P, ctypes.c_void_p, ctypes.c_void_p, c_int_p]),
        ("gkmb200_resident_rows", [P, I, I, c_dbl_p, ctypes.c_long]),
        ("gkmb200_trim", []),
        ("gkmb200_bench_lower_resident", [P, I, I, I, c_dbl_p]),
        ("gkmb200_microbench", [ctypes.c_char_p, c_dbl_p]),
        ("gkmb200_svm_cv", [P, ctypes.c_void_p, ctypes.c_long, I, I, ctypes.POINTER(gkmb200_svm_task), c_int_p,
                            ctypes.POINTER(ctypes.c_byte), c_int_p, ctypes.c_double, ctypes.c_double, I,
                            c_dbl_p, ctypes.POINTER(gkmb200_svm_fit), c_dbl_p]),
        ("gkmb200_svm_cv_ex", [P, ctypes.c_void_p, ctypes.c_long, I, I, ctypes.POINTER(gkmb200_svm_task), c_int_p,
                               ctypes.POINTER(ctypes.c_byte), c_int_p, ctypes.POINTER(gkmb200_svm_options),
                               c_dbl_p, ctypes.POINTER(gkmb200_svm_fit), c_dbl_p, ctypes.POINTER(gkmb200_svm_shrink_stats)]),
        ("gkmb200_lmer_table_get", [P, c_dbl_p]),
        ("gkmb200_lmer_table_scores", [P, P, I, I, ctypes.c_double, c_dbl_p]),
        ("gkmb200_lmer_table_build_ms", [P, c_dbl_p]),
        ("gkmb200_lmer_table_substitutions", [P, P, ctypes.c_longlong, c_int_p, c_int_p, ctypes.c_double, c_dbl_p]),
        ("gkmb200_device_count", []),
        ("gkmb200_set_devices", [c_int_p, I]),
        ("gkmb200_set_option", [ctypes.c_char_p, ctypes.c_char_p]),
        ("gkmb200_set_verbosity", [I]),
        ("gkmb200_abi_version", []),
        ("gkm_main_pywrapper", [ctypes.POINTER(gkmOpt), np.ctypeslib.ndpointer(dtype=np.uintp, ndim=1, flags="C"), c_int_p]),
    ):
        if hasattr(lib, name):
            getattr(lib, name).argtypes = args
            getattr(lib, name).restype = ctypes.c_int
    if hasattr(lib, "gkmb200_lmer_table_new"):
        lib.gkmb200_lmer_table_new.argtypes = [P, I, I, c_dbl_p]
        lib.gkmb200_lmer_table_new.restype = P
        lib.gkmb200_lmer_table_free.argtypes = [P]
        lib.gkmb200_lmer_table_free.restype = None


def last_error(lib=None):
    lib = lib or load()
    msg = lib.gkmb200_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def _check(ret, lib):
    if ret != 0:
        raise GkmError(last_error(lib) or "gkmkern_pylib call failed (%d)" % ret)


def make_param(kernel_type=2, L=11, k=7, d=3, M=50, H=50.0, gamma=1.0, nthreads=1):
    return gkm_parameter(kernel_type, L, k, d, M, H, gamma, nthreads)


def weights(kernel_type, L, k, lib=None):
    lib = lib or load()
    w = np.zeros(L + 1)
    _check(lib.gkmb200_weights(kernel_type, L, k, w.ctypes.data_as(c_dbl_p)), lib)
    return w


def posweights(nk, kernel_type, M, H, lib=None):
    lib = lib or load()
    a = np.zeros(nk, np.uint8)
    b = np.zeros(nk, np.uint8)
    _check(lib.gkmb200_posweights(nk, kernel_type, M, H, a.ctypes.data_as(c_u8_p), b.ctypes.data_as(c_u8_p)), lib)
    return a, b


def check_parameter(lib=None, **kw):
    lib = lib or load()
    p = make_param(**kw)
    msg = lib.gkmb200_check_parameter(ctypes.byref(p))
    return msg.decode() if msg else None


def device_count():
    return load().gkmb200_device_count()


def set_option(key, value):
    lib = load()
    _check(lib.gkmb200_set_option(key.encode(), str(value).encode()), lib)


def microbench(what):
    lib = load()
    r = ctypes.c_double(0.0)
    _check(lib.gkmb200_microbench(what.encode(), ctypes.byref(r)), lib)
    return r.value


class Problem:
    """a parameter set plus sequences, resident on the selected GPUs after upload()"""

    def __init__(self, kernel_type=2, L=11, k=7, d=3, M=50, H=50.0, gamma=1.0, lib=None):
        self.lib = lib or load()
        self.param = make_param(kernel_type, L, k, d, M, H, gamma)
        self.L, self.d, self.kernel_type = L, d, kernel_type
        self.h = self.lib.gkmb200_problem_new(ctypes.byref(self.param))
        if not self.h:
            raise GkmError(last_error(self.lib))
        self.npos = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.gkmb200_problem_free(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def add(self, seq):
        b = seq if isinstance(seq, bytes) else seq.encode("ascii")
        r = self.lib.gkmb200_problem_add(self.h, b, len(b))
        if r < 0:
            raise GkmError(last_error(self.lib))
        return r

    def add_many(self, seqs):
        for s in seqs:
            self.add(s)

    def add_block(self, letters):
        """letters: uint8 matrix [n, len] of ASCII bases (one sequence per row)"""
        a = np.ascontiguousarray(letters, np.uint8)
        r = self.lib.gkmb200_problem_add_block(self.h, a.ctypes.data, a.strides[0], a.shape[0], a.shape[1])
        if r < 0:
            raise GkmError(last_error(self.lib))
        return r

    def read_fasta(self, path):
        r = self.lib.gkmb200_problem_read_fasta(self.h, os.fsencode(path))
        if r < 0:
            raise GkmError(last_error(self.lib))
        return r

    def read(self, posfile, negfile):
        r = self.lib.gkmb200_problem_read(self.h, os.fsencode(posfile), os.fsencode(negfile))
        if r < 0:
            raise GkmError(last_error(self.lib))
        self.npos = r
        return r

    @property
    def n(self):
        return self.lib.gkmb200_problem_size(self.h)

    def seqlen(self, i):
        return self.lib.gkmb200_problem_seqlen(self.h, i)

    def sid(self, i):
        return self.lib.gkmb200_problem_sid(self.h, i)

    def codes(self, i):
        n = self.seqlen(i)
        a = np.zeros(n, np.uint8)
        b = np.zeros(n, np.uint8)
        _check(self.lib.gkmb200_problem_codes(self.h, i, a.ctypes.data_as(c_u8_p), b.ctypes.data_as(c_u8_p)), self.lib)
        return a, b

    def weights(self):
        w = np.zeros(self.d + 1)
        _check(self.lib.gkmb200_problem_get_weights(self.h, w.ctypes.data_as(c_dbl_p)), self.lib)
        return w

    def set_shard(self, rank, world):
        _check(self.lib.gkmb200_problem_set_shard(self.h, rank, world), self.lib)

    def upload(self):
        _check(self.lib.gkmb200_problem_upload(self.h), self.lib)

    def sqnorm(self):
        out = np.zeros(self.n)
        _check(self.lib.gkmb200_problem_sqnorm(self.h, out.ctypes.data_as(c_dbl_p)), self.lib)
        return out

    def kernel_lower(self, kmat=None, copy_threads=4):
        """what gkm_main_pywrapper leaves in kmat: strict lower triangle + unit diagonal"""
        n = self.n
        if kmat is None:
            kmat = np.zeros((n, n))
        rows = (kmat.ctypes.data + np.arange(kmat.shape[0]) * kmat.strides[0]).astype(np.uintp)
        _check(self.lib.gkmb200_kernel_lower(self.h, rows.ctypes.data_as(ctypes.c_void_p), copy_threads), self.lib)
        return kmat

    def kernel_block(self, row0, nrows, col0, ncols, lower=False):
        out = np.zeros((nrows, ncols))
        _check(self.lib.gkmb200_kernel_block(self.h, row0, nrows, col0, ncols, int(lower), out.ctypes.data_as(c_dbl_p), ncols), self.lib)
        return out

    def hist_block(self, row0, nrows, col0, ncols, lower=False):
        out = np.zeros((nrows, ncols, self.d + 1), np.int32)
        _check(self.lib.gkmb200_hist_block(self.h, row0, nrows, col0, ncols, int(lower), out.ctypes.data_as(c_i32_p)), self.lib)
        return out

    def decision_values(self, row0, nrows, col0, ncols, alpha, bias=0.0):
        alpha = np.ascontiguousarray(alpha, np.float64)
        assert alpha.shape == (ncols,)
        out = np.zeros(nrows)
        _check(self.lib.gkmb200_decision_values(self.h, row0, nrows, col0, ncols, alpha.ctypes.data_as(c_dbl_p), bias,
                                                out.ctypes.data_as(c_dbl_p)), self.lib)
        return out

    def lmer_table(self, col0, ncols, alpha):
        """the model sum_c alpha[c - col0] K(., c), c in [col0, col0 + ncols), folded into one weight per L-mer
        (kernel types 0, 1, 2, 4): an LmerTable, built on every GPU of this problem"""
        return LmerTable(self, col0, ncols, alpha)

    def stats(self):
        st = gkmb200_stats()
        _check(self.lib.gkmb200_get_stats(self.h, ctypes.byref(st)), self.lib)
        return st.as_dict()

    def image(self):
        """(planes [n, 3, W] uint32, wend [n, 32 W] uint8 or None): the packed image as it lies on GPU 0"""
        shape = (ctypes.c_int * 2)()
        _check(self.lib.gkmb200_problem_image(self.h, None, None, shape), self.lib)
        n, W = shape[0], shape[1]
        planes = np.zeros((n, 3, W), np.uint32)
        wend = np.zeros((n, 32 * W), np.uint8) if self.kernel_type in (4, 5) else None
        _check(self.lib.gkmb200_problem_image(self.h, planes.ctypes.data, wend.ctypes.data if wend is not None else None, shape), self.lib)
        return planes, wend

    def resident_matrix(self, row0=0, nrows=None):
        """rows of the symmetric kernel matrix kept on the device (computed on first use; what svm_cv(problem=...) consumes);
        nrows = 0 only makes it resident"""
        nrows = self.n - row0 if nrows is None else nrows
        out = np.zeros((max(nrows, 1), self.n))
        _check(self.lib.gkmb200_resident_rows(self.h, row0, nrows, out.ctypes.data_as(c_dbl_p), self.n), self.lib)
        return out[:nrows]

    def index_layout(self):
        """(column blocks, columns per block, first column) of the index variant's last call; (0, 0, 0) otherwise"""
        out = (ctypes.c_int * 3)()
        _check(self.lib.gkmb200_problem_index_layout(self.h, out), self.lib)
        return tuple(out)

    INDEX_BLOCK_FIELDS = ("cb", "ce", "fmt", "postings", "sumsq", "inst", "smem", "launches")

    def index_blocks(self):
        """the index variant's column blocks of the last compute call, on the first GPU: one dict per block with cb, ce
        (columns), fmt (0 P32, 1 C16, 2 W20), postings, sumsq (sum of squared posting-list lengths), inst (bit
        2 RANGE + MINB - 1 for each gkm_index_rows_kernel build that ran), smem (most dynamic shared memory of a launch)
        and launches; [] when another variant ran"""
        n = self.lib.gkmb200_problem_index_blocks(self.h, None, 0)
        if n < 0:
            raise GkmError(last_error(self.lib))
        out = (ctypes.c_longlong * (8 * max(n, 1)))()
        n = self.lib.gkmb200_problem_index_blocks(self.h, out, n)
        if n < 0:
            raise GkmError(last_error(self.lib))
        return [dict(zip(self.INDEX_BLOCK_FIELDS, out[8 * k: 8 * k + 8])) for k in range(n)]

    def launch_shape(self):
        """(variant, TA, TB, dynamic shared memory bytes) of the last bit-sliced, lmer or mma launch for this problem on its
        first GPU (variant 1 lmer, 2 diag, 3 mma; mma: TA = queries per CTA, TB = 8); (0, 0, 0, 0) if none"""
        out = (ctypes.c_int * 4)()
        _check(self.lib.gkmb200_problem_launch_shape(self.h, out), self.lib)
        return tuple(out)

    def bench_lower_resident(self, steps, warmup, flush_l2=True):
        ms = np.zeros(steps)
        _check(self.lib.gkmb200_bench_lower_resident(self.h, steps, warmup, int(flush_l2), ms.ctypes.data_as(c_dbl_p)), self.lib)
        return ms


class LmerTable:
    """a linear gkm-SVM model as 4^L L-mer weights T (gkmb200_lmer_table_new): score(r) = bias + sum over the forward
    L-mers x of r of wt_r(x) T[x] / |r|, at a cost independent of the number of support vectors"""

    def __init__(self, problem, col0, ncols, alpha):
        self.lib, self.L = problem.lib, problem.L
        alpha = np.ascontiguousarray(alpha, np.float64)
        if alpha.shape != (ncols,):
            raise ValueError("alpha must hold ncols = %d values" % ncols)
        self.h = self.lib.gkmb200_lmer_table_new(problem.h, col0, ncols, alpha.ctypes.data_as(c_dbl_p))
        if not self.h:
            raise GkmError(last_error(self.lib))

    def close(self):
        if getattr(self, "h", None):
            self.lib.gkmb200_lmer_table_free(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def weights(self):
        """T as 4^L float64 values in lexicographic L-mer order (A, C, G, T = 0..3, first base most significant)"""
        out = np.zeros(4 ** self.L)
        _check(self.lib.gkmb200_lmer_table_get(self.h, out.ctypes.data_as(c_dbl_p)), self.lib)
        return out

    def scores(self, problem, row0, nrows, bias=0.0):
        """bias + sum_c alpha[c] K(r, c) for the rows [row0, row0 + nrows) of `problem` (same parameters and GPUs)"""
        out = np.zeros(nrows)
        _check(self.lib.gkmb200_lmer_table_scores(self.h, problem.h, row0, nrows, bias, out.ctypes.data_as(c_dbl_p)), self.lib)
        return out

    def substitutions(self, problem, rows, pos, bias=0.0):
        """out[i, v] = bias + the score of row rows[i] of `problem` with base pos[i] replaced by v (A, C, G, T = 0..3), bit for
        bit what scores() gives for a problem holding that mutant; sites in any order, repeats allowed.  (nsites, 4)"""
        rows = np.ascontiguousarray(rows, np.int32)
        pos = np.ascontiguousarray(pos, np.int32)
        if rows.shape != pos.shape or rows.ndim != 1:
            raise ValueError("rows and pos must be 1-D arrays of one length")
        out = np.zeros((len(rows), 4))
        _check(self.lib.gkmb200_lmer_table_substitutions(self.h, problem.h, len(rows), rows.ctypes.data_as(c_int_p),
                                                         pos.ctypes.data_as(c_int_p), bias, out.ctypes.data_as(c_dbl_p)), self.lib)
        return out

    def ism(self, problem, row0, nrows, bias=0.0):
        """in-silico mutagenesis of the rows [row0, row0 + nrows): one (len, 4) array per row, entry [p, v] the score with base p
        replaced by v (the row's own base gives its score), all through one substitutions() call"""
        lens = [problem.seqlen(r) for r in range(row0, row0 + nrows)]
        rows = np.repeat(np.arange(row0, row0 + nrows, dtype=np.int32), lens)
        pos = np.concatenate([np.arange(n, dtype=np.int32) for n in lens]) if lens else np.zeros(0, np.int32)
        out = self.substitutions(problem, rows, pos, bias)
        return np.split(out, np.cumsum(lens)[:-1]) if lens else []

    def build_ms(self):
        """device milliseconds of the build on the first GPU: (S, transform, combine)"""
        out = np.zeros(3)
        _check(self.lib.gkmb200_lmer_table_build_ms(self.h, out.ctypes.data_as(c_dbl_p)), self.lib)
        return tuple(out)


def svm_prepare_tasks(y, splits):
    """(labels 0/1 per sequence, [(train ids, test ids), ...]) -> the flat arrays gkmb200_svm_cv takes.
    Per fit the training ids are grouped by class, label 0 first, in their given order -- the order libsvm's
    svm_group_classes (with sklearn's label sort) gives them -- and that first class is the sub-problem's +1."""
    y = np.asarray(y)
    tasks = (gkmb200_svm_task * len(splits))()
    tr, ty, te = [], [], []
    toff = eoff = 0
    for t, (train, test) in enumerate(splits):
        train = np.asarray(train, np.int32)
        test = np.asarray(test, np.int32)
        lab = y[train]
        if not (np.any(lab == 0) and np.any(lab == 1)) or np.any((lab != 0) & (lab != 1)):
            raise ValueError("fit %d: labels must be 0/1 with both classes present" % t)
        order = np.concatenate((train[lab == 0], train[lab == 1]))
        tr.append(order)
        ty.append(np.where(y[order] == 0, 1, -1).astype(np.int8))
        te.append(test)
        tasks[t].train_off, tasks[t].test_off = toff, eoff
        tasks[t].ntrain, tasks[t].ntest = len(order), len(test)
        toff += len(order)
        eoff += len(test)
    cat = lambda xs, dt: np.ascontiguousarray(np.concatenate(xs) if xs else np.zeros(0), dt)
    return tasks, cat(tr, np.int32), cat(ty, np.int8), cat(te, np.int32)


def svm_cv(y, splits, kmat=None, problem=None, C=1.0, eps=1e-3, max_iter=-1, shrinking=0, stats=False, lib=None):
    """cross-validated C-SVC on the GPU (SURVEY.md 8f/f4).  Either `kmat` (dense symmetric host matrix) or `problem`
    (a capi.Problem whose kernel matrix is computed and kept on the device).  Returns (scores per split, fits, alphas):
    scores are sklearn decision_function values of the test ids, alphas are in the grouped training order.
    shrinking = 1: libsvm's shrinking heuristic, SVC(shrinking=True).  stats=True appends a fourth element, per fit what
    the heuristic did (gkmb200_svm_shrink_stats as a dict)."""
    lib = lib or (problem.lib if problem is not None else load())
    tasks, tr, ty, te = svm_prepare_tasks(y, splits)
    scores = np.zeros(len(te))
    alpha = np.zeros(len(tr))
    fits = (gkmb200_svm_fit * len(splits))()
    if kmat is not None:
        # rows of contiguous doubles are passed in place, with ld = the row stride (a view of a larger buffer: ld > n)
        if not (isinstance(kmat, np.ndarray) and kmat.dtype == np.float64 and kmat.ndim == 2 and kmat.strides[1] == 8
                and kmat.strides[0] % 8 == 0 and kmat.strides[0] >= 8 * kmat.shape[1]):
            kmat = np.ascontiguousarray(kmat, np.float64)
        n, kptr, ld, h = kmat.shape[0], kmat.ctypes.data, kmat.strides[0] // 8, None
    else:
        n, kptr, ld, h = problem.n, None, 0, problem.h
    args = (h, kptr, ld, n, len(splits), tasks, tr.ctypes.data_as(c_int_p), ty.ctypes.data_as(ctypes.POINTER(ctypes.c_byte)),
            te.ctypes.data_as(c_int_p))
    outs = (scores.ctypes.data_as(c_dbl_p), fits, alpha.ctypes.data_as(c_dbl_p))
    st = None
    if shrinking == 0 and not stats:
        _check(lib.gkmb200_svm_cv(*args, C, eps, max_iter, *outs), lib)
    else:
        opt = gkmb200_svm_options(C, eps, max_iter, shrinking, 0)
        st = (gkmb200_svm_shrink_stats * len(splits))()
        _check(lib.gkmb200_svm_cv_ex(*args, ctypes.byref(opt), *outs, st), lib)
    out_s, out_a = [], []
    for t in range(len(splits)):
        out_s.append(scores[tasks[t].test_off: tasks[t].test_off + tasks[t].ntest])
        out_a.append(alpha[tasks[t].train_off: tasks[t].train_off + tasks[t].ntrain])
    out_f = [dict(rho=f.rho, obj=f.obj, nu=f.nu, n_iter=f.n_iter, n_sv=f.n_sv) for f in fits]
    if stats:
        return out_s, out_f, out_a, [x.as_dict() for x in st]
    return out_s, out_f, out_a


def main_pywrapper(posfile, negfile, kernel_type=2, L=11, k=7, d=3, M=50, H=50.0, gamma=1.0,
                   nthreads=1, verbosity=0, nmax=None, kmat=None, lib=None):
    """call gkm_main_pywrapper like scripts/gkmsvm.py:75-88; returns (ret, kmat, npos, nneg)"""
    lib = lib or load()
    if kmat is None:
        kmat = np.zeros((nmax, nmax))
    rows = (kmat.ctypes.data + np.arange(kmat.shape[0]) * kmat.strides[0]).astype(np.uintp)
    narr = np.ones(2, dtype=np.int32)
    opts = gkmOpt(kernel_type, L, k, d, M, H, gamma, os.fsencode(posfile), os.fsencode(negfile), nthreads, verbosity)
    ret = lib.gkm_main_pywrapper(ctypes.byref(opts), rows, narr.ctypes.data_as(c_int_p))
    return ret, kmat, int(narr[0]), int(narr[1])
