"""The launch space of the all-pairs kernels, as test cases (plain Python, no GPU): one definition shared by the CPU lane
emulator tests (test_emu_bitslice.py) and the GPU tier (test_gpu_launch_space.py).

Two launch-time choices decide which device code runs:

* the compiled instance of the bit-sliced kernel, gkm_diag_kernel<L, NB, WEIGHTED, D4> (gkm_bitslice.h: gkm_diag_nb,
  gkm_diag_instance).  INSTANCE_CASES holds one case per instance the parameter gate lets a caller reach (86 of the 105
  compiled ones);
* the tile shape launch_hist (gkm_device.cu) picks from the longest sequence of the problem: (TA, TB) of the bit-sliced
  and lmer kernels (pick_tile, first candidate within 74 KB / 100 KB of shared memory) and the queries per CTA of the
  tcgen05 kernel, QA = min(4, 2176 // L-mers).  SHAPE_CASES holds one case per shape class, its longest sequence at the
  largest length of the class: the shared-memory footprint closest to the limit.

The functions below restate gkm_diag_layout (gkm_diag_kernel.cuh), gkm_lmer_smem_bytes (gkm_lmer_kernel.cuh) and the QA
rule; the GPU tier checks through gkmb200_problem_launch_shape that every case ran the shape it was built for.

Candidates no legal length reaches (sequences hold at most 2 047 bases): lmer (1, 1), unweighted diag (2, 2) and (2, 1),
and pick_tile's second pass (220 KB) for either kernel.
"""
import numpy as np

MAX_LEN = 2047          # longest sequence the reader keeps (libgkm.c:1294-1299)
MAX_BINS = 16           # d <= 15
UNWEIGHTED_TYPES = (0, 1, 2, 3)
WEIGHTED_TYPES = (4, 5)
RBF_TYPES = (3, 5)

DIAG_CAND = ((8, 32), (4, 32), (4, 16), (2, 16), (2, 8), (2, 4), (2, 2), (2, 1))
LMER_CAND = ((8, 8), (4, 4), (2, 2), (1, 1))
DIAG_LIMIT = 74 * 1024
LMER_LIMIT = 100 * 1024
MMA_ROWS_CAP, MMA_QA, MMA_TB = 2176, 4, 8
VARIANT_CODE = {"lmer": 1, "diag": 2, "mma": 3, "index": 4}


# ---- the parameter gate and the instance rule ----
def gate_ok(L, k, d):
    """gkm_param_problem (gkm_weights.c) for 2 <= L <= 16"""
    return 2 <= L <= 16 and 0 <= k <= L and 0 <= d <= L - k and d < MAX_BINS


def diag_nb(d):
    return 4 if d < 4 else 8 if d < 8 else 16


def instance(L, d, weighted):
    """(L, NB, WEIGHTED, D4) of the bit-sliced kernel instance that serves the problem"""
    nb = diag_nb(d)
    return (L, nb, bool(weighted), nb == 8 and not weighted and d == 4)


def compiled_instances():
    """gkm_diag_inst.cu: every L = 2..16 gets NB = 4, 8, 16 x {plain, weighted}, and the unweighted NB = 8 d = 4 one"""
    out = set()
    for L in range(2, 17):
        for nb in (4, 8, 16):
            for w in (False, True):
                out.add((L, nb, w, False))
        out.add((L, 8, False, True))
    return out


def reachable_instances():
    """the instances some (L, k, d) the gate admits is served by, weighted or not"""
    out = set()
    for L in range(2, 17):
        for k in range(0, L + 1):
            for d in range(0, L - k + 1):
                if gate_ok(L, k, d):
                    for w in (False, True):
                        out.add(instance(L, d, w))
    return out


# ---- launch shapes (launch_hist) ----
def image_words(maxlen):
    """(Wmax, Wa): words per plane of the both-strand circular string, 32-position chunks of one strand (gkm_seq.c)"""
    return (2 * maxlen + 31) // 32, (maxlen + 31) // 32


def diag_smem(W, WA, TA, TB, NB, weighted):
    npair = (TA + 1) // 2
    o = 2 * npair * 32 * WA * 16                       # sAp, sAx
    o += TB * 3 * W * 4 + W * 4                        # target planes, zero row
    o += TB * (32 * W + 32) if weighted else 0         # target weights + wrap-around copy
    o += TB * W * 4                                    # lane tasks
    o += 2 * npair * TB * NB * 4                       # histograms
    o += 2 * npair * 4 + TB * 4 + (TB + 1) * 4         # lengths, prefix
    return (o + 15) & ~15


def lmer_smem(WA, TA, TB, nbins, weighted):
    nk = 32 * WA
    o = (TA + 2 * TB) * nk * 4
    if weighted:
        o += (TA + 2 * TB) * nk
    o += TA * TB * nbins * 4 + (TA + TB) * 4
    return (o + 15) & ~15


def _pick(cand, limit, nbytes):
    for ta, tb in cand:
        s = nbytes(ta, tb)
        if s <= limit:
            return (ta, tb, s)
    for ta, tb in cand:
        s = nbytes(ta, tb)
        if s <= 220 * 1024:
            return (ta, tb, s)
    return None


def expected_shape(variant, maxlen, L, d, weighted):
    """(variant code, TA, TB, shared bytes or None) launch_hist picks for a problem whose longest sequence is maxlen"""
    W, WA = image_words(maxlen)
    if variant == "diag":
        ta, tb, s = _pick(DIAG_CAND, DIAG_LIMIT, lambda ta, tb: diag_smem(W, WA, ta, tb, diag_nb(d), weighted))
        return (2, ta, tb, s)
    if variant == "lmer":
        ta, tb, s = _pick(LMER_CAND, LMER_LIMIT, lambda ta, tb: lmer_smem(WA, ta, tb, d + 1, weighted))
        return (1, ta, tb, s)
    assert variant == "mma"
    return (3, min(MMA_QA, MMA_ROWS_CAP // (maxlen - L + 1)), MMA_TB, None)


def shape_classes(variant, L, d, weighted):
    """[(TA, TB), largest maxlen of the class] in order of growing length, over maxlen = L .. MAX_LEN"""
    out = []
    for m in range(L, MAX_LEN + 1):
        sh = expected_shape(variant, m, L, d, weighted)[1:3]
        if out and out[-1][0] == sh:
            out[-1][1] = m
        else:
            out.append([sh, m])
    return [(sh, m) for sh, m in out]


# ---- cases ----
class Case:
    """one problem: parameters, the variant to force, the sequence-set recipe, and (shape cases) the expected launch"""

    def __init__(self, name, kernel_type, L, k, d, variant="diag", maxlen=130, n=45, shape=None):
        assert gate_ok(L, k, d), (L, k, d)
        self.name, self.kernel_type, self.L, self.k, self.d = name, kernel_type, L, k, d
        self.variant, self.maxlen, self.n, self.shape = variant, maxlen, n, shape
        self.weighted = kernel_type in WEIGHTED_TYPES
        self.inst = instance(L, d, self.weighted)

    @property
    def params(self):
        return dict(kernel_type=self.kernel_type, L=self.L, k=self.k, d=self.d, M=50, H=50.0, gamma=0.7)

    def seqs(self, n=None, maxlen=None):
        return case_seqs(self.L, n or self.n, maxlen or self.maxlen, seed=_seed(self.name))

    def __repr__(self):
        return self.name


def _seed(name):
    return sum((i + 1) * ord(c) for i, c in enumerate(name))


def case_seqs(L, n, maxlen, seed):
    """n sequences of L .. maxlen bases, maxlen itself included once: ragged random ones, one of exactly L bases, lengths
    16m - 1, 16m, 16m + 1 (the both-strand circular string ends one base before, on, or one base after a 32-bit word), a
    duplicate, a reverse complement, a homopolymer and a dinucleotide repeat"""
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", np.uint8)

    def rnd(ln):
        return acgt[rng.integers(0, 4, ln)].tobytes().decode()

    m = max(1, (min(maxlen, 3 * L + 40) - 1) // 16)
    edge = [ln for ln in (16 * m - 1, 16 * m, 16 * m + 1) if L <= ln <= maxlen]
    seqs = [rnd(maxlen), rnd(L)] + [rnd(ln) for ln in edge]
    seqs.append(seqs[-1])                                                        # duplicate
    seqs.append(seqs[0][::-1].translate(str.maketrans("ACGT", "TGCA")))          # reverse complement of the longest
    seqs.append("A" * int(rng.integers(L, maxlen + 1)))                          # homopolymer
    seqs.append(("CA" * maxlen)[: int(rng.integers(L, maxlen + 1))])             # dinucleotide repeat
    while len(seqs) < n:
        seqs.append(rnd(int(rng.integers(L, maxlen + 1))))
    seqs = seqs[:n]
    order = rng.permutation(n)                                                   # the longest one anywhere in the tile
    return [seqs[i] for i in order]


def _instance_cases():
    """one case per reachable instance.  Within each class (NB, WEIGHTED, D4) d steps through the values the class
    takes at that L, largest first, so that d = L - 1 and d = L (k = 0) both occur; kernel types rotate over 0..3
    (unweighted) and 4, 5 (weighted)"""
    cases = []
    ti = {False: 0, True: 0}
    classes = sorted({(nb, w, d4) for (_, nb, w, d4) in reachable_instances()})
    for nb, w, d4 in classes:
        Ls = sorted(L for (L, b, ww, dd) in reachable_instances() if (b, ww, dd) == (nb, w, d4))
        for i, L in enumerate(Ls):
            ds = sorted((d for d in range(0, min(L, MAX_BINS - 1) + 1) if instance(L, d, w) == (L, nb, w, d4)), reverse=True)
            d = ds[(5 * i) % len(ds)]
            if nb == 16 and L in (15, 16) and w == (L == 16):
                d = 15                                     # d = 15 at L = 15 (k = 0, unweighted) and L = 16 (weighted)
            types = WEIGHTED_TYPES if w else UNWEIGHTED_TYPES
            kt = types[ti[w] % len(types)]
            ti[w] += 1
            name = "L%d-nb%d-%s%s-d%d-t%d" % (L, nb, "w" if w else "u", "-d4" if d4 else "", d, kt)
            cases.append(Case(name, kt, L, L - d, d))
    return cases


def _shape_cases():
    cases = []
    L, k, d = 11, 7, 3
    for variant, specs in (("diag", ((3, False, 2), (3, True, 4), (8, False, 2), (8, True, 4))),
                           ("lmer", ((3, False, 2), (3, True, 4))),
                           ("mma", ((3, False, 2), (3, True, 4)))):
        for dd, w, kt in specs:
            classes = shape_classes(variant, L, dd, w)
            if dd == 8:
                classes = classes[-2:]                     # NB = 16: its two longest classes
            for (ta, tb), m in classes:
                name = "%s-%s-nb%d-%dx%d-len%d" % (variant, "w" if w else "u", diag_nb(dd), ta, tb, m)
                cases.append(Case(name, kt, L, L - dd if dd > 3 else k, dd, variant=variant, maxlen=m,
                                  n=39 if m > 1000 else 45, shape=expected_shape(variant, m, L, dd, w)))
    return cases


INSTANCE_CASES = _instance_cases()
SHAPE_CASES = _shape_cases()
