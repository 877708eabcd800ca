"""The launch space of the index variant's row kernel, as test cases (plain Python, no GPU): one definition shared by the CPU
tier (test_index_grid.py) and the GPU tier (test_gpu_index_space.py), like launch_grid.py for the all-pairs kernels.

gkm_idx_rows (gkm_index.cu) launches gkm_index_rows_kernel<WEIGHTED, RANGE, FMT, MINB>:
* FMT, the slot format of the column block (gkm_idx_block_fmt): C16 for unit weights, W20 for weights <= 63 on blocks of
  <= 16 352 columns, P32 otherwise or when index_wide is set.  WEIGHTED follows the kernel type, so four (FMT, WEIGHTED)
  pairs exist: C16-u, W20-w, P32-u, P32-w;
* RANGE, set when the wanted columns start inside the block (blo != 0);
* MINB, two CTAs per SM when two full histogram rows of the block fit shared memory (gkm_idx_two_cta), never for P32.
16 instances are compiled, 12 are reachable: P32 never runs two CTAs per SM.  Inside every instance d >= 2 adds the cold
bins (idx_probe_cold and the global scratch of each stream); d <= 1 has none.

The functions below restate index_block_cap and the layout in gkm_launch.cu, gkm_plan_index_blocks (gkm_sched.c),
gkm_idx_block_fmt (gkm_index_host.c), gkm_idx_max_cols, gkm_idx_row_smem and gkm_idx_two_cta (gkm_index.cu).  The skew of a
block (sum of squared posting-list lengths over postings) comes from numpy run lengths of both strands' L-mers.

CASES holds one case per reachable instance with and without cold bins, each built by the cheapest problem that reaches
it; the limits of the slot formats and of shared memory; and each two-CTA boundary at its last column count and at one
warp more, for a single block and for several.  A case is run as a sequence of calls (calls()): the lower triangle
first, whose column range [0, n) every later call sits inside, then rectangles with col0 inside a block and at a block
edge, a lower block off the origin and decision values.  predict() says which instance each block runs for a call, and
with how much dynamic shared memory.
"""
import numpy as np

THREADS = 1024
QCAP, LQCAP = 64, 32
HOT_BINS = 2
TWO_SMEM = 196 * 1024
SMEM_LIMIT = 227 * 1024
SKEW_ONE_CTA = 10.0
MAX_COLS = 0x7FFFFE
C16_MAX_COLS = 0x7FFF
W20_MAX_COLS = 16352
W20_MAX_WEIGHT = 63
W20_MAX_UNITS = 1 << 22
DEFAULT_COLS = 22528          # index_block_cap's default block width
WAVE_ROWS = 148               # rows of one wave; decision values launch 16 waves at a time
DECISION_ROWS = 16 * WAVE_ROWS
P32, C16, W20 = 0, 1, 2
FMT_NAME = {P32: "P32", C16: "C16", W20: "W20"}
WEIGHTED_TYPES = (4, 5)
RBF_TYPES = (3, 5)


# ---- restatements of the host rules ----
def qbytes(c16):
    """GKM_IDX_QBYTES_FMT: the warps' walk queues and long-list counters"""
    return (THREADS // 32) * (QCAP + LQCAP) * (4 if c16 else 8) + (THREADS // 32) * 4


def row_smem(nbins, ldh, maxq, weighted, c16):
    """gkm_idx_row_smem: hot histogram rows, queues, query L-mers (and their weights)"""
    s = min(nbins, HOT_BINS) * ldh * 4 + qbytes(c16) + maxq * 4 + (maxq if weighted else 0)
    return (s + 15) & ~15


def max_cols(nbins, maxq, weighted):
    """gkm_idx_max_cols"""
    budget = SMEM_LIMIT - 1024 - qbytes(False) - maxq * (5 if weighted else 4)
    cols = (budget // (4 * min(nbins, HOT_BINS))) & ~31
    if cols > MAX_COLS:
        cols = MAX_COLS & ~31
    return 0 if cols < 32 else cols


def two_cta(nbins, blk_cols, maxq, weighted, fmt, nblk, skew):
    """gkm_idx_two_cta: 1 when the block's row kernel runs two CTAs per SM"""
    pair = 2 * (row_smem(nbins, (blk_cols + 31) & ~31, maxq, weighted, fmt == C16) + 1280)
    if fmt == P32 or pair > (TWO_SMEM if nblk > 1 else SMEM_LIMIT):
        return 0
    return 0 if weighted and skew > SKEW_ONE_CTA else 1


def block_fmt(weighted, M, ncols, postings, wide):
    """gkm_idx_block_fmt"""
    if wide:
        return P32
    if not weighted:
        return C16 if ncols <= C16_MAX_COLS else P32
    if ncols <= W20_MAX_COLS and M <= W20_MAX_WEIGHT and (4 * postings) // 3 + 64 < 4 * W20_MAX_UNITS:
        return W20
    return P32


def index_block_cap(nbins, maxq, weighted, index_cols=0):
    """index_block_cap (gkm_launch.cu): what fits shared memory, the column limit of the compact format, the option"""
    cap = max_cols(nbins, maxq, weighted)
    if weighted and cap > W20_MAX_COLS:
        cap = W20_MAX_COLS
    if not weighted and cap > (C16_MAX_COLS & ~31):
        cap = C16_MAX_COLS & ~31
    lim = (index_cols & ~31) if index_cols > 0 else DEFAULT_COLS
    return min(cap, lim)


def plan_index_blocks(span, cap, greedy):
    """gkm_plan_index_blocks: (blocks, columns of all but the last)"""
    if span < 1 or cap < 32:
        return 0, 0
    nblk = (span + cap - 1) // cap
    c = (((span + nblk - 1) // nblk) + 31) & ~31
    if c > cap or greedy:
        c = cap & ~31
    return nblk, c


def layout(col0, span, cap, greedy):
    """the blocks [cb, ce) ensure_index cuts the partition [col0, col0 + span) into"""
    nblk, c = plan_index_blocks(span, cap, greedy)
    return [(col0 + k * c, min(col0 + (k + 1) * c, col0 + span)) for k in range(nblk)]


def last_two_cta_cols(nbins, maxq, weighted, fmt, several):
    """the widest block (a multiple of 32 columns) whose row kernel still runs two CTAs per SM"""
    c = 32
    while two_cta(nbins, c + 32, maxq, weighted, fmt, 2 if several else 1, 1.0):
        c += 32
    return c


def inst_bit(rng, minb):
    """the bit of gkm_index_rows_kernel<., RANGE, ., MINB> in gkmb200_problem_index_blocks' instance mask"""
    return 1 << (2 * int(rng) + minb - 1)


def inst_name(fmt, weighted, rng, minb):
    return "%s-%s-R%d-M%d" % (FMT_NAME[fmt], "w" if weighted else "u", int(rng), minb)


def compiled_instances():
    """(fmt, weighted, RANGE, MINB) of the 16 instances gkm_idx_rows can launch"""
    pairs = ((C16, False), (W20, True), (P32, False), (P32, True))
    return {(f, w, r, m) for f, w in pairs for r in (0, 1) for m in (1, 2)}


def reachable_instances():
    return {i for i in compiled_instances() if not (i[0] == P32 and i[3] == 2)}


# ---- sequences and their L-mers ----
ACGT = np.frombuffer(b"ACGT", np.uint8)
_CODE = np.zeros(256, np.int64)
_CODE[np.frombuffer(b"ACGT", np.uint8)] = np.arange(4)


def make_seqs(L, n, length, seed, poly=0, long_rows=0):
    """n sequences of max(L, length // 2) .. length bases: ragged random ones plus one of exactly L bases, a duplicate,
    a reverse complement, a homopolymer and a dinucleotide repeat; `poly` more poly-A rows (long posting lists: skew);
    `long_rows` rows of 2 047 bases near the end (the longest query and the widest shared-memory launch)"""
    rng = np.random.default_rng(seed)
    lo = max(L, length // 2)
    seqs = [ACGT[rng.integers(0, 4, int(ln))].tobytes().decode() for ln in rng.integers(lo, length + 1, n)]
    seqs[1] = seqs[1][:L]
    seqs[3] = seqs[2]
    seqs[4] = seqs[0][::-1].translate(str.maketrans("ACGT", "TGCA"))
    seqs[5] = "A" * length
    seqs[6] = ("CA" * length)[:length - 1]
    for i in range(poly):
        seqs[7 + i * max(1, (n - 8) // max(poly, 1))] = "A" * int(rng.integers(lo, length + 1))
    for i in range(long_rows):
        seqs[n - 3 - 5 * i] = ACGT[rng.integers(0, 4, 2047)].tobytes().decode()
    return seqs


def lmer_codes(seq, L):
    """an integer per L-mer of both strands (the postings of one column)"""
    s = _CODE[np.frombuffer(seq.encode(), np.uint8)]
    both = []
    for t in (s, 3 - s[::-1]):
        w = np.lib.stride_tricks.sliding_window_view(t, L)
        both.append(w @ (4 ** np.arange(L - 1, -1, -1, dtype=np.int64)))
    return np.concatenate(both)


def block_stats(seqs, L, cb, ce):
    """(postings, sum of squared posting-list lengths) of the block [cb, ce)"""
    codes = np.concatenate([lmer_codes(seqs[c], L) for c in range(cb, ce)])
    _, cnt = np.unique(codes, return_counts=True)
    return int(codes.size), int(np.sum(cnt.astype(np.int64) ** 2))


# ---- cases ----
class Call:
    """one compute call: kind in lower (hist_block + kernel_block, lower), rect (hist_block + kernel_block),
    lower_raw (gkmb200_kernel_block, lower, into a NaN-filled buffer with ld > ncols), decision"""

    def __init__(self, kind, row0, nrows, col0, ncols):
        self.kind, self.row0, self.nrows, self.col0, self.ncols = kind, row0, nrows, col0, ncols

    @property
    def lower(self):
        return self.kind in ("lower", "lower_raw")

    def __repr__(self):
        return "%s[%d:+%d, %d:+%d]" % (self.kind, self.row0, self.nrows, self.col0, self.ncols)


class Case:
    """one problem, the options it runs under, and the instance it is built to reach on block `block`"""

    def __init__(self, name, target, kernel_type, L, d, n, M=50, length=40, index_cols=0, wide=0, poly=0, long_rows=0,
                 block=0, decision_rows=0, kind="instance", cold=None):
        self.name, self.target, self.kernel_type, self.L, self.d, self.n, self.M = name, target, kernel_type, L, d, n, M
        self.length, self.index_cols, self.wide, self.poly, self.long_rows = length, index_cols, wide, poly, long_rows
        self.block, self.decision_rows, self.kind = block, decision_rows, kind
        self.weighted = kernel_type in WEIGHTED_TYPES
        self.nbins = d + 1
        self.cold = d >= 2
        assert target[1] == self.weighted, name
        self._seqs = self._stats = None

    def __repr__(self):
        return self.name

    @property
    def params(self):
        return dict(kernel_type=self.kernel_type, L=self.L, k=self.L - self.d, d=self.d, M=self.M, H=50.0, gamma=0.7)

    @property
    def options(self):
        return dict(kernel="index", index_cols=self.index_cols, index_wide=self.wide)

    def seqs(self):
        if self._seqs is None:
            self._seqs = make_seqs(self.L, self.n, self.length, _seed(self.name), self.poly, self.long_rows)
        return self._seqs

    @property
    def maxq(self):
        return 32 * ((max(map(len, self.seqs())) + 31) // 32)

    @property
    def cap(self):
        return index_block_cap(self.nbins, self.maxq, self.weighted, self.index_cols)

    def blocks(self):
        """the partition the first call (the lower triangle over [0, n): greedy) cuts"""
        return layout(0, self.n, self.cap, True)

    def stats(self):
        """per block (postings, sumsq, skew, fmt, MINB)"""
        if self._stats is None:
            bl = self.blocks()
            out = []
            for cb, ce in bl:
                P, sq = block_stats(self.seqs(), self.L, cb, ce)
                fmt = block_fmt(self.weighted, self.M, ce - cb, P, self.wide)
                out.append((P, sq, sq / P, fmt, 2 if two_cta(self.nbins, ce - cb, self.maxq, self.weighted, fmt, len(bl), sq / P) else 1))
            self._stats = out
        return self._stats

    def calls(self):
        n, bl = self.n, self.blocks()
        band = n if n <= 600 else 64                                     # the whole triangle, or bands of it
        cin = bl[self.block][0] + 37                                    # inside the target block
        w = min(200, bl[self.block][1] - cin)
        out = [Call("lower", n - band, band, 0, n)]                      # the partition [0, n): every later call reuses it
        if n > band:
            out.append(Call("lower", n // 2 - 32, 64, 0, n // 2 + 32))
        out.append(Call("rect", max(cin - 24, 0), 48, cin, w))           # col0 inside a block, across the diagonal
        edge = bl[-1][0] if len(bl) > 1 else 0                          # col0 at a block edge
        out.append(Call("rect", max(edge + 40, 0), 48, edge, min(120, n - edge)))
        out.append(Call("lower_raw", cin + w // 2, min(w, n - cin - w // 2), cin, w))
        if self.decision_rows:
            out.append(Call("decision", 0, self.decision_rows, cin, w))
        else:
            out.append(Call("decision", max(cin - 24, 0), min(96, n - max(cin - 24, 0)), cin, w))
        return out

    def predict(self, call):
        """{block: (instance mask, dynamic shared memory)} of the blocks the call launches"""
        out = {}
        st = self.stats()
        for k, (cb, ce) in enumerate(self.blocks()):
            lo, hi = max(call.col0, cb), min(call.col0 + call.ncols, ce)
            if call.lower:
                hi = min(hi, call.row0 + call.nrows - 1)                # columns < row: the last row of the call reaches furthest
            if hi <= lo:
                continue
            fmt, minb = st[k][3], st[k][4]
            out[k] = (inst_bit(lo > cb, minb), row_smem(self.nbins, (hi - lo + 31) & ~31, self.maxq, self.weighted, fmt == C16))
        return out


def _seed(name):
    return sum((i + 1) * ord(c) for i, c in enumerate(name))


def _instance_cases():
    """(instance, cold) -> the cheapest problem: small problems for two CTAs per SM; one CTA per SM through repeats
    (W20: skew > 10), index_wide (P32, unit weights), M = 255 (P32, weights) or a block past the several-block two-CTA
    limit (C16).  RANGE = 0 and 1 use different L, kernel types and seeds; the RANGE one is the target of the rectangle
    whose col0 lies inside the block.  The P32 cases with cold bins take 4 800 rows, so that their decision values span
    three launches."""
    cases = []
    unit_types, w_types = [0, 1, 2, 3], [4, 5]
    i = 0
    c16_one = last_two_cta_cols(3, 64, False, C16, True) + 32         # 10 816 columns per block at 40 bp
    for f, w, r, m in sorted(reachable_instances()):
        for d in (1, 2):
            cold = d >= 2
            L = (10, 8)[r] if d == 1 else (10, 12)[r]
            kt = (w_types if w else unit_types)[i % (2 if w else 4)]
            i += 1
            kw = dict(n=150 + 10 * i)
            if f == C16 and m == 1:
                kw = dict(n=c16_one + 96, index_cols=c16_one, decision_rows=2 * DECISION_ROWS + 64 if cold else 0)
            if f == W20 and m == 1:
                kw.update(poly=24)
            if f == P32 and not w:
                kw.update(wide=1)
            if f == P32 and w:
                kw.update(M=255)
            if f == P32 and cold:
                kw.update(n=4800, decision_rows=2 * DECISION_ROWS + 64)
            name = "%s-%s-L%d-d%d-t%d" % (inst_name(f, w, r, m), "cold" if cold else "hot", L, d, kt)
            cases.append(Case(name, (f, w, r, m), kt, L, d, **kw))
    return cases


def _limit_cases():
    cases = []
    # C16's column limit: a block of 32 736 columns (d = 0: one hot bin), columns up to 0x7FDF in the 15-bit field
    cases.append(Case("limit-C16-32736-cols", (C16, False, 0, 1), 2, 10, 0, 32736, index_cols=32736, kind="limit"))
    # the largest shared-memory launch: unit weights, d >= 1, a 2 047-bp row, a block at gkm_idx_max_cols = 24 800 columns
    cmax = max_cols(2, 2048, False)
    cases.append(Case("limit-smem-P32-%d-cols" % cmax, (P32, False, 0, 1), 2, 10, 1, cmax, index_cols=cmax, wide=1, long_rows=1,
                      kind="limit"))
    cases.append(Case("limit-smem-C16-%d-cols" % cmax, (C16, False, 0, 1), 0, 10, 2, cmax, index_cols=cmax, long_rows=1,
                      kind="limit"))
    # W20's largest weight: M = 63 in its 6-bit field
    cases.append(Case("limit-W20-M63", (W20, True, 1, 2), 4, 10, 2, 300, M=63, kind="limit"))
    return cases


def _boundary_cases():
    """each two-CTA boundary (C16, W20; a single block, several) at its last column count and one warp more"""
    cases = []
    for f, w, kt, d in ((C16, False, 2, 1), (W20, True, 4, 2)):
        for several in (False, True):
            last = last_two_cta_cols(d + 1, 64, w, f, several)
            for cols, m in ((last, 2), (last + 32, 1)):
                n = cols + 96 if several else cols
                dec = 2 * DECISION_ROWS + 64 if (d >= 2 and several and m == 1) else 0
                name = "boundary-%s-%s-%d-cols-M%d" % (FMT_NAME[f], "several" if several else "single", cols, m)
                cases.append(Case(name, (f, w, 0, m), kt, 10, d, n, index_cols=cols if several else 0, decision_rows=dec,
                                  kind="boundary"))
    return cases


INSTANCE_CASES = _instance_cases()
LIMIT_CASES = _limit_cases()
BOUNDARY_CASES = _boundary_cases()
CASES = INSTANCE_CASES + LIMIT_CASES + BOUNDARY_CASES
