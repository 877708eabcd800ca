"""The cuts the device layer makes in one call, as test cases (plain Python, no GPU): one definition shared by the CPU tier
(test_seam_grid.py) and the GPU tier (test_gpu_seams.py).

Before any kernel runs, host code cuts a call into pieces, and every cut has a boundary where a wrong offset, base row,
stream join or buffer size gives wrong numbers without an error:

* compute calls (gkm_compute.cu plan_budget, plan_chunks): chunks of 16-row tiles, at most 65 520 rows (index: 148-row
  waves, at most 592), of at most max(4 MB, output / 16 per GPU) dense bytes, capped by the option chunk_mb;
* decision values (decision_slice): 8 192 rows per launch (index: 2 368), launches alternating the two compute streams;
* the diagonal (gkm_launch.cu launch_diag_rows, behind the sqnorm of an upload and the self histograms of substitutions):
  131 070 rows per launch when the bit-sliced kernel serves it, 1 024 under lmer;
* substitutions (gkm_lmer_table.cu lmer_subst_slice): batches of 2^21 sites, each with the diagonal of its rows
  [rmin, rmax] and its own results offset;
* GPU shares (gkm_dev.h for_each_gpu_share): rows in steps of 8 (decision values, table scores), sites in steps of 1.

This file restates those cuts.  Chunk lists come from the library's exported gkm_plan_chunks_rows with plan_budget
restated; the variant that runs follows launch_grid's rules.  predict() gives, for a call, its pieces, the indices on each
side of every cut and the kernel launches gkmb200_stats.launches must report.  Every case sits one step past a cut;
the first of its `below` calls sits exactly at it (one piece) and the `below` calls together redo the case's work in
calls that stay below the cut.
"""
import ctypes

import numpy as np

import launch_grid

TILE_ROWS, ROW_CAP = 16, 65520          # plan_chunks, bit-sliced / lmer / mma: grid.y <= 65 535 row tiles
WAVE_ROWS, WAVE_CAP = 148, 4 * 148      # plan_chunks, index: whole waves of one CTA per row and SM, 4 per chunk
DECISION_ROWS = {"index": 16 * WAVE_ROWS}  # decision_slice: rows per launch (index: 16 waves)
DECISION_ROWS_DEFAULT = 8192
DIAG_STEP_BITSLICED, DIAG_STEP_OTHER = 131070, 1024  # launch_diag_rows
SUBST_BATCH = 1 << 21                   # GKM_LS_CHUNK: sites per substitution launch
SHARE_ALIGN = {"decision": 8, "scores": 8, "subst": 1}  # for_each_gpu_share
CHUNK_MB_DEFAULT = 128


# ---- the cuts, restated ----
def plan_budget(total_cells, ndev, chunk_mb=CHUNK_MB_DEFAULT, world=1):
    """gkm_compute.cu plan_budget: dense bytes one chunk may hold"""
    want = max(total_cells * 8 // (16 * ndev * world), 4 << 20)
    return min(want, chunk_mb << 20)


class Chunk(ctypes.Structure):
    _fields_ = [("row_begin", ctypes.c_int), ("row_end", ctypes.c_int), ("col_begin", ctypes.c_int),
                ("col_end", ctypes.c_int), ("entries", ctypes.c_longlong)]


def plan_chunks_rows(lib, row0, nrows, col0, ncols, lower, tile_rows, budget, max_rows):
    """the library's own chunk list: [(row_begin, row_end, col_begin, col_end)]"""
    lib.gkm_plan_chunks_rows.argtypes = [ctypes.c_int] * 6 + [ctypes.c_longlong, ctypes.c_int, ctypes.POINTER(Chunk), ctypes.c_int]
    cap = nrows // tile_rows + 2
    buf = (Chunk * cap)()
    n = lib.gkm_plan_chunks_rows(row0, nrows, col0, ncols, int(lower), tile_rows, budget, max_rows, buf, cap)
    assert n >= 0, "chunk planning failed"
    return [(c.row_begin, c.row_end, c.col_begin, c.col_end) for c in buf[:n]]


def plan_chunks(lib, variant, row0, nrows, col0, ncols, lower, ndev=1, chunk_mb=CHUNK_MB_DEFAULT):
    """gkm_compute.cu plan_chunks"""
    total = nrows * ncols // (2 if lower else 1)
    by_rows = variant == "index"
    return plan_chunks_rows(lib, row0, nrows, col0, ncols, lower, WAVE_ROWS if by_rows else TILE_ROWS,
                            plan_budget(total, ndev, chunk_mb), WAVE_CAP if by_rows else ROW_CAP)


def ran_variant(forced, L, d):
    """the variant a compute call runs when `forced` is named (base_variant: mma needs d < L)"""
    return "diag" if forced == "mma" and d >= L else forced


def diag_step(forced):
    """launch_diag_rows: the bit-sliced kernel serves the diagonal but under lmer (pick_variant: mma and index hand the
    diagonal to it)"""
    return DIAG_STEP_OTHER if forced == "lmer" else DIAG_STEP_BITSLICED


def shares(count, ndev, align):
    """for_each_gpu_share: [(begin, end)] per GPU slot"""
    per = -(-(-(-count // ndev)) // align) * align
    return [(min(s * per, count), min(s * per + per, count)) for s in range(ndev)]


def steps(b, e, step):
    """[b, e) cut every `step` items"""
    return [(r, min(r + step, e)) for r in range(b, e, step)]


def seams_of(pieces):
    """the index right before and right after every cut between consecutive pieces"""
    return [(p[1] - 1, p[1]) for p in pieces[:-1]]


# ---- cases ----
class Call:
    """one entry-point call: kind upload | block | lower | decision | scores | subst, and its arguments"""

    def __init__(self, kind, row0=0, nrows=0, col0=0, ncols=0, sites=None, options=None):
        self.kind, self.row0, self.nrows, self.col0, self.ncols = kind, row0, nrows, col0, ncols
        self.sites = sites            # subst: (first site, end site) of the case's site list
        self.options = options or {}

    def __repr__(self):
        if self.kind == "subst":
            return "subst[%d:%d]" % self.sites
        return "%s(%d,+%d)x(%d,+%d)%s" % (self.kind, self.row0, self.nrows, self.col0, self.ncols,
                                           "".join(" %s=%s" % kv for kv in sorted(self.options.items())))


class Case:
    """one problem (parameters, forced variant, sequence recipe), the call that crosses a cut and the calls below it.
    seqs: ("copies", n) n rows cycling over 45 edge-case rows; ("short", n, long_at) rows of L..40 bases, one of 2 047 at
    long_at (or none); ("ragged", n) rows of L..200 bases; ("ism", n) rows of 600 bases"""

    def __init__(self, name, cut, params, variant, seqs, call, below, sites=None, table_cols=0):
        self.name, self.cut, self.params, self.variant, self.recipe = name, cut, params, variant, seqs
        self.call, self.below, self.site_recipe, self.table_cols = call, below, sites, table_cols
        self.L, self.d, self.kernel_type = params["L"], params["d"], params["kernel_type"]
        self.weighted = self.kernel_type in launch_grid.WEIGHTED_TYPES

    def __repr__(self):
        return self.name

    def seqs(self):
        rng = np.random.default_rng(launch_grid._seed(self.name))
        acgt = np.frombuffer(b"ACGT", np.uint8)
        kind, n = self.recipe[0], self.recipe[1]
        if kind == "copies":
            base = launch_grid.case_seqs(self.L, 45, 130, seed=7)
            return [base[i % len(base)] for i in range(n)]
        if kind == "ism":
            return [r.tobytes().decode() for r in acgt[rng.integers(0, 4, (n, 600))]]
        top = 40 if kind == "short" else 200
        lens = rng.integers(self.L, top + 1, n)
        codes = rng.integers(0, 4, int(lens.sum()))
        out, at = [], 0
        for ln in lens:
            out.append(acgt[codes[at:at + ln]].tobytes().decode())
            at += ln
        if kind == "short" and self.recipe[2] is not None:
            out[self.recipe[2]] = acgt[rng.integers(0, 4, launch_grid.MAX_LEN)].tobytes().decode()
        return out

    def lens(self):
        return [len(s) for s in self.seqs()]

    def sites(self, lens):
        """(rows, pos) int32 of the case's whole site list"""
        return self.site_recipe(lens)

    def maxlen(self):
        return max(self.lens())


def predict(case, call, ndev=1, lib=None, lens=None):
    """{"pieces": [(begin, end)], "seams": [(before, after)], "launches": n} of one call of the case on ndev GPUs, the
    problem already uploaded (and, for the index, its column blocks built)"""
    forced = call.options.get("kernel", case.variant)
    if call.kind == "upload":
        n = call.nrows
        pieces = steps(0, n, diag_step(forced))
        return dict(pieces=pieces, seams=seams_of(pieces), launches=ndev * (1 + len(pieces)))   # pack + diagonal
    if call.kind in ("block", "lower"):
        v = ran_variant(forced, case.L, case.d)
        ch = plan_chunks(lib, v, call.row0, call.nrows, call.col0, call.ncols, call.kind == "lower", ndev,
                         call.options.get("chunk_mb", CHUNK_MB_DEFAULT))
        pieces = [(c[0], c[1]) for c in ch]
        assert v != "index"
        return dict(pieces=pieces, seams=seams_of(pieces), launches=sum(1 for c in ch if c[3] > c[2] and c[1] > c[0]))
    if call.kind == "decision":
        v = ran_variant(forced, case.L, case.d)
        per = DECISION_ROWS.get(v, DECISION_ROWS_DEFAULT)
        pieces = []
        for b, e in shares(call.nrows, ndev, SHARE_ALIGN["decision"]):
            pieces += steps(call.row0 + b, call.row0 + e, per)
        blocks = 1 if v != "index" else -(-call.ncols // 22528)
        return dict(pieces=pieces, seams=seams_of(pieces), launches=blocks * len(pieces))
    if call.kind == "scores":
        pieces = [(call.row0 + b, call.row0 + e) for b, e in shares(call.nrows, ndev, SHARE_ALIGN["scores"]) if e > b]
        return dict(pieces=pieces, seams=seams_of(pieces), launches=len(pieces))
    assert call.kind == "subst"
    rows, _ = case.sites(lens)
    s0, s1 = call.sites
    rows = rows[s0:s1]
    pieces, launches = [], 0
    for b, e in shares(len(rows), ndev, SHARE_ALIGN["subst"]):
        for c0, c1 in steps(b, e, SUBST_BATCH):
            r = rows[c0:c1]
            launches += len(steps(int(r.min()), int(r.max()) + 1, diag_step(forced))) + 1
            pieces.append((s0 + c0, s0 + c1))
    return dict(pieces=pieces, seams=seams_of(pieces), launches=launches)


def diag_seams(case, lens):
    """subst: the rows on both sides of each diagonal step inside each batch"""
    rows, _ = case.sites(lens)
    s0, s1 = case.call.sites
    out = []
    for c0, c1 in steps(s0, s1, SUBST_BATCH):
        r = rows[c0:c1]
        out += seams_of(steps(int(r.min()), int(r.max()) + 1, diag_step(case.variant)))
    return out


# ---- the grid ----
def _p(kt, L=10, k=6, d=3):
    return dict(kernel_type=kt, L=L, k=k, d=d, M=50, H=50.0, gamma=0.7)


DEFAULT = _p(4)       # gkmQC's default model: wgkm, L = 10, k = 6, d = 3


def _ism(n):
    """row-ordered in-silico mutagenesis of n rows of 600 bases"""
    def f(lens):
        return np.repeat(np.arange(n, dtype=np.int32), 600), np.tile(np.arange(600, dtype=np.int32), n)
    return f


def _regrow(lens):
    """a first batch of 2^21 sites on rows 0..9, a second one over every row: d_H grows between batches"""
    rng = np.random.default_rng(5)
    r1 = rng.integers(0, 10, SUBST_BATCH).astype(np.int32)
    r2 = np.concatenate([np.arange(len(lens)), rng.integers(0, len(lens), 1000)]).astype(np.int32)
    rows = np.concatenate([r1, r2])
    lens = np.asarray(lens)
    return rows, (rng.integers(0, 1 << 30, len(rows)) % lens[rows]).astype(np.int32)


def _ends(last):
    """sites of row 0 and of row `last` only"""
    def f(lens):
        rows = np.array([0] * 3 + [last] * 3, np.int32)
        return rows, np.array([0, 1, lens[0] - 1, 0, 5, lens[last] - 1], np.int32)
    return f


def _cases():
    cases = []
    n = 2 * DIAG_STEP_OTHER + 37
    for v in ("lmer", "mma", "index", "diag"):
        # the diagonal of an upload: copies of 45 rows on both sides of both 1 024-row cuts (lmer); the other variants
        # hand it to the bit-sliced kernel and take one step
        cases.append(Case("sqnorm-%s" % v, "diag-step", _p(2 if v != "index" else 4), v, ("copies", n),
                          Call("upload", 0, n),
                          [Call("upload", 0, DIAG_STEP_OTHER), Call("upload", 0, n - DIAG_STEP_OTHER)]))
    # lower triangles of 1 000 ragged rows in >= 5 chunks of 1 MB; below: the rows up to 720 and the rest, one chunk of at
    # most 4 MB each
    for v, kt in (("lmer", 2), ("mma", 4)):
        cases.append(Case("lower-%s-t%d" % (v, kt), "chunk-bytes", _p(kt), v, ("ragged", 1000),
                          Call("lower", 0, 1000, 0, 1000, options=dict(chunk_mb=1)),
                          [Call("lower", 0, 720, 0, 720), Call("lower", 720, 280, 0, 1000)]))
    # 65 620 x 8 rectangles: the 65 520-row cap of a chunk, one 2 047-bp row for the smallest row tile
    nr = ROW_CAP + 100
    for v, kt in (("diag", 2), ("lmer", 4), ("mma", 4)):
        cases.append(Case("rect-%s-t%d" % (v, kt), "chunk-rows", _p(kt), v, ("short", nr, 777),
                          Call("block", 0, nr, 3, 8), [Call("block", 0, ROW_CAP, 3, 8), Call("block", ROW_CAP, nr - ROW_CAP, 3, 8)]))
    # decision values: 8 192 + 45 rows from an off-tile row, 40 SVs; index: 2 x 2 368 + 1 rows
    for v, kt in (("diag", 5), ("lmer", 4), ("mma", 3)):
        r0, m = 13, DECISION_ROWS_DEFAULT + 45
        cases.append(Case("dv-%s-t%d" % (v, kt), "decision-rows", _p(kt), v, ("short", r0 + m + 20, None),
                          Call("decision", r0, m, 2, 40),
                          [Call("decision", r0, DECISION_ROWS_DEFAULT, 2, 40), Call("decision", r0 + DECISION_ROWS_DEFAULT, 45, 2, 40)]))
    r0, per = 13, DECISION_ROWS["index"]
    cases.append(Case("dv-index-t2", "decision-rows", _p(2), "index", ("short", r0 + 2 * per + 21, None),
                      Call("decision", r0, 2 * per + 1, 2, 40),
                      [Call("decision", r0, per, 2, 40), Call("decision", r0 + per, per, 2, 40), Call("decision", r0 + 2 * per, 1, 2, 40)]))
    # substitutions past 2^21 sites at gkmQC's default
    ns = 3500 * 600
    for v in ("diag", "lmer"):
        cases.append(Case("subst-ism-%s" % v, "subst-batch", DEFAULT, v, ("ism", 3500), Call("subst", sites=(0, ns)),
                          [Call("subst", sites=(0, SUBST_BATCH)), Call("subst", sites=(SUBST_BATCH, ns))], sites=_ism(3500), table_cols=300))
    nreg = SUBST_BATCH + 3000 + 1000
    cases.append(Case("subst-regrow", "subst-batch", DEFAULT, "diag", ("short", 3000, None), Call("subst", sites=(0, nreg)),
                      [Call("subst", sites=(0, SUBST_BATCH)), Call("subst", sites=(SUBST_BATCH, nreg))], sites=_regrow, table_cols=200))
    nd = DIAG_STEP_BITSLICED + 130
    cases.append(Case("subst-diag-step", "diag-step", DEFAULT, "diag", ("short", nd, None), Call("subst", sites=(0, 6)),
                      [Call("subst", sites=(0, 3)), Call("subst", sites=(3, 6))], sites=_ends(nd - 1), table_cols=100))
    return cases


CASES = _cases()
CUTS = {  # cut -> the variants it applies to
    "diag-step": ("lmer", "diag"),
    "chunk-bytes": ("lmer", "mma"),
    "chunk-rows": ("diag", "lmer", "mma"),
    "decision-rows": ("diag", "lmer", "mma", "index"),
    "subst-batch": ("diag", "lmer"),
}
