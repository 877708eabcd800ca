"""CPU tier: properties of the chunk planner (gkm_sched.c) on generated problems -- the host logic that decides which
rows every launch, every GPU and every rank of a sharded run computes (the reference's counterpart is the row
interleave of gkmkern_pylib.c:70-90).  Whatever the shape: the chunks tile the rows exactly once, their entries add up
to the block, a chunk of more than one row tile respects both the byte budget and the row bound, and round-robin
ownership leaves no rank more than one chunk's worth above its share."""
import ctypes

import pytest

from gkmqc_b200 import capi

hypothesis = pytest.importorskip("hypothesis")
from hypothesis import given, settings  # noqa: E402
from hypothesis import strategies as st  # noqa: E402

# derandomize: every run draws the same fixed sequence of examples (a test tier must not be a lottery); the wider sweeps
# named in DESIGN.md were run once by raising max_examples.


class Chunk(ctypes.Structure):
    _fields_ = [("row_begin", ctypes.c_int), ("row_end", ctypes.c_int), ("col_begin", ctypes.c_int),
                ("col_end", ctypes.c_int), ("entries", ctypes.c_longlong)]


def plan(row0, nrows, col0, ncols, lower, tile_rows, budget, max_rows, cap=1 << 16):
    lib = capi.load()
    lib.gkm_plan_chunks_rows.argtypes = [ctypes.c_int] * 6 + [ctypes.c_longlong, ctypes.c_int, ctypes.POINTER(Chunk), ctypes.c_int]
    buf = (Chunk * cap)()
    n = lib.gkm_plan_chunks_rows(row0, nrows, col0, ncols, lower, tile_rows, budget, max_rows, buf, cap)
    return n, [(c.row_begin, c.row_end, c.col_begin, c.col_end, c.entries) for c in buf[:max(n, 0)]]


def entries_of(rb, re_, col0, cend, lower):
    tot = 0
    for a in range(rb, re_):
        hi = min(cend, a) if lower else cend
        tot += max(0, hi - col0)
    return tot


@settings(derandomize=True, max_examples=300, deadline=None)
@given(row0=st.integers(0, 5000), nrows=st.integers(0, 3000), col0=st.integers(0, 5000), ncols=st.integers(0, 3000),
       lower=st.booleans(), tile_rows=st.sampled_from([1, 2, 16, 148]), budget=st.sampled_from([8, 4096, 1 << 20, 1 << 27]),
       max_rows=st.sampled_from([0, 148, 592, 65520]))
def test_chunks_tile_any_block(row0, nrows, col0, ncols, lower, tile_rows, budget, max_rows):
    n, chunks = plan(row0, nrows, col0, ncols, int(lower), tile_rows, budget, max_rows)
    assert n == len(chunks) and n >= 0
    assert n <= nrows // tile_rows + 2          # the bound gkm_dev_compute sizes its arrays with
    cursor = row0
    for rb, re_, cb, ce, ent in chunks:
        assert rb == cursor and re_ > rb, "contiguous, non-empty, in row order"
        cursor = re_
        assert cb == col0
        want_ce = min(col0 + ncols, re_) if lower else col0 + ncols
        assert ce == max(want_ce, col0)
        assert ent == entries_of(rb, re_, col0, col0 + ncols, lower)
        assert (re_ - rb) % tile_rows == 0 or re_ == row0 + nrows, "whole row tiles, but for the last chunk"
        if re_ - rb > tile_rows:                # a chunk of several tiles obeys both bounds; a single tile may be over
            assert (re_ - rb) * (ce - cb) * 8 <= budget
            assert max_rows == 0 or re_ - rb <= max_rows
    assert cursor == row0 + nrows
    assert sum(c[4] for c in chunks) == entries_of(row0, row0 + nrows, col0, col0 + ncols, lower)


@settings(derandomize=True, max_examples=60, deadline=None)
@given(n=st.integers(2000, 60000), world=st.sampled_from([1, 2, 3, 4, 8]), index=st.booleans())
def test_round_robin_ownership_is_balanced(n, world, index):
    """the plan gkm_dev_compute makes for a lower triangle (tile 148 rows and at most 592 per chunk for the index variant,
    16 and the grid bound otherwise; budget min(128 MB, total / (16 x ranks))), chunks dealt c % world"""
    lib = capi.load()
    total = n * (n - 1) // 2
    budget = min(128 << 20, max(4 << 20, n * n // 2 * 8 // (16 * world)))
    nch, chunks = plan(0, n, 0, n, 1, 148 if index else 16, budget, 4 * 148 if index else 65520)
    assert nch > 0
    share = [0] * world
    rows = [0] * world
    for c, ch in enumerate(chunks):
        r = lib.gkm_chunk_owner(c, nch, world)
        assert 0 <= r < world and r == c % world
        share[r] += ch[4]
        rows[r] += ch[1] - ch[0]
    assert sum(share) == total
    biggest = max(ch[4] for ch in chunks)
    if index:   # every row costs the same there: rows are what has to balance.  Chunk sizes never grow with the row index
        # (the byte budget bites harder the wider the rows are), so a round of the deal differs by at most first - last
        # chunk over all rounds together (<= 592 rows) and the ragged last round adds at most one more chunk
        sizes = [ch[1] - ch[0] for ch in chunks[:-1]]
        assert all(a >= b for a, b in zip(sizes, sizes[1:]))
        assert max(rows) - min(rows) <= 2 * 592
    else:
        assert max(share) <= total / world + biggest


def index_blocks(span, cap, greedy):
    lib = capi.load()
    lib.gkm_plan_index_blocks.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
    cols = ctypes.c_int(-1)
    nblk = lib.gkm_plan_index_blocks(span, cap, int(greedy), ctypes.byref(cols))
    return nblk, cols.value


def test_index_blocks_of_the_gpu_layout_tests():
    """the layouts the GPU tier reads back (gkmb200_problem_index_layout), stated without a GPU: 150 columns under
    index_cols = 128, and 20 000 columns under 16 384 (unit weights) or the compact weighted slots' 16 352"""
    assert index_blocks(150, 128, False) == (2, 96)
    assert index_blocks(150, 128, True) == (2, 128)
    assert index_blocks(20000, 16384, False) == (2, 10016)
    assert index_blocks(20000, 16384, True) == (2, 16384)
    assert index_blocks(20000, 16352, True) == (2, 16352)


@settings(derandomize=True, max_examples=300, deadline=None)
@given(span=st.integers(1, 200000), cap=st.integers(1, 1024).map(lambda x: 32 * x), greedy=st.booleans())
def test_index_blocks_tile_the_columns(span, cap, greedy):
    """block k holds columns [k cols, min((k + 1) cols, span)) (ensure_index): every column in exactly one block, none
    wider than the cap (a multiple of 32, as index_block_cap gives it), whole warps of columns but for the last block"""
    nblk, cols = index_blocks(span, cap, greedy)
    assert nblk == -(-span // cap) and cols % 32 == 0 and 0 < cols <= cap
    blocks = [(k * cols, min((k + 1) * cols, span)) for k in range(nblk)]
    assert blocks[-1][1] == span and all(ce > cb for cb, ce in blocks), "every block non-empty, the last ends the span"
    if greedy:
        assert cols == cap
