/* gkm_sched.c -- how the kernel matrix is cut into chunks of row tiles and which process owns
 * which chunk, and the index variant's column blocks.  Pure host logic (tested on CPU, world_size 2).
 *
 * The reference interleaves single rows over pthreads (gkmkern_pylib.c:70-90,
 * row a = i*NTHREADS + t) because row a costs ~a.  Here the unit is a chunk of
 * whole row tiles sized by output bytes, so chunks near the bottom of the triangle
 * hold fewer rows; ownership alternates so every shard gets the same share of
 * entries to within one chunk.  No chunk needs data from another: K(i,j) depends on
 * sequences i and j only, so shards never communicate.
 */
#include "gkm_internal.h"

int gkm_plan_chunks(int row0, int nrows, int col0, int ncols, int lower, int tile_rows,
                    long long max_chunk_bytes, gkm_chunk *out, int max_chunks)
{
    return gkm_plan_chunks_rows(row0, nrows, col0, ncols, lower, tile_rows, max_chunk_bytes, 0, out, max_chunks);
}

/* max_rows > 0 also bounds the rows of a chunk.  The "index" kernel variant costs the same for every row
 * whatever the number of columns (it probes the whole index), so its chunks are cut by rows, which keeps
 * round-robin ownership balanced there too. */
int gkm_plan_chunks_rows(int row0, int nrows, int col0, int ncols, int lower, int tile_rows,
                         long long max_chunk_bytes, int max_rows, gkm_chunk *out, int max_chunks)
{
    if (nrows < 0 || ncols < 0 || tile_rows < 1 || max_chunks < 1) return -1;
    int n = 0;
    int r = row0;
    const int rend = row0 + nrows;
    while (r < rend) {
        /* grow the chunk tile by tile while its dense output stays under the byte budget */
        int e = r;
        long long entries = 0;
        for (;;) {
            int ne = e + tile_rows;
            if (ne > rend) ne = rend;
            int cend = col0 + ncols;
            if (lower && cend > ne) cend = ne; /* columns j < last row of the chunk */
            long long width = (long long) (cend > col0 ? cend - col0 : 0);
            long long bytes = (long long) (ne - r) * width * 8;
            if (e > r && (bytes > max_chunk_bytes || (max_rows > 0 && ne - r > max_rows))) break;
            e = ne;
            if (e >= rend) break;
        }
        int cend = col0 + ncols;
        if (lower && cend > e) cend = e;
        if (cend < col0) cend = col0;
        for (int a = r; a < e; a++) {
            int hi = cend;
            if (lower && hi > a) hi = a;
            if (hi > col0) entries += hi - col0;
        }
        if (n >= max_chunks) return -1;
        out[n].row_begin = r; out[n].row_end = e;
        out[n].col_begin = col0; out[n].col_end = cend;
        out[n].entries = entries;
        n++;
        r = e;
    }
    return n;
}

/* round-robin ownership; chunks are produced in row order with near-equal byte
 * size, so plain modulo balances entries to within one chunk per shard */
int gkm_chunk_owner(int chunk_index, int nchunks, int world)
{
    (void) nchunks;
    if (world <= 1) return 0;
    return chunk_index % world;
}

/* span columns in blocks of at most cap (a multiple of 32), block k = [k cols, min((k + 1) cols, span)): equal shares of
 * whole warps of columns, or -- greedy -- full blocks first and the rest in the last one: in a lower triangle row a probes
 * only the blocks that start below it, so the earlier a block ends the fewer rows pay for the next one. */
int gkm_plan_index_blocks(int span, int cap, int greedy, int *cols)
{
    if (span < 1 || cap < 32) { *cols = 0; return 0; }
    const int nblk = (span + cap - 1) / cap;
    int c = (((span + nblk - 1) / nblk) + 31) & ~31;
    if (c > cap || greedy) c = cap & ~31;
    *cols = c;
    return nblk;
}
