/* gkm_seq.c -- sequences of a problem: FASTA input, base coding, the shape of the 2-bit plane image.
 *
 * Host-side counterpart of gkmkernel_new_object (libgkm.c:841-938) and
 * read_fasta_file (libgkm.c:1251-1314).  What the reference keeps per sequence as
 * byte arrays (seq, seq_rc, wt, wt_rc) becomes the image the kernels read: two bit
 * planes per strand (bit p of plane b = bit b of the base code at position p,
 * A,C,G,T = 0,1,2,3) and, for the weighted kernel types, the positional weights
 * re-indexed by window END position (gkm_pack.h).  The GPU packs it (gkm_device.cu);
 * gkm_pack_problem builds the same image here for the CPU emulators.  sqnorm is NOT
 * computed here -- it is the diagonal of the kernel and comes from the GPU.
 */
#include <ctype.h>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "gkm_internal.h"
#include "gkm_pack.h"

gkmb200_problem *gkmb200_problem_new(const gkm_parameter *param)
{
    if (!param) { gkm_set_error("null parameter"); return NULL; }
    const char *bad = gkm_param_problem(param, GKM_MAX_L);
    if (bad) { gkm_set_error("%s", bad); return NULL; }
    gkmb200_problem *p = (gkmb200_problem *) calloc(1, sizeof(*p));
    if (!p) { gkm_set_error("out of memory"); return NULL; }
    p->param = *param;
    p->nbins = param->d + 1;
    p->weighted = (param->kernel_type == EST_TRUNC_PW || param->kernel_type == EST_TRUNC_PW_RBF);
    /* every problem computes all of its chunks unless told otherwise (gkmb200_problem_set_shard, or the
     * environment for gkm_main_pywrapper's own problem: gkm_problem_shard_from_env) */
    p->shard_rank = 0;
    p->shard_world = 1;
    if (gkm_calc_weights(param->kernel_type, param->L, param->k, p->w)) {
        gkm_set_error("cannot compute weights for L=%d k=%d", param->L, param->k);
        free(p);
        return NULL;
    }
    return p;
}

/* One process per GPU (torchrun-style launches): GKM_SHARD="rank/world" makes this process compute only the
 * chunks it owns.  Read for the problem of gkm_main_pywrapper alone -- the caller that set the variable knows that
 * its matrix is partial; the problems behind the libgkm ABI (gkmkernel_kernelfunc_batch_all: one row, one chunk)
 * and the CLI would silently return zeros on every rank but one. */
void gkm_problem_shard_from_env(gkmb200_problem *p)
{
    const char *sh = getenv("GKM_SHARD");
    int r = 0, w = 1;
    if (sh && sscanf(sh, "%d/%d", &r, &w) == 2 && w >= 1 && r >= 0 && r < w) { p->shard_rank = r; p->shard_world = w; }
}

void gkmb200_problem_free(gkmb200_problem *p)
{
    if (!p) return;
    gkm_dev_release(p);
    gkm_unpack_problem(p);
    for (int i = 0; i < p->n; i++) if (p->sid) free(p->sid[i]);
    free(p->arena);
    free(p->off);
    free(p->sid);
    free(p->len);
    free(p);
}

int gkm_problem_reserve(gkmb200_problem *p, int extra)
{
    if (p->n + extra <= p->cap) return 0;
    int cap = p->cap ? p->cap : 256;
    while (cap < p->n + extra) cap *= 2;
    int *len = (int *) realloc(p->len, sizeof(int) * (size_t) cap);
    if (!len) return 1;
    p->len = len;
    size_t *off = (size_t *) realloc(p->off, sizeof(size_t) * (size_t) cap);
    if (!off) return 1;
    p->off = off;
    char **sid = (char **) realloc(p->sid, sizeof(char *) * (size_t) cap);
    if (!sid) return 1;
    for (int i = p->cap; i < cap; i++) sid[i] = NULL;
    p->sid = sid;
    p->cap = cap;
    return 0;
}

/* room for `extra` more bases (+ 16 of slack: the SSE2 coder stores whole vectors) */
static int arena_reserve(gkmb200_problem *p, size_t extra)
{
    if (p->arena_len + extra + 16 <= p->arena_cap) return 0;
    size_t cap = p->arena_cap ? p->arena_cap : ((size_t) 1 << 16);
    while (cap < p->arena_len + extra + 16) cap *= 2;
    uint8_t *a = (uint8_t *) realloc(p->arena, cap);
    if (!a) return 1;
    p->arena = a;
    p->arena_cap = cap;
    return 0;
}

int gkmb200_problem_add(gkmb200_problem *p, const char *seq, int len)
{
    if (!p || !seq) { gkm_set_error("null argument"); return -1; }
    if (len < 0) len = (int) strlen(seq);
    if (len > GKM_MAX_BASES) len = GKM_MAX_BASES;
    if (len < p->param.L) {
        gkm_set_error("sequence %d has %d bases, fewer than L=%d", p->n, len, p->param.L);
        return -1;
    }
    if (gkm_problem_reserve(p, 1) || arena_reserve(p, (size_t) len)) { gkm_set_error("out of memory"); return -1; }
    /* the letters go into the arena as they are (the GPU codes and packs them); the host only looks for letters that are
     * not nucleotides, sixteen at a time, to name them like the reference does (libgkm.c:864-875) */
    uint8_t *c = p->arena + p->arena_len;
    memcpy(c, seq, (size_t) len);
    int any_bad = 0, i = 0;
#if defined(__SSE2__)
    {
        const __m128i up = _mm_set1_epi8((char) 0xDF);
        const __m128i cA = _mm_set1_epi8('A'), cC = _mm_set1_epi8('C'), cG = _mm_set1_epi8('G'), cT = _mm_set1_epi8('T');
        __m128i all_ok = _mm_set1_epi8((char) 0xFF);
        for (; i + 16 <= len; i += 16) {
            const __m128i u = _mm_and_si128(_mm_loadu_si128((const __m128i *) (seq + i)), up);
            const __m128i ok = _mm_or_si128(_mm_or_si128(_mm_cmpeq_epi8(u, cA), _mm_cmpeq_epi8(u, cC)),
                                            _mm_or_si128(_mm_cmpeq_epi8(u, cG), _mm_cmpeq_epi8(u, cT)));
            all_ok = _mm_and_si128(all_ok, ok);
        }
        any_bad |= _mm_movemask_epi8(all_ok) != 0xFFFF;
    }
#endif
    for (; i < len; i++) {
        const unsigned u = (unsigned char) seq[i] & 0xDFu;
        any_bad |= !(u == 'A' || u == 'C' || u == 'G' || u == 'T');
    }
    if (any_bad) { /* rare: name the offenders like the reference does; they count as 'A' wherever codes are made */
        for (int j = 0; j < len; j++) {
            const unsigned u = (unsigned char) seq[j] & 0xDFu;
            if (u == 'A' || u == 'C' || u == 'G' || u == 'T') continue;
            if (p->nonacgt < 10)
                gkm_log(GKM_LOG_WARN, "'%c' at sequence %d(%d) is not a valid nucleotide. Only ACGT are allowed", seq[j], p->n, j);
            p->nonacgt++;
        }
    }
    p->len[p->n] = len;
    p->off[p->n] = p->arena_len;
    p->arena_len += (size_t) len;
    p->sid[p->n] = NULL;
    gkm_unpack_problem(p); /* packed image is stale now */
    return p->n++;
}

/* n sequences of `len` bases each, `stride` bytes apart in one buffer (a numpy uint8 matrix of letters): the in-memory
 * entry point for batches (SURVEY.md 8f/f2) */
int gkmb200_problem_add_block(gkmb200_problem *p, const char *bases, long stride, int n, int len)
{
    if (!p || !bases || n < 0 || len < 0 || stride < len) { gkm_set_error("bad sequence block"); return -1; }
    if (gkm_problem_reserve(p, n)) { gkm_set_error("out of memory"); return -1; }
    for (int i = 0; i < n; i++)
        if (gkmb200_problem_add(p, bases + (size_t) i * (size_t) stride, len) < 0) return -1;
    return p->n;
}

static int fasta_add(gkmb200_problem *p, const char *seq, int seqlen, const char *id, int idlen)
{
    const int i = gkmb200_problem_add(p, seq, seqlen);
    if (i >= 0 && id) {
        char *s = (char *) malloc((size_t) idlen + 1);
        if (s) { memcpy(s, id, (size_t) idlen); s[idlen] = '\0'; }
        p->sid[i] = s;
    }
    return i;
}

/* one FASTA file; the line discipline of libgkm.c:1207-1225,1268-1304:
 * a line ends at the first CR or LF, '>' in column 0 opens a record, all other
 * lines extend the current record up to 2047 bases, text before the first
 * record is ignored. */
int gkmb200_problem_read_fasta(gkmb200_problem *p, const char *path)
{
    if (!p || !path) { gkm_set_error("null argument"); return -1; }
    FILE *fp = fopen(path, "rb");
    if (!fp) { gkm_set_error("can't open file %s", path); return -1; }
    /* the whole file in one buffer (bins of gkmQC are a few MB), then one pass with memchr */
    size_t cap = (size_t) 1 << 20, got = 0;
    if (fseek(fp, 0, SEEK_END) == 0) {
        long sz = ftell(fp);
        if (sz > 0) cap = (size_t) sz + 1;
        rewind(fp);
    }
    char *buf = (char *) malloc(cap);
    char *seq = (char *) malloc(GKM_MAX_BASES + 1);
    if (!buf || !seq) { free(buf); free(seq); fclose(fp); gkm_set_error("out of memory reading %s", path); return -1; }
    for (;;) {
        size_t r = fread(buf + got, 1, cap - got, fp);
        got += r;
        if (got < cap) break;
        char *nb = (char *) realloc(buf, cap * 2);
        if (!nb) { free(buf); free(seq); fclose(fp); gkm_set_error("out of memory reading %s", path); return -1; }
        buf = nb;
        cap *= 2;
    }
    fclose(fp);
    int seqlen = 0, open_rec = 0, added = 0, warned = 0, fail = 0;
    const char *id0 = NULL; int idlen = 0; /* id of the open record: the first token of its header line behind '>' */
    const char *cur = buf, *end = buf + got;
    while (!fail && cur < end) {
        const char *nl = (const char *) memchr(cur, '\n', (size_t) (end - cur));
        const char *next = nl ? nl + 1 : end;
        const char *le = nl ? nl : end;
        /* the line ends at the first CR, LF or NUL (libgkm.c:1207-1225 reads lines as C strings) */
        const char *cr = (const char *) memchr(cur, '\r', (size_t) (le - cur));
        if (cr) le = cr;
        const char *nul = (const char *) memchr(cur, '\0', (size_t) (le - cur));
        if (nul) le = nul;
        if (le > cur && cur[0] == '>') {
            if (open_rec) {
                if (fasta_add(p, seq, seqlen, id0, idlen) < 0) fail = 1; else added++;
            }
            if ((added % 1000) == 0) gkm_log(GKM_LOG_INFO, "reading... %d", added);
            open_rec = 1; seqlen = 0; warned = 0;
            /* strtok(line, " \t\r\n") then +1 (libgkm.c:1287-1292): the token that starts with '>' */
            id0 = cur + 1; idlen = 0;
            while (id0 + idlen < le && id0[idlen] != ' ' && id0[idlen] != '\t') idlen++;
        } else if (open_rec && seqlen < GKM_MAX_BASES) {
            size_t ll = (size_t) (le - cur);
            if ((size_t) seqlen + ll > GKM_MAX_BASES) {
                if (!warned)
                    gkm_log(GKM_LOG_WARN, "maximum sequence length allowed is %d. The first %d nucleotides of record %d will only be used",
                            GKM_MAX_BASES, GKM_MAX_BASES, added);
                warned = 1;
                ll = (size_t) (GKM_MAX_BASES - seqlen);
            }
            memcpy(seq + seqlen, cur, ll);
            seqlen += (int) ll;
        }
        cur = next;
    }
    if (!fail && open_rec) {
        if (fasta_add(p, seq, seqlen, id0, idlen) < 0) fail = 1; else added++;
    }
    gkm_log(GKM_LOG_INFO, "reading... done");
    free(buf);
    free(seq);
    return fail ? -1 : added;
}

/* positives get ids 0..n_pos-1, negatives follow (libgkm.c:1316-1333).  The two files are independent: the
 * negatives are parsed by a helper thread into a scratch problem while this thread parses the positives, then
 * appended (1 of the 2 ms the reads took at 10k sequences). */
struct read_job { gkmb200_problem *q; const char *path; int n; char err[512]; };

static void *read_worker(void *arg)
{
    struct read_job *j = (struct read_job *) arg;
    j->n = gkmb200_problem_read_fasta(j->q, j->path);
    if (j->n < 0) snprintf(j->err, sizeof(j->err), "%s", gkmb200_last_error()); /* the message is thread-local */
    return NULL;
}

int gkmb200_problem_read(gkmb200_problem *p, const char *posfile, const char *negfile)
{
    if (!p || !posfile || !negfile) { gkm_set_error("null argument"); return -1; }
    struct read_job job;
    memset(&job, 0, sizeof(job));
    job.path = negfile;
    job.q = gkmb200_problem_new(&p->param);
    pthread_t th;
    const int threaded = job.q && pthread_create(&th, NULL, read_worker, &job) == 0;
    gkm_log(GKM_LOG_INFO, "reading sequences from %s", posfile);
    int np = gkmb200_problem_read_fasta(p, posfile);
    int nn = -1;
    if (threaded) {
        pthread_join(th, NULL);
        nn = job.n;
        if (np >= 0 && nn >= 0) {
            gkm_log(GKM_LOG_INFO, "reading sequences from %s", negfile);
            if (gkm_problem_reserve(p, job.q->n) || arena_reserve(p, job.q->arena_len)) { gkm_set_error("out of memory"); nn = -1; }
            else {
                memcpy(p->arena + p->arena_len, job.q->arena, job.q->arena_len); /* 1.5 MB per 5 000 x 300 bp */
                for (int i = 0; i < job.q->n; i++) {
                    p->len[p->n] = job.q->len[i];
                    p->off[p->n] = p->arena_len + job.q->off[i];
                    p->sid[p->n] = job.q->sid[i];
                    job.q->sid[i] = NULL;
                    p->n++;
                }
                p->arena_len += job.q->arena_len;
                p->nonacgt += job.q->nonacgt;
                gkm_unpack_problem(p);
            }
        } else if (np >= 0) {
            gkm_set_error("%s", job.err);
        }
    } else if (np >= 0) {
        gkm_log(GKM_LOG_INFO, "reading sequences from %s", negfile);
        nn = gkmb200_problem_read_fasta(p, negfile);
    }
    if (job.q) gkmb200_problem_free(job.q);
    if (np < 0 || nn < 0) return -1;
    p->npos = np;
    return np;
}

int gkmb200_problem_size(const gkmb200_problem *p) { return p ? p->n : -1; }

int gkmb200_problem_seqlen(const gkmb200_problem *p, int i)
{
    if (!p || i < 0 || i >= p->n) return -1;
    return p->len[i];
}

/* id of a record read from FASTA (gkm_data.sid: the first token behind '>', libgkm.c:1287-1292); NULL for in-memory sequences */
const char *gkmb200_problem_sid(const gkmb200_problem *p, int i)
{
    if (!p || i < 0 || i >= p->n) return NULL;
    return p->sid[i];
}

/* the byte arrays the reference would hold in gkm_data.seq / seq_rc (codes 1..4) */
int gkmb200_problem_codes(const gkmb200_problem *p, int i, uint8_t *fwd, uint8_t *rc)
{
    if (!p || i < 0 || i >= p->n) return 1;
    const int n = p->len[i];
    for (int j = 0; j < n; j++) {
        if (fwd) fwd[j] = (uint8_t) (gkm_base_code(gkm_letters(p, i)[j]) + 1);
        if (rc) rc[j] = (uint8_t) (4 - gkm_base_code(gkm_letters(p, i)[n - 1 - j]));
    }
    return 0;
}

int gkmb200_problem_get_weights(const gkmb200_problem *p, double *w)
{
    if (!p || !w) return 1;
    for (int m = 0; m < p->nbins; m++) w[m] = p->w[m];
    return 0;
}

int gkmb200_problem_set_shard(gkmb200_problem *p, int rank, int world)
{
    if (!p || world < 1 || rank < 0 || rank >= world) { gkm_set_error("bad shard %d/%d", rank, world); return 1; }
    p->shard_rank = rank;
    p->shard_world = world;
    return 0;
}

void gkm_unpack_problem(gkmb200_problem *p)
{
    if (!p->packed) return;
    free(p->planes); p->planes = NULL;
    free(p->wend); p->wend = NULL;
    free(p->sqnorm); p->sqnorm = NULL;
    p->packed = 0;
    p->have_sqnorm = 0;
    p->host_sqnorm = 0;
}

/* shape of the image: words per plane and the sqnorm buffer; the image itself is built on the device */
int gkm_shape_problem(gkmb200_problem *p)
{
    if (p->packed) return 0;
    if (p->n == 0) { gkm_set_error("problem has no sequences"); return 1; }
    int maxlen = 0;
    for (int i = 0; i < p->n; i++) if (p->len[i] > maxlen) maxlen = p->len[i];
    p->Wmax = (2 * maxlen + 31) / 32;
    p->Wa = (maxlen + 31) / 32;
    p->maxlen = maxlen;
    p->sqnorm = (double *) calloc((size_t) p->n, sizeof(double));
    if (!p->sqnorm) { gkm_set_error("out of memory"); return 1; }
    p->packed = 1;
    p->have_sqnorm = 0;
    return 0;
}

/* the image of every sequence on the host, by the rule the device packer applies (gkm_pack.h): for the CPU emulators of
 * the test tier only, so one position at a time */
int gkm_pack_problem(gkmb200_problem *p)
{
    if (p->packed && p->planes) return 0;
    if (gkm_shape_problem(p)) return 1;
    const int W = p->Wmax, L = p->param.L;
    p->planes = (uint32_t *) calloc((size_t) p->n * 3 * (size_t) W, sizeof(uint32_t));
    if (p->weighted) p->wend = (uint8_t *) calloc((size_t) p->n * 32 * (size_t) W, 1);
    if (!p->planes || (p->weighted && !p->wend)) {
        gkm_unpack_problem(p);
        gkm_set_error("out of memory packing %d sequences", p->n);
        return 1;
    }
    uint8_t tab[GKM_MAX_BASES + 1];
    if (p->weighted) gkm_posweight_table(p->param.kernel_type, p->param.M, p->param.H, tab);
    for (int i = 0; i < p->n; i++) {
        const int len = p->len[i], centre = (len - L + 1) / 2;
        uint32_t *pl = p->planes + (size_t) i * 3 * (size_t) W;
        for (int wi = 0; wi < W; wi++)
            for (int b = 0; b < 32; b++) {
                const int j = wi * 32 + b;
                int s;
                const uint32_t code = gkm_pack_code(gkm_letters(p, i), len, L, j, &s);
                pl[wi] |= (code & 1u) << b;
                pl[W + wi] |= (code >> 1) << b;
                pl[2 * W + wi] |= (uint32_t) (s >= 0) << b;
                if (p->weighted) p->wend[(size_t) i * 32 * (size_t) W + (size_t) j] = gkm_pack_weight(tab, centre, s);
            }
    }
    return 0;
}
