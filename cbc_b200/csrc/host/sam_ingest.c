/* sam_ingest.c -- see sam_ingest.h. Files are mapped whole and split with memchr: no per-line buffers, so the
 * reference's 1024-byte line limit (src/sam_file_allocation.c:444) and its "MD must not be the last field"
 * trap (:507-511) do not exist here. */
#define _GNU_SOURCE
#include "sam_ingest.h"

#include <fcntl.h>
#include <pthread.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>

static int fail(char *err, size_t n, int rc, const char *fmt, ...) {
    if (err && n) { va_list ap; va_start(ap, fmt); vsnprintf(err, n, fmt, ap); va_end(ap); }
    return rc;
}

typedef struct { const uint8_t *p; size_t n; int fd; } mapped;
static int map_file(const char *path, mapped *m) {
    m->p = NULL; m->n = 0;
    m->fd = open(path, O_RDONLY);
    if (m->fd < 0) return -1;
    struct stat st;
    if (fstat(m->fd, &st)) { close(m->fd); return -1; }
    m->n = (size_t)st.st_size;
    if (m->n == 0) return 0;
    void *p = mmap(NULL, m->n, PROT_READ, MAP_PRIVATE | MAP_POPULATE, m->fd, 0);   /* page tables filled once, not by faults of the workers */
    if (p == MAP_FAILED) { close(m->fd); return -1; }
    madvise(p, m->n, MADV_SEQUENTIAL);
    m->p = (const uint8_t *)p;
    return 0;
}
static void unmap_file(mapped *m) { if (m->p) munmap((void *)m->p, m->n); if (m->fd >= 0) close(m->fd); m->p = NULL; }

/* ------------------------------------------------------------------ FASTA */
int cbch_read_fasta(const char *path, cbch_fasta *out, char *err, size_t errlen) {
    memset(out, 0, sizeof *out);
    mapped m;
    if (map_file(path, &m)) return fail(err, errlen, CBCH_ERR_IO, "cannot open %s", path);
    uint32_t cap = 0;
    const uint8_t *p = m.p, *end = m.p + m.n;
    int rc = CBCH_OK;
    while (p < end) {
        const uint8_t *nl = memchr(p, '\n', (size_t)(end - p));
        const uint8_t *le = nl ? nl : end;
        if (p < le && *p == '>') {
            if (out->n == cap) {
                cap = cap ? cap * 2 : 32;
                out->names = realloc(out->names, cap * sizeof *out->names);
                out->bases = realloc(out->bases, cap * sizeof *out->bases);
                out->len = realloc(out->len, cap * sizeof *out->len);
                if (!out->names || !out->bases || !out->len) { rc = CBCH_ERR_NOMEM; break; }
            }
            const uint8_t *q = p + 1;
            while (q < le && *q != ' ' && *q != '\t' && *q != '\r') q++;
            size_t nl_len = (size_t)(q - (p + 1));
            char *name = malloc(nl_len + 1);
            if (!name) { rc = CBCH_ERR_NOMEM; break; }
            memcpy(name, p + 1, nl_len); name[nl_len] = 0;
            /* record body: up to the next '>' at a line start; size bound = bytes until then */
            const uint8_t *body = nl ? nl + 1 : end, *scan = body, *next = end;
            while (scan < end) {
                if (*scan == '>') { next = scan; break; }
                const uint8_t *e2 = memchr(scan, '\n', (size_t)(end - scan));
                if (!e2) break;
                scan = e2 + 1;
            }
            uint8_t *bases = malloc((size_t)(next - body) + 1);
            if (!bases) { free(name); rc = CBCH_ERR_NOMEM; break; }
            uint64_t len = 0;
            for (const uint8_t *s = body; s < next;) {
                const uint8_t *e2 = memchr(s, '\n', (size_t)(next - s));
                const uint8_t *le2 = e2 ? e2 : next;
                size_t k = (size_t)(le2 - s);
                if (k && s[k - 1] == '\r') k--;
                memcpy(bases + len, s, k); len += k;
                s = e2 ? e2 + 1 : next;
            }
            out->names[out->n] = name; out->bases[out->n] = bases; out->len[out->n] = len; out->n++;
            p = next;
            continue;
        }
        p = nl ? nl + 1 : end;
    }
    unmap_file(&m);
    if (rc) { cbch_free_fasta(out); return fail(err, errlen, rc, "out of memory reading %s", path); }
    if (out->n == 0) return fail(err, errlen, CBCH_ERR_PARSE, "%s holds no FASTA record", path);
    return CBCH_OK;
}
void cbch_free_fasta(cbch_fasta *fa) {
    for (uint32_t i = 0; i < fa->n; i++) { free(fa->names[i]); free(fa->bases[i]); }
    free(fa->names); free(fa->bases); free(fa->len);
    memset(fa, 0, sizeof *fa);
}

/* ------------------------------------------------------------------ SAM */
static int grow(void **p, uint64_t *cap, uint64_t need, size_t elem) {
    if (need <= *cap) return 0;
    uint64_t c = *cap ? *cap : 1024;
    while (c < need) c += c / 2 + 1024;
    void *q = realloc(*p, (size_t)(c * elem));
    if (!q) return -1;
    *p = q; *cap = c;
    return 0;
}
static int reserve_reads(cbch_batch *b, uint64_t n, int with_md) {
    if (n <= b->cap) return 0;
    uint64_t c = b->cap ? b->cap : 4096;
    while (c < n) c += c / 2;
#define RS(field, extra) do { void *q = realloc(b->field, (size_t)((c + extra) * sizeof *b->field)); if (!q) return -1; b->field = q; } while (0)
    RS(pos, 0); RS(flag, 0); RS(seq_len, 0); RS(chr, 0); RS(seq_off, 1); RS(cigar_off, 1);
    if (with_md) RS(md_off, 1);
#undef RS
    b->cap = c;
    return 0;
}
static int parse_u32(const uint8_t *s, const uint8_t *e, uint32_t *v) {
    if (s >= e) return -1;
    uint64_t x = 0;
    for (; s < e; s++) { if (*s < '0' || *s > '9') return -1; x = x * 10 + (uint64_t)(*s - '0'); if (x > 0xffffffffull) return -1; }
    *v = (uint32_t)x;
    return 0;
}

/* One worker's share of the file: the lines of [begin, end) parsed into its own batch (pool offsets from 0), plus what
 * the merge needs to restate whole-file facts: the SEQ lengths of its first two records (get_read_length looks at the
 * file's second record, mapped or not) and its line count (error messages carry whole-file line numbers). */
typedef struct {
    const uint8_t *begin, *end;
    const cbch_fasta *fa;
    uint32_t flags;                      /* CBCH_DERIVE_MD: MD tags are not looked for, the part has no MD arrays */
    cbch_batch part;
    uint64_t records; uint32_t len1, len2;
    int rc; uint64_t err_line; char err[200];
} ingest_part;

static int part_fail(ingest_part *w, int rc, const char *fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(w->err, sizeof w->err, fmt, ap); va_end(ap);
    w->rc = rc; w->err_line = w->part.n_lines;
    return rc;
}

static void parse_range(ingest_part *w) {
    cbch_batch *b = &w->part;
    const cbch_fasta *fa = w->fa;
    memset(b, 0, sizeof *b);
    w->records = 0; w->len1 = w->len2 = 0; w->rc = CBCH_OK; w->err_line = 0; w->err[0] = 0;
    const uint8_t *p = w->begin, *end = w->end;
    int rc = CBCH_OK;
    uint32_t last_chr = 0; const uint8_t *last_name = NULL; size_t last_name_len = 0;
    /* sized from the range once (a record is at least 22 bytes of text, its SEQ / CIGAR / MD are substrings of it): no
       reallocation while parsing; untouched pages cost nothing */
    const uint64_t range = (uint64_t)(end - p);
    const int with_md = !(w->flags & CBCH_DERIVE_MD);
    if (reserve_reads(b, range / 22u + 16u, with_md) || grow((void **)&b->seq, &b->seq_cap, range + 64, 1) ||
        grow((void **)&b->cigar, &b->cigar_cap, range / 2u + 64, 1) || (with_md && grow((void **)&b->md, &b->md_cap, range / 2u + 64, 1))) rc = part_fail(w, CBCH_ERR_NOMEM, "out of memory");
    uint64_t so = 0, co = 0, mo = 0;
    while (!rc && p < end) {
        const uint8_t *nl = memchr(p, '\n', (size_t)(end - p));
        const uint8_t *le = nl ? nl : end;
        const uint8_t *line = p;
        p = nl ? nl + 1 : end;
        if (le > line && le[-1] == '\r') le--;
        b->n_lines++;
        if (le == line || *line == '@') continue;                 /* header (get_read_length skips them, :40-46) */
        /* the 11 mandatory fields */
        const uint8_t *f[12]; int nf = 0;
        const uint8_t *s = line;
        while (nf < 11) {
            const uint8_t *t = memchr(s, '\t', (size_t)(le - s));
            f[nf++] = s;
            if (!t) { s = le + 1; break; }
            s = t + 1;
        }
        if (nf < 11) { rc = part_fail(w, CBCH_ERR_PARSE, "fewer than 11 fields"); break; }
        f[11] = s;                                                /* start of the optional fields (or le + 1) */
#define FEND(i) ((i) < 10 ? f[(i) + 1] - 1 : (f[11] > le ? le : f[11] - 1))
        uint32_t flag, pos;
        if (parse_u32(f[1], FEND(1), &flag) || flag > 0xffffu || parse_u32(f[3], FEND(3), &pos)) { rc = part_fail(w, CBCH_ERR_PARSE, "bad FLAG or POS"); break; }
        const uint32_t seqlen = (uint32_t)(FEND(9) - f[9]);
        w->records++;
        if (w->records == 1) w->len1 = seqlen;
        if (w->records == 2) w->len2 = seqlen;
        if (flag & 4u) { b->n_unmapped++; continue; }             /* src/compression.c:50 */
        if (seqlen > 0xffffu) { rc = part_fail(w, CBCH_ERR_PARSE, "SEQ too long"); break; }
        /* RNAME -> ordinal (consecutive records mostly share it) */
        const uint8_t *rn = f[2]; size_t rl = (size_t)(FEND(2) - f[2]);
        uint32_t chr = last_chr;
        if (!(last_name && rl == last_name_len && !memcmp(rn, last_name, rl))) {
            uint32_t c;
            for (c = 0; c < fa->n; c++) if (strlen(fa->names[c]) == rl && !memcmp(fa->names[c], rn, rl)) break;
            if (c == fa->n) { rc = part_fail(w, CBCH_ERR_RNAME, "RNAME %.*s is not in the reference", (int)rl, rn); break; }
            chr = c; last_chr = c; last_name = rn; last_name_len = rl;
        }
        /* MD:Z among the optional fields (CBCH_DERIVE_MD: not looked for) */
        const uint8_t *md = NULL; size_t mdl = 0;
        for (const uint8_t *o = f[11]; with_md && o < le;) {
            const uint8_t *t = memchr(o, '\t', (size_t)(le - o));
            const uint8_t *oe = t ? t : le;
            if (oe - o >= 5 && o[0] == 'M' && o[1] == 'D' && o[2] == ':' && o[3] == 'Z' && o[4] == ':') { md = o + 5; mdl = (size_t)(oe - md); break; }
            o = oe + 1;
        }
        if (with_md && !md) { rc = part_fail(w, CBCH_ERR_NO_MD, "no MD:Z tag (README.md:25-29 requires it; -M derives it on the GPU)"); break; }
        const size_t cgl = (size_t)(FEND(5) - f[5]);
        if (reserve_reads(b, b->n_reads + 1, with_md) || grow((void **)&b->seq, &b->seq_cap, so + seqlen + 64, 1) ||
            grow((void **)&b->cigar, &b->cigar_cap, co + cgl + 64, 1) || (with_md && grow((void **)&b->md, &b->md_cap, mo + mdl + 64, 1))) { rc = part_fail(w, CBCH_ERR_NOMEM, "out of memory"); break; }
        const uint64_t r = b->n_reads++;
        b->pos[r] = pos; b->flag[r] = (uint16_t)flag; b->seq_len[r] = (uint16_t)seqlen; b->chr[r] = chr;
        b->seq_off[r] = so; memcpy(b->seq + so, f[9], seqlen); so += seqlen;
        b->cigar_off[r] = co; memcpy(b->cigar + co, f[5], cgl); co += cgl;
        if (with_md) { b->md_off[r] = mo; memcpy(b->md + mo, md, mdl); mo += mdl; }
        if (seqlen > b->max_len) b->max_len = seqlen;
    }
    if (!rc) { b->seq_off[b->n_reads] = so; b->cigar_off[b->n_reads] = co; if (with_md) b->md_off[b->n_reads] = mo; }
}

/* second phase of the threaded ingest: every worker copies its part to its place in the merged batch */
typedef struct { ingest_part *w; cbch_batch *dst; uint64_t r0, s0, c0, m0; } merge_job;
static void merge_part(merge_job *j) {
    const cbch_batch *s = &j->w->part; cbch_batch *d = j->dst;
    const uint64_t n = s->n_reads;
    if (!n) return;
    memcpy(d->pos + j->r0, s->pos, n * sizeof *d->pos); memcpy(d->flag + j->r0, s->flag, n * sizeof *d->flag);
    memcpy(d->seq_len + j->r0, s->seq_len, n * sizeof *d->seq_len); memcpy(d->chr + j->r0, s->chr, n * sizeof *d->chr);
    for (uint64_t r = 0; r < n; r++) { d->seq_off[j->r0 + r] = s->seq_off[r] + j->s0; d->cigar_off[j->r0 + r] = s->cigar_off[r] + j->c0; }
    memcpy(d->seq + j->s0, s->seq, s->seq_off[n]); memcpy(d->cigar + j->c0, s->cigar, s->cigar_off[n]);
    if (d->md_off) {                                              /* NULL: a batch without MD (CBCH_DERIVE_MD) */
        for (uint64_t r = 0; r < n; r++) d->md_off[j->r0 + r] = s->md_off[r] + j->m0;
        memcpy(d->md + j->m0, s->md, s->md_off[n]);
    }
    cbch_free_batch(&j->w->part);                                 /* every worker returns its own part (unmapping them one after the other on the caller's thread was a sixth of the ingest) */
}
static double now_s(void) { struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return (double)t.tv_sec + (double)t.tv_nsec * 1e-9; }
static void *parse_thread(void *arg) { parse_range((ingest_part *)arg); return NULL; }
static void *merge_thread(void *arg) { merge_part((merge_job *)arg); return NULL; }

int cbch_default_threads(void) {
    const char *e = getenv("CBCH_THREADS");
    long t = e ? atol(e) : sysconf(_SC_NPROCESSORS_ONLN);
    if (t < 1) t = 1;
    if (t > 64) t = 64;
    return (int)t;
}

int cbch_read_sam(const char *path, const cbch_fasta *fa, int var_length, cbch_batch *b, char *err, size_t errlen) {
    return cbch_read_sam_ex(path, fa, var_length, cbch_default_threads(), 0u, b, err, errlen);
}

/* The file is cut at line starts into n_threads ranges of about equal bytes; every worker parses its range into its own
 * batch, then copies it to its place in the merged one (two rounds of threads, no locks). The result does not depend
 * on n_threads. */
int cbch_map(const char *path, int populate, cbch_mapped *out) {
    out->p = NULL; out->n = 0;
    out->fd = open(path, O_RDONLY);
    if (out->fd < 0) return CBCH_ERR_IO;
    struct stat st;
    if (fstat(out->fd, &st)) { close(out->fd); out->fd = -1; return CBCH_ERR_IO; }
    out->n = (uint64_t)st.st_size;
    if (out->n == 0) return CBCH_OK;
    void *p = mmap(NULL, (size_t)out->n, PROT_READ, MAP_PRIVATE | (populate ? MAP_POPULATE : 0), out->fd, 0);
    if (p == MAP_FAILED) { close(out->fd); out->fd = -1; return CBCH_ERR_IO; }
    madvise(p, (size_t)out->n, MADV_SEQUENTIAL);
    out->p = (const uint8_t *)p;
    return CBCH_OK;
}
void cbch_unmap(cbch_mapped *m) { if (m->p) munmap((void *)m->p, (size_t)m->n); if (m->fd >= 0) close(m->fd); m->p = NULL; m->fd = -1; }
const uint8_t *cbch_next_line(const uint8_t *p, const uint8_t *end) {
    const uint8_t *nl = p < end ? memchr(p, '\n', (size_t)(end - p)) : NULL;
    return nl ? nl + 1 : end;
}

int cbch_read_sam_mt(const char *path, const cbch_fasta *fa, int var_length, int n_threads, cbch_batch *b, char *err, size_t errlen) {
    return cbch_read_sam_ex(path, fa, var_length, n_threads, 0u, b, err, errlen);
}
int cbch_read_sam_ex(const char *path, const cbch_fasta *fa, int var_length, int n_threads, uint32_t flags, cbch_batch *b, char *err, size_t errlen) {
    memset(b, 0, sizeof *b);
    mapped m;
    if (map_file(path, &m)) return fail(err, errlen, CBCH_ERR_IO, "cannot open %s", path);
    const int rc = cbch_ingest_range_ex(m.p, m.p + m.n, fa, var_length, n_threads, 0, flags, b, err, errlen);
    unmap_file(&m);
    return rc;
}

/* The lines of [begin, end) (begin at a line start). header_len != 0: the read length of the stream header is given
 * (a later batch of a file takes the first batch's: get_read_length looks at the file's second record). */
int cbch_ingest_range(const uint8_t *begin, const uint8_t *range_end, const cbch_fasta *fa, int var_length, int n_threads, uint32_t header_len,
                      cbch_batch *b, char *err, size_t errlen) {
    return cbch_ingest_range_ex(begin, range_end, fa, var_length, n_threads, header_len, 0u, b, err, errlen);
}
int cbch_ingest_range_ex(const uint8_t *begin, const uint8_t *range_end, const cbch_fasta *fa, int var_length, int n_threads, uint32_t header_len,
                         uint32_t flags, cbch_batch *b, char *err, size_t errlen) {
    memset(b, 0, sizeof *b);
    const int with_md = !(flags & CBCH_DERIVE_MD);
    const char *path = "the SAM input";
    struct { const uint8_t *p; size_t n; } m = { begin, (size_t)(range_end - begin) };
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 64) n_threads = 64;
    if (m.n < (size_t)n_threads * 4096u) n_threads = (int)(m.n / 4096u) + 1;       /* small files: fewer workers */
    ingest_part *w = calloc((size_t)n_threads, sizeof *w);
    merge_job *jobs = calloc((size_t)n_threads, sizeof *jobs);
    pthread_t *th = calloc((size_t)n_threads, sizeof *th);
    if (!w || !jobs || !th) { free(w); free(jobs); free(th); return fail(err, errlen, CBCH_ERR_NOMEM, "out of memory"); }
    const uint8_t *end = m.p + m.n, *cur = m.p;
    for (int t = 0; t < n_threads; t++) {
        const uint8_t *stop = end;
        if (t + 1 < n_threads) {
            const uint8_t *guess = m.p + m.n / (size_t)n_threads * (size_t)(t + 1);
            if (guess < cur) guess = cur;
            const uint8_t *nl = guess < end ? memchr(guess, '\n', (size_t)(end - guess)) : NULL;
            stop = nl ? nl + 1 : end;
        }
        w[t].begin = cur; w[t].end = stop; w[t].fa = fa; w[t].flags = flags;
        cur = stop;
    }
    const int trace = getenv("CBCH_TRACE") != NULL;
    const double t_begin = now_s();
    int started = 0;
    for (int t = 1; t < n_threads; t++) { if (pthread_create(&th[t], NULL, parse_thread, &w[t])) break; started = t; }
    for (int t = started + 1; t < n_threads; t++) parse_range(&w[t]);           /* threads that could not start: here */
    parse_range(&w[0]);
    for (int t = 1; t <= started; t++) pthread_join(th[t], NULL);
    const double t_parsed = now_s();

    /* whole-file facts, and the first error in file order */
    int rc = CBCH_OK;
    uint64_t lines = 0, records = 0, n = 0, so = 0, co = 0, mo = 0; uint32_t lens[2] = { 0, 0 };
    for (int t = 0; t < n_threads && !rc; t++) {
        if (w[t].rc) {
            rc = w[t].rc;
            if (rc == CBCH_ERR_NOMEM) fail(err, errlen, rc, "out of memory reading %s", path);
            else fail(err, errlen, rc, "line %llu: %s", (unsigned long long)(lines + w[t].err_line), w[t].err);
            break;
        }
        if (records < 2 && w[t].records) { lens[records] = w[t].len1; if (records == 0 && w[t].records >= 2) lens[1] = w[t].len2; }
        records += w[t].records;
        jobs[t].w = &w[t]; jobs[t].dst = b; jobs[t].r0 = n; jobs[t].s0 = so; jobs[t].c0 = co; jobs[t].m0 = mo;
        n += w[t].part.n_reads; lines += w[t].part.n_lines; b->n_unmapped += w[t].part.n_unmapped;
        if (w[t].part.n_reads) { so += w[t].part.seq_off[w[t].part.n_reads]; co += w[t].part.cigar_off[w[t].part.n_reads]; if (with_md) mo += w[t].part.md_off[w[t].part.n_reads]; }
        if (w[t].part.max_len > b->max_len) b->max_len = w[t].part.max_len;
    }
    if (!rc) {
        if (reserve_reads(b, n + 1, with_md) || grow((void **)&b->seq, &b->seq_cap, so + 64, 1) || grow((void **)&b->cigar, &b->cigar_cap, co + 64, 1) ||
            (with_md && grow((void **)&b->md, &b->md_cap, mo + 64, 1))) rc = fail(err, errlen, CBCH_ERR_NOMEM, "out of memory reading %s", path);
    }
    if (!rc) {
        b->n_reads = n; b->n_lines = lines;
        started = 0;
        for (int t = 1; t < n_threads; t++) { if (pthread_create(&th[t], NULL, merge_thread, &jobs[t])) break; started = t; }
        for (int t = started + 1; t < n_threads; t++) merge_part(&jobs[t]);
        merge_part(&jobs[0]);
        for (int t = 1; t <= started; t++) pthread_join(th[t], NULL);
        b->seq_off[n] = so; b->cigar_off[n] = co; if (with_md) b->md_off[n] = mo;
        /* get_read_length (:47-53): fixed-length mode takes the SECOND record's SEQ length; -l takes the maximum */
        b->read_len_header = var_length ? b->max_len : header_len ? header_len : (records >= 2 ? lens[1] : lens[0]);
    }
    const double t_merged = now_s();
    for (int t = 0; t < n_threads; t++) cbch_free_batch(&w[t].part);
    free(w); free(jobs); free(th);
    if (trace) fprintf(stderr, "[cbch ingest] %d workers: parse %.1f ms, merge %.1f ms, free %.1f ms\n", n_threads, (t_parsed - t_begin) * 1e3,
                       (t_merged - t_parsed) * 1e3, (now_s() - t_merged) * 1e3);
    if (rc) { cbch_free_batch(b); return rc; }
    return CBCH_OK;
}

void cbch_free_batch(cbch_batch *b) {
    free(b->pos); free(b->flag); free(b->seq_len); free(b->chr); free(b->seq_off); free(b->cigar_off); free(b->md_off);
    free(b->seq); free(b->cigar); free(b->md);
    memset(b, 0, sizeof *b);
}

void cbch_batch_view(const cbch_batch *b, cbcg_batch *v) {
    v->n_reads = b->n_reads; v->pos = b->pos; v->flag = b->flag; v->seq_len = b->seq_len; v->chr = b->chr;
    v->seq_off = b->seq_off; v->seq = b->seq; v->cigar_off = b->cigar_off; v->cigar = b->cigar; v->md_off = b->md_off; v->md = b->md;
}


/* ------------------------------------------------------------------------------------------------ compact batches */
typedef struct {
    const cbcg_batch *b; cbch_compact *c; uint64_t r0, r1;
    uint8_t *seq2; uint16_t *cl, *ml; uint64_t *so;
    uint32_t *pos; uint16_t *flag, *sl; uint8_t *cig, *md;      /* every worker also copies its reads' fixed fields and CIGAR / MD text */
    uint64_t n_exc; uint32_t *er; uint16_t *eb; uint8_t *ec; uint64_t exc_cap; int oom;
} pack_job;
static inline unsigned base2(uint8_t ch) { return ch == 'A' ? 0u : ch == 'C' ? 1u : ch == 'G' ? 2u : ch == 'T' ? 3u : 4u; }
/* Eight bases at once: the 2-bit code of A / C / G / T is ((c >> 1) ^ (c >> 2)) & 3 (A 0, C 1, G 2, T 3, the order of
 * base2 and of the device's unpack); the ASCII letter is rebuilt from the code and compared with the input, so anything that
 * is not one of the four upper-case letters sends the group to the byte-by-byte path (which lists it as an exception).
 * Bases k = 0 .. 3 of a byte sit at bits 2k, as below. Returns 0 when the group needs the slow path. */
static inline int pack8(const uint8_t *s, uint8_t *d2) {
    uint64_t x; memcpy(&x, s, 8);
#if defined(__BYTE_ORDER__) && __BYTE_ORDER__ != __ORDER_LITTLE_ENDIAN__
    return 0;
#endif
    const uint64_t L = 0x0101010101010101ull;
    const uint64_t y = ((x >> 1) ^ (x >> 2)) & (3u * L);
    const uint64_t c0 = y & L, c1 = (y >> 1) & L, both = c0 & c1;
    const uint64_t e = (0x40u * L) | (both << 4) | (c1 << 2) | ((c1 ^ c0) << 1) | (both ^ L);
    if (x != e) return 0;
    const uint32_t lo = (uint32_t)y, hi = (uint32_t)(y >> 32);
    d2[0] = (uint8_t)(lo | (lo >> 6) | (lo >> 12) | (lo >> 18));
    d2[1] = (uint8_t)(hi | (hi >> 6) | (hi >> 12) | (hi >> 18));
    return 1;
}
static void pack_part(pack_job *j) {
    const cbcg_batch *b = j->b;
    if (j->r1 > j->r0) {
        const uint64_t m = j->r1 - j->r0, c0 = b->cigar_off[0];
        memcpy(j->pos + j->r0, b->pos + j->r0, m * 4); memcpy(j->flag + j->r0, b->flag + j->r0, m * 2); memcpy(j->sl + j->r0, b->seq_len + j->r0, m * 2);
        memcpy(j->cig + (b->cigar_off[j->r0] - c0), b->cigar + b->cigar_off[j->r0], b->cigar_off[j->r1] - b->cigar_off[j->r0]);
        if (b->md_off) memcpy(j->md + (b->md_off[j->r0] - b->md_off[0]), b->md + b->md_off[j->r0], b->md_off[j->r1] - b->md_off[j->r0]);
    }
    for (uint64_t r = j->r0; r < j->r1; r++) {
        const uint8_t *s = b->seq + b->seq_off[r];
        const uint32_t len = b->seq_len[r];
        uint8_t *d = j->seq2 + j->so[r];
        for (uint32_t i = 0; i < len; i += 4) {
            if (i + 8u <= len && !(i & 4u) && pack8(s + i, d + (i >> 2))) { i += 4; continue; }   /* two bytes done: skip the second group too */
            unsigned byte = 0;
            for (uint32_t k = 0; k < 4 && i + k < len; k++) {
                unsigned c2 = base2(s[i + k]);
                if (c2 > 3u) {
                    if (j->n_exc == j->exc_cap) {
                        uint64_t nc = j->exc_cap ? j->exc_cap * 2 : 1024;
                        uint32_t *er = realloc(j->er, nc * 4); uint16_t *eb = realloc(j->eb, nc * 2); uint8_t *ec = realloc(j->ec, nc);
                        if (!er || !eb || !ec) { j->oom = 1; free(er ? er : j->er); free(eb ? eb : j->eb); free(ec ? ec : j->ec); j->er = NULL; j->eb = NULL; j->ec = NULL; return; }
                        j->er = er; j->eb = eb; j->ec = ec; j->exc_cap = nc;
                    }
                    j->er[j->n_exc] = (uint32_t)r; j->eb[j->n_exc] = (uint16_t)(i + k); j->ec[j->n_exc] = s[i + k]; j->n_exc++;
                    c2 = 0;
                }
                byte |= c2 << (2 * k);
            }
            d[i >> 2] = (uint8_t)byte;
        }
        j->cl[r] = (uint16_t)(b->cigar_off[r + 1] - b->cigar_off[r]);
        if (b->md_off) j->ml[r] = (uint16_t)(b->md_off[r + 1] - b->md_off[r]);
    }
}
static void *pack_thread(void *arg) { pack_part((pack_job *)arg); return NULL; }

void cbch_free_compact(cbch_compact *c) {
    if (!c) return;
    void (*rel)(void *) = c->release ? c->release : free;
    cbcg_batch_compact *v = &c->v;
    rel((void *)v->pos); rel((void *)v->flag); rel((void *)v->seq_len); rel((void *)v->cigar_len); rel((void *)v->md_len);
    rel((void *)v->run_first); rel((void *)v->run_chr); rel((void *)v->seq2); rel((void *)v->exc_read); rel((void *)v->exc_base); rel((void *)v->exc_char);
    rel((void *)v->cigar); rel((void *)v->md);
    rel((void *)v->tile_base);
    memset(c, 0, sizeof *c);
}

int cbch_pack_batch(const cbcg_batch *b, int n_threads, void *(*alloc)(size_t), void (*release)(void *), cbch_compact *out) {
    memset(out, 0, sizeof *out);
    if (!alloc) { alloc = malloc; release = free; }
    out->alloc = alloc; out->release = release;
    const uint64_t n = b->n_reads;
    cbcg_batch_compact *v = &out->v;
    v->n_reads = n;
    if (!n) return CBCH_OK;
    if (n_threads <= 0) n_threads = cbch_default_threads();
    if ((uint64_t)n_threads > n) n_threads = (int)n;
    const int trace = getenv("CBCH_TRACE") != NULL;
    const double t_begin = now_s();
    uint64_t *so = malloc((n + 1) * 8);
    if (!so) return CBCH_ERR_NOMEM;
    uint64_t o = 0, n_runs = 0;
    uint32_t mx = 0, mn = 0xffffffffu;
    for (uint64_t r = 0; r < n; r++) {
        const uint32_t l = b->seq_len[r];
        so[r] = o; o += ((uint64_t)l + 3u) >> 2;
        if (l > mx) mx = l;
        if (l < mn) mn = l;
        if (r == 0 || b->chr[r] != b->chr[r - 1]) n_runs++;
    }
    so[n] = o;
    const int with_md = b->md_off != NULL;                    /* without MD: md_len = md = NULL and a zero MD column */
    const uint64_t s0 = b->seq_off[0], c0 = b->cigar_off[0], m0 = with_md ? b->md_off[0] : 0, co_n = b->cigar_off[n] - c0, mo_n = with_md ? b->md_off[n] - m0 : 0;
    {   /* one entry per tile of 128 reads, and the totals */
        const uint64_t tiles = (n + 127u) / 128u;
        uint64_t *tb = alloc((tiles + 1) * 32);
        v->tile_base = tb;
        if (!tb) { free(so); return CBCH_ERR_NOMEM; }
        for (uint64_t t = 0; t <= tiles; t++) { const uint64_t r = t * 128u < n ? t * 128u : n; tb[4 * t] = b->seq_off[r] - s0; tb[4 * t + 1] = so[r]; tb[4 * t + 2] = b->cigar_off[r] - c0; tb[4 * t + 3] = with_md ? b->md_off[r] - m0 : 0; }
        v->max_len = mx; v->min_len = mn;
    }
    uint32_t *pos = alloc(n * 4); uint16_t *flag = alloc(n * 2), *sl = alloc(n * 2), *cl = alloc(n * 2), *ml = with_md ? alloc(n * 2) : NULL;
    uint64_t *rf = alloc(n_runs * 8); uint32_t *rc = alloc(n_runs * 4);
    uint8_t *seq2 = alloc(o + 64), *cig = alloc(co_n + 64), *md = with_md ? alloc(mo_n + 64) : NULL;
    v->pos = pos; v->flag = flag; v->seq_len = sl; v->cigar_len = cl; v->md_len = ml; v->run_first = rf; v->run_chr = rc; v->seq2 = seq2; v->cigar = cig; v->md = md;
    if (!pos || !flag || !sl || !cl || (with_md && (!ml || !md)) || !rf || !rc || !seq2 || !cig) { free(so); cbch_free_compact(out); return CBCH_ERR_NOMEM; }
    { uint64_t k = 0; for (uint64_t r = 0; r < n; r++) if (r == 0 || b->chr[r] != b->chr[r - 1]) { rf[k] = r; rc[k] = b->chr[r]; k++; } v->n_runs = (uint32_t)n_runs; }
    const double t_head = now_s();
    pack_job *jobs = calloc((size_t)n_threads, sizeof *jobs);
    pthread_t *th = calloc((size_t)n_threads, sizeof *th);
    if (!jobs || !th) { free(jobs); free(th); free(so); cbch_free_compact(out); return CBCH_ERR_NOMEM; }
    for (int t = 0; t < n_threads; t++) {
        jobs[t].b = b; jobs[t].c = out; jobs[t].r0 = n * (uint64_t)t / (uint64_t)n_threads; jobs[t].r1 = n * (uint64_t)(t + 1) / (uint64_t)n_threads;
        jobs[t].seq2 = seq2; jobs[t].cl = cl; jobs[t].ml = ml; jobs[t].so = so;
        jobs[t].pos = pos; jobs[t].flag = flag; jobs[t].sl = sl; jobs[t].cig = cig; jobs[t].md = md;
    }
    int started = 0;
    for (int t = 1; t < n_threads; t++) { if (pthread_create(&th[t], NULL, pack_thread, &jobs[t])) break; started = t; }
    for (int t = started + 1; t < n_threads; t++) pack_part(&jobs[t]);
    pack_part(&jobs[0]);
    for (int t = 1; t <= started; t++) pthread_join(th[t], NULL);
    if (trace) fprintf(stderr, "[cbch pack] %d workers: offsets + copies %.1f ms, bases %.1f ms\n", n_threads, (t_head - t_begin) * 1e3, (now_s() - t_head) * 1e3);
    uint64_t n_exc = 0; int oom = 0;
    for (int t = 0; t < n_threads; t++) { n_exc += jobs[t].n_exc; oom |= jobs[t].oom; }
    if (!oom && n_exc) {
        uint32_t *er = alloc(n_exc * 4); uint16_t *eb = alloc(n_exc * 2); uint8_t *ec = alloc(n_exc);
        v->exc_read = er; v->exc_base = eb; v->exc_char = ec;
        if (!er || !eb || !ec) oom = 1;
        else { uint64_t k = 0; for (int t = 0; t < n_threads; t++) { memcpy(er + k, jobs[t].er, jobs[t].n_exc * 4); memcpy(eb + k, jobs[t].eb, jobs[t].n_exc * 2); memcpy(ec + k, jobs[t].ec, jobs[t].n_exc); k += jobs[t].n_exc; } }
    }
    v->n_exc = oom ? 0 : n_exc;
    for (int t = 0; t < n_threads; t++) { free(jobs[t].er); free(jobs[t].eb); free(jobs[t].ec); }
    free(jobs); free(th);
    out->bytes = n * (4 + 2 + 2 + 2 + (with_md ? 2 : 0)) + o + co_n + mo_n + n_runs * 12 + n_exc * 7 + ((n + 127u) / 128u + 1) * 32;
    free(so);
    if (oom) { cbch_free_compact(out); return CBCH_ERR_NOMEM; }
    return CBCH_OK;
}
