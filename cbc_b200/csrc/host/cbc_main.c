/*
 * cbc_main.c -- the reference's command line over the B200 path.
 *
 *   cbc -c <sam> <out> <ref.fa>     compress   (README.md:59;  checked-in spelling `-c <ratio> ...`, src/main.c:114-123, also accepted)
 *   cbc -d <in>  <out> <ref.fa>     decompress (README.md:67;  checked-in spelling `-x`, src/main.c:136-139, also accepted)
 * options: -b N     reads per block (default: sized by the library, CBCG_BLOCK_AUTO; the container is the blocked "CBCB" format)
 *          -1       single-block mode: the reference's own stream, byte-identical to `program -c 1` built with -DDEBUG
 *          -l       variable-length reads: header read length = longest SEQ (src/main.c -l)
 *          -g LIST  CUDA devices, e.g. `-g 0,1,2,3`: batches (region shards of the sorted input) are dealt out to them
 *          -B MB    SAM text per batch (default 2048): memory is bounded by three batches whatever the file size
 *          -M       -c only: the input's MD:Z tags are not read (records need none); every read's MD is derived on the GPU from its
 *                   CIGAR, SEQ and the reference (cbcg.h, "a batch without MD"), so an aligner's output without --MD codes as it
 *                   would after `samtools calmd`. The container is the one the derived MD gives, and nothing in it records -M.
 *                   A read whose CIGAR's query length is not its SEQ length is refused. Without -M a record without MD:Z is an error.
 *          -C       CIGAR recovery (SURVEY.md 8f row 4; cbcg_cigar_pack / cbcg_cigar_unpack): -c also writes <out>.cig, the side
 *                   sections of the batches (u64 length + section each); -d reads <in>.cig and writes "CIGAR<TAB>SEQ" lines
 *          -r NAME[:START[-END]]   -d only, repeatable: write only the reads that overlap one of the regions (1-based, inclusive;
 *                   cbcg_decode_region), each once, in file order. The region is split at the last ':', so record names that
 *                   contain one still work. Every batch of a "CBCS" file gets the same regions; a batch that none of them
 *                   touches (cbcg_region_plan: no blocks) makes no device call. Not with -C unless with -S.
 *          -S       -d only: write SAM (cbcg_decode_sam): a header, then one alignment record per read (QNAME, MAPQ, mate fields
 *                   and QUAL are not stored: `*`, 255, `*`, 0, 0, `*`), with NM and MD recomputed against the reference. The
 *                   header is written once: for a "CBCB" or "CBCS" input from batch 0's chromosome table (cbcg_sam_header; a
 *                   later batch whose table differs is an error), for a single-block stream from the reference; LN comes
 *                   from the reference. With -C the CIGARs are the input's (<in>.cig), else the ones the indels imply.
 *                   With -r only the region's records.
 *
 * Host C only: SAM/FASTA ingest (sam_ingest.c) and file I/O; the coding runs on the GPU through include/cbcg.h.
 * Where the reference's compress() (src/compression.c:112-170) reads a line, codes it and moves on, this driver
 * pipelines: an ingest thread parses and packs batch k + 1 (all host cores) while a device thread per GPU codes batch
 * k and the main thread writes batch k - 1; GPU start-up (context, reference upload) runs beside the first ingest.
 * One batch: the output is a "CBCB" container. Several: a "CBCS" file, one self-contained container per batch
 * (cbc_b200/shard.py reads and writes the same layout). Prints the reference's progress lines
 * (src/compression.c:157,166,206). Returns 0 on success (the reference's main returns 1, src/main.c:370).
 */
#define _GNU_SOURCE
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <sys/mman.h>

#include "cbcg.h"
#include "sam_ingest.h"

#define MAX_DEV 16
#define CBCS_MAGIC 0x53434243u

static uint32_t rd_u32(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }
static double now(void) { struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec; }

static int usage(void) {
    fprintf(stderr, "usage: cbc -c [-1] [-l] [-C] [-M] [-b reads_per_block] [-g devices] [-B batch_MB] <sam> <out> <ref.fa>\n"
                    "       cbc -d [-C] [-g devices] <in> <out> <ref.fa>\n"
                    "       cbc -d -r NAME[:START[-END]] [-r ...] [-g devices] <in> <out> <ref.fa>\n"
                    "       cbc -d -S [-C] [-r NAME[:START[-END]] ...] [-g devices] <in> <out.sam> <ref.fa>\n");
    return 2;
}

/* ---- a unit of work travelling ingest -> device -> writer */
typedef struct job {
    uint64_t index;
    /* compress */
    cbch_batch hb; cbch_compact cb; int have_compact;
    /* decompress */
    const uint8_t *in; uint64_t in_len; int legacy;
    /* CIGAR recovery (-C): compress: the batch's side section; decompress: in = its section, out = the CIGAR lines */
    const uint8_t *cig_in; uint64_t cig_in_len;
    uint8_t *cig; uint64_t cig_len;
    /* result */
    uint8_t *out; uint64_t out_len; uint64_t n_reads; float device_ms; uint64_t n_blocks;
    int rc; char err[256];
    int done, written;
    uint64_t bound, seq_bases; uint32_t header_len;
} job;

typedef struct shared {
    pthread_mutex_t mu; pthread_cond_t cv;
    job **jobs; uint64_t n_jobs;                /* all jobs, by index */
    uint64_t produced;                          /* jobs [0, produced) are ready for a device */
    uint64_t next_take;                         /* next job a device thread takes */
    int producer_failed;
    /* run parameters */
    int mode, single, var_length, with_cigar, sam, derive_md; uint32_t block_reads;
    const cbch_fasta *fa; int fa_ready;
    const cbcg_region *regions; uint32_t n_regions;     /* -r: region decode */
    double t_gpu_ready;
} shared;

typedef struct devthread { shared *S; int device; pthread_t th; int rc; char err[256]; double create_s, setref_s, call_s, alloc_s; } devthread;

static void *device_main(void *arg) {
    devthread *D = (devthread *)arg;
    shared *S = D->S;
    cbcg_ctx *ctx = NULL;
    double tq = now();
    int rc = cbcg_create(D->device, &ctx);                       /* context creation runs beside the FASTA / SAM ingest */
    D->create_s = now() - tq;
    if (rc) { snprintf(D->err, sizeof D->err, "device %d: %s", D->device, cbcg_strerror(rc)); D->rc = rc; }
    pthread_mutex_lock(&S->mu);
    while (!S->fa_ready) pthread_cond_wait(&S->cv, &S->mu);
    pthread_mutex_unlock(&S->mu);
    tq = now();
    if (!rc) {
        rc = cbcg_set_reference(ctx, S->fa->n, (const char *const *)S->fa->names, (const uint8_t *const *)S->fa->bases, S->fa->len);
        if (rc) { snprintf(D->err, sizeof D->err, "device %d: %s", D->device, cbcg_last_error(ctx)); D->rc = rc; }
    }
    D->setref_s = now() - tq;
    pthread_mutex_lock(&S->mu);
    if (S->t_gpu_ready == 0) S->t_gpu_ready = now();
    pthread_mutex_unlock(&S->mu);
    for (;;) {
        pthread_mutex_lock(&S->mu);
        while (S->next_take >= S->produced && S->next_take < S->n_jobs && !S->producer_failed) pthread_cond_wait(&S->cv, &S->mu);
        if (S->next_take >= S->n_jobs || (S->producer_failed && S->next_take >= S->produced)) { pthread_mutex_unlock(&S->mu); break; }
        job *J = S->jobs[S->next_take++];
        pthread_mutex_unlock(&S->mu);
        if (D->rc) { J->rc = D->rc; snprintf(J->err, sizeof J->err, "%s", D->err); }
        else if (S->mode == 'c') {
            cbcg_encode_opts o = { J->header_len ? J->header_len : 1u, S->single ? 0u : S->block_reads, S->single ? 0u : 1u, 0u };
            cbcg_batch v; cbch_batch_view(&J->hb, &v);
            uint64_t cap = J->bound, n = 0;
            tq = now();
            J->out = (uint8_t *)malloc(cap ? cap : 1);
            if (!J->out) { J->rc = CBCG_ERR_NOMEM; snprintf(J->err, sizeof J->err, "out of memory"); }
            else {
                rc = J->have_compact ? cbcg_encode_compact(ctx, &J->cb.v, &o, J->out, cap, &n) : cbcg_encode(ctx, &v, &o, J->out, cap, &n);
                if (rc == CBCG_ERR_CAPACITY && n > cap) { free(J->out); J->out = (uint8_t *)malloc(n); rc = J->out ? cbcg_fetch_container(ctx, J->out, n, &n) : CBCG_ERR_NOMEM; }
                if (rc) { J->rc = rc; snprintf(J->err, sizeof J->err, "%s", cbcg_last_error(ctx)); }
                J->out_len = n;
                D->call_s += now() - tq;
                cbcg_stats st; cbcg_get_stats(ctx, &st); J->device_ms = st.ms_total; J->n_blocks = st.n_blocks;
                if (!rc && S->with_cigar) {                       /* the batch is still whole (ingest kept it) */
                    uint64_t ccap = cbcg_cigar_bound(&v), cn = 0;
                    J->cig = (uint8_t *)malloc(ccap ? ccap : 1);
                    rc = J->cig ? cbcg_cigar_pack(ctx, &v, J->cig, ccap, &cn) : CBCG_ERR_NOMEM;
                    if (rc) { J->rc = rc; snprintf(J->err, sizeof J->err, "%s", cbcg_last_error(ctx)); }
                    J->cig_len = cn;
                }
            }
            if (J->have_compact) cbch_free_compact(&J->cb);
        } else if (S->sam) {                                      /* SAM records; the writer adds the header */
            uint64_t nb = 1, n_reads = 0, pb = 0, cap = 0, n = 0;
            if (S->n_regions) {
                rc = cbcg_region_plan(J->in, J->in_len, J->legacy, S->regions, S->n_regions, &nb, &n_reads, &pb, &cap);
                if (rc) { J->rc = rc; snprintf(J->err, sizeof J->err, "region plan: %s", cbcg_strerror(rc)); nb = 0; }
            }
            if (nb) {                                             /* a batch that no region touches costs no device call */
                if (J->legacy || cbcg_decoded_size(J->in, J->in_len, &n_reads, &cap) != CBCG_OK) cap = 1u << 20;
                cap = 2 * cap + (1u << 16);                       /* SAM lines: about SEQ + 60 bytes */
                tq = now();
                J->out = (uint8_t *)malloc(cap);
                rc = J->out ? cbcg_decode_sam(ctx, J->in, J->in_len, J->legacy, S->with_cigar ? J->cig_in : NULL, S->with_cigar ? J->cig_in_len : 0,
                                              S->n_regions ? S->regions : NULL, S->n_regions, 0u, J->out, cap, &n, NULL, 0, &n_reads) : CBCG_ERR_NOMEM;
                if (rc == CBCG_ERR_CAPACITY && n > cap) { free(J->out); J->out = (uint8_t *)malloc(n); rc = J->out ? cbcg_fetch_decoded(ctx, J->out, n, &n) : CBCG_ERR_NOMEM; }
                if (rc) { J->rc = rc; snprintf(J->err, sizeof J->err, "%s", ctx ? cbcg_last_error(ctx) : "no context"); }
                J->out_len = n; J->n_reads = n_reads;
                D->call_s += now() - tq;
                cbcg_stats st; cbcg_get_stats(ctx, &st); J->device_ms = st.ms_total;
            }
        } else if (S->n_regions) {
            uint64_t nb = 0, n_reads = 0, pb = 0, cap = 0, n = 0;
            rc = cbcg_region_plan(J->in, J->in_len, J->legacy, S->regions, S->n_regions, &nb, &n_reads, &pb, &cap);
            if (rc) { J->rc = rc; snprintf(J->err, sizeof J->err, "region plan: %s", cbcg_strerror(rc)); }
            else if (nb) {                                        /* a batch that no region touches costs no device call */
                if (J->legacy) cap = 1u << 20;
                tq = now();
                J->out = (uint8_t *)malloc(cap ? cap : 1);
                rc = J->out ? cbcg_decode_region(ctx, J->in, J->in_len, J->legacy, S->regions, S->n_regions, J->out, cap, &n, NULL, 0, &n_reads) : CBCG_ERR_NOMEM;
                if (rc == CBCG_ERR_CAPACITY && n > cap) { free(J->out); J->out = (uint8_t *)malloc(n); rc = J->out ? cbcg_fetch_decoded(ctx, J->out, n, &n) : CBCG_ERR_NOMEM; }
                if (rc) { J->rc = rc; snprintf(J->err, sizeof J->err, "%s", ctx ? cbcg_last_error(ctx) : "no context"); }
                J->out_len = n; J->n_reads = n_reads;
                D->call_s += now() - tq;
                cbcg_stats st; cbcg_get_stats(ctx, &st); J->device_ms = st.ms_total;
            }
        } else {
            uint64_t n_reads = 0, cap = 0, n = 0;
            if (!J->legacy && cbcg_decoded_size(J->in, J->in_len, &n_reads, &cap) != CBCG_OK) { J->rc = CBCG_ERR_FORMAT; snprintf(J->err, sizeof J->err, "malformed container"); }
            else {
                if (J->legacy) cap = 1u << 20;
                tq = now();
                J->out = (uint8_t *)malloc(cap ? cap : 1);
                rc = J->out ? cbcg_decode(ctx, J->in, J->in_len, J->legacy, J->out, cap, &n, &n_reads) : CBCG_ERR_NOMEM;
                if (rc == CBCG_ERR_CAPACITY && n > cap) { free(J->out); J->out = (uint8_t *)malloc(n); rc = J->out ? cbcg_fetch_decoded(ctx, J->out, n, &n) : CBCG_ERR_NOMEM; }
                if (rc) { J->rc = rc; snprintf(J->err, sizeof J->err, "%s", ctx ? cbcg_last_error(ctx) : "no context"); }
                J->out_len = n; J->n_reads = n_reads;
                D->call_s += now() - tq;
                cbcg_stats st; cbcg_get_stats(ctx, &st); J->device_ms = st.ms_total;
                if (!rc && S->with_cigar) {
                    uint64_t ccap = J->in_len * 4 + (1u << 16), cn = 0, nr2 = 0;
                    J->cig = (uint8_t *)malloc(ccap);
                    rc = J->cig ? cbcg_cigar_unpack(ctx, J->in, J->in_len, J->legacy, J->cig_in, J->cig_in_len, J->cig, ccap, &cn, &nr2) : CBCG_ERR_NOMEM;
                    if (rc == CBCG_ERR_CAPACITY && cn > ccap) {
                        free(J->cig); J->cig = (uint8_t *)malloc(cn); ccap = cn;
                        rc = J->cig ? cbcg_cigar_unpack(ctx, J->in, J->in_len, J->legacy, J->cig_in, J->cig_in_len, J->cig, ccap, &cn, &nr2) : CBCG_ERR_NOMEM;
                    }
                    if (rc) { J->rc = rc; snprintf(J->err, sizeof J->err, "%s", cbcg_last_error(ctx)); }
                    J->cig_len = cn;
                }
            }
        }
        pthread_mutex_lock(&S->mu);
        J->done = 1;
        pthread_cond_broadcast(&S->cv);
        pthread_mutex_unlock(&S->mu);
    }
    if (ctx) cbcg_destroy(ctx);
    return NULL;
}

static void publish(shared *S, int failed) {
    pthread_mutex_lock(&S->mu);
    if (failed) S->producer_failed = 1; else S->produced++;
    pthread_cond_broadcast(&S->cv);
    pthread_mutex_unlock(&S->mu);
}
static job *wait_done(shared *S, uint64_t k) {
    pthread_mutex_lock(&S->mu);
    while (!S->jobs[k]->done && !(S->producer_failed && k >= S->produced)) pthread_cond_wait(&S->cv, &S->mu);
    job *J = S->jobs[k]->done ? S->jobs[k] : NULL;
    pthread_mutex_unlock(&S->mu);
    return J;
}

/* ---- compress: the ingest thread */
typedef struct ingest_arg { shared *S; const cbch_mapped *map; const uint8_t **cut; double ingest_s; uint64_t n_unmapped; int rc; char err[256]; uint64_t window; } ingest_arg;
static void *ingest_main(void *arg) {
    ingest_arg *A = (ingest_arg *)arg;
    shared *S = A->S;
    uint32_t header_len = 0;
    for (uint64_t k = 0; k < S->n_jobs; k++) {
        /* at most `window` batches between ingest and the writer: memory stays bounded */
        pthread_mutex_lock(&S->mu);
        while (k >= A->window && !S->jobs[k - A->window]->written && !S->producer_failed) pthread_cond_wait(&S->cv, &S->mu);
        pthread_mutex_unlock(&S->mu);
        job *J = S->jobs[k];
        const double t0 = now();
        int rc = cbch_ingest_range_ex(A->cut[k], A->cut[k + 1], S->fa, S->var_length, cbch_default_threads(), header_len,
                                      S->derive_md ? CBCH_DERIVE_MD : 0u, &J->hb, A->err, sizeof A->err);
        if (!rc) {
            cbcg_batch v; cbch_batch_view(&J->hb, &v);
            cbcg_encode_opts o = { J->hb.read_len_header ? J->hb.read_len_header : 1u, S->single ? 0u : S->block_reads, S->single ? 0u : 1u, 0u };
            J->bound = cbcg_encode_bound(&v, &o);
            J->seq_bases = J->hb.n_reads ? J->hb.seq_off[J->hb.n_reads] : 0; J->header_len = J->hb.read_len_header; J->n_reads = J->hb.n_reads;
            if (!S->single && !S->with_cigar && J->hb.n_reads && cbch_pack_batch(&v, 0, NULL, NULL, &J->cb) == CBCH_OK) {   /* 2 bits per base on the link */
                J->have_compact = 1;
                const uint64_t unm = J->hb.n_unmapped;
                cbch_free_batch(&J->hb);                          /* the packed form is all the device thread needs */
                J->hb.n_unmapped = unm;
            }
        }
        A->ingest_s += now() - t0;
        if (rc) { A->rc = rc; publish(S, 1); return NULL; }
        if (!header_len) header_len = J->header_len;
        A->n_unmapped += J->hb.n_unmapped;
        publish(S, 0);
    }
    return NULL;
}

/* The SAM header: @HD and the @SQ lines of batch 0's chromosome table (a single-block stream: of the reference), each with
 * LN from the reference when it holds the name. */
static int write_sam_header(FILE *fo, const job *J0, const cbch_fasta *fa) {
    uint8_t *h = NULL; uint64_t n = 0;
    if (!J0->legacy) {
        if (cbcg_sam_header(J0->in, J0->in_len, NULL, 0, &n) != CBCG_ERR_CAPACITY || !(h = (uint8_t *)malloc(n)) ||
            cbcg_sam_header(J0->in, J0->in_len, h, n, &n) != CBCG_OK) { free(h); return 1; }
    } else {
        uint64_t cap = 64;
        for (uint32_t k = 0; k < fa->n; k++) cap += strlen(fa->names[k]) + 16;
        if (!(h = (uint8_t *)malloc(cap))) return 1;
        n = (uint64_t)snprintf((char *)h, cap, "@HD\tVN:1.6\tSO:coordinate\n");
        for (uint32_t k = 0; k < fa->n; k++) n += (uint64_t)snprintf((char *)h + n, cap - n, "@SQ\tSN:%s\n", fa->names[k]);
    }
    int rc = 0;
    for (const uint8_t *l = h, *e = h + n; l < e && !rc;) {
        const uint8_t *nl = (const uint8_t *)memchr(l, '\n', (size_t)(e - l));
        if (!nl) nl = e;
        if (fwrite(l, 1, (size_t)(nl - l), fo) != (size_t)(nl - l)) rc = 1;
        if (nl - l > 7 && !memcmp(l, "@SQ\tSN:", 7))
            for (uint32_t k = 0; k < fa->n; k++)
                if (strlen(fa->names[k]) == (size_t)(nl - l - 7) && !memcmp(fa->names[k], l + 7, (size_t)(nl - l - 7))) {
                    fprintf(fo, "\tLN:%llu", (unsigned long long)fa->len[k]); break;
                }
        if (fputc('\n', fo) == EOF) rc = 1;
        l = nl + 1;
    }
    free(h);
    return rc;
}
/* 1 when batch k's chromosome table differs from batch 0's */
static int sam_table_differs(const job *J0, const job *J) {
    uint64_t a = 0, b = 0;
    if (cbcg_sam_header(J0->in, J0->in_len, NULL, 0, &a) != CBCG_ERR_CAPACITY || cbcg_sam_header(J->in, J->in_len, NULL, 0, &b) != CBCG_ERR_CAPACITY || a != b) return 1;
    uint8_t *x = (uint8_t *)malloc(a), *y = (uint8_t *)malloc(b);
    int d = !x || !y || cbcg_sam_header(J0->in, J0->in_len, x, a, &a) || cbcg_sam_header(J->in, J->in_len, y, b, &b) || memcmp(x, y, a);
    free(x); free(y);
    return d;
}

/* NAME[:START[-END]], split at the last ':' when what follows it is START or START-END (else the whole text is the name) */
static int parse_region(const char *a, cbcg_region *r) {
    const char *c = strrchr(a, ':');
    size_t name_len = strlen(a);
    unsigned long long s = 1, t = UINT64_MAX;
    if (c && c != a && c[1] >= '0' && c[1] <= '9') {
        char *e;
        const unsigned long long s1 = strtoull(c + 1, &e, 10);
        unsigned long long t1 = UINT64_MAX;
        int ok = !*e || *e == '-';
        if (ok && *e == '-') { const char *q = e + 1; t1 = (*q >= '0' && *q <= '9') ? strtoull(q, &e, 10) : 0; ok = *q >= '0' && *q <= '9' && !*e; }
        if (ok) {
            if (s1 == 0 || t1 < s1) return -1;
            name_len = (size_t)(c - a); s = s1; t = t1;
        }
    }
    char *name = strndup(a, name_len);
    if (!name) return -1;
    r->name = name; r->start = s; r->end = t;
    return 0;
}

static int parse_devices(const char *s, int *dev) {
    int n = 0;
    while (*s && n < MAX_DEV) {
        char *e; long v = strtol(s, &e, 10);
        if (e == s || v < 0) return -1;
        dev[n++] = (int)v;
        if (*e == ',') e++;
        s = e;
    }
    return n;
}

int main(int argc, char **argv) {
    int mode = 0, single = 0, var_length = 0, with_cigar = 0, sam = 0, derive_md = 0, n_dev = 1, dev[MAX_DEV] = { 0 };
    uint32_t block_reads = CBCG_BLOCK_AUTO;
    uint64_t batch_mb = 2048;
    const char *files[4]; int nfiles = 0;
    cbcg_region *regions = NULL; uint32_t n_regions = 0;
    for (int i = 1; i < argc; i++) {
        const char *a = argv[i];
        if (!strcmp(a, "-c")) mode = 'c';
        else if (!strcmp(a, "-d") || !strcmp(a, "-x")) mode = 'd';
        else if (!strcmp(a, "-1")) single = 1;
        else if (!strcmp(a, "-l")) var_length = 1;
        else if (!strcmp(a, "-C")) with_cigar = 1;
        else if (!strcmp(a, "-S")) sam = 1;
        else if (!strcmp(a, "-M")) derive_md = 1;
        else if (!strcmp(a, "-b") && i + 1 < argc) block_reads = (uint32_t)strtoul(argv[++i], NULL, 10);
        else if (!strcmp(a, "-B") && i + 1 < argc) batch_mb = strtoull(argv[++i], NULL, 10);
        else if (!strcmp(a, "-r") && i + 1 < argc) {
            cbcg_region *g = (cbcg_region *)realloc(regions, (n_regions + 1) * sizeof *regions);
            if (!g) return 1;
            regions = g;
            if (parse_region(argv[++i], &regions[n_regions])) { fprintf(stderr, "cbc: bad region '%s' (NAME[:START[-END]], 1 <= START <= END)\n", argv[i]); return 2; }
            n_regions++;
        }
        else if (!strcmp(a, "-g") && i + 1 < argc) { n_dev = parse_devices(argv[++i], dev); if (n_dev < 1) return usage(); }
        else if (a[0] == '-' && a[1]) return usage();
        else if (nfiles < 4) files[nfiles++] = a;
        else return usage();
    }
    /* the checked-in reference wants a ratio before the file names (`-c 1 sam out ref`, 1 = lossless): accept and drop it */
    if (mode == 'c' && nfiles == 4) {
        char *e; (void)strtod(files[0], &e);
        if (*e != 0) return usage();
        files[0] = files[1]; files[1] = files[2]; files[2] = files[3]; nfiles = 3;
    }
    if (!mode || nfiles != 3) { fprintf(stderr, "Missing required filenames\n"); return usage(); }
    if (n_regions && mode != 'd') { fprintf(stderr, "cbc: -r selects reads to decode: it goes with -d\n"); return usage(); }
    if (sam && mode != 'd') { fprintf(stderr, "cbc: -S writes SAM: it goes with -d\n"); return usage(); }
    if (derive_md && mode != 'c') { fprintf(stderr, "cbc: -M derives MD for encoding: it goes with -c\n"); return usage(); }
    if (n_regions && with_cigar && !sam) { fprintf(stderr, "cbc: -r cannot be combined with -C: CIGAR recovery rebuilds every read of a batch\n"); return 2; }
    if (!single && block_reads == 0) block_reads = CBCG_BLOCK_AUTO;
    if (batch_mb < 1) batch_mb = 1;

    const double t0 = now();
    shared S; memset(&S, 0, sizeof S);
    pthread_mutex_init(&S.mu, NULL); pthread_cond_init(&S.cv, NULL);
    S.mode = mode; S.single = single; S.var_length = var_length; S.block_reads = block_reads; S.with_cigar = with_cigar;
    S.regions = regions; S.n_regions = n_regions; S.sam = sam; S.derive_md = derive_md;
    devthread D[MAX_DEV]; memset(D, 0, sizeof D);

    /* ---- the input, cut into jobs (before the device threads start: they index S.jobs) */
    cbch_mapped map; memset(&map, 0, sizeof map); map.fd = -1;
    const uint8_t **cut = NULL;
    const uint8_t *in = NULL; uint8_t *cig_file = NULL; uint64_t in_len = 0;
    if (mode == 'c') {
        printf("Compressing...\n");
        const uint64_t batch_bytes = batch_mb << 20;
        if (cbch_map(files[0], 0, &map)) { fprintf(stderr, "cbc: cannot open %s\n", files[0]); return 1; }
        S.n_jobs = single ? 1 : (map.n + batch_bytes - 1) / batch_bytes;
        if (S.n_jobs == 0) S.n_jobs = 1;
        cut = (const uint8_t **)calloc(S.n_jobs + 1, sizeof *cut);
        const uint8_t *end = map.p + map.n;
        cut[0] = map.p;
        for (uint64_t k = 1; k < S.n_jobs; k++) { const uint8_t *g = map.p + k * batch_bytes; cut[k] = g < end ? cbch_next_line(g, end) : end; if (cut[k] < cut[k - 1]) cut[k] = cut[k - 1]; }
        cut[S.n_jobs] = end;
    } else {
        printf("Decompressing...\n");
        /* mapped, not read: the payload pages a region query does not need are never read from disk */
        if (cbch_map(files[0], 0, &map)) { fprintf(stderr, "cbc: cannot open %s\n", files[0]); return 1; }
        in = map.p; in_len = map.n;
        if (n_regions && in_len) madvise((void *)map.p, (size_t)in_len, MADV_RANDOM);   /* no read-ahead past the blocks a query needs */
        uint32_t h[4] = { 0, 0, 0, 0 };
        if (in_len >= 16) memcpy(h, in, 16);
        S.n_jobs = (h[0] == CBCS_MAGIC && h[2] > 0 && 16 + 16ull * h[2] <= in_len) ? h[2] : 1;
    }
    S.jobs = (job **)calloc(S.n_jobs, sizeof *S.jobs);
    for (uint64_t k = 0; k < S.n_jobs; k++) { S.jobs[k] = (job *)calloc(1, sizeof(job)); S.jobs[k]->index = k; }
    if (mode == 'd') {
        uint64_t nr, cap;
        if (S.n_jobs == 1 && !(in_len >= 16 && rd_u32(in) == CBCS_MAGIC)) {
            S.jobs[0]->in = in; S.jobs[0]->in_len = in_len;
            S.jobs[0]->legacy = cbcg_decoded_size(in, in_len, &nr, &cap) != CBCG_OK;            /* no "CBCB" header: a reference stream */
        } else for (uint64_t k = 0; k < S.n_jobs; k++) {
            uint64_t off, len; memcpy(&off, in + 16 + 16 * k, 8); memcpy(&len, in + 24 + 16 * k, 8);
            if (off > in_len || len > in_len - off) { fprintf(stderr, "cbc: truncated CBCS file\n"); return 1; }
            S.jobs[k]->in = in + off; S.jobs[k]->in_len = len;
        }
        if (with_cigar) {                                      /* <in>.cig: u64 length + section per batch, in batch order */
            char path[4096]; snprintf(path, sizeof path, "%s.cig", files[0]);
            FILE *fc = fopen(path, "rb");
            if (!fc) { fprintf(stderr, "cbc: cannot open %s\n", path); return 1; }
            fseek(fc, 0, SEEK_END); long csz = ftell(fc); fseek(fc, 0, SEEK_SET);
            cig_file = (uint8_t *)malloc(csz > 0 ? (size_t)csz : 1);
            if (!cig_file || fread(cig_file, 1, (size_t)csz, fc) != (size_t)csz) { fprintf(stderr, "cbc: cannot read %s\n", path); return 1; }
            fclose(fc);
            uint64_t o = 0;
            for (uint64_t k = 0; k < S.n_jobs; k++) {
                uint64_t l = 0;
                if (o + 8 > (uint64_t)csz) { fprintf(stderr, "cbc: %s holds fewer sections than the input has batches\n", path); return 1; }
                memcpy(&l, cig_file + o, 8); o += 8;
                if (l > (uint64_t)csz - o) { fprintf(stderr, "cbc: truncated %s\n", path); return 1; }
                S.jobs[k]->cig_in = cig_file + o; S.jobs[k]->cig_in_len = l; o += l;
            }
        }
        S.produced = S.n_jobs;
    }
    if ((uint64_t)n_dev > S.n_jobs) n_dev = (int)S.n_jobs;
    for (int d = 0; d < n_dev; d++) { D[d].S = &S; D[d].device = dev[d]; pthread_create(&D[d].th, NULL, device_main, &D[d]); }

    /* ---- the reference genome (device threads are creating their contexts meanwhile) */
    char err[256] = "";
    cbch_fasta fa;
    const double t_fa0 = now();
    if (cbch_read_fasta(files[2], &fa, err, sizeof err)) { fprintf(stderr, "cbc: %s\n", err); return 1; }
    const double fasta_s = now() - t_fa0;
    pthread_mutex_lock(&S.mu); S.fa = &fa; S.fa_ready = 1; pthread_cond_broadcast(&S.cv); pthread_mutex_unlock(&S.mu);

    int status = 0;
    uint64_t total_reads = 0, total_out = 0, total_blocks = 0; double device_ms = 0;
    FILE *fo = fopen(files[1], "wb");
    if (!fo) { fprintf(stderr, "cbc: cannot write %s\n", files[1]); status = 1; }
    FILE *fcig = NULL; uint64_t cig_bytes = 0;
    if (with_cigar && mode == 'c' && !status) {
        char path[4096]; snprintf(path, sizeof path, "%s.cig", files[1]);
        fcig = fopen(path, "wb");
        if (!fcig) { fprintf(stderr, "cbc: cannot write %s\n", path); status = 1; }
    }
    ingest_arg IA; memset(&IA, 0, sizeof IA);
    pthread_t ith; int have_ith = 0;
    const double t1 = now();
    if (mode == 'c' && !status) {
        IA.S = &S; IA.map = &map; IA.cut = cut; IA.window = (uint64_t)n_dev + 2;
        pthread_create(&ith, NULL, ingest_main, &IA); have_ith = 1;
    }
    /* ---- the writer: results in order */
    const int sharded = mode == 'c' && S.n_jobs > 1;
    uint64_t *shard_off = NULL, *shard_len = NULL, filepos = 0, seq_bases = 0;
    if (sharded && !status) {
        shard_off = (uint64_t *)calloc(S.n_jobs, 8); shard_len = (uint64_t *)calloc(S.n_jobs, 8);
        filepos = 16 + 16 * S.n_jobs;
        if (fseek(fo, (long)filepos, SEEK_SET)) status = 1;
    }
    for (uint64_t k = 0; k < S.n_jobs && !status; k++) {
        job *J = wait_done(&S, k);
        if (!J) { fprintf(stderr, "cbc: %s\n", IA.err[0] ? IA.err : "ingest failed"); status = 1; break; }
        if (J->rc) { fprintf(stderr, "cbc: %s\n", J->err); status = 1; break; }
        if (sam && k == 0 && write_sam_header(fo, J, &fa)) { fprintf(stderr, "cbc: cannot write the SAM header of %s\n", files[0]); status = 1; break; }
        if (sam && k > 0 && sam_table_differs(S.jobs[0], J)) { fprintf(stderr, "cbc: batch %llu names other chromosomes than batch 0: one SAM header cannot describe both\n", (unsigned long long)k); status = 1; break; }
        if (with_cigar && mode == 'd' && !sam) {                         /* "CIGAR<TAB>SEQ" per read: the two texts hold one line per read each */
            const uint8_t *c = J->cig, *ce = J->cig + J->cig_len, *q = J->out, *qe = J->out + J->out_len;
            while (c < ce && q < qe) {
                const uint8_t *cn = (const uint8_t *)memchr(c, '\n', (size_t)(ce - c)), *qn = (const uint8_t *)memchr(q, '\n', (size_t)(qe - q));
                if (!cn || !qn) break;
                if (fwrite(c, 1, (size_t)(cn - c), fo) != (size_t)(cn - c) || fputc('\t', fo) == EOF || fwrite(q, 1, (size_t)(qn - q + 1), fo) != (size_t)(qn - q + 1)) { status = 1; break; }
                c = cn + 1; q = qn + 1;
            }
            if (!status && (c != ce || q != qe)) { fprintf(stderr, "cbc: CIGAR and SEQ line counts differ\n"); status = 1; }
            if (status) break;
        } else if (J->out_len && fwrite(J->out, 1, J->out_len, fo) != J->out_len) { fprintf(stderr, "cbc: cannot write %s\n", files[1]); status = 1; break; }
        if (fcig) {
            if (fwrite(&J->cig_len, 1, 8, fcig) != 8 || (J->cig_len && fwrite(J->cig, 1, J->cig_len, fcig) != J->cig_len)) { fprintf(stderr, "cbc: cannot write the CIGAR sections\n"); status = 1; break; }
            cig_bytes += 8 + J->cig_len;
        }
        if (sharded) { shard_off[k] = filepos; shard_len[k] = J->out_len; filepos += J->out_len; }
        total_reads += J->n_reads; total_out += J->out_len; total_blocks += J->n_blocks; device_ms += J->device_ms;
        if (mode == 'c') { seq_bases += J->seq_bases; cbch_free_batch(&J->hb); }
        pthread_mutex_lock(&S.mu);
        free(J->out); J->out = NULL; free(J->cig); J->cig = NULL; J->written = 1;     /* frees a slot of the ingest window */
        pthread_cond_broadcast(&S.cv);
        pthread_mutex_unlock(&S.mu);
    }
    if (status) { pthread_mutex_lock(&S.mu); S.producer_failed = 1; S.next_take = S.n_jobs; pthread_cond_broadcast(&S.cv); pthread_mutex_unlock(&S.mu); }
    if (sharded && !status) {
        uint32_t h[4] = { CBCS_MAGIC, 1u, (uint32_t)S.n_jobs, 0u };
        if (fseek(fo, 0, SEEK_SET) || fwrite(h, 1, 16, fo) != 16) status = 1;
        for (uint64_t k = 0; k < S.n_jobs && !status; k++) if (fwrite(&shard_off[k], 1, 8, fo) != 8 || fwrite(&shard_len[k], 1, 8, fo) != 8) status = 1;
        total_out += 16 + 16 * S.n_jobs;
    }
    if (fo && fclose(fo)) status = 1;
    if (fcig && fclose(fcig)) status = 1;
    const double t2 = now();
    if (have_ith) pthread_join(ith, NULL);
    for (int d = 0; d < n_dev; d++) pthread_join(D[d].th, NULL);
    if (!status) {
        if (mode == 'c') {
            printf("Final Size: %llu\n", (unsigned long long)total_out);
            if (with_cigar) printf("CIGAR sections: %llu bytes\n", (unsigned long long)cig_bytes);
            printf("Compression took %f\n", t2 - t1);
            printf("reads %llu (unmapped skipped %llu), blocks %llu, batches %llu on %d device(s), %.4f bits/base, fasta %.3f s, ingest %.3f s (%.2f GB/s), gpu ready %.3f s, device %.3f ms\n",
                   (unsigned long long)total_reads, (unsigned long long)IA.n_unmapped, (unsigned long long)total_blocks, (unsigned long long)S.n_jobs, n_dev,
                   seq_bases ? 8.0 * (double)total_out / (double)seq_bases : 0.0, fasta_s, IA.ingest_s, IA.ingest_s > 0 ? (double)map.n / IA.ingest_s / 1e9 : 0.0,
                   S.t_gpu_ready - t0, device_ms);
        } else {
            printf("Decompression took %f\n", t2 - t1);
            printf("reads %llu, shards %llu on %d device(s), gpu ready %.3f s, device %.3f ms\n", (unsigned long long)total_reads, (unsigned long long)S.n_jobs, n_dev, S.t_gpu_ready - t0, device_ms);
        }
    }
    if (getenv("CBC_TRACE")) for (int d = 0; d < n_dev; d++)
        fprintf(stderr, "[cbc] device %d: context %.3f s, reference upload %.3f s, coding calls %.3f s; writer done at %.3f s\n", dev[d], D[d].create_s, D[d].setref_s, D[d].call_s, t2 - t0);
    for (uint64_t k = 0; k < S.n_jobs; k++) { free(S.jobs[k]->out); free(S.jobs[k]->cig); free(S.jobs[k]); }
    free(S.jobs); free(cut); free(cig_file); free(shard_off); free(shard_len);
    for (uint32_t k = 0; k < n_regions; k++) free((void *)regions[k].name);
    free(regions);
    cbch_unmap(&map);
    cbch_free_fasta(&fa);
    printf("Total time elapsed: %f seconds.\n", now() - t0);
    return status;
}
