/*
 * sam_ingest.h -- host-side SAM / FASTA ingest into the SoA batch of include/cbcg.h.
 *
 * Replaces, for the read path, load_sam_line + get_read_length (src/sam_file_allocation.c:26-79,
 * 437-529) and the FASTA half of store_reference_in_memory (src/read_decompression.c:17-53). Plain C,
 * no CUDA: the CLI hands the result to the C ABI; the CPU tests check it against the generator.
 */
#ifndef CBC_SAM_INGEST_H
#define CBC_SAM_INGEST_H
#include <stddef.h>
#include <stdint.h>
#include "cbcg.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct cbch_fasta {
    uint32_t n;
    char **names;            /* record names: text after '>' up to the first blank */
    uint8_t **bases;         /* as in the file (case kept; the device upper-cases) */
    uint64_t *len;
} cbch_fasta;

typedef struct cbch_batch {
    uint64_t n_reads, cap;
    uint32_t *pos; uint16_t *flag; uint16_t *seq_len; uint32_t *chr;
    uint64_t *seq_off, *cigar_off, *md_off;
    uint8_t *seq, *cigar, *md;
    uint64_t seq_cap, cigar_cap, md_cap;
    uint32_t read_len_header;     /* get_read_length: SEQ length of the 2nd record, or the maximum (var_length) */
    uint32_t max_len;
    uint64_t n_unmapped;          /* records skipped: FLAG & 4 (src/compression.c:50) */
    uint64_t n_lines;
} cbch_batch;

enum { CBCH_OK = 0, CBCH_ERR_IO = -1, CBCH_ERR_NOMEM = -2, CBCH_ERR_PARSE = -3, CBCH_ERR_RNAME = -4, CBCH_ERR_NO_MD = -5 };
/* Ingest flags. CBCH_DERIVE_MD: MD:Z tags are not looked for (a record without one is accepted, one that has one is read as
 * if it had none); the batch's md_off and md stay NULL, a batch without MD that the library derives MD for (cbcg.h). */
#define CBCH_DERIVE_MD 1u

int  cbch_read_fasta(const char *path, cbch_fasta *out, char *err, size_t errlen);
void cbch_free_fasta(cbch_fasta *fa);
/* Mapped records of a SAM file; RNAME is resolved against the FASTA record names. */
int  cbch_read_sam(const char *path, const cbch_fasta *fa, int var_length, cbch_batch *out, char *err, size_t errlen);
/* The same with an explicit worker count (cbch_read_sam uses CBCH_THREADS or the online cores, at most 64): the file is
 * cut at line starts, the ranges are parsed in parallel and merged; the result does not depend on the count. */
int  cbch_read_sam_mt(const char *path, const cbch_fasta *fa, int var_length, int n_threads, cbch_batch *out, char *err, size_t errlen);
/* The same with ingest flags (CBCH_DERIVE_MD); cbch_read_sam and cbch_read_sam_mt are this with flags 0. */
int  cbch_read_sam_ex(const char *path, const cbch_fasta *fa, int var_length, int n_threads, uint32_t flags, cbch_batch *out, char *err, size_t errlen);
int  cbch_default_threads(void);
/* Streaming: the file mapped once (populate: fault it all in now, for files that fit in memory), cut at line starts with
 * cbch_next_line, ingested range by range. header_len != 0 overrides the fixed-length header value (later batches of a
 * file take the first batch's). */
typedef struct cbch_mapped { const uint8_t *p; uint64_t n; int fd; } cbch_mapped;
int  cbch_map(const char *path, int populate, cbch_mapped *out);
void cbch_unmap(cbch_mapped *m);
const uint8_t *cbch_next_line(const uint8_t *p, const uint8_t *end);
int  cbch_ingest_range(const uint8_t *begin, const uint8_t *end, const cbch_fasta *fa, int var_length, int n_threads, uint32_t header_len,
                       cbch_batch *out, char *err, size_t errlen);
/* The same with ingest flags (CBCH_DERIVE_MD); cbch_ingest_range is this with flags 0. */
int  cbch_ingest_range_ex(const uint8_t *begin, const uint8_t *end, const cbch_fasta *fa, int var_length, int n_threads, uint32_t header_len,
                          uint32_t flags, cbch_batch *out, char *err, size_t errlen);
void cbch_free_batch(cbch_batch *b);
void cbch_batch_view(const cbch_batch *b, cbcg_batch *view);

/* The compact form of a batch (cbcg_batch_compact, include/cbcg.h): what crosses the host-device link (a batch without MD:
 * md_len = md = NULL and a zero MD column in tile_base). All arrays are
 * allocated with `alloc` (NULL: malloc; pass cbcg_host_alloc for page-locked memory) and released with cbch_free_compact
 * through `release`. n_threads <= 0: the default worker count. */
typedef struct cbch_compact {
    cbcg_batch_compact v;                 /* the view handed to cbcg_encode_compact */
    void *(*alloc)(size_t); void (*release)(void *);
    uint64_t bytes;                       /* what will cross the link */
} cbch_compact;
int  cbch_pack_batch(const cbcg_batch *b, int n_threads, void *(*alloc)(size_t), void (*release)(void *), cbch_compact *out);
void cbch_free_compact(cbch_compact *c);

#ifdef __cplusplus
}
#endif
#endif
