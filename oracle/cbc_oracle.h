/*
 * oracle/cbc_oracle.h -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU restatement (plain C) of the reference's aligned-read coding path, used only
 * as the checker by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg.
 * Nothing under cbc_b200/ may include, link or call it.
 *
 * Parity pinning: the reference ships no golden vectors (SURVEY.md section 4), so this
 * restatement is pinned against outputs of the reference itself, built unmodified
 * into oracle/_ref/ (cbc_ref, cbc_trace): byte-identical streams and identical
 * symbol traces, see tests/test_oracle_vs_reference.py and tests/golden/.
 */
#ifndef CBC_ORACLE_H
#define CBC_ORACLE_H

#include <stdint.h>
#include <stddef.h>
#include "cbcg_format.h"

#ifdef __cplusplus
extern "C" {
#endif

/* SoA batch: what load_sam_line (src/sam_file_allocation.c:437-529) yields per record. */
typedef struct cbco_batch {
    uint64_t n_reads;
    const uint32_t *pos;        /* POS, 1-based */
    const uint16_t *flag;       /* FLAG */
    const uint16_t *seq_len;    /* strlen(SEQ) */
    const uint32_t *chr;        /* chromosome ordinal (index into the reference table) */
    const uint64_t *seq_off;    /* n_reads+1 offsets into seq */
    const uint8_t  *seq;
    const uint64_t *cigar_off;  /* n_reads+1 */
    const uint8_t  *cigar;
    const uint64_t *md_off;     /* n_reads+1; MD:Z payload */
    const uint8_t  *md;
} cbco_batch;

/* Reference genome: upper-cased bases per record, as store_reference_in_memory
 * (src/read_decompression.c:17-53) leaves them. */
typedef struct cbco_genome {
    uint32_t n_chr;
    const uint8_t *const *bases;
    const uint64_t *len;
    const char *const *name;
} cbco_genome;

typedef struct cbco_buf { uint8_t *data; uint64_t size, cap; } cbco_buf;
void cbco_buf_free(cbco_buf *b);

/* Edit extraction (compress_edits + add_snps_to_array, src/read_compression.c:265-701).
 * recs[n_reads]; edits needs room for sum(n_dels+n_snps+n_ins) entries. A read carries up to 255
 * deletions whatever its length, and, when its CIGAR and MD agree with its SEQ, at most len SNPs
 * and insertions together: CBCO_EDITS_PER_READ(len) entries (8 spare) per read are always enough.
 * Returns number of edit entries, -2 when they do not fit in edits_cap, or <0 on an input outside
 * the reference's contract. Nothing is written past edits_cap. */
#define CBCO_EDITS_PER_READ(len) ((uint64_t)(len) + 255u + 8u)
int64_t cbco_extract(const cbco_batch *b, const cbco_genome *g, cbcg_read_rec *recs,
                     uint16_t *edits, uint64_t edits_cap);

/* Read reconstruction (reconstruct_read + print_line, src/read_decompression.c:339-529,
 * src/compression.c:16-40). Writes SEQ + '\n' per read into out. */
int64_t cbco_reconstruct(uint64_t n_reads, const cbcg_read_rec *recs, const uint16_t *edits,
                         const uint32_t *chr, const cbco_genome *g, uint8_t *out, uint64_t out_cap);

/* Legacy single stream, byte-identical to `program -c 1` built with -DDEBUG.
 * read_len_header: what get_read_length returns (second record's SEQ length, or max with -l).
 * If trace != NULL it receives the (key, symbol) sequence exactly as the tracer logs it. */
int cbco_encode_legacy(const cbco_batch *b, const cbco_genome *g, uint32_t read_len_header,
                       cbco_buf *out, cbco_buf *trace);

/* Decode a legacy stream to SEQ lines (`program -x`). recs/edits/chr optional (may be NULL). */
int cbco_decode_legacy(const uint8_t *stream, uint64_t stream_len, const cbco_genome *g,
                       cbco_buf *seq_out, uint64_t *n_reads_out);

/* Raw symbol list of a read range [r0, r1) coded as ONE block with block-local state:
 * same per-read symbol order as the reference, POS emitted as CBCG_S_POS_X raw values.
 * legacy != 0: prepend the 136 header symbols and append the end marker, chr changes
 * emit RNAME symbols (whole-stream semantics). Used to check K1/K1b. */
int cbco_symbols(const cbco_batch *b, const cbco_genome *g, const cbcg_read_rec *recs,
                 const uint16_t *edits, uint64_t r0, uint64_t r1, uint32_t read_len_header,
                 int legacy, cbco_buf *symbols);

/* Blocked container ("CBCB", our design): independent blocks of block_reads reads, cut at
 * chromosome changes, each with its own coder; model snapshots per generation (n_gens >= 1). */
int cbco_encode_blocked(const cbco_batch *b, const cbco_genome *g, uint32_t read_len_header,
                        uint32_t block_reads, uint32_t gen_mode, cbco_buf *out);
/* The batch coded with the block cut (per-block read counts, generations, header words) of an existing container. */
int cbco_encode_like(const uint8_t *container, uint64_t len, const cbco_batch *b, const cbco_genome *g, cbco_buf *out);
/* Same container with an explicit generation schedule (experiments; gen_mode 1 uses CBCG_GEN_*). */
int cbco_encode_scheduled(const cbco_batch *b, const cbco_genome *g, uint32_t read_len_header, uint32_t block_reads,
                          uint32_t n_sched, const uint32_t *sched_count, const uint32_t *sched_reads, cbco_buf *out);
int cbco_decode_blocked(const uint8_t *container, uint64_t len, const cbco_genome *g,
                        cbco_buf *seq_out, uint64_t *n_reads_out);

#ifdef __cplusplus
}
#endif
#endif
