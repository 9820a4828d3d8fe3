/*
 * cbcg.h -- C ABI of the B200 implementation of cbc's aligned-read coding path.
 *
 * This is the drop-in boundary: plain C, plain pointers and sizes, no CUDA or torch
 * types. The reference (1mishra/cbc) has no plugin/FFI interface; its seams are ordinary
 * C functions over process-global state (SURVEY.md section 8b). Each entry point below
 * names the reference function(s) it replaces. All functions return 0 on success or a
 * negative cbcg_status; nothing asserts or exits (the reference does:
 * src/stream_model.c:62,71, src/read_compression.c:41, src/main.c:248-250).
 *
 * Threading: one host thread per context; one context per GPU. No globals.
 * Ownership: the caller owns every host buffer; the context owns all device memory.
 * There is no CPU fallback: cbcg_create fails if no sm_100 device is usable.
 */
#ifndef CBCG_H
#define CBCG_H

#include <stdint.h>
#include <stddef.h>
#include "cbcg_format.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef enum cbcg_status {
    CBCG_OK              = 0,
    CBCG_ERR_ARG         = -1,   /* bad argument / NULL */
    CBCG_ERR_CUDA        = -2,   /* CUDA runtime error (cbcg_last_error has the text) */
    CBCG_ERR_NO_DEVICE   = -3,   /* no usable sm_100 GPU: there is no CPU path */
    CBCG_ERR_NOMEM       = -4,
    CBCG_ERR_CAPACITY    = -5,   /* caller's output buffer too small */
    CBCG_ERR_INPUT       = -6,   /* a read is outside what the reference can code (SURVEY.md 8c):
                                    POS 0, length 0 or > 252, reference span (length - insertions
                                    + deletions) past the chromosome's end, CIGAR '*'/'N'/junk,
                                    > 255 edits of a kind, unsorted positions, zero-probability symbol
                                    (src/stream_model.c:71: e.g. L SNPs in a read at header length L), and,
                                    in the single-block stream only, a POS step pos - prev_pos + 1 above
                                    5 000 000 (CBCG_MAX_POS_X; the first read of a chromosome steps from 0).
                                    Blocked containers code any POS step. */
    CBCG_ERR_NO_REFERENCE = -7,  /* cbcg_set_reference not called / chromosome ordinal out of range */
    CBCG_ERR_FORMAT      = -8,   /* container header / index malformed */
    CBCG_ERR_CORRUPT     = -9,   /* bitstream decodes to an impossible symbol */
    CBCG_ERR_LIMIT       = -10,  /* internal table limit (distinct FLAG values per block) */
    CBCG_ERR_INTERNAL    = -11
} cbcg_status;

typedef struct cbcg_ctx cbcg_ctx;

/* SoA batch of aligned reads: the product of load_sam_line (src/sam_file_allocation.c:437-529)
 * for n_reads records. Offsets arrays have n_reads + 1 entries; pools are plain bytes. */
typedef struct cbcg_batch {
    uint64_t n_reads;
    const uint32_t *pos;        /* POS, 1-based (sam_line_t.pos) */
    const uint16_t *flag;       /* FLAG */
    const uint16_t *seq_len;    /* strlen(SEQ) */
    const uint32_t *chr;        /* chromosome ordinal into the table given to cbcg_set_reference */
    const uint64_t *seq_off;    const uint8_t *seq;     /* SEQ */
    const uint64_t *cigar_off;  const uint8_t *cigar;   /* CIGAR text */
    const uint64_t *md_off;     const uint8_t *md;      /* MD:Z payload (read_line_t.edits) */
} cbcg_batch;

/* The same batch in the form that crosses the host-device link (about 60 bytes per 150-base read instead of 196): SEQ at
 * 2 bits per base, every read starting on a byte (ceil(len / 4) bytes; base i in bits 2 (i & 3) of byte i >> 2;
 * A C G T = 0 1 2 3), whatever is not A, C, G or T listed apart (packed as 0); CIGAR and MD text as lengths, not offsets;
 * chromosomes as runs (reads are sorted). tile_base holds, for every tile of 128 reads and once more for the end of the
 * batch, the bytes of SEQ, seq2, CIGAR and MD text that precede it (4 x u64 per entry): the library cuts the batch
 * into pipeline chunks at tile boundaries with it, the per-read offsets are rebuilt on the device (which also checks
 * the lengths against it), where the batch is unpacked into the cbcg_batch layout before K1 reads it.
 * cbch_pack_batch (csrc/host/sam_ingest.h) makes one from a cbcg_batch; the SAM ingest can fill one directly. */
typedef struct cbcg_batch_compact {
    uint64_t n_reads;
    const uint32_t *pos;
    const uint16_t *flag;
    const uint16_t *seq_len;
    const uint16_t *cigar_len;
    const uint16_t *md_len;
    uint32_t n_runs; uint32_t pad;
    const uint64_t *run_first;  /* first read ordinal of each chromosome run, ascending; run_first[0] == 0 */
    const uint32_t *run_chr;    /* its chromosome ordinal */
    const uint8_t *seq2;
    uint64_t n_exc;             /* bases that are not A / C / G / T */
    const uint32_t *exc_read;   /* read ordinal, ascending */
    const uint16_t *exc_base;   /* index of the base in the read */
    const uint8_t *exc_char;    /* the character */
    const uint8_t *cigar;
    const uint8_t *md;
    const uint64_t *tile_base;  /* ((n_reads + 127) / 128 + 1) x { SEQ bytes, seq2 bytes, CIGAR bytes, MD bytes } before the tile */
    uint32_t max_len, min_len;  /* longest / shortest SEQ */
} cbcg_batch_compact;

/* block_reads value that lets the library size blocks so that the last generation fills the GPU's resident
 * block slots a whole number of times (reads per block <= CBCG_BLOCK_AUTO_MAX). The choice is written to the
 * container header like any other block size. */
#define CBCG_BLOCK_AUTO      0xffffffffu
#define CBCG_BLOCK_AUTO_MAX  1280u

typedef struct cbcg_encode_opts {
    uint32_t read_len_header;   /* what get_read_length returns (src/sam_file_allocation.c:26-79):
                                   the alphabet size of the snps/indels/var models */
    uint32_t block_reads;       /* reads per independently coded block; 0 = ONE block holding the whole
                                   input in the reference's own stream layout (byte-identical to
                                   `program -c 1` built with -DDEBUG): the verification mode */
    uint32_t gen_mode;          /* 0: every block starts from the reference's initial model state;
                                   1: generation-primed blocks (see DESIGN.md) */
    uint32_t substreams;        /* blocked containers: 0 / 1: one arithmetic-coded stream per block (every symbol of a read in
                                   the reference's order); 4: four substreams per block (CBCG_MODE_SPLIT4, cbcg_format.h) */
} cbcg_encode_opts;

/* Per-call device timings (CUDA events on the library's stream), for bench.py / profiling. */
typedef struct cbcg_stats {
    float ms_h2d, ms_extract, ms_plan, ms_code, ms_gather, ms_reconstruct, ms_d2h, ms_total;
    float ms_k1, ms_k3;         /* K1 / K3 kernel alone (events tight around the launch; ms_extract and
                                   ms_reconstruct also hold the host round trip that reads the totals) */
    uint64_t n_reads, n_blocks, n_symbols, n_edits, payload_bytes, container_bytes;
    uint64_t h2d_bytes, d2h_bytes;
    uint32_t kernel_launches;
    uint32_t retried;           /* 1: the call started in an overlapped order, found on the device that the sizes projected
                                   from the head of the batch were too small, and ran again in the one-stream order */
} cbcg_stats;

/* ---- lifetime */
int  cbcg_create(int device, cbcg_ctx **out);
void cbcg_destroy(cbcg_ctx *ctx);
const char *cbcg_strerror(int status);
const char *cbcg_last_error(const cbcg_ctx *ctx);      /* detail of the last failure on this context */
int  cbcg_abi_version(void);
int  cbcg_get_stats(const cbcg_ctx *ctx, cbcg_stats *out);   /* stats of the last call */

/* Page-locked host memory for batches and outputs: host<->device copies of pageable memory are staged
 * and run at a fraction of the link rate. Optional; any host pointer is accepted everywhere. */
void *cbcg_host_alloc(size_t bytes);
void  cbcg_host_free(void *p);

/* ---- reference genome. Replaces store_reference_in_memory (src/read_decompression.c:17-53) and the
 * chromosome switch in compress_line/decompress_line (src/compression.c:58-64,91-101): all records are
 * resident at once, upper-cased on upload, addressed by ordinal. names are used for the container. */
int cbcg_set_reference(cbcg_ctx *ctx, uint32_t n_chr, const char *const *names,
                       const uint8_t *const *bases, const uint64_t *len);

/* ---- K1: edit extraction. Replaces compress_edits + add_snps_to_array
 * (src/read_compression.c:265-606, 613-701), without the symbol emission. recs[n_reads];
 * edits_cap entries of u16; *n_edits receives the number written. */
int cbcg_extract(cbcg_ctx *ctx, const cbcg_batch *batch, cbcg_read_rec *recs,
                 uint16_t *edits, uint64_t edits_cap, uint64_t *n_edits);

/* ---- symbol streams, for parity tests: the (stream, ctx, symbol) sequence compress_read hands to
 * send_value_to_as (src/read_compression.c:15-44, 557-600; src/stream_model.c:53), one list per block.
 * POS is reported as the raw value x = pos - prevPos + 1 under CBCG_S_POS_X. block_reads == 0 gives the
 * whole-stream sequence including the 136 header symbols, RNAME symbols and the end marker.
 * block_sym_count (optional) receives one count per block; *n_blocks the number of blocks. */
int cbcg_extract_symbols(cbcg_ctx *ctx, const cbcg_batch *batch, const cbcg_encode_opts *opts,
                         cbcg_symbol *symbols, uint64_t symbols_cap, uint64_t *n_symbols,
                         uint64_t *block_sym_count, uint64_t blocks_cap, uint64_t *n_blocks);

/* ---- K1 + K2: encode. Replaces compress() (src/compression.c:112-170) from the first compress_line
 * on, including the header ints of alloc_sam_models (src/sam_file_allocation.c:363-404) in
 * single-block mode. out receives the whole container (or the bare reference stream when
 * opts->block_reads == 0). */
int cbcg_encode(cbcg_ctx *ctx, const cbcg_batch *batch, const cbcg_encode_opts *opts,
                uint8_t *out, uint64_t out_cap, uint64_t *out_len);
uint64_t cbcg_encode_bound(const cbcg_batch *batch, const cbcg_encode_opts *opts);
/* The same from a compact batch: a third of the bytes on the link, the same container byte for byte. */
int cbcg_encode_compact(cbcg_ctx *ctx, const cbcg_batch_compact *batch, const cbcg_encode_opts *opts,
                        uint8_t *out, uint64_t out_cap, uint64_t *out_len);
int cbcg_batch_upload_compact(cbcg_ctx *ctx, const cbcg_batch_compact *batch);   /* becomes the resident batch */

/* ---- K2 + K3: decode. Replaces decompress() + print_line (src/compression.c:173-216, 16-40):
 * seq_out receives SEQ + '\n' per read. legacy != 0: `in` is a bare reference stream. */
int cbcg_decode(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, int legacy,
                uint8_t *seq_out, uint64_t seq_cap, uint64_t *seq_len, uint64_t *n_reads);
/* Output size of a container without decoding it (header only); 0 on a malformed header. */
int cbcg_decoded_size(const uint8_t *in, uint64_t in_len, uint64_t *n_reads, uint64_t *max_seq_bytes);

/* Decode to edit records instead of text (what decompress_read yields before reconstruct_read writes
 * the bases): for parity tests of the block decoder alone. */
int cbcg_decode_edits(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, int legacy,
                      cbcg_read_rec *recs, uint64_t recs_cap, uint32_t *chr, uint16_t *edits,
                      uint64_t edits_cap, uint64_t *n_reads, uint64_t *n_edits);

/* ---- K3: read reconstruction from edit records. Replaces reconstruct_read + print_line
 * (src/read_decompression.c:339-529, src/compression.c:16-40). */
int cbcg_reconstruct(cbcg_ctx *ctx, uint64_t n_reads, const cbcg_read_rec *recs, const uint32_t *chr,
                     const uint16_t *edits, uint64_t n_edits, uint8_t *seq_out, uint64_t seq_cap,
                     uint64_t *seq_len);

/* ---- CIGAR recovery (SURVEY.md 8f row 4). Upstream declares reconstructCigar / cigarFlags (include/sam_block.h:179,443)
 * and sketches decompress_cigar (src/read_decompression.c:91-113: a per-read flag "the CIGAR is the one the indels
 * imply", the text itself otherwise) without implementing either; the coded stream therefore returns SEQ only. These two
 * calls add the rest as a side section that travels beside the container (the CLI appends it with -C): reads whose
 * CIGAR is what their deletions and insertions imply -- every read of configs 1-4 -- cost nothing, reads whose end
 * operations are soft clips (coded as insertions by the reference, src/read_compression.c:358-479) cost two bytes, any
 * other CIGAR (=, X, H, P, ...) is kept verbatim. cbcg_cigar_pack runs K1 on the batch and classifies every read on the
 * device; cbcg_cigar_unpack decodes the container to edit records and writes every read's CIGAR + '\n' in read order
 * (section == NULL: the implied CIGARs alone). State: cbcg_cigar_pack uploads `batch` (it becomes the resident batch, like
 * cbcg_batch_upload) and cbcg_cigar_unpack is a decode (it invalidates "the last encode", like cbcg_decode of a foreign
 * container); neither touches the container's bytes. Section layout ("CBCC" v1): api.cu, above cbcg_cigar_bound. */
uint64_t cbcg_cigar_bound(const cbcg_batch *batch);
int cbcg_cigar_pack(cbcg_ctx *ctx, const cbcg_batch *batch, uint8_t *out, uint64_t out_cap, uint64_t *out_len);
int cbcg_cigar_unpack(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, int legacy, const uint8_t *section, uint64_t section_len,
                      uint8_t *cigar_out, uint64_t cigar_cap, uint64_t *cigar_len, uint64_t *n_reads);

/* ---- region decode (DESIGN.md, "Region decode"): the reads of a blocked container that overlap genomic intervals,
 * without decoding the whole container. The blocks of generation g start from the snapshot that merges every block of the
 * generations before g, so the call decodes every block of every generation before the latest generation g* that a region
 * touches, then only the touched blocks of g* (gen_mode 0: only the touched blocks). A legacy stream is one block: it is
 * decoded whole and then filtered.
 *   overlap: a read overlaps [start, end] on its chromosome if pos <= end and pos + span - 1 >= start, span = len - n_ins +
 *     n_dels from the decoded record (deletions and insertions counted per base; the reference codes soft clips as
 *     insertions, so clipped bases are not part of the span): the alignment end samtools computes for M/I/D/S CIGARs.
 *   several regions give their union: a read is returned once however many regions it overlaps; they need not be sorted.
 *     A name that is not in the container (legacy: not in the loaded reference) matches nothing; that is not an error.
 *   errors: start == 0, start > end, a NULL name or n_regions == 0 -> CBCG_ERR_ARG; a malformed header or index ->
 *     CBCG_ERR_FORMAT; a block that has to be decoded names a chromosome missing from the loaded reference ->
 *     CBCG_ERR_NO_REFERENCE (blocks that are not decoded may).
 *   capacity: as cbcg_decode. seq_cap or ids_cap too small -> CBCG_ERR_CAPACITY with *seq_len / *n_reads set to the sizes
 *     needed; cbcg_fetch_decoded then returns the text.
 *   statistics: cbcg_get_stats's n_blocks and n_reads are what the block decoder decoded (more than is returned);
 *     the returned count is *n_reads.
 *   state: a decode; it invalidates "the last encode" as cbcg_decode of a foreign container does. */
/* A genomic interval: 1-based, both ends inclusive; end = UINT64_MAX means "to the end of the record".
 * name: a reference record name as stored in the container. */
typedef struct cbcg_region { const char *name; uint64_t start, end; } cbcg_region;

/* What cbcg_decode_region would do with this container and these regions, computed on the host from the header and the
 * block index alone (no context, no device, no payload bytes read): blocks and reads it decodes, payload bytes it
 * reads, and an upper bound on the text it returns. A legacy stream does not store its read count: *n_blocks = 1,
 * *payload_bytes = in_len, *n_reads = *max_seq_bytes = UINT64_MAX (unknown). */
int cbcg_region_plan(const uint8_t *in, uint64_t in_len, int legacy, const cbcg_region *regions, uint32_t n_regions,
                     uint64_t *n_blocks, uint64_t *n_reads, uint64_t *payload_bytes, uint64_t *max_seq_bytes);

/* The reads that overlap at least one region, each once, in container order: SEQ + '\n' per read, like cbcg_decode,
 * and (read_ids != NULL) each read's ordinal in the container. */
int cbcg_decode_region(cbcg_ctx *ctx, const uint8_t *in, uint64_t in_len, int legacy,
                       const cbcg_region *regions, uint32_t n_regions,
                       uint8_t *seq_out, uint64_t seq_cap, uint64_t *seq_len,
                       uint64_t *read_ids, uint64_t ids_cap, uint64_t *n_reads);

/* ---- device-resident variants (inputs already in HBM when the timed region starts): upload once,
 * run many times. Results stay on the device until fetched. Used by bench.py for `value`. */
int cbcg_batch_upload(cbcg_ctx *ctx, const cbcg_batch *batch);                 /* replaces the resident batch */
int cbcg_encode_resident(cbcg_ctx *ctx, const cbcg_encode_opts *opts);         /* K1 + plan + K2e + gather */
int cbcg_decode_resident(cbcg_ctx *ctx);                                       /* K2d + K3 on the last encode's blocks */
int cbcg_fetch_container(cbcg_ctx *ctx, uint8_t *out, uint64_t out_cap, uint64_t *out_len);
int cbcg_fetch_decoded(cbcg_ctx *ctx, uint8_t *seq_out, uint64_t seq_cap, uint64_t *seq_len);
/* Container header + per-block index of the last encode, without the payload: what one shard contributes
 * to a multi-GPU container index (SURVEY.md 8e). *payload_bytes (optional) receives the payload size. */
int cbcg_fetch_index(cbcg_ctx *ctx, uint8_t *out, uint64_t out_cap, uint64_t *out_len, uint64_t *payload_bytes);

/* ---- timing marks: CUDA events on the library's own stream (slots 0..3), for bench.py. */
int cbcg_mark(cbcg_ctx *ctx, int slot);
int cbcg_elapsed_ms(cbcg_ctx *ctx, int from, int to, float *ms);

#ifdef __cplusplus
}
#endif
#endif /* CBCG_H */
