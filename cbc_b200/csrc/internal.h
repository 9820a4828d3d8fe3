/* internal.h -- device-side data layout shared by the kernels and the host API (api.cu). */
#pragma once
#include <stdint.h>
#include "cbcg.h"

/* Read batch resident in HBM: the SoA arrays of cbcg_batch, pools padded by POOL_PAD bytes so that
 * 16-byte-aligned bulk copies may over-read past the last record. */
#define POOL_PAD 64u

struct DevBatch {
    uint64_t n_reads;
    const uint32_t *pos;
    const uint16_t *flag;
    const uint16_t *seq_len;
    const uint32_t *chr;
    const uint64_t *seq_off;   const uint8_t *seq;
    const uint64_t *cigar_off; const uint8_t *cigar;
    const uint64_t *md_off;    const uint8_t *md;
    uint32_t max_len;                      /* max(seq_len) */
    uint32_t ref_cap;                      /* K1: bytes of reference a tile of 128 reads is expected to span, with margin (0: no estimate) */
};

/* Reference genome resident in HBM: one byte per base, upper-cased, records concatenated with
 * each record start aligned to 256 bytes and REF_PAD bytes of 'N' after each record. */
#define REF_PAD 1024u
#define MAX_CHR 4096u

struct DevGenome {
    uint32_t n_chr;
    const uint8_t *bases;                  /* whole buffer */
    const uint64_t *chr_off;               /* [n_chr] byte offset of each record in `bases` */
    const uint64_t *chr_len;               /* [n_chr] */
};

/* One independently coded block of position-ordered reads. */
struct BlockDesc {
    uint32_t first_read;                   /* ordinal of its first read in the shard */
    uint32_t n_reads;
    uint32_t chr;
    uint32_t base_pos;                     /* prevPos at block start: POS of its first read (0 in single-block mode) */
    uint32_t n_edits;                      /* edit entries of the block: bounds its var rows */
    uint32_t gen;                          /* generation (0: reference initial state) */
    uint32_t payload_bytes;                /* coded size (encoder output / decoder input) */
    uint32_t n_symbols;
    uint64_t edit_base;                    /* first edit entry of the block in the edit array */
    uint64_t payload_off;                  /* decoder: offset of the block's bytes in the payload buffer;
                                              encoder: offset of its scratch output region */
    uint64_t ws_off;                       /* offset of its model workspace (bytes) */
    uint64_t sym_off;                      /* symbol-list mode: first entry of its list */
    uint32_t pos_card;                     /* primed blocks, out: final POS alphabet size */
    uint32_t n_rows;                       /*   var rows created */
    uint32_t pa_touched;                   /*   pos_alpha models instantiated */
    uint32_t pad;
    uint32_t sub_bytes[CBCG_N_SUB];        /* blocked containers (v4): coded size of each substream, A | B | C | D back to back */
};

/* Coder launch parameters. */
struct CoderParams {
    uint32_t block_begin;                  /* this launch codes blocks [block_begin, block_begin + n_blocks) */
    uint32_t n_blocks;
    uint32_t L;                            /* header read length = alphabet of snps / indels / var */
    uint32_t legacy;                       /* 1: single block in the reference's own stream layout */
    uint32_t mode;                         /* 0 encode, 1 decode, 2 symbol list */
    BlockDesc *blocks;
    cbcg_read_rec *recs;                   /* in (encode, list) / out (decode) */
    uint16_t *edits;                       /* in / out */
    uint32_t *chr;                         /* per read: in (encode) / out (decode) */
    DevGenome genome;
    uint8_t *ws;                           /* model workspace */
    uint8_t *payload;                      /* encode: per-block scratch regions; decode: compact payload */
    cbcg_symbol *symbols;                  /* list mode */
    const uint8_t *chr_names;              /* legacy: NUL-terminated names, MAX_NAME bytes each */
    unsigned long long *err;
    uint32_t lean;                         /* blocked containers: same_ref and length bytes 1..3 are not coded */
    uint32_t short_flush;                  /* blocked containers: 1 + scale3 closing bits instead of the reference's 26+ */
    uint32_t primed;                       /* gen_mode 1: models start from `snap` instead of the initial state */
    uint32_t fixed_len;                    /* CBCG_MODE_FIXED_LEN: every read is L bases, the length symbol is not coded */
    uint32_t no_merge;                     /* the blocks of this launch are not merged into a snapshot afterwards (the last generation): their final
                                              model states are not needed */
    uint32_t indel_heavy;                  /* host estimate: the batch's CIGAR text per read says most reads carry indels / clips */
    uint32_t n_sub;                        /* blocked containers: substreams of the blocks of THIS launch (one generation): 1 or CBCG_N_SUB */
    uint32_t layout_mode;                  /* the container's layout bits (CBCG_MODE_SPLIT4, split generations): CBCG_BLOCK_NSUB(layout_mode, gen) per block */
    const uint8_t *snap;                   /* snapshot S_{g-1} (snapshot_bytes(L) bytes); blocked containers always start from one */
    uint8_t *fin;                          /* per block (absolute index): its image of the small models (WarpModels), read by the merges */
    struct K2Tri *tri;                       /* encode, one-stream blocks: the symbols' intervals, written by the model kernel and coded by the
                                              interval kernel (k2_tri_off / K2_TRI_*) */
};
struct alignas(16) K2Tri { uint32_t lo, cnt, n, flags; };   /* moved as one 16-byte word (uint4) by the kernels */
/* Interval buffer of a two-kernel encode, in slots of 16 bytes (cumulative count, count, total, flags). Block b owns
 * [k2_tri_off(b), + 12 n_reads + 2 n_edits + 8): slot 0 holds the number of main slots, main slots from slot 1 (<= 8 per
 * read + 2 per edit, in stream order), then the escape list (<= 4 per read: the byte symbols of POS escapes, in order
 * of appearance). */
#ifdef __CUDACC__
#define CBCG_HD __host__ __device__
#else
#define CBCG_HD
#endif
static inline CBCG_HD uint64_t k2_tri_off(const BlockDesc &B, uint32_t b) { return 12ull * B.first_read + 2ull * B.edit_base + 8ull * b; }
static inline CBCG_HD uint64_t k2_tri_esc(const BlockDesc &B) { return 1ull + 8ull * B.n_reads + 2ull * B.n_edits; }
static inline uint64_t k2_tri_slots(uint64_t n_reads, uint64_t edits_cap, uint64_t n_blocks) { return 12ull * n_reads + 2ull * edits_cap + 8ull * n_blocks + 64ull; }
#define MAX_NAME 256u

/* Host-callable launchers (defined in the .cu files). */
int launch_extract(const DevBatch &b, const DevGenome &g, cbcg_read_rec *recs, uint16_t *edits,
                   uint64_t edits_cap, uint64_t *tile_desc, uint32_t *ticket, uint64_t *total_edits,
                   unsigned long long *err, cudaStream_t st, cudaEvent_t ev_start, cudaEvent_t ev_stop,
                   uint64_t r_begin = 0, uint64_t r_end = ~0ull, const uint64_t *edit_base = nullptr);
int launch_reconstruct(uint64_t n_reads, const cbcg_read_rec *recs, const uint32_t *chr, const uint16_t *edits,
                       const DevGenome &g, uint8_t *out, uint64_t out_cap, uint32_t max_len, uint32_t fixed_len,
                       uint64_t *tile_desc, uint32_t *ticket, uint64_t *total_bytes,
                       unsigned long long *err, cudaStream_t st, cudaEvent_t ev_start, cudaEvent_t ev_stop, uint32_t ref_cap_hint = 0);
/* k0_unpack.cu: reads [r_begin, r_end) of a compact batch (r_begin a multiple of 128) -> the SoA batch */
int launch_unpack(uint64_t r_begin, uint64_t r_end, uint64_t n_reads, const uint16_t *seq_len, const uint16_t *cigar_len, const uint16_t *md_len,
                  const uint8_t *seq2, const uint64_t *tile_base, const uint64_t *run_first, const uint32_t *run_chr, uint32_t n_runs,
                  uint64_t *seq_off, uint64_t *cigar_off, uint64_t *md_off, uint8_t *seq, uint32_t *chr, unsigned long long *err, cudaStream_t st);
int launch_patch(const uint32_t *exc_read, const uint16_t *exc_base, const uint8_t *exc_char, uint64_t n_exc, const uint64_t *seq_off, uint8_t *seq, cudaStream_t st);
/* k4_cigar.cu: CIGAR recovery. cls: per read, 0 implied / 1, 2, 3 end operations are soft clips / 4 verbatim */
int launch_cigar_class(uint64_t n_reads, const cbcg_read_rec *recs, const uint16_t *edits, const uint64_t *cigar_off,
                       const uint8_t *cigar, uint8_t *cls, cudaStream_t st);
uint64_t cigar_num_tiles(uint64_t n_reads);
int launch_cigar_emit(uint64_t n_reads, const cbcg_read_rec *recs, const uint16_t *edits, const uint8_t *cls,
                      const uint64_t *exc_read, const uint64_t *exc_off, const uint8_t *exc_text, uint64_t n_exc,
                      uint8_t *out, uint64_t out_cap, uint64_t *tile_desc, uint32_t *ticket, uint64_t *total_bytes,
                      unsigned long long *err, cudaStream_t st);
uint64_t extract_num_tiles(uint64_t n_reads);
uint64_t reconstruct_num_tiles(uint64_t n_reads);
int launch_plan(const CoderParams &p, uint32_t n_reads_total, uint64_t n_edits_total, uint64_t ws_cap,
                uint64_t payload_cap, uint64_t *totals, cudaStream_t st,
                const uint64_t *carry_in = nullptr, const uint64_t *n_edits_dev = nullptr);
int launch_coder(const CoderParams &p, cudaStream_t st);
uint32_t coder_resident_blocks(int device);     /* blocks (warps) of the warp kernel the whole GPU holds at once */
int launch_gather(BlockDesc *blocks, uint32_t n_blocks, const uint8_t *scratch, uint8_t *out,
                  uint64_t *out_off, int blocked, uint32_t layout_mode, cudaStream_t st);   /* blocked: CBCG_BLOCK_NSUB(layout_mode, gen) pieces per block */
uint32_t coder_launches(const CoderParams &p);  /* kernel launches launch_coder(p) makes */
uint64_t coder_ws_bytes_bound(uint32_t L, uint64_t n_reads, uint64_t n_edits, uint64_t n_blocks, int legacy, int primed);
/* generation snapshots (gen_mode 1) */
uint64_t snapshot_bytes(uint32_t L);
uint64_t fin_stride_bytes(void);
int launch_snapshot_init(uint8_t *snap, uint32_t L, cudaStream_t st);
int launch_merge(const BlockDesc *blocks, uint32_t block_begin, uint32_t n_blocks, uint32_t L, const uint8_t *prev,
                 uint8_t *next, const uint8_t *fin, const uint8_t *ws, unsigned long long *err, uint32_t flag_target, cudaStream_t st);
int launch_code_kernel(const CoderParams &p, cudaStream_t st); /* k2_blocks.cu: the interval half of a two-kernel encode */
void set_carveout_all(int pct);                 /* -1: driver default per kernel; 0..100: one split for every kernel */
int launch_copy16(void *dst, const void *src, uint64_t bytes, cudaStream_t st);
int launch_d2h_bytes(void *dst_host, const void *src_dev, uint64_t bytes, cudaStream_t st);   /* dst: mapped pinned host memory, any alignment */
int launch_copy_words(void *dst, const void *src, uint32_t n_words, cudaStream_t st);          /* <= 32 64-bit words */
uint64_t coder_payload_bound(uint64_t n_reads, uint64_t n_edits, uint64_t n_blocks, int legacy);
/* k5_region.cu: region select and compaction. iv: the query's intervals (genome ordinals), sorted by (chr, start), overlaps
   merged; runs: n_runs pairs (dense ordinal of a run's first read, its ordinal in the container), ascending. *total
   receives the number of reads kept. */
struct RegionIv { uint32_t chr, pad; uint64_t start, end; };   /* 1-based, both ends inclusive */
uint64_t region_num_tiles(uint64_t n_reads);
int launch_region_select(uint64_t n_reads, const cbcg_read_rec *recs, const uint32_t *chr, const RegionIv *iv, uint32_t n_iv,
                         const uint64_t *runs, uint32_t n_runs, cbcg_read_rec *out_recs, uint32_t *out_chr, uint64_t *out_ids,
                         uint64_t *tile_desc, uint32_t *ticket, uint64_t *total, unsigned long long *err, cudaStream_t st);
/* k6_sam.cu: SAM lines from records + K3's text (seq_text, SEQ + '\n' per read; fixed_len: every read that long). names: MAX_NAME
   bytes per genome record, name_len their lengths. ids (optional): container ordinal per read, the index into cls (optional,
   per container read: CIGAR class); exc_*: the class-4 reads' texts by ascending container ordinal. tile_desc: 2 x
   sam_num_tiles(n_reads) words. *total_bytes receives the text's size. */
uint64_t sam_num_tiles(uint64_t n_reads);
int launch_sam(uint64_t n_reads, const cbcg_read_rec *recs, const uint32_t *chr, const uint16_t *edits, const DevGenome &g,
               const uint8_t *names, const uint32_t *name_len, const uint8_t *seq_text, uint32_t max_len, uint32_t fixed_len,
               const uint64_t *ids, const uint8_t *cls, const uint64_t *exc_read, const uint64_t *exc_off, const uint8_t *exc_text,
               uint64_t n_exc, uint8_t *out, uint64_t out_cap, uint64_t *tile_desc, uint32_t *ticket, uint64_t *total_bytes,
               unsigned long long *err, cudaStream_t st);
/* k7_md.cu: the MD of reads [r_begin, r_end) of a batch that carries none, into md / md_off (md_cap bytes of pool; a read
   whose MD does not fit gets an empty one at md_cap and CBCG_ERR_CAPACITY). md_base (optional): MD bytes of the reads
   before r_begin. *total_md receives md_base + the range's MD bytes, exact even when they do not fit. tile_desc:
   md_num_tiles(r_end - r_begin) words. */
uint64_t md_num_tiles(uint64_t n_reads);
int launch_md(const DevBatch &b, const DevGenome &g, uint64_t *md_off, uint8_t *md, uint64_t md_cap, uint64_t *tile_desc,
              uint32_t *ticket, uint64_t *total_md, unsigned long long *err, cudaStream_t st, uint64_t r_begin, uint64_t r_end,
              const uint64_t *md_base);
/* k8_pileup.cu: per-position counts over regions. iv: the merged request intervals (genome ordinals, clipped to the record
   lengths), iv_slot: the accumulator slot of each one's first position (each takes end - start + 2 slots); acc: 8 columns of
   n_pad u32 (n_pad a multiple of K8_SCAN_TILE, zeroed by the caller). reg: per requested region with rows, its first output
   row, chromosome, first position and first slot, ascending by row. cls / exc_*: as launch_sam; seq_text: K3's text of the
   reads (needed only when cls lists class-4 reads, else NULL). rows: n_rows x CBCG_PU_COLS u32. tile_desc: max(
   pileup_num_tiles(n_reads), 2 n_pad / K8_SCAN_TILE) words. *n_counted receives the reads counted. */
#define K8_SCAN_TILE 1024u
struct PileupReg { uint64_t row0, start, slot0; uint32_t chr, pad; };
uint64_t pileup_num_tiles(uint64_t n_reads);
int launch_pileup(uint64_t n_reads, const cbcg_read_rec *recs, const uint32_t *chr, const uint16_t *edits, const DevGenome &g,
                  const RegionIv *iv, const uint64_t *iv_slot, uint32_t n_iv, uint32_t flag_exclude, const uint64_t *ids, const uint8_t *cls,
                  const uint64_t *exc_read, const uint64_t *exc_off, const uint8_t *exc_text, uint64_t n_exc, const uint8_t *seq_text,
                  uint32_t max_len, uint32_t fixed_len, uint32_t *acc, uint64_t n_pad, uint64_t n_slots, const PileupReg *reg, uint32_t n_reg,
                  uint32_t *rows, uint64_t n_rows, uint64_t *tile_desc, uint32_t *ticket, uint64_t *n_counted, unsigned long long *err,
                  cudaStream_t st);
/* k9_bam.cu: BAM records in BGZF blocks. launch_bam_records: K6's inputs (ref_id: per genome ordinal, its index in the
   header's name list, -1 for none) -> the uncompressed record stream (stream_cap bytes), rec_off (n_reads + 1 offsets: each
   record's, then the stream's size) and block_first (the first record of each BGZF block, then n_reads; <= stream_cap /
   K9_BLOCK_CUT + 2 entries); totals[0] receives the stream's size and totals[1] the block count. tile_desc: 2 x
   bam_num_tiles(n_reads) words. launch_bgzf: those blocks -> out, back to back; *total_bytes receives their size.
   tile_desc: n_blocks words. */
#define K9_BLOCK_CUT 49152u
uint64_t bam_num_tiles(uint64_t n_reads);
int launch_bam_records(uint64_t n_reads, const cbcg_read_rec *recs, const uint32_t *chr, const uint16_t *edits, const DevGenome &g,
                       const int32_t *ref_id, const uint8_t *seq_text, uint32_t max_len, uint32_t fixed_len, const uint64_t *ids,
                       const uint8_t *cls, const uint64_t *exc_read, const uint64_t *exc_off, const uint8_t *exc_text, uint64_t n_exc,
                       uint8_t *stream, uint64_t stream_cap, uint64_t *rec_off, uint32_t *block_first, uint64_t *tile_desc, uint32_t *ticket,
                       uint64_t *totals, unsigned long long *err, cudaStream_t st);
int launch_bgzf(const uint8_t *stream, const uint64_t *rec_off, const uint32_t *block_first, uint32_t n_blocks, uint8_t *out,
                uint64_t *tile_desc, uint32_t *ticket, uint64_t *total_bytes, unsigned long long *err, cudaStream_t st);
/* k10_bam_in.cu: BAM input (DESIGN.md 5g). BgzfMember: one BGZF member, found by the host's walk of the header chain: its raw
   deflate bytes in[in_off, + in_len), its output out[out_off, + isize) and its CRC32. launch_inflate: a warp per member;
   CBCG_ERR_CORRUPT (item: the member) on any deflate, ISIZE or CRC problem. launch_bam_boundaries: the whole records of the
   stream [0, T) cut into n_seg segments at seg[0 .. n_seg] (seg[0] = 0, seg[n_seg] = T); work: 5 n_seg words; rec_start: the
   offset of every whole record (rec_cap entries; T / 36 + 1 suffice: a chain stops at a block_size below 32, and one that
   reaches it is CBCG_ERR_FORMAT); words[0] receives the record count, [1] the start of the bytes after the last whole
   record, [2] the segments walked again. launch_bam_count / launch_bam_write: the mapped records (map: refID ->
   genome ordinal, -1 for none) into the batch b (b.n_reads records' room for launch_bam_count, then the pools sized from
   words[3..6]: reads, SEQ, CIGAR and MD bytes; derive: no MD is looked for); tile_desc: 4 x bam_in_num_tiles words; lens:
   l_seq of records 0 and 1, 0xffffffff - the shortest and the longest read. src / md_at: a word per record. run_first /
   run_last: room for b.n_reads pairs of words each ((first read | chromosome << 32, POS), (last read, POS)); words[7] / [8]
   receive their counts. */
struct BgzfMember { uint64_t in_off, out_off; uint32_t in_len, isize, crc, pad; };
int launch_inflate(const uint8_t *in, const BgzfMember *mem, uint32_t n_members, uint8_t *out, unsigned long long *err, cudaStream_t st);
int launch_bam_boundaries(const uint8_t *stream, uint64_t T, const uint64_t *seg, uint32_t n_seg, int32_t n_ref, uint64_t *work,
                          uint64_t *rec_start, uint64_t rec_cap, uint64_t *words, unsigned long long *err, cudaStream_t st);
uint64_t bam_in_num_tiles(uint64_t n_records);
int launch_bam_count(const uint8_t *stream, const uint64_t *rec_start, uint64_t n_rec, const int32_t *map, int32_t n_ref, uint32_t derive,
                     const DevBatch &b, uint64_t *src, uint64_t *md_at, uint64_t *tile_desc, uint32_t *ticket, uint64_t *words, uint32_t *lens,
                     unsigned long long *err, cudaStream_t st);
int launch_bam_write(const uint8_t *stream, const DevBatch &b, uint32_t derive, const uint64_t *src, const uint64_t *md_at, uint64_t *run_first,
                     uint64_t *run_last, uint64_t *words, cudaStream_t st);
