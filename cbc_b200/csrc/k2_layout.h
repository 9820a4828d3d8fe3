/*
 * k2_layout.h -- memory layouts of the block coder shared by its kernels (k2_coder.cu: the warp kernels; k2_blocks.cu:
 * the interval kernel of a two-kernel encode), its scalar twin (k2_roles.cuh), the generation merges and the host API:
 * per-block model workspace, per-block image of the small models, generation snapshot. Plain C++ (host + device).
 */
#pragma once
#include <stdint.h>
#include <stddef.h>
#include "cbcg.h"

#ifdef __CUDACC__
#define K2_HD __host__ __device__ __forceinline__
#else
#define K2_HD inline
#endif

#define K2_WARPS    4u
#define K2_MIN_CTAS 5          /* resident CTAs per SM the register allocation is held to: 96 registers, no spills
                                  (cold per-warp values live in shared memory, WarpCold); 6 spills and is slower */
#define K2_THREADS  (K2_WARPS * 32u)
#define LIKELY(c)   __builtin_expect(!!(c), 1)
#define UNLIKELY(c) __builtin_expect(!!(c), 0)
#define FLAG_CAP    CBCG_FLAG_ADAPT_MAX   /* distinct FLAG values a block / a snapshot adapts (the sparse table's size, a format constant: rules F1 / F2 in cbcg_format.h; 128 -> 256 measured time-neutral) */
#define PA_STRIDE   260u              /* words per 256-symbol model row: 256 counts, n, padding to 16 bytes */
#define VAR_DIRECT_MIN_EDITS 32768u       /* blocks with more edits index var rows directly by context */
#define VAR_DEFERRED 0x80000000u           /* hash value: row not built yet, low 16 bits = the one symbol coded in it */

enum { MODE_ENC = 0, MODE_DEC = 1, MODE_LIST = 2 };

#define SYNCW() __syncwarp()

/* ------------------------------------------------------------------------------------------------
 * per-block workspace layout in HBM (u32 units unless noted) */
struct WsLayout {
    uint64_t pos_cnt, pos_val;     /* pos_cap each */
    uint64_t pos_alpha;            /* 4 x 257 */
    uint64_t var_hash;             /* u64 x hash_cap, or init bitmap (2048 u32) in direct mode */
    uint64_t var_rows;             /* rows x Lp */
    uint64_t codebook;             /* legacy: 4 x 257 */
    uint64_t rname;                /* legacy: 256 x 257 */
    uint64_t total;                /* bytes */
    uint32_t pos_cap, hash_cap, rows_cap, Lp, direct;
};

K2_HD uint32_t pow2_ceil(uint32_t x) { uint32_t p = 32; while (p < x) p <<= 1; return p; }

K2_HD WsLayout ws_layout(uint32_t L, uint64_t n_reads, uint64_t n_edits, int legacy, int primed) {
    WsLayout w;
    w.Lp = (L + 1u + 31u) & ~31u;
    w.pos_cap = (uint32_t)(n_reads + 34u) + (primed ? CBCG_SNAP_POS_MAX : 0u);
    w.direct = (!primed && (legacy || n_edits >= VAR_DIRECT_MIN_EDITS)) ? 1u : 0u;
    w.rows_cap = w.direct ? CBCG_VAR_CONTEXTS : (uint32_t)n_edits;
    w.hash_cap = w.direct ? 1024u : pow2_ceil((uint32_t)(2u * n_edits + 2u));   /* u64 slots */
    uint64_t o = 0;                                                            /* in bytes, 16-aligned pieces */
    w.pos_cnt = o;   o += ((uint64_t)w.pos_cap * 4u + 15u) & ~15ull;
    w.pos_val = o;   o += ((uint64_t)w.pos_cap * 4u + 15u) & ~15ull;
    w.pos_alpha = o; o += 4u * PA_STRIDE * 4u + 16u;
    w.var_hash = o;  o += (uint64_t)w.hash_cap * 8u;
    w.var_rows = o;  o += (uint64_t)w.rows_cap * w.Lp * 4u;
    w.codebook = o;  if (legacy) o += 4u * PA_STRIDE * 4u + 16u;
    w.rname = o;     if (legacy) o += 256u * PA_STRIDE * 4u + 16u;
    if (legacy) o += 2u * 65536u * 4u;                                         /* FLAG table beyond FLAG_CAP entries: keys, then counts, right behind rname (Coder::flag_spill) */
    w.total = (o + 255u) & ~255ull;
    return w;
}

/* Scratch room of substream q of a block (encoder): symbols x 20 bits (count >= 1, n <= 2^20) + slack, 16-byte
 * aligned. A: POS + an escape's 4 bytes per read; B: length byte + FLAG; C: match, SNP count, 3 indel counts;
 * D: position + base per edit. */
K2_HD uint64_t k2_sub_cap(uint32_t q, uint64_t n_reads, uint64_t n_edits) {
    const uint64_t syms = q == CBCG_SUB_POS ? 5u * n_reads : q == CBCG_SUB_FLAG ? 2u * n_reads : q == CBCG_SUB_COUNTS ? 5u * n_reads : 2u * n_edits;
    return ((syms * 20u) / 8u + 64u + 15u) & ~15ull;
}
/* Room for a block's coded bytes (encoder). layout 0: four substream regions; 1: one stream per block (<= 12 symbols
 * per read + 2 per edit, <= 20 bits each); 2: the reference's own stream (+ header ints and names). */
K2_HD uint64_t payload_cap_bytes(uint64_t n_reads, uint64_t n_edits, int layout) {
    if (layout == 0) return k2_sub_cap(0, n_reads, n_edits) + k2_sub_cap(1, n_reads, n_edits) + k2_sub_cap(2, n_reads, n_edits) + k2_sub_cap(3, n_reads, n_edits);
    const uint64_t syms = (layout == 2 ? 16u : 12u) * n_reads + 2u * n_edits + (layout == 2 ? 136u + 4096u : 0u) + 8u;
    return ((syms * 20u) / 8u + 64u + 15u) & ~15ull;
}
K2_HD uint64_t symlist_cap(uint64_t n_reads, uint64_t n_edits, int legacy) {
    return 12u * n_reads + 2u * n_edits + (legacy ? 136u + 2048u : 0u) + 8u;
}


/* ------------------------------------------------------------------------------------------------
 * shared-memory models of one warp. Dense model = counts[card] followed by n at [card]. */
struct WarpModels {
    uint32_t snps[256];            /* card L, n at [L]                (initialize_stream_model_snps :243) */
    uint32_t indels[256];          /* card L                          (:277) */
    uint32_t rlen0[256];           /* card 255: length byte 0         (initialize_stream_model_id(.,4,255) :583) */
    uint32_t chars[6][8];          /* card 5                          (:350-411) */
    uint32_t match[4][4];          /* card 2                          (:204) */
    uint32_t same_ref[4];          /* card 2                          (:617) */
    uint32_t rlenk[3][2];          /* length bytes 1..3, always symbol 0: (count[0], n) */
    uint32_t flag_key[FLAG_CAP];   /* FLAG model (:96-130), sparse: touched values, ascending */
    uint32_t flag_cnt[FLAG_CAP];
    uint32_t flag_used, flag_n;
    uint16_t cumdel[256];          /* decoder: cumulative deletion offsets of the current read */
};

/* Per-warp values the hot loop rarely needs (once per 32 payload bits, per POS escape, per decoded SNP): kept in
 * shared memory behind the models instead of in registers. */
struct WarpCold {
    uint8_t *io;                   /* the block's payload: written by the encoder, read by the decoder */
    const uint8_t *ref;            /* decoder: the block's chromosome */
    uint64_t ref_len, edits_cap_abs;
    uint32_t io_cap;               /* encoder: room in io; decoder: payload bytes */
    uint32_t pos_cap, rows_cap, pad;
};
struct WarpShared { WarpModels m; WarpCold c; };

/* ------------------------------------------------------------------------------------------------
 * generation snapshot (gen_mode 1): the state every block of the next generation starts from. */
struct SnapLayout { uint64_t small, pos_hdr, pos_val, pos_cnt, pos_alpha, bitmap, flag_prev, flag_acc, ones, var, total; uint32_t Lp; };
K2_HD SnapLayout snap_layout(uint32_t L) {
    SnapLayout s; uint64_t o = 0;
    s.Lp = (L + 1u + 31u) & ~31u;
    s.small = o;     o += (sizeof(WarpModels) + 15u) & ~15ull;
    s.pos_hdr = o;   o += 16u;                                         /* card, n */
    s.pos_val = o;   o += (uint64_t)(CBCG_SNAP_POS_MAX + 32u) * 4u;
    s.pos_cnt = o;   o += (uint64_t)(CBCG_SNAP_POS_MAX + 32u) * 4u;
    s.pos_alpha = o; o += 4u * PA_STRIDE * 4u + 16u;
    s.bitmap = o;    o += 2048u * 4u;
    s.flag_prev = o; o += 65536u * 4u;                                 /* merge scratch: dense FLAG counts */
    s.flag_acc = o;  o += 65536u * 4u;
    s.ones = o;      o += (uint64_t)s.Lp * 4u;                         /* the initial state of a var row, read only */
    s.var = o;       o += (uint64_t)CBCG_VAR_CONTEXTS * s.Lp * 4u;
    s.total = (o + 255u) & ~255ull;
    return s;
}

K2_HD uint64_t fin_stride_dev() { return (sizeof(WarpModels) + 15u) & ~15ull; }

/* Only `var` (the last piece) moves with L: every other offset is a compile-time constant, so the block coder keeps
 * one base pointer and forms the addresses where it uses them (registers are what bounds its occupancy). */
struct SnapView {
    const uint8_t *base; uint32_t Lp;
    K2_HD SnapView() {}
    K2_HD SnapView(const uint8_t *b, uint32_t L) : base(b), Lp((L + 1u + 31u) & ~31u) {}
    K2_HD const uint32_t *at(uint64_t off) const { return (const uint32_t *)(base + off); }
    K2_HD const uint32_t *small() const { return at(snap_layout(1).small); }
    K2_HD const uint32_t *pos_hdr() const { return at(snap_layout(1).pos_hdr); }
    K2_HD const uint32_t *pos_val() const { return at(snap_layout(1).pos_val); }
    K2_HD const uint32_t *pos_cnt() const { return at(snap_layout(1).pos_cnt); }
    K2_HD const uint32_t *pos_alpha() const { return at(snap_layout(1).pos_alpha); }
    K2_HD const uint32_t *bitmap() const { return at(snap_layout(1).bitmap); }
    K2_HD const uint32_t *ones() const { return at(snap_layout(1).ones); }
    K2_HD const uint32_t *var_row(uint32_t ctx) const { return at(snap_layout(1).ones + (uint64_t)Lp * 4u) + (uint64_t)ctx * Lp; }
};

