/*
 * k2_coder.cu -- K2: adaptive context models + arithmetic coder, one warp per block (hot path part 2).
 *
 * Replaces, bit for bit:
 *   stream_model.c   update_model :31-51, send_value_to_as :53-76, read_value_from_as :78-117
 *   Arithmetic_stream.c  arithmetic_encoder_step :274-345, encoder_last_step :348-364,
 *                        arithmetic_get_symbol_range :373-381, arithmetic_decoder_step :389-454,
 *                        the MSB-first bit packer :155-194
 *   read_compression.c   compress_read :15-44, compress_pos(_alpha) :75-159, compress_flag :50-70,
 *                        compress_match/snps/indels/var/chars :164-260, the emission half of
 *                        compress_edits :557-600, compute_delta_to_first_snp :703-718
 *   read_decompression.c decompress_read :59-86 and the decoding half of reconstruct_read :339-458
 *   id_compression.c     compress_rname / decompress_rname :39-94 (single-block mode)
 *   qv_codebook.c        compress_int / decompress_int :14-95 (stream header, single-block mode)
 * with the initial model states of sam_models.c (:56-411, :562-586, :611-620, :734-770).
 *
 * B200 design. Each block of position-ordered reads is an independent coder instance run by ONE
 * WARP; K2_WARPS blocks share a CTA. All 32 lanes carry the coder interval redundantly (uniform
 * registers, no divergence); the lanes cooperate on what is a serial scan in the reference:
 *   - cumulative counts: strided partial sums + __reduce_add_sync (encode), 32-wide inclusive
 *     shuffle scan + ballot (decode search);
 *   - the 65 536-symbol FLAG model and the 255-symbol length models are kept SPARSE (all-ones
 *     initial state is closed under the reference's halve-and-increment rescale), so a FLAG step is
 *     one pass over <= 128 touched values in shared memory instead of a 65 536-entry scan;
 *   - the first 32 slots of the growing POS alphabet live one per lane in registers;
 *   - var rows (65 535 contexts x L counts) are created on first touch in a per-block arena in HBM,
 *     found through a 32-wide probed hash table (one coalesced 256 B load per lookup);
 *   - small dense models (snps, indels, chars, match, length byte 0) live in shared memory;
 *   - the SNP-site memory snpInRef[] (300 MB global array in the reference) is a 1024-bit ring held
 *     one word per lane: reads are position-sorted, so only [pos-1, pos+L) is ever consulted;
 *   - renormalisation is closed-form (ac_core.h): no bit-at-a-time loop.
 * The coder is latency-bound integer work, not HBM-bound: throughput comes from the number of
 * resident warps (blocks), see DESIGN.md.
 */
#include <algorithm>
#include "common.cuh"
#include "internal.h"
#include "ac_core.h"

#include "k2_layout.h"

uint64_t coder_ws_bytes_bound(uint32_t L, uint64_t n_reads, uint64_t n_edits, uint64_t n_blocks, int legacy, int primed) {
    if (legacy) return ws_layout(L, n_reads, n_edits, 1, 0).total + 256;
    const uint64_t Lp = (L + 1u + 31u) & ~31u;
    /* per block: pos 2 x (n+34) x 4 (+32), pos_alpha 4128, hash <= max(32, 4 n_edits + 4) x 8, rows n_edits x Lp x 4;
       a block in direct mode replaces hash + rows by 8 KB + 65535 rows: bounded by its own n_edits >= 32768 rows. */
    uint64_t b = n_blocks * (2u * (34u * 4u + 16u) + 4u * PA_STRIDE * 4u + 16u + 32u * 8u + 8192u + 512u);
    b += n_reads * 8u + n_edits * 32u + n_edits * Lp * 4u;
    if (primed) b += n_blocks * (uint64_t)CBCG_SNAP_POS_MAX * 8u;
    return 2u * b + 4096u;                                   /* direct blocks use <= 2 x their hashed size */
}
uint64_t coder_payload_bound(uint64_t n_reads, uint64_t n_edits, uint64_t n_blocks, int legacy) {
    return payload_cap_bytes(n_reads, n_edits, legacy ? 2 : 0) + n_blocks * 512u;   /* per block: four substream regions, each with its own slack and alignment */
}
uint64_t snapshot_bytes(uint32_t L) { return snap_layout(L).total; }
uint64_t fin_stride_bytes(void) { return (sizeof(WarpModels) + 15u) & ~15ull; }

/* All-ones initial state of a dense model (every initialize_stream_model_* of sam_models.c but chars).
 * Out of line on purpose: it is cold code, and the block coder's loop has to fit the instruction cache. */
__device__ __noinline__ void fill_ones(uint32_t *m, uint32_t card, uint32_t lane) {
    for (uint32_t i = lane; i < card; i += 32u) m[i] = 1u;
    if (lane == 0) m[card] = card;
}

/* Cold paths, out of line for the same reason. */
struct WarpModels;
/* update_model's rescale (src/stream_model.c:38-49): halve-and-increment every count; returns the new total. */
__device__ __noinline__ uint32_t rescale_counts(uint32_t *m, uint32_t card, uint32_t lane) {
    uint32_t s = 0;
    for (uint32_t i = lane; i < card; i += 32u) { const uint32_t c = (m[i] >> 1) + 1u; m[i] = c; s += c; }
    return __reduce_add_sync(FULL_MASK, s);
}
/* A FLAG value seen for the first time in this block: insert (x, 1 + 8) into the ascending sparse table. */
__device__ __noinline__ void flag_insert(uint32_t *key, uint32_t *cnt, uint32_t used, uint32_t x, uint32_t lane) {
    uint32_t p = 0;                                        /* insertion point: touched values below x */
    for (uint32_t base = 0; base < used; base += 32u) {
        const uint32_t i = base + lane;
        p += (uint32_t)__popc(__ballot_sync(FULL_MASK, i < used && key[i] < x));
    }
    if (used > p) {
        for (int base = (int)((used - 1u) & ~31u); base >= 0; base -= 32) {
            const uint32_t i = (uint32_t)base + lane;
            const bool mv = (i >= p && i < used);
            uint32_t k = 0, c = 0;
            if (mv) { k = key[i]; c = cnt[i]; }
            __syncwarp();
            if (mv) { key[i + 1u] = k; cnt[i + 1u] = c; }
            __syncwarp();
            if ((uint32_t)base <= p) break;
        }
    }
    if (lane == 0) { key[p] = x; cnt[p] = 1u + 8u; }
    __syncwarp();
}

/* A var row built from its read-only source with one touch (count of x and the total, +step) already applied. */
__device__ __noinline__ void copy_row_touched(uint32_t *row, const uint32_t *src, uint32_t L, uint32_t x, uint32_t step, uint32_t lane) {
    for (uint32_t i = lane; i <= L; i += 32u) row[i] = src[i] + ((i == x || i == L) ? step : 0u);
}
/* The last 1..3 bytes of a block's payload, zeros behind them (big-endian word). */
__device__ __noinline__ uint32_t refill_tail(const uint8_t *in, uint32_t in_pos, uint32_t in_len) {
    uint32_t w = 0;
    for (uint32_t i = 0; i < 4u; i++) { w <<= 8; if (in_pos + i < in_len) w |= (uint32_t)in[in_pos + i]; }
    return w;
}
/* Bit packer state, passed to the out-of-line long-run emitter. */
struct BitSink { uint64_t acc; uint32_t nacc, out_pos, out_cap; uint8_t *out; int err; };
__device__ __forceinline__ void sink_put(BitSink &b, uint32_t v, uint32_t k, uint32_t lane) {
    if (k == 0) return;
    b.acc = (b.acc << k) | (uint64_t)v;
    b.nacc += k;
    if (b.nacc >= 32u) {
        const uint32_t w = (uint32_t)(b.acc >> (b.nacc - 32u));
        if (b.out_pos + 4u <= b.out_cap) { if (lane == 0) *reinterpret_cast<uint32_t *>(b.out + b.out_pos) = __byte_perm(w, 0u, 0x0123); }
        else b.err = CBCG_ERR_CAPACITY;
        b.out_pos += 4u;
        b.nacc -= 32u;
        b.acc &= (1ull << b.nacc) - 1ull;
    }
}
/* b0, then `run` inverse bits (more than fit one 32-bit put: a long E3 run), then the low rest_bits of rest. */
__device__ __noinline__ void emit_long(BitSink *bs, uint32_t b0, uint32_t run, uint32_t rest, uint32_t rest_bits, uint32_t lane) {
    BitSink b = *bs;
    const uint32_t inv = b0 ? 0u : 0xffffffffu;
    uint32_t r = run < 31u ? run : 31u;
    sink_put(b, (b0 << r) | (inv & ((1u << r) - 1u)), r + 1u, lane);
    run -= r;
    while (run) { r = run < 32u ? run : 32u; sink_put(b, r == 32u ? inv : (inv & ((1u << r) - 1u)), r, lane); run -= r; }
    sink_put(b, rest, rest_bits, lane);
    *bs = b;
}

/* ------------------------------------------------------------------------------------------------ */
/* TRI: the encoder's model half on its own (k2_model_kernel): every coder step is replaced by a store of the symbol's
   interval (cumulative count, count, model total) for the interval kernel (k2_code_kernel) to code. */
#define TRI_ESC 1u                             /* on a POS interval: the escape's four byte symbols follow (in the block's escape list) */
/* The decoder's coder step as ONE copy of code: interval update, renormalisation shape, the next k + m stream bits, the
 * tag -- 40 % of the instructions the decoder executes, which the direct call sites of the state machine would otherwise
 * each hold inline (six hot sites: a hot loop of 24 KB walked by warps that are rarely at the same place, 23 % of the
 * decoder's stall samples waiting for instruction fetch). State travels by value in registers (whole-program
 * compilation: ptxas gives a non-inlined device function its own register convention, no stack). */
struct AcDecState { uint32_t l, u, t, dcnt, in_pos; uint64_t dbuf; };
__device__ __noinline__ AcDecState ac_decode_step_shared(AcDecState s, uint32_t lo, uint32_t cnt, uint32_t n, double rn, const WarpCold *cold) {
    AcInterval a = { s.l, s.u };
    ac_narrow_r(a, lo, lo + cnt, n, rn);
    uint32_t k, bits, m; AcInterval nx;
    ac_renorm_shape(a, k, bits, m, nx);
    uint32_t left = k + m;                                                /* up to 51 bits; the tag keeps the last 26 */
    s.l = nx.l; s.u = nx.u;
    if (left == 0u) return s;
    if (LIKELY(left < 32u)) {
        /* nearly every step: fewer than 32 bits, one top-up at most, and 32-bit arithmetic for the tag (bits shifted past
           bit 31 are past the 26 the tag keeps) */
        if (UNLIKELY(s.dcnt < left)) {
            uint32_t w = 0;
            const uint8_t *in = cold->io; const uint32_t in_len = cold->io_cap;
            if (s.in_pos + 4u <= in_len) {
                w = ((uint32_t)in[s.in_pos] << 24) | ((uint32_t)in[s.in_pos + 1u] << 16) | ((uint32_t)in[s.in_pos + 2u] << 8) | (uint32_t)in[s.in_pos + 3u];
            } else if (s.in_pos < in_len) w = refill_tail(in, s.in_pos, in_len);
            s.in_pos += 4u;
            s.dbuf |= (uint64_t)w << (32u - s.dcnt);
            s.dcnt += 32u;
        }
        const uint32_t in32 = (uint32_t)(s.dbuf >> 32) >> (32u - left);
        s.dbuf <<= left;
        s.dcnt -= left;
        uint32_t r = ((s.t << left) | in32) & CBCG_AC_TOP;
        if (m) r ^= CBCG_AC_MSB;
        s.t = r;
        return s;
    }
    uint64_t in64 = 0;
    while (left) {
        const uint32_t take = left < 32u ? left : 32u;
        if (UNLIKELY(s.dcnt < take)) {
            uint32_t w = 0;
            const uint8_t *in = cold->io; const uint32_t in_len = cold->io_cap;
            if (s.in_pos + 4u <= in_len) {
                w = ((uint32_t)in[s.in_pos] << 24) | ((uint32_t)in[s.in_pos + 1u] << 16) | ((uint32_t)in[s.in_pos + 2u] << 8) | (uint32_t)in[s.in_pos + 3u];
            } else if (s.in_pos < in_len) w = refill_tail(in, s.in_pos, in_len);
            s.in_pos += 4u;
            s.dbuf |= (uint64_t)w << (32u - s.dcnt);
            s.dcnt += 32u;
        }
        in64 = (in64 << take) | (uint32_t)(s.dbuf >> (64u - take));
        s.dbuf <<= take;
        s.dcnt -= take;
        left -= take;
    }
    s.t = ac_tag_shift(s.t, k, m, (uint32_t)in64);
    return s;
}

template <int MODE, bool TRI = false>
struct Coder {
    /* --- TRI: where the next interval goes, and the flag bits that go with it */
    uint4 *tri_at; uint32_t tri_flag;
    /* --- arithmetic coder state (uniform across the warp) */
    AcInterval a;
    uint32_t t;
    int32_t scale3;
    /* encoder bit packer */
    uint64_t acc; uint32_t nacc;
    uint32_t out_pos;
    /* decoder bit reader */
    uint32_t in_pos, dcnt; uint64_t dbuf;
    /* symbol list */
    cbcg_symbol *list; uint32_t list_n, list_cap;

    uint32_t lane;
    int err;
    uint32_t n_symbols;
    uint32_t last_lo, last_n;              /* interval start and model total of the last dense symbol */

    /* --- models */
    WarpModels *M;
    uint32_t L, Lp;
    /* pos: slots 0..31 one per lane, the rest in HBM */
    uint32_t pos_rv, pos_rc, pos_card, pos_n;
    bool pa_init;
    /* var */
    uint64_t *var_hash; uint32_t hash_mask; uint32_t n_rows; bool var_direct;
    /* the rest of the block's workspace, addressed from var_hash (ws_layout: pos_cnt | pos_val | pos_alpha | var_hash | var_rows) */
    WarpCold *coldp;
    __device__ __forceinline__ WarpCold &cold() const { return *coldp; }
    __device__ __forceinline__ uint32_t pos_stride() const { return (uint32_t)((((uint64_t)cold().pos_cap * 4u + 15u) & ~15ull) >> 2); }
    __device__ __forceinline__ uint32_t *pos_alpha() const { return reinterpret_cast<uint32_t *>(var_hash) - (4u * PA_STRIDE + 4u); }
    __device__ __forceinline__ uint32_t *pos_gval() const { return pos_alpha() - pos_stride(); }
    __device__ __forceinline__ uint32_t *pos_gcnt() const { return pos_alpha() - 2u * pos_stride(); }
    __device__ __forceinline__ uint32_t *var_rows() const { return reinterpret_cast<uint32_t *>(var_hash + hash_mask + 1u); }
    __device__ __forceinline__ uint32_t *var_bitmap() const { return reinterpret_cast<uint32_t *>(var_hash); }
    bool var_defer, var_ro; uint32_t defer_idx, defer_key;   /* deferred rows of the last generation (var_row) */
    /* legacy-only */
    uint32_t *codebook, *rname;
    __device__ __forceinline__ uint32_t *flag_spill() const { return rname + 256u * PA_STRIDE + 4u; }   /* ws_layout: 2 x 65 536 words behind rname */
    /* primed blocks */
    bool primed, lean; SnapView snap;
    /* SNP-site ring: word (p >> 5) & 31 lives in lane; covers [ring_base, ring_base + 1024) */
    uint32_t ring; uint32_t ring_word;     /* ring_word = ring_base >> 5 */

    /* ============================================================ bit I/O */
    __device__ __forceinline__ void put_bits(uint32_t v, uint32_t k) {       /* k <= 32 */
        if (k == 0) return;
        acc = (acc << k) | (uint64_t)v;
        nacc += k;
        if (UNLIKELY(nacc >= 32u)) {
            uint32_t w = (uint32_t)(acc >> (nacc - 32u));
            if (out_pos + 4u <= cold().io_cap) { if (lane == 0) *reinterpret_cast<uint32_t *>(cold().io + out_pos) = __byte_perm(w, 0u, 0x0123); }
            else err = CBCG_ERR_CAPACITY;
            out_pos += 4u;
            nacc -= 32u;
            acc &= (1ull << nacc) - 1ull;
        }
    }
    /* One bit b0, then `run` copies of its inverse (the pending E3 bits, src/Arithmetic_stream.c:318-322), then the
       low rest_bits of rest. The usual case is one put; long runs go out of line: the hot loop has to fit the
       instruction cache. */
    __device__ __forceinline__ void emit(uint32_t b0, uint32_t run, uint32_t rest, uint32_t rest_bits) {
        if (LIKELY(run + 1u + rest_bits <= 32u)) {
            const uint32_t inv = b0 ? 0u : 0xffffffffu;
            put_bits((b0 << (run + rest_bits)) | ((inv & ((1u << run) - 1u)) << rest_bits) | rest, run + 1u + rest_bits);
        } else {
            BitSink b = { acc, nacc, out_pos, cold().io_cap, cold().io, err };
            emit_long(&b, b0, run, rest, rest_bits, lane);
            acc = b.acc; nacc = b.nacc; out_pos = b.out_pos; err = b.err;
        }
    }
    /* stream_finish_byte (:189-194): the byte in progress always goes out, even an empty one */
    __device__ __forceinline__ void finish_bits(bool always_last = true) {
        uint32_t full = nacc >> 3, rem = nacc & 7u;
        for (uint32_t i = 0; i < full; i++) {
            uint32_t byte = (uint32_t)(acc >> (nacc - 8u * (i + 1u))) & 0xffu;
            if (out_pos < cold().io_cap) { if (lane == 0) cold().io[out_pos] = (uint8_t)byte; } else err = CBCG_ERR_CAPACITY;
            out_pos++;
        }
        if (rem || always_last) {
            uint32_t last = rem ? (((uint32_t)acc & ((1u << rem) - 1u)) << (8u - rem)) : 0u;
            if (out_pos < cold().io_cap) { if (lane == 0) cold().io[out_pos] = (uint8_t)last; } else err = CBCG_ERR_CAPACITY;
            out_pos++;
        }
        nacc = 0; acc = 0;
    }
    /* next k bits of the input, first bit most significant; zeros past the end (the reference's
       zero-filled buffer, src/Arithmetic_stream.c:30,117). dbuf holds the upcoming bits left-aligned;
       it is topped up 32 bits at a time, so a symbol costs shifts, not loads. */
    __device__ __forceinline__ uint32_t get_bits(uint32_t k) {               /* k <= 32 */
        if (k == 0) return 0u;
        if (UNLIKELY(dcnt < k)) {
            uint32_t w = 0;
            const uint8_t *in = cold().io; const uint32_t in_len = cold().io_cap;
            if (in_pos + 4u <= in_len) {
                w = ((uint32_t)in[in_pos] << 24) | ((uint32_t)in[in_pos + 1u] << 16) | ((uint32_t)in[in_pos + 2u] << 8) | (uint32_t)in[in_pos + 3u];
            } else if (in_pos < in_len) w = refill_tail(in, in_pos, in_len);
            in_pos += 4u;
            dbuf |= (uint64_t)w << (32u - dcnt);
            dcnt += 32u;
        }
        const uint32_t r = (uint32_t)(dbuf >> (64u - k));
        dbuf <<= k;
        dcnt -= k;
        return r;
    }

    /* ============================================================ arithmetic coder */
    __device__ __forceinline__ void ac_init() {
        a.l = 0; a.u = CBCG_AC_TOP; scale3 = 0; t = 0; acc = 0; nacc = 0; out_pos = 0; in_pos = 0; dcnt = 0; dbuf = 0;
        if (MODE == MODE_DEC) t = get_bits(CBCG_AC_BITS);                    /* :262 */
    }
    __device__ __forceinline__ void ac_encode(uint32_t lo, uint32_t cnt, uint32_t n) {
        if (UNLIKELY(cnt == 0u || n == 0u)) { err = CBCG_ERR_INPUT; return; }          /* reference: assert :71 / :293 */
        ac_narrow(a, lo, lo + cnt, n);
        uint32_t k, bits, m; AcInterval nx;
        ac_renorm_shape(a, k, bits, m, nx);
        if (k) {
            emit((bits >> (k - 1u)) & 1u, (uint32_t)scale3, bits & ((1u << (k - 1u)) - 1u), k - 1u);
            scale3 = 0;
        }
        scale3 += (int32_t)m;
        a = nx;
    }
    __device__ __forceinline__ void ac_decode_step(uint32_t lo, uint32_t cnt, uint32_t n, double rn) {
        const AcDecState r = ac_decode_step_shared(AcDecState{ a.l, a.u, t, dcnt, in_pos, dbuf }, lo, cnt, n, rn, coldp);
        a.l = r.l; a.u = r.u; t = r.t; dcnt = r.dcnt; in_pos = r.in_pos; dbuf = r.dbuf;
    }
    /* encoder_last_step (:348-364) */
    __device__ __forceinline__ void ac_flush() {
        emit(a.l >> (CBCG_AC_BITS - 1u), (uint32_t)scale3, a.l & CBCG_AC_LOWMASK, CBCG_AC_BITS - 1u);
        scale3 = 0;
        finish_bits();
    }

    /* Blocked containers: after renormalisation l < 2^25 <= u, so the value 2^25 -- "1", the pending E3 bits as
       "0", zeros ever after -- lies in [l, u]; the decoder reads zeros past the end of a block. */
    __device__ __forceinline__ void ac_flush_short() {
        emit(1u, (uint32_t)scale3, 0u, 0u);
        scale3 = 0;
        finish_bits(false);
    }

    /* Decoder search without the division of arithmetic_get_symbol_range (:373-381): target = floor(A / range) with
       A = (t - l + 1) n - 1, and for an integer cumulative count c,  c <= target  <=>  c * range <= A.  The 32 lanes
       test their candidates with one 64-bit multiply each instead of waiting for a reciprocal and a corrected quotient. */
    __device__ __forceinline__ uint64_t dec_A(uint32_t n) const { return (uint64_t)(t - a.l + 1u) * n - 1ull; }
    __device__ __forceinline__ uint32_t dec_range() const { return a.u - a.l + 1u; }
#define DEC_LE(c) ((uint64_t)(c) * range <= A)               /* c <= target */

    /* one coder step given the symbol's interval; decode: caller found (lo, cnt) from the target */
    /* decoder: the reciprocal of the model total, formed before the search so that it is ready when the symbol is */
    __device__ __forceinline__ double dec_rcp(uint32_t n) const { return MODE == MODE_DEC ? ac_rcp(n) : 0.0; }
    __device__ __forceinline__ void code_interval(uint32_t lo, uint32_t cnt, uint32_t n) { code_interval(lo, cnt, n, dec_rcp(n)); }
    __device__ __forceinline__ void code_interval(uint32_t lo, uint32_t cnt, uint32_t n, double rn) {
        if (TRI) {
            if (UNLIKELY(cnt == 0u || n == 0u)) { err = CBCG_ERR_INPUT; return; }          /* reference: assert :71 / :293 */
            if (lane == 0) *tri_at = make_uint4(lo, cnt, n, tri_flag);
            tri_flag = 0u;
        } else if (MODE == MODE_ENC) ac_encode(lo, cnt, n); else ac_decode_step(lo, cnt, n, rn);
        n_symbols++;
    }

    /* ============================================================ dense models (counts[card], n at [card]) */
    /* cnt and n are the symbol's count and the model total the caller just coded with: no reload on the dependent
       chain. A deferred var row (var_ro, see var_row) is not written: the touch is noted in its hash slot instead. */
    template <bool IS_VAR>
    __device__ __forceinline__ void dense_update(uint32_t *m, uint32_t card, uint32_t step, uint32_t x, uint32_t cnt, uint32_t n) {
        n += step;
        if (IS_VAR && UNLIKELY(var_ro)) {
            var_ro = false;
            if (n < CBCG_RESCALE) {
                if (lane == 0) var_hash[defer_idx] = ((uint64_t)defer_key << 32) | VAR_DEFERRED | x;
                SYNCW();
                return;
            }
            /* the touch rescales the row: build it after all (cold) */
            if (n_rows >= cold().rows_cap) { err = CBCG_ERR_INTERNAL; return; }
            uint32_t *row = var_rows() + (uint64_t)n_rows * Lp;
            copy_row_touched(row, m, L, x, step, lane);
            if (lane == 0) var_hash[defer_idx] = ((uint64_t)defer_key << 32) | n_rows;
            n_rows++;
            SYNCW();
            const uint32_t s = rescale_counts(row, card, lane);
            SYNCW();
            if (lane == 0) row[card] = s;
            SYNCW();
            return;
        }
        SYNCW();
        if (lane == 0) { m[x] = cnt + step; m[card] = n; }
        SYNCW();
        if (UNLIKELY(n >= CBCG_RESCALE)) {                                   /* update_model :38-49 */
            const uint32_t s = rescale_counts(m, card, lane);
            SYNCW();
            if (lane == 0) m[card] = s;
            SYNCW();
        }
    }
    /* Four counts per lane per step (rows are 16-byte aligned): 128 symbols of cumulative count in one load,
       where the reference walks them one by one (src/stream_model.c:64-67, :96-99). */
    __device__ __forceinline__ uint4 load4(const uint32_t *m, uint32_t i, uint32_t card) {
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (i < card) {
            v = *reinterpret_cast<const uint4 *>(m + i);
            if (i + 1u >= card) v.y = 0u;
            if (i + 2u >= card) v.z = 0u;
            if (i + 3u >= card) v.w = 0u;
        }
        return v;
    }
    /* pre: the caller already knows the symbol and its cumulative count (pre_lo); no scan.
       SMALL (call sites whose alphabet is a constant 2 or 5: match bit, bases): the first four counts always resolve
       the symbol (card 5: or it is symbol 4), so the scan code is not instantiated there. IS_VAR: the model may be a
       deferred var row. Both only prune code: every instantiation computes the same thing. */
    template <int SMALL, bool IS_VAR>
    __device__ __forceinline__ uint32_t sym_dense(uint32_t *m, uint32_t card, uint32_t step, uint32_t x, bool pre, uint32_t pre_lo) {
        if (err) return 0u;
        const uint32_t n = m[card];
        const double rn = dec_rcp(n);
        uint32_t lo = 0, cnt = 0;
        if (pre) { lo = pre_lo; cnt = m[x]; }
        else if (MODE == MODE_ENC) {
            if (UNLIKELY(x >= card)) { err = CBCG_ERR_INPUT; return 0u; }    /* reference: assert :62 */
            if (SMALL == 2 || LIKELY(x < 4u)) {                                      /* most symbols are small: one broadcast load */
                const uint4 v = load4(m, 0u, card);
                lo = (x > 0u ? v.x : 0u) + (x > 1u ? v.y : 0u) + (x > 2u ? v.z : 0u);
                cnt = x == 0u ? v.x : (x == 1u ? v.y : (x == 2u ? v.z : v.w));
            } else if (SMALL == 5) {                                         /* symbol 4 of 5 */
                const uint4 v = load4(m, 0u, card);
                lo = v.x + v.y + v.z + v.w; cnt = m[4];
            } else {
                uint32_t s = 0;
                for (uint32_t base = 0; base < x; base += 128u) {
                    const uint32_t i = base + 4u * lane;
                    const uint4 v = load4(m, i, card);
                    s += (i < x ? v.x : 0u) + (i + 1u < x ? v.y : 0u) + (i + 2u < x ? v.z : 0u) + (i + 3u < x ? v.w : 0u);
                }
                lo = warp_sum(s); cnt = m[x];
            }
        } else {
            const uint64_t A = dec_A(n); const uint32_t range = dec_range();
            const uint4 f = load4(m, 0u, card);
            const uint32_t s1 = f.x, s2 = s1 + f.y, s3 = s2 + f.z, s4 = s3 + f.w;
            if (LIKELY(!DEC_LE(s4))) {                                       /* resolved by the first four counts: no scan */
                const uint32_t q = (uint32_t)DEC_LE(s1) + (uint32_t)DEC_LE(s2) + (uint32_t)DEC_LE(s3);
                lo = q == 0u ? 0u : (q == 1u ? s1 : (q == 2u ? s2 : s3));
                cnt = q == 0u ? f.x : (q == 1u ? f.y : (q == 2u ? f.z : f.w));
                x = q;
            } else if (SMALL == 2) { err = CBCG_ERR_CORRUPT; return 0u; }   /* target beyond the model total */
            else if (SMALL == 5) {
                x = 4u; lo = s4; cnt = m[4];
                if (DEC_LE(s4 + cnt)) { err = CBCG_ERR_CORRUPT; return 0u; }
            } else {
                uint32_t carry = 0; bool found = false;
                x = 0;
                for (uint32_t base = 0; base < card; base += 128u) {
                    const uint32_t i = base + 4u * lane;
                    const uint4 v = load4(m, i, card);
                    const uint32_t mine = v.x + v.y + v.z + v.w;
                    const uint32_t incl = warp_incl_scan(mine) + carry;
                    const uint32_t hit = __ballot_sync(FULL_MASK, !DEC_LE(incl));     /* lanes past the row add 0: never first */
                    if (hit) {
                        const uint32_t h = (uint32_t)__ffs(hit) - 1u;
                        const uint32_t before = __shfl_sync(FULL_MASK, incl - mine, h);
                        const uint32_t c0 = __shfl_sync(FULL_MASK, v.x, h), c1 = __shfl_sync(FULL_MASK, v.y, h);
                        const uint32_t c2 = __shfl_sync(FULL_MASK, v.z, h), c3 = __shfl_sync(FULL_MASK, v.w, h);
                        const uint32_t t1 = before + c0, t2 = t1 + c1, t3 = t2 + c2;
                        const uint32_t q = (uint32_t)DEC_LE(t1) + (uint32_t)DEC_LE(t2) + (uint32_t)DEC_LE(t3);
                        lo = q == 0u ? before : (q == 1u ? t1 : (q == 2u ? t2 : t3));
                        cnt = q == 0u ? c0 : (q == 1u ? c1 : (q == 2u ? c2 : c3));
                        x = base + 4u * h + q; found = true;
                        break;
                    }
                    carry = __shfl_sync(FULL_MASK, incl, 31);
                }
                if (!found) { err = CBCG_ERR_CORRUPT; return 0u; }
            }
            if (UNLIKELY(x >= card)) { err = CBCG_ERR_CORRUPT; return 0u; }
        }
        last_lo = lo; last_n = n;
        code_interval(lo, cnt, n, rn);
        if (UNLIKELY(err)) return 0u;
        dense_update<IS_VAR>(m, card, step, x, cnt, n);
        return x;
    }

    __device__ __forceinline__ void dense_init_ones(uint32_t *m, uint32_t card) { fill_ones(m, card, lane); }

    /* ============================================================ length bytes 1..3 (always symbol 0) */
    __device__ __forceinline__ uint32_t sym_rlenk(uint32_t k, uint32_t x) {
        if (err) return 0u;
        uint32_t c0 = M->rlenk[k][0], n = M->rlenk[k][1];
        if (MODE == MODE_ENC) { if (x != 0u) { err = CBCG_ERR_INPUT; return 0u; } }
        else { const uint64_t A = dec_A(n); const uint32_t range = dec_range(); if (DEC_LE(c0)) { err = CBCG_ERR_CORRUPT; return 0u; } }
        code_interval(0u, c0, n);
        c0 += 10u; n += 10u;
        if (n >= CBCG_RESCALE) { c0 = (c0 >> 1) + 1u; n = c0 + 254u; }
        SYNCW();
        if (lane == 0) { M->rlenk[k][0] = c0; M->rlenk[k][1] = n; }
        SYNCW();
        return 0u;
    }

    /* ============================================================ FLAG (65 536 symbols, sparse) */
    __device__ __forceinline__ uint32_t sym_flag(uint32_t x) {
        if (err) return 0u;
        const uint32_t used = M->flag_used, n = M->flag_n;
        const double rn = dec_rcp(n);
        uint32_t lo, cnt; int found_idx = -1;
        /* The table lives in shared memory while it has fewer than FLAG_CAP entries. Blocked containers never grow it
           further (rule F1); the single-block mode is the reference's own stream, whose model adapts all 65 536 values
           (src/sam_models.c:96-130): there the table moves to the workspace when it reaches FLAG_CAP entries. */
        const bool unbounded = !lean && MODE != MODE_LIST;
        uint32_t *fkey = M->flag_key, *fcnt = M->flag_cnt;
        if (unbounded && UNLIKELY(used >= FLAG_CAP)) { fkey = flag_spill(); fcnt = fkey + 65536u; }
        if (MODE == MODE_ENC) {
            if (x > 0xffffu) { err = CBCG_ERR_INPUT; return 0u; }
            uint32_t extra = 0; cnt = 1u;
            for (uint32_t base = 0; base < used; base += 32u) {
                const uint32_t i = base + lane;
                const uint32_t k = (i < used) ? fkey[i] : 0xffffffffu;
                const uint32_t c = (i < used) ? fcnt[i] : 1u;
                if (k < x) extra += c - 1u;
                const uint32_t hit = __ballot_sync(FULL_MASK, k == x);
                if (hit) { const uint32_t h = (uint32_t)__ffs(hit) - 1u; cnt = __shfl_sync(FULL_MASK, c, h); found_idx = (int)(base + h); }
            }
            lo = x + warp_sum(extra);
        } else {
            /* the touched values are tested with DEC_LE; the target itself (one division) is only needed when the
               symbol turns out to be an untouched value, whose ordinal is target minus the extras below it */
            const uint64_t A = dec_A(n); const uint32_t range = dec_range();
            uint32_t carry = 0; bool done = false;
            lo = 0; cnt = 1u; x = 0;
            for (uint32_t base = 0; base < used && !done; base += 32u) {
                const uint32_t i = base + lane;
                const bool valid = i < used;
                const uint32_t k = valid ? fkey[i] : 0xffffffffu;
                const uint32_t c = valid ? fcnt[i] : 1u;
                const uint32_t e = c - 1u;
                const uint32_t incl = warp_incl_scan(e) + carry;
                const uint32_t E = incl - e;                       /* extras of all touched values below this one */
                const uint32_t Ak = k + E;                         /* cumulative count at the start of value k */
                const uint32_t below = __ballot_sync(FULL_MASK, valid && DEC_LE(Ak + c));
                const uint32_t nb = (uint32_t)__popc(below);
                if (nb == 32u) { carry = __shfl_sync(FULL_MASK, incl, 31); continue; }
                const uint32_t Ec = __shfl_sync(FULL_MASK, E, nb);
                const uint32_t Ac = __shfl_sync(FULL_MASK, Ak, nb);
                const uint32_t cc = __shfl_sync(FULL_MASK, c, nb);
                const uint32_t kc = __shfl_sync(FULL_MASK, k, nb);
                const bool vc = (base + nb) < used;
                if (vc && DEC_LE(Ac)) { x = kc; lo = Ac; cnt = cc; found_idx = (int)(base + nb); }
                else { const uint32_t target = ac_target(a, t, n); x = target - Ec; lo = target; cnt = 1u; }
                carry = Ec; done = true;
            }
            if (!done) { const uint32_t target = ac_target(a, t, n); x = target - carry; lo = target; cnt = 1u; }   /* every touched value lies below */
            if (x > 0xffffu) { err = CBCG_ERR_CORRUPT; return 0u; }
        }
        code_interval(lo, cnt, n, rn);
        if (err) return 0u;
        /* update_model with step 8 */
        SYNCW();
        uint32_t nused = used;
        if (found_idx >= 0) { if (lane == 0) fcnt[found_idx] += 8u; }
        else {
            if (UNLIKELY(used >= FLAG_CAP) && !unbounded) return x;                  /* rule F1 (cbcg_format.h): coded at count 1, model unchanged */
            flag_insert(fkey, fcnt, used, x, lane);
            if (lane == 0) M->flag_used = used + 1u;
            nused = used + 1u;
            if (unbounded && UNLIKELY(nused == FLAG_CAP)) {                         /* the table outgrows shared memory: on to the workspace */
                SYNCW();
                uint32_t *sk = flag_spill();
                for (uint32_t i = lane; i < FLAG_CAP; i += 32u) { sk[i] = M->flag_key[i]; sk[65536u + i] = M->flag_cnt[i]; }
                fcnt = sk + 65536u;
            }
        }
        uint32_t nn = n + 8u;
        SYNCW();
        if (UNLIKELY(nn >= CBCG_RESCALE)) nn = rescale_counts(fcnt, nused, lane) + (65536u - nused);
        if (lane == 0) M->flag_n = nn;
        SYNCW();
        return x;
    }

    /* ============================================================ POS (growing alphabet) */
    __device__ __forceinline__ void pos_load(uint32_t base, uint32_t &v, uint32_t &c) {
        const uint32_t i = base + lane;
        if (base == 0u) { v = pos_rv; c = (i < pos_card) ? pos_rc : 0u; }
        else if (i < pos_card) { v = pos_gval()[i]; c = pos_gcnt()[i]; }
        else { v = 0u; c = 0u; }
    }
    __device__ __forceinline__ void pos_update(uint32_t slot) {                 /* update_model, step 10 */
        if (slot < 32u) { if (lane == slot) pos_rc += 10u; }
        else if (lane == 0) pos_gcnt()[slot] += 10u;
        pos_n += 10u;
        SYNCW();
        if (UNLIKELY(pos_n >= CBCG_RESCALE)) {
            uint32_t s = 0;
            if (lane < pos_card) { pos_rc = (pos_rc >> 1) + 1u; s += pos_rc; }
            { uint32_t *gc = pos_gcnt(); for (uint32_t i = 32u + lane; i < pos_card; i += 32u) { uint32_t c = (gc[i] >> 1) + 1u; gc[i] = c; s += c; } }
            pos_n = warp_sum(s);
            SYNCW();
        }
    }
    __device__ __forceinline__ void pos_append(uint32_t x) {                    /* new symbol, count 0, then updated (:147-153) */
        const uint32_t slot = pos_card;
        if (slot >= cold().pos_cap) { err = CBCG_ERR_INTERNAL; return; }
        if (slot < 32u) { if (lane == slot) { pos_rv = x; pos_rc = 0u; } }
        else if (lane == 0) { pos_gval()[slot] = x; pos_gcnt()[slot] = 0u; }
        pos_card = slot + 1u;
        SYNCW();
        pos_update(slot);
    }
    __device__ __forceinline__ void pa_ensure() {
        if (!pa_init) {
            uint32_t *pa = pos_alpha();
            if (primed) { for (uint32_t i = lane; i < 4u * PA_STRIDE; i += 32u) pa[i] = snap.pos_alpha()[i]; }
            else for (uint32_t k = 0; k < 4u; k++) dense_init_ones(pa + k * PA_STRIDE, 256u);
            pa_init = true;
            SYNCW();
        }
    }
    /* compress_pos / decompress_pos, the POS symbol itself: x = pos - prevPos + 1. Returns the value (decode:
       0 when the escape was decoded) and the slot; the caller codes the 4 escape bytes and calls pos_append. */
    __device__ __forceinline__ uint32_t sym_pos_main(uint32_t x, uint32_t &slot) {
        slot = 0;
        if (err) return 0u;
        const double rn = dec_rcp(pos_n);
        uint32_t lo = 0, cnt = 0;
        if (MODE == MODE_ENC) {
            bool found = false;
            for (uint32_t base = 0; base < pos_card; base += 32u) {
                uint32_t v, c; pos_load(base, v, c);
                const uint32_t i = base + lane;
                const uint32_t hit = __ballot_sync(FULL_MASK, i >= 1u && i < pos_card && v == x);
                if (hit) {
                    const uint32_t h = (uint32_t)__ffs(hit) - 1u;
                    lo += warp_sum(lane < h ? c : 0u);
                    cnt = __shfl_sync(FULL_MASK, c, h);
                    slot = base + h; found = true;
                    break;
                }
                lo += warp_sum(c);
            }
            if (!found) { slot = 0; lo = 0; cnt = __shfl_sync(FULL_MASK, pos_rc, 0); if (TRI) tri_flag = TRI_ESC; }
        } else {
            const uint64_t A = dec_A(pos_n); const uint32_t range = dec_range();
            uint32_t carry = 0; bool found = false;
            for (uint32_t base = 0; base < pos_card; base += 32u) {
                uint32_t v, c; pos_load(base, v, c);
                const uint32_t incl = warp_incl_scan(c) + carry;
                const uint32_t hit = __ballot_sync(FULL_MASK, (base + lane) < pos_card && !DEC_LE(incl));
                if (hit) {
                    const uint32_t h = (uint32_t)__ffs(hit) - 1u;
                    cnt = __shfl_sync(FULL_MASK, c, h);
                    lo = __shfl_sync(FULL_MASK, incl, h) - cnt;
                    slot = base + h; x = __shfl_sync(FULL_MASK, v, h); found = true;
                    break;
                }
                carry = __shfl_sync(FULL_MASK, incl, 31);
            }
            if (!found) { err = CBCG_ERR_CORRUPT; return 0u; }
        }
        code_interval(lo, cnt, pos_n, rn);
        if (err) return 0u;
        pos_update(slot);
        return x;
    }

    /* ============================================================ var rows */
    __device__ __forceinline__ uint32_t *var_row(uint32_t ctx) {
        if (ctx >= CBCG_VAR_CONTEXTS) { err = (MODE == MODE_ENC) ? CBCG_ERR_INPUT : CBCG_ERR_CORRUPT; return nullptr; }
        if (var_direct) {
            uint32_t *row = var_rows() + (uint64_t)ctx * Lp;
            const uint32_t w = var_bitmap()[ctx >> 5];
            if (!((w >> (ctx & 31u)) & 1u)) {
                dense_init_ones(row, L);
                SYNCW();
                if (lane == 0) var_bitmap()[ctx >> 5] = w | (1u << (ctx & 31u));
                SYNCW();
            }
            return row;
        }
        const uint32_t key = ctx + 1u;
        uint32_t h = (ctx * 0x9E3779B1u) >> 7;
        const uint32_t snap_w = primed ? snap.bitmap()[ctx >> 5] : 0u;           /* in flight with the probe */
        for (uint32_t probes = 0; probes <= hash_mask; probes += 32u, h += 32u) {
            const uint32_t idx = (h + lane) & hash_mask;
            const uint64_t s = var_hash[idx];
            const uint32_t k = (uint32_t)(s >> 32);
            const uint32_t mm = __ballot_sync(FULL_MASK, k == key);
            const uint32_t ee = __ballot_sync(FULL_MASK, k == 0u);
            if (mm && (!ee || __ffs(mm) < __ffs(ee))) {
                const uint32_t hl = (uint32_t)__ffs(mm) - 1u;
                const uint32_t r = __shfl_sync(FULL_MASK, (uint32_t)s, hl);
                if (!(r & VAR_DEFERRED)) return var_rows() + (uint64_t)r * Lp;
                /* second touch of a deferred row: build it now, with the first touch's update applied */
                if (n_rows >= cold().rows_cap) { err = CBCG_ERR_INTERNAL; return nullptr; }
                const uint32_t nr = n_rows++, x1 = r & 0xffffu;
                uint32_t *row = var_rows() + (uint64_t)nr * Lp;
                const uint32_t *src = ((snap_w >> (ctx & 31u)) & 1u) ? snap.var_row(ctx) : snap.ones();
                copy_row_touched(row, src, L, x1, 10u, lane);
                if (lane == hl) var_hash[idx] = ((uint64_t)key << 32) | nr;
                SYNCW();
                return row;
            }
            if (ee) {
                const uint32_t el = (uint32_t)__ffs(ee) - 1u;
                const bool in_snap = primed && ((snap_w >> (ctx & 31u)) & 1u);
                if (var_defer) {
                    /* Last generation: nobody merges this block's rows, and most contexts are touched once per block.
                       Code straight from the snapshot's row (read only) and note the touch in the hash slot
                       (dense_update); the row is only built if the context comes back. */
                    defer_idx = (h + el) & hash_mask; defer_key = key; var_ro = true;
                    return const_cast<uint32_t *>(in_snap ? snap.var_row(ctx) : snap.ones());
                }
                if (n_rows >= cold().rows_cap) { err = CBCG_ERR_INTERNAL; return nullptr; }
                const uint32_t r = n_rows++;
                uint32_t *row = var_rows() + (uint64_t)r * Lp;
                if (lane == el) var_hash[idx] = ((uint64_t)key << 32) | r;
                if (in_snap) {                                                       /* copy on first touch */
                    const uint32_t *src = snap.var_row(ctx);
                    for (uint32_t i = lane; i <= L; i += 32u) row[i] = src[i];
                } else dense_init_ones(row, L);
                SYNCW();
                return row;
            }
        }
        err = CBCG_ERR_INTERNAL;
        return nullptr;
    }
    /* ============================================================ SNP-site ring (snpInRef) */
    __device__ __forceinline__ void ring_reset() { ring = 0u; ring_word = 0u; }
    __device__ __forceinline__ void ring_advance(uint32_t pos) {               /* window must start at or below pos - 1 */
        const uint32_t nw = (pos - 1u) >> 5;
        if (nw > ring_word) {
            const uint32_t adv = nw - ring_word;
            if (adv >= 32u || ((lane - ring_word) & 31u) < adv) ring = 0u;     /* words that rotate out and back in */
            ring_word = nw;
        }
    }
    __device__ __forceinline__ void ring_set(uint32_t p) {                      /* snpInRef[p] = 1 */
        if ((p >> 5) - ring_word < 32u && lane == ((p >> 5) & 31u)) ring |= 1u << (p & 31u);
    }
    /* compute_delta_to_first_snp (:703-718): distance from position s to the first marked site in
       [s, e), else `none` */
    __device__ __forceinline__ uint32_t ring_first(uint32_t s, uint32_t e, uint32_t none) {
        uint32_t best = 0xffffffffu;
        if (e > s) {
            const uint32_t sw = s >> 5;
            const uint32_t w = sw + ((lane - sw) & 31u);                        /* this lane's word at or after s */
            if (w - ring_word < 32u && (w << 5) < e) {
                uint32_t bitsw = ring;
                if (w == sw) bitsw &= 0xffffffffu << (s & 31u);
                if (((w + 1u) << 5) > e) bitsw &= (e & 31u) ? ((1u << (e & 31u)) - 1u) : 0xffffffffu;
                if (bitsw) best = (w << 5) + (uint32_t)__ffs(bitsw) - 1u;
            }
        }
        best = warp_min(best);
        return best == 0xffffffffu ? none : best - s;
    }

    /* ============================================================ symbol dispatch */
    __device__ __forceinline__ void list_put(uint32_t stream, uint32_t ctx, uint32_t x) {
        if (list_n < list_cap) { if (lane == 0) { list[list_n].key = CBCG_SYM_KEY(stream, ctx); list[list_n].value = x; } }
        else err = CBCG_ERR_CAPACITY;
        list_n++;
        n_symbols++;
    }
    /* ============================================================ model initial states */
    __device__ __forceinline__ void init_L_models() {          /* the models whose alphabet is the header read length */
        dense_init_ones(M->snps, L);
        dense_init_ones(M->indels, L);
        SYNCW();
    }
    __device__ __forceinline__ void init_from_snapshot() {
        uint32_t *dst = reinterpret_cast<uint32_t *>(M);
        for (uint32_t i = lane; i < (uint32_t)(sizeof(WarpModels) / 4u); i += 32u) dst[i] = snap.small()[i];
        pos_card = snap.pos_hdr()[0]; pos_n = snap.pos_hdr()[1];
        pos_rv = (lane < pos_card) ? snap.pos_val()[lane] : 0u;
        pos_rc = (lane < pos_card) ? snap.pos_cnt()[lane] : 0u;
        for (uint32_t i = 32u + lane; i < pos_card; i += 32u) { pos_gval()[i] = snap.pos_val()[i]; pos_gcnt()[i] = snap.pos_cnt()[i]; }
        pa_init = false;
        n_rows = 0;
        for (uint32_t i = lane; i <= hash_mask; i += 32u) var_hash[i] = 0ull;
        SYNCW();
    }
    __device__ __forceinline__ void init_models(bool legacy) {
        if (MODE == MODE_LIST) return;
        dense_init_ones(M->rlen0, 255u);
        if (lane < 6u) {                                        /* initialize_stream_model_chars :350-411 */
            uint32_t n = 0;
            for (uint32_t i = 0; i < 4u; i++) { uint32_t c = (i == lane) ? 0u : 8u; M->chars[lane][i] = c; n += c; }
            M->chars[lane][4] = 1u; n += 1u;
            if (lane < 4u) {
                const uint32_t f0 = (lane == 0u || lane == 3u) ? 1u : 0u, f1 = (lane == 0u || lane == 3u) ? 2u : 3u;
                M->chars[lane][f0] += 8u; M->chars[lane][f1] += 8u; n += 16u;
            }
            M->chars[lane][5] = n;
        }
        if (lane < 4u) { M->match[lane][0] = 1u; M->match[lane][1] = 1u; M->match[lane][2] = 2u; }
        if (lane == 0) {
            M->same_ref[0] = 1u; M->same_ref[1] = 1u; M->same_ref[2] = 2u;
            for (uint32_t k = 0; k < 3u; k++) { M->rlenk[k][0] = 1u; M->rlenk[k][1] = 255u; }
            M->flag_used = 0u; M->flag_n = 65536u;
        }
        pos_rv = 0u; pos_rc = (lane == 0u) ? 1u : 0u; pos_card = 1u; pos_n = 1u;   /* escape only (:132-162) */
        pa_init = false;
        n_rows = 0;
        if (var_direct) { for (uint32_t i = lane; i < 2048u; i += 32u) var_bitmap()[i] = 0u; }
        else { for (uint32_t i = lane; i <= hash_mask; i += 32u) var_hash[i] = 0ull; }
        if (legacy) {
            for (uint32_t k = 0; k < 4u; k++) dense_init_ones(codebook + k * PA_STRIDE, 256u);
            for (uint32_t k = 0; k < 256u; k++) dense_init_ones(rname + k * PA_STRIDE, 256u);
        }
        SYNCW();
    }
};

/* ------------------------------------------------------------------------------------------------
 * The block coder proper: ONE loop that walks the reference's symbol order as a state machine, so that every
 * model kind (dense, FLAG, POS) has a single call site in the generated code. (Inlining the coder at each
 * of the reference's ~30 emission sites made a 28 000-instruction kernel that spent a third of its time
 * waiting for instruction fetch.) States follow compress_read / decompress_read (src/read_compression.c:15-44,
 * src/read_decompression.c:59-86), the emission / decoding half of compress_edits / reconstruct_read
 * (:557-600 / :339-458), compress_rname / decompress_rname (src/id_compression.c:39-94) and the stream
 * header (src/sam_file_allocation.c:363-404, src/compression.c:139,152). State the reference keeps in statics
 * is explicit: prev_pos (src/read_compression.c:115), prev_m (:167), prev_char (src/id_compression.c:42). */
enum : uint32_t { ST_HDR, ST_READ, ST_SAMEREF, ST_RNAME, ST_RLEN0, ST_RLENK, ST_POS, ST_POSESC, ST_FLAG, ST_MATCH, ST_SNPS,
                  ST_INDELS, ST_DEL, ST_SNPVAR, ST_SNPCHAR, ST_INSVAR, ST_INSCHAR, ST_READ_END, ST_ENDMARK, ST_DONE };
enum : uint32_t { K_NONE, K_DENSE, K_RLENK, K_FLAG, K_POS };

template <int MODE, bool LEGACY>
__global__ void __launch_bounds__(K2_THREADS, K2_MIN_CTAS)
k2_coder_kernel(CoderParams P) {
    __shared__ __align__(16) WarpShared sshared[K2_WARPS];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t bl = blockIdx.x * K2_WARPS + warp;
    if (bl >= P.n_blocks) return;
    if (*reinterpret_cast<volatile unsigned long long *>(P.err)) return;   /* an earlier stage failed (e.g. the plan ran out of workspace): offsets may be out of range */
    const uint32_t b = P.block_begin + bl;
    BlockDesc &B = P.blocks[b];
    constexpr bool legacy = LEGACY;                     /* single-block mode is its own instantiation: its header, RNAME and
                                                           end-marker states stay out of the blocked kernels' instruction stream */
    const bool primed = !LEGACY && P.primed != 0 && MODE != MODE_LIST;
    constexpr bool lean = !LEGACY && MODE != MODE_LIST;  /* blocked containers never code same_ref / length bytes 1..3 */
    const bool fixed = lean && P.fixed_len != 0;         /* ... nor length byte 0 when every read is L bases long */

    Coder<MODE> C;
    C.lane = lane; C.err = 0; C.n_symbols = 0; C.M = &sshared[warp].m; C.coldp = &sshared[warp].c;
    C.primed = primed; C.lean = lean;
    C.var_defer = primed; C.var_ro = false; C.defer_idx = 0; C.defer_key = 0;   /* merge_add adds a deferred slot's one update */
    if (primed) C.snap = SnapView(P.snap, P.L);
    C.L = P.L; C.Lp = (P.L + 1u + 31u) & ~31u;
    /* workspace */
    const uint64_t ws_edits = (MODE == MODE_DEC && legacy) ? 0xffffffffull : B.n_edits;
    uint32_t decode_L = P.L;
    {
        const WsLayout w = ws_layout(P.L ? P.L : 252u, B.n_reads, ws_edits, legacy, primed);
        uint8_t *base = P.ws + B.ws_off;
        C.var_hash = reinterpret_cast<uint64_t *>(base + w.var_hash);
        C.codebook = reinterpret_cast<uint32_t *>(base + w.codebook);
        C.rname = reinterpret_cast<uint32_t *>(base + w.rname);
        C.hash_mask = w.hash_cap - 1u; C.var_direct = w.direct != 0u;
        C.Lp = w.Lp;
        if (lane == 0) {
            WarpCold &W = C.cold();
            W.pos_cap = w.pos_cap; W.rows_cap = w.rows_cap;
            W.io = P.payload + B.payload_off;
            W.io_cap = (MODE == MODE_DEC) ? B.payload_bytes : (uint32_t)payload_cap_bytes(B.n_reads, B.n_edits, legacy ? 2 : 1);
            W.ref = nullptr; W.ref_len = 0;
            if (!legacy && B.chr < P.genome.n_chr) { W.ref = P.genome.bases + P.genome.chr_off[B.chr]; W.ref_len = P.genome.chr_len[B.chr]; }
            W.edits_cap_abs = B.edit_base + B.n_edits;
        }
        SYNCW();
    }
    C.list = P.symbols + B.sym_off; C.list_n = 0; C.list_cap = (uint32_t)symlist_cap(B.n_reads, B.n_edits, legacy);
    if (primed) C.init_from_snapshot(); else C.init_models(legacy);
    C.ring_reset();
    if (MODE != MODE_LIST) C.ac_init();
    if (!legacy && MODE != MODE_LIST && !primed) C.init_L_models();
    if (!legacy && MODE == MODE_DEC && B.chr >= P.genome.n_chr) C.err = CBCG_ERR_NO_REFERENCE;

    /* ---- machine state */
    uint32_t state = legacy ? ST_HDR : ST_READ;
    uint32_t k = 0;                                      /* sub-index inside a state (header byte, edit ordinal ...) */
    uint32_t prev_pos = B.base_pos, prev_m = 0u, prev_char = 0u;
    uint32_t cur_chr = legacy ? 0xffffffffu : B.chr, chr = cur_chr;
    const uint64_t r0 = B.first_read;
    const uint32_t n_reads = B.n_reads;                 /* legacy decode: capacity, the end marker stops the loop */
    uint64_t e_cursor = B.edit_base;
    uint32_t i = 0, n_done = 0;
    /* the read in flight */
    uint32_t pos = 0, len = 0, flag = 0, match = 0, ns = 0, nd = 0, ni = 0, strand = 0, samepos = 0, posx = 0, acc = 0;
    uint32_t prev = 0, ne = 0, ed = 0, edp = 0, refb = 0, change = 0, hdr_L = 0;
    uint32_t rl_x = 0xffffffffu, rl_lo = 0;             /* remembered length symbol and its cumulative count */
    const uint16_t *e_in = P.edits;
    const uint8_t *name = P.chr_names;

    /* The machine is threaded with gotos: every state has a set-up block S_x (describe its symbol, then CODE) and a
       post block P_x (consume the value, jump straight to the next state's set-up). One dispatch per symbol --
       CODE's switch on `state` -- instead of a loop with a set-up switch and a post switch. */
    uint32_t card, step, x, key, ctx, pre_lo, y, slot;
    uint32_t *m;
    bool is_var, pre;
#define SYMBOL(KIND, M, CARD, STEP, X, KEY) do { m = (M); card = (CARD); step = (STEP); x = (X); key = (KEY); is_var = false; pre = false; pre_lo = 0; } while (0)
#define VAR_SYMBOL(CTX, X) do { m = nullptr; ctx = (CTX); card = C.L; step = 10u; x = (X); key = CBCG_SYM_KEY(CBCG_S_VAR, ctx); is_var = true; pre = false; pre_lo = 0; } while (0)
    card = step = x = key = ctx = pre_lo = y = 0; slot = 1u; m = nullptr; is_var = pre = false;
    if (C.err) goto M_DONE;
    if (legacy) goto S_HDR;
    goto S_READ;

    /* ================================================ code the described symbol: one call site per model kind */
    /* POS, FLAG and the constant length bytes have one state each: their coder call sits in that state and continues
       straight to its post block (CODE_DIRECT), no dispatch at all. Every other symbol is a dense model and comes here. */
#define CODE_DIRECT(CALL, STREAM, CTXV, XV, NEXT) do { \
        y = (XV); slot = 1u; \
        if (MODE == MODE_LIST) C.list_put((STREAM), (CTXV), (XV)); else y = (CALL); \
        if (UNLIKELY(C.err)) goto M_DONE; \
        goto NEXT; } while (0)
    /* The four dense symbols of nearly every read (match bit, SNP count, SNP position, SNP base) get their own coder
       call too; the rare states share the CODE site below and its dispatch. */
#define DENSE_DIRECT(SMALL, IS_VAR, M, CARD, STEP, STREAM, CTXV, XV, NEXT) do { \
        y = (XV); \
        if (MODE == MODE_LIST) C.list_put((STREAM), (CTXV), (XV)); else y = C.template sym_dense<SMALL, IS_VAR>((M), (CARD), (STEP), (XV), false, 0u); \
        if (UNLIKELY(C.err)) goto M_DONE; \
        goto NEXT; } while (0)
CODE:
    if (is_var && MODE != MODE_LIST) { m = C.var_row(ctx); if (!m) goto M_DONE; }
    y = x;
    if (MODE == MODE_LIST) C.list_put(key >> 24, key & 0xffffffu, x);
    else y = C.template sym_dense<0, true>(m, card, step, x, pre, pre_lo);
    if (C.err) goto M_DONE;
    switch (state) {
        case ST_HDR: goto P_HDR;       case ST_SAMEREF: goto P_SAMEREF; case ST_RNAME: goto P_RNAME;   case ST_RLEN0: goto P_RLEN0;
        case ST_POSESC: goto P_POSESC;
        case ST_INDELS: goto P_INDELS; case ST_DEL: goto P_DEL;
        case ST_INSVAR: goto P_INSVAR; case ST_INSCHAR: goto P_INSCHAR;
        case ST_ENDMARK: goto P_ENDMARK;
        default: C.err = CBCG_ERR_INTERNAL; goto M_DONE;
    }

    /* ---- stream header: 34 ints x 4 bytes, MSB first, through codebook[0..3] (compress_int) */
S_HDR: {
        const uint32_t word = k >> 2, byte = k & 3u;
        const uint32_t v = word == 0u ? P.L : (word == 33u ? CBCG_LOSSLESS : CBCG_WELL_DEBUG);
        state = ST_HDR;
        SYMBOL(K_DENSE, C.codebook + byte * PA_STRIDE, 256u, 1u, (v >> (24u - 8u * byte)) & 0xffu, CBCG_SYM_KEY(CBCG_S_CODEBOOK, byte));
        goto CODE;
    }
P_HDR:
    if (MODE == MODE_DEC) {
        const uint32_t word = k >> 2, byte = k & 3u;
        if (word == 0u) hdr_L |= y << (24u - 8u * byte);
        else if (word == 33u && y != ((CBCG_LOSSLESS >> (24u - 8u * byte)) & 0xffu)) { C.err = CBCG_ERR_FORMAT; goto M_DONE; }
    }
    if (++k < 136u) goto S_HDR;
    if (MODE == MODE_DEC) {
        if (hdr_L == 0u || hdr_L > CBCG_MAX_READ_LEN) { C.err = CBCG_ERR_FORMAT; goto M_DONE; }
        C.L = hdr_L; decode_L = hdr_L;
    }
    if (MODE != MODE_LIST) C.init_L_models();                 /* alloc_read_models_t runs after the header int (:371-375) */
    goto S_READ;

    /* ---- next read (not a symbol) */
S_READ:
    if (!(legacy && MODE == MODE_DEC) && i >= n_reads) {
        if (legacy && MODE != MODE_DEC) { k = 0; goto S_ENDMARK; }
        goto M_DONE;
    }
    if (MODE != MODE_DEC) {
        const uint4 v = reinterpret_cast<const uint4 *>(P.recs)[r0 + i];
        if (i + 1u < n_reads) {                                            /* next read's record: hide its latency */
            asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const uint4 *>(P.recs) + r0 + i + 1u));
        }
        pos = v.x; flag = v.y & 0xffffu; len = v.y >> 16; match = v.w & 0xffu;
        ns = (v.w >> 8) & 0xffu; nd = (v.w >> 16) & 0xffu; ni = v.w >> 24;
        e_in = P.edits + v.z;
        if (!match) asm volatile("prefetch.global.L1 [%0];" ::"l"(e_in));
        if (legacy) {
            chr = P.chr[r0 + i];
            if (chr >= P.genome.n_chr) { C.err = CBCG_ERR_NO_REFERENCE; goto M_DONE; }
            change = chr != cur_chr;
            goto S_SAMEREF;
        }
        if (cur_chr >= P.genome.n_chr) { C.err = CBCG_ERR_NO_REFERENCE; goto M_DONE; }   /* blocks never span chromosomes: the host cut them */
        change = 0;
        if (lean) {
            if (!fixed) goto S_RLEN0;
            if (len != P.L) { C.err = CBCG_ERR_INPUT; goto M_DONE; }        /* the host checked the batch */
            goto S_POS;
        }
        goto S_SAMEREF;
    }
    change = 0;
    if (legacy || !lean) goto S_SAMEREF;
    if (fixed) { len = P.L; goto S_POS; }                                      /* CBCG_MODE_FIXED_LEN: no length symbol */
    goto S_RLEN0;

    /* ---- compress_rname / decompress_rname (src/id_compression.c:39-94) */
S_SAMEREF:
    state = ST_SAMEREF;
    SYMBOL(K_DENSE, C.M->same_ref, 2u, 10u, change, CBCG_SYM_KEY(CBCG_S_SAME_REF, 0u));
    goto CODE;
P_SAMEREF:
    if (MODE == MODE_DEC) {
        if (!legacy) { if (y != 0u) { C.err = CBCG_ERR_CORRUPT; goto M_DONE; } }
        else change = y;
    }
    if (change) { k = 0; if (MODE != MODE_DEC) name = P.chr_names + (uint64_t)chr * MAX_NAME; goto S_RNAME; }
    if (legacy && MODE == MODE_DEC) {
        if (cur_chr == 0xffffffffu) { C.err = CBCG_ERR_CORRUPT; goto M_DONE; }
        if (i >= n_reads) { C.err = CBCG_ERR_CAPACITY; goto M_DONE; }
    }
    goto S_RLEN0;
S_RNAME:                                                      /* name bytes then 0, context = previous byte (never reset) */
    state = ST_RNAME;
    SYMBOL(K_DENSE, C.rname + prev_char * PA_STRIDE, 256u, 10u, (MODE != MODE_DEC && k < MAX_NAME) ? (uint32_t)name[k] : 0u,
           CBCG_SYM_KEY(CBCG_S_RNAME, prev_char));
    goto CODE;
P_RNAME: {
        bool name_done = false;
        if (MODE == MODE_DEC) {
            if (y == (uint32_t)'\n') goto M_DONE;                           /* end marker (decompress_rname :82-84) */
            if (y == 0u) { name_done = true; chr = cur_chr + 1u; }           /* records are taken in FASTA order */
            else prev_char = y;
        } else { if (x == 0u) name_done = true; else { prev_char = x; k++; } }
        if (!name_done) goto S_RNAME;
        if (chr >= P.genome.n_chr) { C.err = CBCG_ERR_NO_REFERENCE; goto M_DONE; }
        if (MODE == MODE_DEC && i >= n_reads) { C.err = CBCG_ERR_CAPACITY; goto M_DONE; }
        cur_chr = chr; prev_pos = 0u; C.ring_reset();                       /* src/compression.c:58-64 */
        SYNCW();
        if (lane == 0) { C.cold().ref = P.genome.bases + P.genome.chr_off[chr]; C.cold().ref_len = P.genome.chr_len[chr]; }
        SYNCW();
        goto S_RLEN0;
    }

    /* ---- length: byte 0 carries it, bytes 1..3 are always 0 (src/read_compression.c:29-33) */
S_RLEN0:
    state = ST_RLEN0;
    SYMBOL(K_DENSE, C.M->rlen0, 255u, 10u, len & 0xffu, CBCG_SYM_KEY(CBCG_S_RLENGTH, 0u));
    /* fixed-length input codes the same symbol every read; its cumulative count only moves when a smaller symbol is
       coded or the model rescales, so it is remembered instead of re-summed */
    if (MODE != MODE_LIST && rl_x < 255u) {
        if (MODE == MODE_ENC) pre = (x == rl_x);
        else {
            const uint64_t A = C.dec_A(m[255]); const uint32_t range = C.dec_range();
            pre = DEC_LE(rl_lo) && !DEC_LE(rl_lo + m[rl_x]);
            if (pre) x = rl_x;
        }
        pre_lo = rl_lo;
    }
    goto CODE;
P_RLEN0:
    if (MODE == MODE_DEC) len = y;
    if (MODE != MODE_LIST) { rl_x = (C.last_n + 10u >= CBCG_RESCALE) ? 0xffffffffu : y; rl_lo = C.last_lo; }
    if (lean) goto S_POS;
    k = 1;
S_RLENK:
    state = ST_RLENK;
    CODE_DIRECT(C.sym_rlenk(k - 1u, 0u), CBCG_S_RLENGTH, k, 0u, P_RLENK);
P_RLENK:
    if (MODE == MODE_DEC) len |= y << (8u * k);
    if (++k < 4u) goto S_RLENK;

    /* ---- position (src/read_compression.c:113-159): x = pos - prevPos + 1 through the growing alphabet */
S_POS:
    state = ST_POS;
    x = 0u;
    if (MODE != MODE_DEC) {
        if (pos == 0u || len == 0u || len > CBCG_MAX_READ_LEN) { C.err = CBCG_ERR_INPUT; goto M_DONE; }
        /* the reference's POS alphabet bounds the step of its own stream only; a blocked container codes any 32-bit step */
        if (pos < prev_pos || (LEGACY && pos - prev_pos + 1u > CBCG_MAX_POS_X)) { C.err = CBCG_ERR_INPUT; goto M_DONE; }
        x = pos - prev_pos + 1u;
    }
    CODE_DIRECT(C.sym_pos_main(x, slot), CBCG_S_POS_X, 0u, x, P_POS);
P_POS:
    posx = (MODE == MODE_DEC) ? y : x;
    if (MODE == MODE_LIST || slot != 0u) goto M_POS_DONE;
    acc = 0; k = 0;
S_POSESC:                                                     /* the escaped value, 4 bytes MSB first (compress_pos_alpha :75-108) */
    state = ST_POSESC;
    if (k == 0u) C.pa_ensure();
    SYMBOL(K_DENSE, C.pos_alpha() + k * PA_STRIDE, 256u, 10u, (posx >> (24u - 8u * k)) & 0xffu, CBCG_SYM_KEY(CBCG_S_POS_ALPHA, k));
    goto CODE;
P_POSESC:
    acc |= y << (24u - 8u * k);
    if (++k < 4u) goto S_POSESC;
    if (MODE == MODE_DEC) posx = acc;
    C.pos_append(posx);
    if (C.err) goto M_DONE;
M_POS_DONE:
    if (MODE == MODE_DEC) {
        if (posx == 0u) { C.err = CBCG_ERR_CORRUPT; goto M_DONE; }
        pos = prev_pos + posx - 1u;
        if (pos == 0u || len == 0u || len > CBCG_MAX_READ_LEN) { C.err = CBCG_ERR_CORRUPT; goto M_DONE; }
    }
    samepos = posx == 1u;
    prev_pos = pos;
    C.ring_advance(pos);

    /* ---- flag, match */
    state = ST_FLAG;
    x = flag;
    CODE_DIRECT(C.sym_flag(x), CBCG_S_FLAG, 0u, x, P_FLAG);
P_FLAG:
    flag = y; strand = (flag >> 4) & 1u;                                   /* :57-60 */
    state = ST_MATCH;
    ctx = (samepos << 1) | prev_m;
    x = match;
    DENSE_DIRECT(2, false, C.M->match[ctx], 2u, 1u, CBCG_S_MATCH, ctx, x, P_MATCH);
P_MATCH:
    match = y; prev_m = y; ne = 0;
    if (MODE == MODE_DEC) { ns = nd = ni = 0; }
    if (match) goto M_READ_END;
    if (MODE == MODE_DEC) {
        /* the decoder needs the reference base under every SNP it decodes (the context of the base symbol): a
           dependent byte load from HBM per SNP unless the read's stretch of the reference is already on its way */
        const uint8_t *rp = C.cold().ref + (pos - 1u);
        asm volatile("prefetch.global.L1 [%0];" ::"l"(rp));
        asm volatile("prefetch.global.L1 [%0];" ::"l"(rp + 128));
        if (len > 128u) asm volatile("prefetch.global.L1 [%0];" ::"l"(rp + 256));
    }

    /* ---- counts (:557-565) */
    state = ST_SNPS;
    x = ((nd | ni) == 0u) ? ns : 0u;
    DENSE_DIRECT(0, false, C.M->snps, C.L, 10u, CBCG_S_SNPS, 0u, x, P_SNPS);
P_SNPS:
    if (MODE == MODE_DEC) { ns = y; nd = ni = 0; if (y != 0u) goto M_COUNTS_DONE; }
    else if ((nd | ni) == 0u) goto M_COUNTS_DONE;
    k = 0;
S_INDELS:
    state = ST_INDELS;
    SYMBOL(K_DENSE, C.M->indels, C.L, 16u, k == 0u ? ns : (k == 1u ? nd : ni), CBCG_SYM_KEY(CBCG_S_INDELS, 0u));
    goto CODE;
P_INDELS:
    if (MODE == MODE_DEC) { if (k == 0u) ns = y; else if (k == 1u) nd = y; else ni = y; }
    if (++k < 3u) goto S_INDELS;
M_COUNTS_DONE:
    if (MODE == MODE_DEC) {
        if (ni > len || ns > 255u || nd > 255u || ni > 255u) { C.err = CBCG_ERR_CORRUPT; goto M_DONE; }
        if ((uint64_t)(ns + nd + ni) > C.cold().edits_cap_abs - e_cursor) { C.err = CBCG_ERR_CAPACITY; goto M_DONE; }
    }
    prev = 0; k = 0; ne = 0;
    if (nd) goto S_DEL;
    if (ns) goto S_SNPVAR;
    if (ni) goto S_INSVAR;
    goto M_READ_END;

    /* ---- deletions (:568-572) */
S_DEL:
    state = ST_DEL;
    if (MODE != MODE_DEC) ed = e_in[k];
    VAR_SYMBOL((prev << 1) | strand, CBCG_EDIT_DELTA(ed));
    goto CODE;
P_DEL:
    prev += y;
    if (MODE == MODE_DEC && lane == 0) { P.edits[e_cursor + ne] = CBCG_EDIT(y, 0, 0); C.M->cumdel[k] = (uint16_t)min(prev, 0xffffu); }
    ne++;
    if (++k < nd) goto S_DEL;
    if (MODE == MODE_DEC) SYNCW();
    prev = 0; k = 0;
    if (ns) goto S_SNPVAR;
    if (ni) goto S_INSVAR;
    goto M_READ_END;

    /* ---- SNPs (:573-593) */
S_SNPVAR: {
        state = ST_SNPVAR;
        if (MODE != MODE_DEC) ed = e_in[nd + k];
        const uint32_t delta = C.ring_first(pos - 1u + prev, (prev < len) ? pos - 1u + len : pos - 1u + prev, len + 2u);
        ctx = (((delta << CBCG_BITS_DELTA) + prev) << 1) | strand;
        x = CBCG_EDIT_DELTA(ed);
        m = nullptr;
        if (MODE != MODE_LIST) { m = C.var_row(ctx); if (!m) goto M_DONE; }
        DENSE_DIRECT(0, true, m, C.L, 10u, CBCG_S_VAR, ctx, x, P_SNPVAR);
    }
P_SNPVAR: {
        edp = y;
        const uint32_t idx = prev + y;                                         /* index in the insertion-free read */
        prev += y + 1u;
        C.ring_set(pos + prev - 2u);                                           /* :589 */
        if (MODE == MODE_DEC) {
            uint32_t skipped = 0;                                              /* deletions at or before idx (:426-437) */
            if (nd) {
                for (uint32_t q = lane; q < nd; q += 32u) skipped += (C.M->cumdel[q] <= idx);
                skipped = warp_sum(skipped);
            }
            const uint64_t ri = (uint64_t)pos - 1u + idx + skipped;
            refb = base_code(ri < C.cold().ref_len ? (uint32_t)C.cold().ref[ri] : 0u);
        } else refb = CBCG_EDIT_REFB(ed);
        state = ST_SNPCHAR;
        x = CBCG_EDIT_TARGET(ed);
        DENSE_DIRECT(5, false, C.M->chars[refb], 5u, 8u, CBCG_S_CHARS, refb, x, P_SNPCHAR);
    }
P_SNPCHAR:
    if (MODE == MODE_DEC && lane == 0) P.edits[e_cursor + ne] = CBCG_EDIT(edp, y, refb);
    ne++;
    if (++k < ns) goto S_SNPVAR;
    prev = 0; k = 0;
    if (ni) goto S_INSVAR;
    goto M_READ_END;

    /* ---- insertions (:594-600) */
S_INSVAR:
    state = ST_INSVAR;
    if (MODE != MODE_DEC) ed = e_in[nd + ns + k];
    VAR_SYMBOL((prev << 1) | strand, CBCG_EDIT_DELTA(ed));
    goto CODE;
P_INSVAR:
    edp = y; prev += y;
    state = ST_INSCHAR;
    SYMBOL(K_DENSE, C.M->chars[CBCG_BP_O], 5u, 8u, CBCG_EDIT_TARGET(ed), CBCG_SYM_KEY(CBCG_S_CHARS, CBCG_BP_O));
    goto CODE;
P_INSCHAR:
    if (MODE == MODE_DEC && lane == 0) P.edits[e_cursor + ne] = CBCG_EDIT(edp, y, CBCG_BP_O);
    ne++;
    if (++k < ni) goto S_INSVAR;

M_READ_END:
    if (MODE == MODE_DEC) {
        if (lane == 0) {
            uint4 v;
            v.x = pos; v.y = flag | (len << 16); v.z = (uint32_t)e_cursor;
            v.w = match | (match ? 0u : ((ns << 8) | (nd << 16) | (ni << 24)));
            reinterpret_cast<uint4 *>(P.recs)[r0 + i] = v;
            P.chr[r0 + i] = cur_chr;
        }
        e_cursor += ne;
    }
    n_done++; i++;
    goto S_READ;

    /* ---- end of stream: name "\n" (src/compression.c:152) */
S_ENDMARK:
    state = ST_ENDMARK;
    if (k == 0u) SYMBOL(K_DENSE, C.M->same_ref, 2u, 10u, 1u, CBCG_SYM_KEY(CBCG_S_SAME_REF, 0u));
    else SYMBOL(K_DENSE, C.rname + prev_char * PA_STRIDE, 256u, 10u, k == 1u ? (uint32_t)'\n' : 0u, CBCG_SYM_KEY(CBCG_S_RNAME, prev_char));
    goto CODE;
P_ENDMARK:
    if (k == 1u) prev_char = '\n';
    if (++k < 3u) goto S_ENDMARK;

M_DONE:
#undef SYMBOL
#undef VAR_SYMBOL
#undef CODE_DIRECT
#undef DENSE_DIRECT

    if (MODE == MODE_ENC && !C.err) { if (P.short_flush && !legacy) C.ac_flush_short(); else C.ac_flush(); }
    if (C.err) dev_set_error(P.err, C.err, ((uint64_t)b << 20) | (n_done & 0xfffffu));
    if (primed && P.fin && !C.err) {                     /* final state for the generation merge */
        SYNCW();
        uint32_t *dst = reinterpret_cast<uint32_t *>(P.fin + (uint64_t)b * fin_stride_dev());
        const uint32_t *src = reinterpret_cast<const uint32_t *>(C.M);
        for (uint32_t q = lane; q < (uint32_t)(sizeof(WarpModels) / 4u); q += 32u) dst[q] = src[q];
        if (lane < C.pos_card) { C.pos_gval()[lane] = C.pos_rv; C.pos_gcnt()[lane] = C.pos_rc; }
        if (lane == 0) { B.pos_card = C.pos_card; B.n_rows = C.n_rows; B.pa_touched = C.pa_init ? 1u : 0u; }
    }
    if (lane == 0) {
        B.n_symbols = (MODE == MODE_LIST) ? C.list_n : C.n_symbols;
        if (MODE == MODE_ENC) { B.payload_bytes = C.out_pos; B.sub_bytes[0] = C.out_pos; }
        if (MODE == MODE_DEC) { B.n_reads = n_done; B.n_edits = (uint32_t)(e_cursor - B.edit_base); B.pad = decode_L; }
    }
}


/* ================================================================================================
 * Blocked containers (format v4): ONE CTA PER BLOCK, ONE WARP PER SUBSTREAM.
 *
 * The four substreams of a block (cbcg_format.h: POS | length + FLAG | match + counts | var + bases) are independent
 * arithmetic-coded streams over disjoint groups of models, so the block is four short chains instead of one long
 * one, and each warp runs a small loop over ONE kind of symbol -- no state machine, no dispatch, an instruction
 * footprint of a few hundred instructions per role (round 1's single chain through every model was 5 900
 * instructions walked by 20 warps per SM, a third of its stall samples waiting for instruction fetch).
 * Encode: the four warps never talk. Decode: the match context needs samePos, the edit loops need the counts and the
 * strand, so the roles run as a software pipeline through a ring in shared memory: POS and FLAG run ahead, the counts
 * follow one read behind them, the edits one read behind the counts; a block takes the time of its longest substream
 * instead of their sum. Lanes cooperate inside a symbol exactly as in round 1 (Coder<>: strided cumulative counts,
 * 32-wide hash probe, POS slots in registers). The block's small models live once in shared memory, each field
 * owned by one role. The scalar twin of these loops (k2_roles.cuh) is what the CPU harness checks against the oracle. */
#define K2B_WARPS 4u
#define K2B_MIN_CTAS 5
#define K2B_RING 256u
struct K2BEntry { uint32_t pos, flaglen, counts; };
struct K2BShared {
    WarpModels m;
    WarpCold c[K2B_WARPS];
    K2BEntry ring[K2B_RING];                   /* decode: what the roles hand each other, by read ordinal mod K2B_RING */
    volatile uint32_t progress[K2B_WARPS];      /* decode: reads finished by each role */
    volatile int failed;
    unsigned long long err_seen;
};
/* wait until role `r` has finished read i (returns false when the block has failed) */
__device__ __forceinline__ bool k2b_wait(K2BShared &S, uint32_t r, uint32_t i, uint32_t &seen) {
    if (i < seen) return true;
    for (;;) {
        const uint32_t v = S.progress[r];
        if (v > i) { seen = v; return true; }
        if (S.failed) return false;
        __nanosleep(40);
    }
}
/* a producer may run at most K2B_RING reads ahead of the edits role (the last consumer) */
__device__ __forceinline__ bool k2b_room(K2BShared &S, uint32_t i, uint32_t &seen_d) {
    if (i < seen_d + K2B_RING) return true;
    for (;;) {
        const uint32_t v = S.progress[CBCG_SUB_EDITS];
        if (i < v + K2B_RING) { seen_d = v; return true; }
        if (S.failed) return false;
        __nanosleep(100);
    }
}
__device__ __forceinline__ void k2b_publish(K2BShared &S, uint32_t r, uint32_t done, uint32_t lane) {
    __syncwarp();
    if (lane == 0) { __threadfence_block(); S.progress[r] = done; }
}
__device__ __forceinline__ void k2b_copy(uint32_t *dst, const uint32_t *src, uint32_t n, uint32_t lane) { for (uint32_t i = lane; i < n; i += 32u) dst[i] = src[i]; }

template <int MODE>
__global__ void __launch_bounds__(K2B_WARPS * 32u, K2B_MIN_CTAS)
k2_block_kernel(CoderParams P) {
    __shared__ __align__(16) K2BShared S;
    const uint32_t role = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    if (threadIdx.x == 0) { S.err_seen = *reinterpret_cast<volatile unsigned long long *>(P.err); S.failed = 0; }
    if (threadIdx.x < K2B_WARPS) S.progress[threadIdx.x] = 0u;
    __syncthreads();
    if (S.err_seen) return;                              /* an earlier stage failed: offsets may be out of range */
    const uint32_t b = P.block_begin + blockIdx.x;
    BlockDesc &B = P.blocks[b];
    const WsLayout w = ws_layout(P.L, B.n_reads, B.n_edits, 0, 1);
    uint8_t *wsb = P.ws + B.ws_off;
    const uint32_t L = P.L, n_reads = B.n_reads;
    const bool fixed = P.fixed_len != 0;
    const uint64_t r0 = B.first_read;

    Coder<MODE> C;
    C.lane = lane; C.err = 0; C.n_symbols = 0; C.M = &S.m; C.coldp = &S.c[role];
    C.primed = true; C.lean = true; C.var_defer = true; C.var_ro = false; C.defer_idx = 0; C.defer_key = 0;
    C.snap = SnapView(P.snap, L);
    C.L = L; C.Lp = w.Lp;
    C.var_hash = reinterpret_cast<uint64_t *>(wsb + w.var_hash); C.hash_mask = w.hash_cap - 1u; C.var_direct = false;
    C.codebook = nullptr; C.rname = nullptr; C.list = nullptr; C.list_n = 0; C.list_cap = 0;
    C.n_rows = 0; C.pa_init = false; C.pos_card = 1u; C.pos_n = 1u; C.pos_rv = 0u; C.pos_rc = 0u;
    C.last_lo = 0; C.last_n = 0;
    if (lane == 0) {
        WarpCold &W = S.c[role];
        W.pos_cap = w.pos_cap; W.rows_cap = w.rows_cap; W.pad = 0;
        if (MODE == MODE_ENC) {
            uint64_t o = B.payload_off;
            for (uint32_t q = 0; q < role; q++) o += k2_sub_cap(q, n_reads, B.n_edits);
            W.io = P.payload + o; W.io_cap = (uint32_t)k2_sub_cap(role, n_reads, B.n_edits);
        } else {
            uint64_t o = B.payload_off;
            for (uint32_t q = 0; q < role; q++) o += B.sub_bytes[q];
            W.io = P.payload + o; W.io_cap = B.sub_bytes[role];
        }
        W.ref = nullptr; W.ref_len = 0;
        if (B.chr < P.genome.n_chr) { W.ref = P.genome.bases + P.genome.chr_off[B.chr]; W.ref_len = P.genome.chr_len[B.chr]; }
        W.edits_cap_abs = B.edit_base + B.n_edits;
    }
    __syncwarp();
    const WarpModels *SM = reinterpret_cast<const WarpModels *>(C.snap.small());
    WarpModels *FM = reinterpret_cast<WarpModels *>(P.fin + (uint64_t)b * fin_stride_dev());
    C.ring_reset();
    uint32_t i = 0, seen_a = 0, seen_b = 0, seen_c = 0, seen_d = 0;
    bool bailed = false;                                 /* another role failed: leave without an error of our own */
#define K2B_FAIL(code) do { C.err = (code); goto role_done; } while (0)

    if (role == CBCG_SUB_POS) {
        /* ---- A: POS through the growing alphabet (compress_pos :113-159, compress_pos_alpha :75-108) */
        C.pos_card = C.snap.pos_hdr()[0]; C.pos_n = C.snap.pos_hdr()[1];
        if (C.pos_card > w.pos_cap) K2B_FAIL(CBCG_ERR_INTERNAL);
        C.pos_rv = (lane < C.pos_card) ? C.snap.pos_val()[lane] : 0u;
        C.pos_rc = (lane < C.pos_card) ? C.snap.pos_cnt()[lane] : 0u;
        for (uint32_t q = 32u + lane; q < C.pos_card; q += 32u) { C.pos_gval()[q] = C.snap.pos_val()[q]; C.pos_gcnt()[q] = C.snap.pos_cnt()[q]; }
        __syncwarp();
        C.ac_init();
        uint32_t prev_pos = B.base_pos;
        for (; i < n_reads; i++) {
            uint32_t x = 0, pos = 0, slot = 1u;
            if (MODE == MODE_ENC) {
                pos = P.recs[r0 + i].pos;
                if (pos == 0u || pos < prev_pos) K2B_FAIL(CBCG_ERR_INPUT);
                x = pos - prev_pos + 1u;
            } else if (!k2b_room(S, i, seen_d)) { bailed = true; break; }
            const uint32_t y = C.sym_pos_main(x, slot);
            if (C.err) break;
            if (MODE == MODE_DEC) x = y;
            if (slot == 0u) {                                /* escape: the value itself, 4 bytes MSB first, then a new slot */
                C.pa_ensure();
                uint32_t acc = 0;
                for (uint32_t k = 0; k < 4u; k++) {
                    const uint32_t yk = C.template sym_dense<0, false>(C.pos_alpha() + k * PA_STRIDE, 256u, 10u, (x >> (24u - 8u * k)) & 0xffu, false, 0u);
                    acc |= yk << (24u - 8u * k);
                }
                if (C.err) break;
                if (MODE == MODE_DEC) x = acc;
                C.pos_append(x);
                if (C.err) break;
            }
            if (MODE == MODE_DEC) {
                if (x == 0u) K2B_FAIL(CBCG_ERR_CORRUPT);
                pos = prev_pos + x - 1u;
                if (pos == 0u) K2B_FAIL(CBCG_ERR_CORRUPT);
                if (lane == 0) { P.recs[r0 + i].pos = pos; P.chr[r0 + i] = B.chr; S.ring[i & (K2B_RING - 1u)].pos = pos; }
                k2b_publish(S, role, i + 1u, lane);
            }
            prev_pos = pos;
        }
    } else if (role == CBCG_SUB_FLAG) {
        /* ---- B: length byte 0 (variable-length containers) and FLAG (compress_read :29-33, compress_flag :50-70) */
        k2b_copy(S.m.rlen0, SM->rlen0, 256u, lane);
        k2b_copy(S.m.same_ref, SM->same_ref, 4u + 6u, lane);             /* same_ref, rlenk: never coded here, the merge reads the image */
        { const uint32_t used = SM->flag_used; k2b_copy(S.m.flag_key, SM->flag_key, used, lane); k2b_copy(S.m.flag_cnt, SM->flag_cnt, used, lane);
          if (lane == 0) { S.m.flag_used = used; S.m.flag_n = SM->flag_n; } }
        __syncwarp();
        C.ac_init();
        for (; i < n_reads; i++) {
            uint32_t len = L, flag = 0;
            if (MODE == MODE_ENC) {
                const uint32_t v = reinterpret_cast<const uint32_t *>(P.recs + r0 + i)[1];
                flag = v & 0xffffu; len = v >> 16;
                if (len == 0u || len > CBCG_MAX_READ_LEN || (fixed && len != L)) K2B_FAIL(CBCG_ERR_INPUT);
            } else if (!k2b_room(S, i, seen_d)) { bailed = true; break; }
            if (!fixed) len = C.template sym_dense<0, false>(S.m.rlen0, 255u, 10u, len & 0xffu, false, 0u);
            flag = C.sym_flag(flag);
            if (C.err) break;
            if (MODE == MODE_DEC) {
                if (len == 0u || len > CBCG_MAX_READ_LEN) K2B_FAIL(CBCG_ERR_CORRUPT);
                const uint32_t v = flag | (len << 16);
                if (lane == 0) { reinterpret_cast<uint32_t *>(P.recs + r0 + i)[1] = v; S.ring[i & (K2B_RING - 1u)].flaglen = v; }
                k2b_publish(S, role, i + 1u, lane);
            }
        }
    } else if (role == CBCG_SUB_COUNTS) {
        /* ---- C: match bit, SNP count, indel counts (compress_match :164-188, compress_snps / compress_indels :193-228) */
        k2b_copy(S.m.snps, SM->snps, 512u, lane);                        /* snps, indels */
        k2b_copy(&S.m.match[0][0], &SM->match[0][0], 16u, lane);
        __syncwarp();
        C.ac_init();
        uint32_t prev_pos = B.base_pos, prev_m = 0u;
        uint64_t edits_left = B.n_edits;
        for (; i < n_reads; i++) {
            uint32_t pos, len = L, match = 0, ns = 0, nd = 0, ni = 0;
            if (MODE == MODE_ENC) {
                const uint4 v = reinterpret_cast<const uint4 *>(P.recs)[r0 + i];
                pos = v.x; len = v.y >> 16; match = v.w & 0xffu; ns = (v.w >> 8) & 0xffu; nd = (v.w >> 16) & 0xffu; ni = v.w >> 24;
            } else {
                if (!k2b_wait(S, CBCG_SUB_POS, i, seen_a) || !k2b_wait(S, CBCG_SUB_FLAG, i, seen_b) || !k2b_room(S, i, seen_d)) { bailed = true; break; }
                const volatile K2BEntry &e = S.ring[i & (K2B_RING - 1u)];
                pos = e.pos; len = e.flaglen >> 16;
            }
            const uint32_t samepos = pos == prev_pos ? 1u : 0u;          /* deltaP == 1 (:170) */
            prev_pos = pos;
            match = C.template sym_dense<2, false>(S.m.match[(samepos << 1) | prev_m], 2u, 1u, match, false, 0u);
            if (C.err) break;
            prev_m = match;
            if (!match) {
                uint32_t x = ((nd | ni) == 0u) ? ns : 0u;
                x = C.template sym_dense<0, false>(S.m.snps, L, 10u, x, false, 0u);
                if (MODE == MODE_DEC) { ns = x; nd = ni = 0; }
                if (!C.err && (MODE == MODE_DEC ? x == 0u : (nd | ni) != 0u)) {          /* :560-565 */
                    ns = C.template sym_dense<0, false>(S.m.indels, L, 16u, ns, false, 0u);
                    nd = C.template sym_dense<0, false>(S.m.indels, L, 16u, nd, false, 0u);
                    ni = C.template sym_dense<0, false>(S.m.indels, L, 16u, ni, false, 0u);
                }
                if (C.err) break;
                if (MODE == MODE_DEC) {
                    if (ni > len || ns > 255u || nd > 255u || ni > 255u) K2B_FAIL(CBCG_ERR_CORRUPT);
                    if ((uint64_t)(ns + nd + ni) > edits_left) K2B_FAIL(CBCG_ERR_CAPACITY);
                    edits_left -= ns + nd + ni;
                }
            } else if (MODE == MODE_DEC) { ns = nd = ni = 0; }
            if (MODE == MODE_DEC) {
                const uint32_t v = match | (ns << 8) | (nd << 16) | (ni << 24);
                if (lane == 0) { reinterpret_cast<uint32_t *>(P.recs + r0 + i)[3] = v; S.ring[i & (K2B_RING - 1u)].counts = v; }
                k2b_publish(S, role, i + 1u, lane);
            }
        }
    } else {
        /* ---- D: edit positions through the var rows, bases through chars (:568-600; compute_delta_to_first_snp :703-718) */
        k2b_copy(&S.m.chars[0][0], &SM->chars[0][0], 48u, lane);
        for (uint32_t q = lane; q <= C.hash_mask; q += 32u) C.var_hash[q] = 0ull;
        __syncwarp();
        C.ac_init();
        if (MODE == MODE_DEC && B.chr >= P.genome.n_chr) K2B_FAIL(CBCG_ERR_NO_REFERENCE);
        uint64_t e_cursor = B.edit_base;
        for (; i < n_reads; i++) {
            uint32_t pos, len, flag, match, ns, nd, ni;
            const uint16_t *e_in = P.edits;
            if (MODE == MODE_ENC) {
                const uint4 v = reinterpret_cast<const uint4 *>(P.recs)[r0 + i];
                pos = v.x; flag = v.y & 0xffffu; len = v.y >> 16; match = v.w & 0xffu; ns = (v.w >> 8) & 0xffu; nd = (v.w >> 16) & 0xffu; ni = v.w >> 24;
                e_in = P.edits + v.z;
                if (!match) asm volatile("prefetch.global.L1 [%0];" ::"l"(e_in));
            } else {
                if (!k2b_wait(S, CBCG_SUB_COUNTS, i, seen_c)) { bailed = true; break; }
                const volatile K2BEntry &e = S.ring[i & (K2B_RING - 1u)];
                pos = e.pos; flag = e.flaglen & 0xffffu; len = e.flaglen >> 16;
                const uint32_t cw = e.counts;
                match = cw & 0xffu; ns = (cw >> 8) & 0xffu; nd = (cw >> 16) & 0xffu; ni = cw >> 24;
                if (lane == 0) reinterpret_cast<uint32_t *>(P.recs + r0 + i)[2] = (uint32_t)e_cursor;
            }
            const uint32_t strand = (flag >> 4) & 1u;                    /* :57-60 */
            C.ring_advance(pos);
            if (!match) {
                if (MODE == MODE_DEC) {                                  /* the reference bases under this read: the context of every decoded base */
                    const uint8_t *rp = C.cold().ref + (pos - 1u);
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(rp));
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(rp + 128));
                }
                uint32_t prev = 0, ne = 0;
                for (uint32_t k = 0; k < nd; k++) {                       /* deletions (:568-572) */
                    uint32_t *m = C.var_row((prev << 1) | strand);
                    if (!m) break;
                    const uint32_t d = C.template sym_dense<0, true>(m, L, 10u, MODE == MODE_ENC ? CBCG_EDIT_DELTA(e_in[k]) : 0u, false, 0u);
                    if (C.err) break;
                    prev += d;
                    if (MODE == MODE_DEC && lane == 0) { P.edits[e_cursor + ne] = CBCG_EDIT(d, 0, 0); S.m.cumdel[k] = (uint16_t)min(prev, 0xffffu); }
                    ne++;
                }
                if (MODE == MODE_DEC) __syncwarp();
                prev = 0;
                for (uint32_t k = 0; k < ns && !C.err; k++) {             /* SNPs (:573-593) */
                    const uint32_t ed = MODE == MODE_ENC ? e_in[nd + k] : 0u;
                    const uint32_t delta = C.ring_first(pos - 1u + prev, (prev < len) ? pos - 1u + len : pos - 1u + prev, len + 2u);
                    uint32_t *m = C.var_row((((delta << CBCG_BITS_DELTA) + prev) << 1) | strand);
                    if (!m) break;
                    const uint32_t p = C.template sym_dense<0, true>(m, L, 10u, CBCG_EDIT_DELTA(ed), false, 0u);
                    if (C.err) break;
                    const uint32_t idx = prev + p;                        /* index in the insertion-free read */
                    prev += p + 1u;
                    C.ring_set(pos + prev - 2u);                          /* :589 */
                    uint32_t refb;
                    if (MODE == MODE_DEC) {
                        uint32_t skipped = 0;                             /* deletions at or before idx (:426-437) */
                        if (nd) { for (uint32_t q = lane; q < nd; q += 32u) skipped += (S.m.cumdel[q] <= idx); skipped = warp_sum(skipped); }
                        const uint64_t ri = (uint64_t)pos - 1u + idx + skipped;
                        refb = base_code(ri < C.cold().ref_len ? (uint32_t)C.cold().ref[ri] : 0u);
                    } else refb = CBCG_EDIT_REFB(ed);
                    if (refb > 5u) K2B_FAIL(CBCG_ERR_INPUT);
                    const uint32_t tgt = C.template sym_dense<5, false>(S.m.chars[refb], 5u, 8u, CBCG_EDIT_TARGET(ed), false, 0u);
                    if (MODE == MODE_DEC && lane == 0) P.edits[e_cursor + ne] = CBCG_EDIT(p, tgt, refb);
                    ne++;
                }
                prev = 0;
                for (uint32_t k = 0; k < ni && !C.err; k++) {             /* insertions (:594-600) */
                    const uint32_t ed = MODE == MODE_ENC ? e_in[nd + ns + k] : 0u;
                    uint32_t *m = C.var_row((prev << 1) | strand);
                    if (!m) break;
                    const uint32_t p = C.template sym_dense<0, true>(m, L, 10u, CBCG_EDIT_DELTA(ed), false, 0u);
                    prev += p;
                    const uint32_t tgt = C.template sym_dense<5, false>(S.m.chars[CBCG_BP_O], 5u, 8u, CBCG_EDIT_TARGET(ed), false, 0u);
                    if (MODE == MODE_DEC && lane == 0) P.edits[e_cursor + ne] = CBCG_EDIT(p, tgt, CBCG_BP_O);
                    ne++;
                }
                if (C.err) break;
                e_cursor += ne;
            }
            if (MODE == MODE_DEC) k2b_publish(S, role, i + 1u, lane);
        }
        if (MODE == MODE_DEC && !C.err && !bailed && e_cursor - B.edit_base != B.n_edits) C.err = CBCG_ERR_CORRUPT;   /* the index said otherwise */
    }
role_done:
#undef K2B_FAIL
    if (C.err) {
        dev_set_error(P.err, C.err, ((uint64_t)b << 20) | (i & 0xfffffu));
        S.failed = 1;                                        /* releases the roles that wait for this one */
        return;
    }
    if (bailed) return;
    /* ---- close the substream, leave the final model state where the merge kernels read it */
    if (MODE == MODE_ENC) {
        uint32_t bytes = 0;
        if (C.n_symbols) { C.ac_flush_short(); bytes = C.out_pos; }       /* nothing coded: nothing stored */
        if (C.err) { dev_set_error(P.err, C.err, (uint64_t)b << 20); return; }
        if (lane == 0) B.sub_bytes[role] = bytes;
    }
    __syncwarp();
    if (role == CBCG_SUB_POS) {
        if (lane < C.pos_card) { C.pos_gval()[lane] = C.pos_rv; C.pos_gcnt()[lane] = C.pos_rc; }
        if (lane == 0) { B.pos_card = C.pos_card; B.pa_touched = C.pa_init ? 1u : 0u; }
    } else if (role == CBCG_SUB_FLAG) {
        k2b_copy(FM->rlen0, S.m.rlen0, 256u, lane); k2b_copy(FM->same_ref, S.m.same_ref, 10u, lane);
        const uint32_t used = S.m.flag_used;
        k2b_copy(FM->flag_key, S.m.flag_key, used, lane); k2b_copy(FM->flag_cnt, S.m.flag_cnt, used, lane);
        if (lane == 0) { FM->flag_used = used; FM->flag_n = S.m.flag_n; }
    } else if (role == CBCG_SUB_COUNTS) {
        k2b_copy(FM->snps, S.m.snps, 512u, lane); k2b_copy(&FM->match[0][0], &S.m.match[0][0], 16u, lane);
    } else {
        k2b_copy(&FM->chars[0][0], &S.m.chars[0][0], 48u, lane);
        if (lane == 0) B.n_rows = C.n_rows;
    }
    if (lane == 0) atomicAdd(&B.n_symbols, C.n_symbols);
}

int launch_block_kernel(const CoderParams &p, cudaStream_t st) {
    if (p.n_blocks == 0) return 0;
    if (p.mode == MODE_ENC) k2_block_kernel<MODE_ENC><<<p.n_blocks, K2B_WARPS * 32u, 0, st>>>(p);
    else k2_block_kernel<MODE_DEC><<<p.n_blocks, K2B_WARPS * 32u, 0, st>>>(p);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

/* ================================================================================================
 * Encode of one-stream blocks in TWO KERNELS: models (here), then intervals (k2_code_kernel, k2_blocks.cu).
 *
 * An encoder knows every symbol and every context before it codes anything: the adaptive models (stream_model.c
 * :31-76) never look at the coder's interval, only the coder (Arithmetic_stream.c:274-345) does. The warp kernel above,
 * as a one-kernel encoder, ran both behind each other, 175 warp instructions per symbol, all 32 lanes repeating the
 * interval arithmetic, every block one chain of ~4 700 dependent symbols. Here
 *   - the model half runs as FOUR INDEPENDENT CHAINS per block (POS | length + FLAG | match + counts | var + bases: the
 *     model groups of cbcg_format.h), a warp each, lanes cooperating inside a symbol as before; a chain is a short loop
 *     over one kind of symbol -- no state machine, no interval arithmetic, no bit packer -- and writes each symbol's
 *     interval (cumulative count, count, total: 20 bits each) to the slot the symbol has in the block's stream order
 *     (slot = running sum over the reads' symbol counts, which every chain forms for itself from the records);
 *   - the interval half is one THREAD per block: 32 blocks per warp run the same ~60 instructions per symbol on
 *     different data (closed-form renormalisation: no data-dependent loop), reading their slots in order.
 * Same models, same order, same intervals: the container is byte-identical to the oracle's. POS escapes are the one
 * symbol whose presence the other chains cannot know: the POS triple carries a flag and the four byte symbols go to an
 * escape list that the interval kernel splices in. */
#define K2M_MIN_CTAS 8
/* chains of a block: POS | length + FLAG | match + counts | edit positions + bases (CBCG_SUB_*; the grid runs them from
   the last to the first: the longest chain is scheduled first) */
#define K2M_ROLES      CBCG_N_SUB
__device__ __forceinline__ uint32_t k2m_slots(uint32_t cw, uint32_t lead) {       /* symbols of one read in stream order */
    const uint32_t match = cw & 0xffu, ns = (cw >> 8) & 0xffu, nd = (cw >> 16) & 0xffu, ni = cw >> 24;
    return lead + 3u + (match ? 0u : 1u + ((nd | ni) ? 3u : 0u) + nd + 2u * ns + 2u * ni);
}
/* GROUPED: the edit positions of an unmerged generation by context (below); its own instantiation, so that the serial walk
   of the other keeps its registers (the two together spill into the serial loop: config 5 +5 %). */
template <bool GROUPED>
__global__ void __launch_bounds__(K2_THREADS, K2M_MIN_CTAS)
k2_model_kernel(CoderParams P, uint32_t role_mask) {
    __shared__ __align__(16) WarpShared sh[K2_WARPS];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t role = (K2M_ROLES - 1u) - blockIdx.y;                  /* the longest chain (edit positions) is scheduled first */
    if (!((role_mask >> role) & 1u)) return;                              /* timing experiments only (CBCG_K2M_ROLES) */
    const uint32_t bl = blockIdx.x * K2_WARPS + warp;
    if (bl >= P.n_blocks) return;
    if (*reinterpret_cast<volatile unsigned long long *>(P.err)) return;   /* an earlier stage failed: offsets may be out of range */
    const uint32_t b = P.block_begin + bl;
    BlockDesc &B = P.blocks[b];
    const WsLayout w = ws_layout(P.L, B.n_reads, B.n_edits, 0, 1);
    uint8_t *wsb = P.ws + B.ws_off;
    const uint32_t L = P.L, n_reads = B.n_reads;
    const bool fixed = P.fixed_len != 0;
    const uint32_t lead = fixed ? 0u : 1u;                                 /* the length symbol of variable-length containers */
    const uint64_t r0 = B.first_read;
    WarpModels &S = sh[warp].m;

    Coder<MODE_ENC, true> C;
    C.lane = lane; C.err = 0; C.n_symbols = 0; C.M = &S; C.coldp = &sh[warp].c;
    C.primed = true; C.lean = true; C.var_defer = true; C.var_ro = false; C.defer_idx = 0; C.defer_key = 0;
    C.snap = SnapView(P.snap, L);
    C.L = L; C.Lp = w.Lp;
    C.var_hash = reinterpret_cast<uint64_t *>(wsb + w.var_hash); C.hash_mask = w.hash_cap - 1u; C.var_direct = false;
    C.codebook = nullptr; C.rname = nullptr; C.list = nullptr; C.list_n = 0; C.list_cap = 0;
    C.n_rows = 0; C.pa_init = false; C.pos_card = 1u; C.pos_n = 1u; C.pos_rv = 0u; C.pos_rc = 0u;
    C.last_lo = 0; C.last_n = 0; C.tri_flag = 0u;
    if (lane == 0) {
        WarpCold &W = sh[warp].c;
        W.pos_cap = w.pos_cap; W.rows_cap = w.rows_cap; W.pad = 0; W.io = nullptr; W.io_cap = 0; W.ref = nullptr; W.ref_len = 0;
        W.edits_cap_abs = B.edit_base + B.n_edits;
    }
    __syncwarp();
    uint4 *T = reinterpret_cast<uint4 *>(P.tri) + k2_tri_off(B, b);
    uint4 *slots = T + 1;
    const WarpModels *SM = reinterpret_cast<const WarpModels *>(C.snap.small());
    WarpModels *FM = reinterpret_cast<WarpModels *>(P.fin + (uint64_t)b * fin_stride_dev());
    const uint4 *recs = reinterpret_cast<const uint4 *>(P.recs) + r0;
    uint32_t i = 0, slot = 0;
#define K2M_FAIL(code) do { C.err = (code); goto chain_done; } while (0)

    if (B.chr >= P.genome.n_chr) K2M_FAIL(CBCG_ERR_NO_REFERENCE);         /* blocks never span chromosomes: the host cut them */
    if (role == CBCG_SUB_POS) {
        /* ---- POS through the growing alphabet (compress_pos :113-159, compress_pos_alpha :75-108) */
        C.pos_card = C.snap.pos_hdr()[0]; C.pos_n = C.snap.pos_hdr()[1];
        if (C.pos_card > w.pos_cap) K2M_FAIL(CBCG_ERR_INTERNAL);
        C.pos_rv = (lane < C.pos_card) ? C.snap.pos_val()[lane] : 0u;
        C.pos_rc = (lane < C.pos_card) ? C.snap.pos_cnt()[lane] : 0u;
        for (uint32_t q = 32u + lane; q < C.pos_card; q += 32u) { C.pos_gval()[q] = C.snap.pos_val()[q]; C.pos_gcnt()[q] = C.snap.pos_cnt()[q]; }
        __syncwarp();
        uint4 *esc = T + k2_tri_esc(B);
        uint32_t prev_pos = B.base_pos;
        uint4 v = n_reads ? recs[0] : make_uint4(0u, 0u, 0u, 0u);
        for (; i < n_reads; i++) {
            const uint4 nx = (i + 1u < n_reads) ? recs[i + 1u] : v;        /* next read's record: off the chain */
            const uint32_t pos = v.x;
            if (pos == 0u || pos < prev_pos) K2M_FAIL(CBCG_ERR_INPUT);
            const uint32_t x = pos - prev_pos + 1u;
            uint32_t s = 1u;
            C.tri_at = slots + slot + lead;
            C.sym_pos_main(x, s);
            if (C.err) break;
            if (s == 0u) {                                   /* escape: the value itself, 4 bytes MSB first, then a new slot */
                C.pa_ensure();
                for (uint32_t k = 0; k < 4u; k++) {
                    C.tri_at = esc++;
                    C.template sym_dense<0, false>(C.pos_alpha() + k * PA_STRIDE, 256u, 10u, (x >> (24u - 8u * k)) & 0xffu, false, 0u);
                }
                if (C.err) break;
                C.pos_append(x);
                if (C.err) break;
            }
            prev_pos = pos;
            slot += k2m_slots(v.w, lead);
            v = nx;
        }
    } else if (role == CBCG_SUB_FLAG) {
        /* ---- length byte 0 (variable-length containers) and FLAG (compress_read :29-33, compress_flag :50-70).
           While the sparse FLAG table has <= 32 touched values it lives one entry per lane, ascending like the table in
           shared memory: key, count, and the extras (count - 1) of all entries below, kept up to date by a predicated add
           per update -- so a symbol's cumulative count x + extras(below x) is two ballots and two shuffles, no scan. An
           insertion into a full warp or a rescale writes the entries to shared memory and carries on there (sym_flag). */
        k2b_copy(S.rlen0, SM->rlen0, 256u, lane);
        k2b_copy(S.same_ref, SM->same_ref, 4u + 6u, lane);                 /* same_ref, rlenk: never coded here, the merge reads the image */
        uint32_t used = SM->flag_used, fn = SM->flag_n;
        k2b_copy(S.flag_key, SM->flag_key, used, lane); k2b_copy(S.flag_cnt, SM->flag_cnt, used, lane);
        if (lane == 0) { S.flag_used = used; S.flag_n = fn; }
        __syncwarp();
        bool in_regs = used <= 32u;
        uint32_t fk = 0xffffffffu, fc = 1u, fE = 0u, etot = 0u;
#define K2M_FLAG_LOAD() do { \
            fk = (lane < used) ? S.flag_key[lane] : 0xffffffffu; fc = (lane < used) ? S.flag_cnt[lane] : 1u; \
            const uint32_t e1_ = fc - 1u, in_ = warp_incl_scan(e1_); fE = in_ - e1_; etot = __shfl_sync(FULL_MASK, in_, 31); } while (0)
#define K2M_FLAG_STORE() do { \
            if (lane < used) { S.flag_key[lane] = fk; S.flag_cnt[lane] = fc; } \
            if (lane == 0) { S.flag_used = used; S.flag_n = fn; } \
            __syncwarp(); } while (0)
        if (in_regs) K2M_FLAG_LOAD();
        uint4 v = n_reads ? recs[0] : make_uint4(0u, 0u, 0u, 0u);
        for (; i < n_reads; i++) {
            const uint4 nx = (i + 1u < n_reads) ? recs[i + 1u] : v;
            const uint32_t flag = v.y & 0xffffu, len = v.y >> 16;
            if (len == 0u || len > CBCG_MAX_READ_LEN || (fixed && len != L)) K2M_FAIL(CBCG_ERR_INPUT);
            if (!fixed) { C.tri_at = slots + slot; C.template sym_dense<0, false>(S.rlen0, 255u, 10u, len & 0xffu, false, 0u); }
            uint4 *at = slots + slot + lead + 1u;
            bool coded = false;
            if (LIKELY(in_regs)) {
                const uint32_t p = (uint32_t)__popc(__ballot_sync(FULL_MASK, fk < flag));       /* entries below: lanes 0 .. p-1 */
                const bool found = __ballot_sync(FULL_MASK, fk == flag) != 0u;
                const uint32_t Ep = __shfl_sync(FULL_MASK, fE, p & 31u), cp = __shfl_sync(FULL_MASK, fc, p & 31u);
                const uint32_t below = p < used ? Ep : etot;
                if (found || used < 32u) {
                    if (lane == 0) *at = make_uint4(flag + below, found ? cp : 1u, fn, 0u);
                    C.n_symbols++;
                    if (found) { if (lane == p) fc += 8u; }                  /* update_model, step 8 */
                    else {                                                   /* first touch: (flag, 1 + 8) enters at p */
                        const uint32_t ku = __shfl_up_sync(FULL_MASK, fk, 1), cu = __shfl_up_sync(FULL_MASK, fc, 1), eu = __shfl_up_sync(FULL_MASK, fE, 1);
                        if (lane > p) { fk = ku; fc = cu; fE = eu; }
                        if (lane == p) { fk = flag; fc = 9u; fE = below; }
                        used++;
                    }
                    if (lane > p) fE += 8u;
                    etot += 8u; fn += 8u;
                    if (UNLIKELY(fn >= CBCG_RESCALE)) {                      /* update_model :38-49, on the table in shared memory */
                        K2M_FLAG_STORE();
                        fn = rescale_counts(S.flag_cnt, used, lane) + (65536u - used);
                        __syncwarp();
                        K2M_FLAG_LOAD();
                    }
                    coded = true;
                } else { K2M_FLAG_STORE(); in_regs = false; }                /* a 33rd value: the table moves to shared memory */
            }
            if (!coded) {
                C.tri_at = at;
                C.sym_flag(flag);
                if (C.err) break;
            }
            slot += k2m_slots(v.w, lead);
            v = nx;
        }
        if (!C.err && in_regs) K2M_FLAG_STORE();
#undef K2M_FLAG_LOAD
#undef K2M_FLAG_STORE
        if (!C.err && lane == 0) T[0] = make_uint4(slot, 0u, 0u, 0u);   /* the block's main slots: what the interval kernel walks */
    } else if (role == CBCG_SUB_COUNTS) {
        /* ---- match bit, SNP count, indel counts (compress_match :164-188, compress_snps / compress_indels :193-228) */
        k2b_copy(S.snps, SM->snps, 512u, lane);                            /* snps, indels */
        k2b_copy(&S.match[0][0], &SM->match[0][0], 16u, lane);
        __syncwarp();
        uint32_t prev_pos = B.base_pos, prev_m = 0u;
        uint4 v = n_reads ? recs[0] : make_uint4(0u, 0u, 0u, 0u);
        for (; i < n_reads; i++) {
            const uint4 nx = (i + 1u < n_reads) ? recs[i + 1u] : v;
            const uint32_t pos = v.x, match = v.w & 0xffu, ns = (v.w >> 8) & 0xffu, nd = (v.w >> 16) & 0xffu, ni = v.w >> 24;
            const uint32_t samepos = pos == prev_pos ? 1u : 0u;            /* deltaP == 1 (:170) */
            prev_pos = pos;
            uint4 *at = slots + slot + lead + 2u;
            C.tri_at = at;
            C.template sym_dense<2, false>(S.match[(samepos << 1) | prev_m], 2u, 1u, match, false, 0u);
            if (C.err) break;
            prev_m = match;
            if (!match) {
                C.tri_at = at + 1;
                C.template sym_dense<0, false>(S.snps, L, 10u, ((nd | ni) == 0u) ? ns : 0u, false, 0u);
                if (!C.err && (nd | ni) != 0u) {                           /* :560-565 */
                    C.tri_at = at + 2; C.template sym_dense<0, false>(S.indels, L, 16u, ns, false, 0u);
                    C.tri_at = at + 3; C.template sym_dense<0, false>(S.indels, L, 16u, nd, false, 0u);
                    C.tri_at = at + 4; C.template sym_dense<0, false>(S.indels, L, 16u, ni, false, 0u);
                }
                if (C.err) break;
            }
            slot += k2m_slots(v.w, lead);
            v = nx;
        }
    } else if (GROUPED && 8ull * n_reads + 2ull * B.n_edits + 8ull < (1ull << 24)) {     /* slot indices are packed in 24 bits below */
        /* ---- edit positions and bases of a generation that nobody merges (the last one: 92 % of the reads), WITHOUT the
           serial walk through the var rows. A var context's model is touched by a handful of symbols per block and is
           independent of every other context's; what orders the symbols is only the SNP-site ring (input alone) and the
           earlier symbols of the SAME context. So:
             A. one sequential pass over the reads forms every position symbol's context (ring_first / ring_set as in
                compute_delta_to_first_snp :703-718), lists (context, symbol, slot) and codes the bases through chars
                (shared memory, cheap) on the way;
             B. the list is linked by context, 32 symbols a step: each symbol learns the previous symbol of its context
                (warp match for the ones in the same step, a hash of last occurrences for the earlier ones);
             C. a LANE per symbol: cumulative count and count from the snapshot's row (read only; all-ones for a context
                the snapshot lacks), plus 10 for every earlier symbol of the context below / at the symbol (update_model's
                step) -- no row is copied, no row is written, no symbol waits for another context's.
           A context whose total would reach the rescale threshold inside the block sends the block through the serial
           walk below instead (never seen on the named shapes: totals start far from 2^20). */
        /* Step C walks back over the earlier symbols of a symbol's context: fine for the handful a context sees in a
           block, quadratic for a context that thousands of symbols share -- the first deletion / insertion of a read has
           context (0, strand) whatever the read. Indel-heavy blocks take the serial walk (config 5: measured twice as slow
           here), and so does any block in which a context turns out to be shared by more than K2M_CTX_MAX symbols. */
#define K2M_INDEL_MAX 1024u
#define K2M_CTX_MAX   1023u
        {
            uint32_t indels = 0;
            for (uint32_t q = lane; q < n_reads; q += 32u) { const uint32_t cw = recs[q].w; if (!(cw & 0xffu)) indels += ((cw >> 16) & 0xffu) + (cw >> 24); }
            if (warp_sum(indels) > K2M_INDEL_MAX) goto edits_serial;
        }
        k2b_copy(&S.chars[0][0], &SM->chars[0][0], 48u, lane);
        for (uint32_t q = lane; q <= C.hash_mask; q += 32u) C.var_hash[q] = 0ull;
        __syncwarp();
        C.ring_reset();
        uint32_t *it_ctx = C.var_rows();                                    /* the rows' room in the workspace: 4 words per symbol of <= n_edits */
        uint32_t *it_xs = it_ctx + B.n_edits, *it_prev = it_xs + B.n_edits, *it_ord = it_prev + B.n_edits;
        uint32_t K = 0, max_ord = 0;
        uint4 v = n_reads ? recs[0] : make_uint4(0u, 0u, 0u, 0u);
        for (; i < n_reads; i++) {                                          /* ---- A */
            const uint4 nx = (i + 1u < n_reads) ? recs[i + 1u] : v;
            const uint32_t pos = v.x, flag = v.y & 0xffffu, len = v.y >> 16, match = v.w & 0xffu;
            const uint32_t ns = (v.w >> 8) & 0xffu, nd = (v.w >> 16) & 0xffu, ni = v.w >> 24;
            if (pos == 0u) K2M_FAIL(CBCG_ERR_INPUT);
            if (!(nx.w & 0xffu)) asm volatile("prefetch.global.L1 [%0];" ::"l"(P.edits + nx.z));
            const uint32_t strand = (flag >> 4) & 1u;                      /* :57-60 */
            C.ring_advance(pos);
            if (!match) {
                const uint16_t *e_in = P.edits + v.z;
                uint32_t at = slot + lead + 4u + ((nd | ni) ? 3u : 0u);     /* slot index of the read's first edit symbol */
                if (K + nd + ns + ni > B.n_edits) K2M_FAIL(CBCG_ERR_INTERNAL);
#define K2M_ITEM(CTX, X) do { const uint32_t c_ = (CTX), x_ = (X); \
                    if (c_ >= CBCG_VAR_CONTEXTS || x_ >= L) K2M_FAIL(CBCG_ERR_INPUT); \
                    if (lane == 0) { it_ctx[K] = c_; it_xs[K] = (at << 8) | x_; } K++; at++; } while (0)
                uint32_t prev = 0;
                for (uint32_t k = 0; k < nd; k++) {                         /* deletions (:568-572) */
                    const uint32_t d = CBCG_EDIT_DELTA((uint32_t)e_in[k]);
                    K2M_ITEM((prev << 1) | strand, d);
                    prev += d;
                }
                prev = 0;
                for (uint32_t k = 0; k < ns; k++) {                         /* SNPs (:573-593) */
                    const uint32_t ed = e_in[nd + k];
                    const uint32_t delta = C.ring_first(pos - 1u + prev, (prev < len) ? pos - 1u + len : pos - 1u + prev, len + 2u);
                    const uint32_t p = CBCG_EDIT_DELTA(ed);
                    K2M_ITEM((((delta << CBCG_BITS_DELTA) + prev) << 1) | strand, p);
                    prev += p + 1u;
                    C.ring_set(pos + prev - 2u);                            /* :589 */
                    const uint32_t refb = CBCG_EDIT_REFB(ed);
                    if (refb > 5u) K2M_FAIL(CBCG_ERR_INPUT);
                    C.tri_at = slots + at; at++;
                    C.template sym_dense<5, false>(S.chars[refb], 5u, 8u, CBCG_EDIT_TARGET(ed), false, 0u);
                    if (C.err) break;
                }
                prev = 0;
                for (uint32_t k = 0; k < ni && !C.err; k++) {               /* insertions (:594-600) */
                    const uint32_t ed = e_in[nd + ns + k];
                    const uint32_t p = CBCG_EDIT_DELTA(ed);
                    K2M_ITEM((prev << 1) | strand, p);
                    prev += p;
                    C.tri_at = slots + at; at++;
                    C.template sym_dense<5, false>(S.chars[CBCG_BP_O], 5u, 8u, CBCG_EDIT_TARGET(ed), false, 0u);
                }
#undef K2M_ITEM
                if (C.err) break;
            }
            slot += k2m_slots(v.w, lead);
            v = nx;
        }
        if (C.err) goto chain_done;
        __syncwarp();
        for (uint32_t base = 0; base < K; base += 32u) {                    /* ---- B */
            const uint32_t kk = base + lane;
            const bool valid = kk < K;
            const uint32_t c = valid ? it_ctx[kk] : 0xffffff00u + lane;    /* lanes past the list: a group of their own */
            const uint32_t peers = __match_any_sync(FULL_MASK, c);
            const uint32_t below = peers & ((1u << lane) - 1u);
            const bool top = (peers >> lane) == 1u;                         /* the group's last symbol of this step: it updates the hash */
            uint32_t prev = 0xffffffffu;
            if (valid) {
                const uint64_t key = (uint64_t)(c + 1u) << 32;
                uint32_t h = (c * 0x9E3779B1u) >> 7;
                for (;;) {
                    const uint32_t idx = h & C.hash_mask;
                    const uint64_t e = C.var_hash[idx];
                    if ((e >> 32) == (uint64_t)(c + 1u)) { prev = (uint32_t)e; if (top) C.var_hash[idx] = key | kk; break; }
                    if (e == 0ull) {
                        if (!top) break;                                    /* nothing earlier; the top lane makes the entry */
                        if (atomicCAS(reinterpret_cast<unsigned long long *>(&C.var_hash[idx]), 0ull, key | kk) == 0ull) break;
                        continue;                                           /* another context took the slot in this step: look again */
                    }
                    h++;
                }
                /* ordinal of the symbol within its context: the ones of this step, and those before the step's first */
                const uint32_t ord = (uint32_t)__popc(below) + (prev != 0xffffffffu ? it_ord[prev] + 1u : 0u);
                if (below) prev = base + 31u - (uint32_t)__clz(below);      /* the nearest earlier symbol of the context is in this step */
                it_prev[kk] = prev; it_ord[kk] = ord;
                max_ord = max(max_ord, ord);
            }
            __syncwarp();
        }
        if (warp_sum(max_ord > K2M_CTX_MAX ? 1u : 0u)) { i = 0; slot = 0; goto edits_serial; }
        __threadfence_block();
        __syncwarp();
        bool redo = false;
        for (uint32_t base = 0; base < K; base += 32u) {                    /* ---- C */
            const uint32_t kk = base + lane;
            if (kk < K) {
                const uint32_t c = it_ctx[kk], xs = it_xs[kk], x = xs & 0xffu;
                const uint32_t *row = ((C.snap.bitmap()[c >> 5] >> (c & 31u)) & 1u) ? C.snap.var_row(c) : C.snap.ones();
                uint32_t n = row[L], cnt = row[x], lo = 0;
                uint32_t j = 0;
                for (; j + 4u <= x; j += 4u) { const uint4 q = *reinterpret_cast<const uint4 *>(row + j); lo += q.x + q.y + q.z + q.w; }
                if (j < x) { const uint4 q = *reinterpret_cast<const uint4 *>(row + j); lo += q.x + (j + 1u < x ? q.y : 0u) + (j + 2u < x ? q.z : 0u); }
                for (uint32_t e = it_prev[kk]; e != 0xffffffffu; e = it_prev[e]) {   /* earlier symbols of the context: update_model, step 10 */
                    const uint32_t xe = it_xs[e] & 0xffu;
                    n += 10u; lo += xe < x ? 10u : 0u; cnt += xe == x ? 10u : 0u;
                }
                if (n + 10u >= CBCG_RESCALE) redo = true;
                else if (cnt == 0u || n == 0u) C.err = CBCG_ERR_INPUT;       /* reference: assert :71 / :293 */
                else slots[xs >> 8] = make_uint4(lo, cnt, n, 0u);
            }
        }
        if (__any_sync(FULL_MASK, C.err != 0)) { if (!C.err) C.err = CBCG_ERR_INPUT; goto chain_done; }
        if (__any_sync(FULL_MASK, redo)) {                                  /* a total reaches the threshold: the serial walk, from the top */
            i = 0; slot = 0;
            goto edits_serial;
        }
        if (lane == 0) B.n_rows = 0u;
        goto chain_done;
    } else {
        /* ---- edit positions through the var rows, bases through chars (:568-600; compute_delta_to_first_snp :703-718).
           Measured and dropped: the bases as a fifth chain of their own (220 M more warp instructions for the second walk
           over the records, 0.24 ms slower: the kernel as a whole is bound by instruction issue, not by its longest chain);
           asking for the next context's hash line and snapshot row one symbol ahead (the contexts depend on the input
           alone): this chain alone 1.65 -> 1.79 ms. */
edits_serial:
        k2b_copy(&S.chars[0][0], &SM->chars[0][0], 48u, lane);
        for (uint32_t q = lane; q <= C.hash_mask; q += 32u) C.var_hash[q] = 0ull;
        __syncwarp();
        C.ring_reset();
        uint4 v = n_reads ? recs[0] : make_uint4(0u, 0u, 0u, 0u);
        for (; i < n_reads; i++) {
            const uint4 nx = (i + 1u < n_reads) ? recs[i + 1u] : v;
            const uint32_t pos = v.x, flag = v.y & 0xffffu, len = v.y >> 16, match = v.w & 0xffu;
            const uint32_t ns = (v.w >> 8) & 0xffu, nd = (v.w >> 16) & 0xffu, ni = v.w >> 24;
            if (pos == 0u) K2M_FAIL(CBCG_ERR_INPUT);
            if (!(nx.w & 0xffu)) asm volatile("prefetch.global.L1 [%0];" ::"l"(P.edits + nx.z));
            const uint32_t strand = (flag >> 4) & 1u;                      /* :57-60 */
            C.ring_advance(pos);
            if (!match) {
                const uint16_t *e_in = P.edits + v.z;
                uint4 *at = slots + slot + lead + 4u + ((nd | ni) ? 3u : 0u);
                uint32_t prev = 0;
                for (uint32_t k = 0; k < nd; k++) {                         /* deletions (:568-572) */
                    uint32_t *m = C.var_row((prev << 1) | strand);
                    if (!m) break;
                    const uint32_t d = CBCG_EDIT_DELTA((uint32_t)e_in[k]);
                    C.tri_at = at++;
                    C.template sym_dense<0, true>(m, L, 10u, d, false, 0u);
                    if (C.err) break;
                    prev += d;
                }
                prev = 0;
                for (uint32_t k = 0; k < ns && !C.err; k++) {               /* SNPs (:573-593) */
                    const uint32_t ed = e_in[nd + k];
                    const uint32_t delta = C.ring_first(pos - 1u + prev, (prev < len) ? pos - 1u + len : pos - 1u + prev, len + 2u);
                    uint32_t *m = C.var_row((((delta << CBCG_BITS_DELTA) + prev) << 1) | strand);
                    if (!m) break;
                    const uint32_t p = CBCG_EDIT_DELTA(ed);
                    C.tri_at = at++;
                    C.template sym_dense<0, true>(m, L, 10u, p, false, 0u);
                    if (C.err) break;
                    prev += p + 1u;
                    C.ring_set(pos + prev - 2u);                            /* :589 */
                    const uint32_t refb = CBCG_EDIT_REFB(ed);
                    if (refb > 5u) K2M_FAIL(CBCG_ERR_INPUT);
                    C.tri_at = at++;
                    C.template sym_dense<5, false>(S.chars[refb], 5u, 8u, CBCG_EDIT_TARGET(ed), false, 0u);
                }
                prev = 0;
                for (uint32_t k = 0; k < ni && !C.err; k++) {               /* insertions (:594-600) */
                    const uint32_t ed = e_in[nd + ns + k];
                    uint32_t *m = C.var_row((prev << 1) | strand);
                    if (!m) break;
                    const uint32_t p = CBCG_EDIT_DELTA(ed);
                    C.tri_at = at++;
                    C.template sym_dense<0, true>(m, L, 10u, p, false, 0u);
                    prev += p;
                    C.tri_at = at++;
                    C.template sym_dense<5, false>(S.chars[CBCG_BP_O], 5u, 8u, CBCG_EDIT_TARGET(ed), false, 0u);
                }
                if (C.err) break;
            }
            slot += k2m_slots(v.w, lead);
            v = nx;
        }
    }
chain_done:
#undef K2M_FAIL
    if (C.err) { dev_set_error(P.err, C.err, ((uint64_t)b << 20) | (i & 0xfffffu)); return; }
    /* ---- leave the final model state where the merge kernels read it */
    __syncwarp();
    if (role == CBCG_SUB_POS) {
        if (lane < C.pos_card) { C.pos_gval()[lane] = C.pos_rv; C.pos_gcnt()[lane] = C.pos_rc; }
        if (lane == 0) { B.pos_card = C.pos_card; B.pa_touched = C.pa_init ? 1u : 0u; }
    } else if (role == CBCG_SUB_FLAG) {
        k2b_copy(FM->rlen0, S.rlen0, 256u, lane); k2b_copy(FM->same_ref, S.same_ref, 10u, lane);
        const uint32_t used = S.flag_used;
        k2b_copy(FM->flag_key, S.flag_key, used, lane); k2b_copy(FM->flag_cnt, S.flag_cnt, used, lane);
        if (lane == 0) { FM->flag_used = used; FM->flag_n = S.flag_n; }
    } else if (role == CBCG_SUB_COUNTS) {
        k2b_copy(FM->snps, S.snps, 512u, lane); k2b_copy(&FM->match[0][0], &S.match[0][0], 16u, lane);
    } else {
        k2b_copy(&FM->chars[0][0], &S.chars[0][0], 48u, lane);
        if (lane == 0) B.n_rows = C.n_rows;
    }
}

/* one-stream blocks, encode: the model kernel, then the interval kernel (k2_blocks.cu) */
static int launch_split_encode(const CoderParams &p, cudaStream_t st) {
    const dim3 grid((p.n_blocks + K2_WARPS - 1u) / K2_WARPS, K2M_ROLES);
    const char *rm = getenv("CBCG_K2M_ROLES");                          /* timing experiments: chains to run (tools/role_times.py) */
    const uint32_t role_mask = rm ? (uint32_t)atoi(rm) : 0xfu;
    /* indel-heavy input (the host's estimate from the CIGAR text per read): every block would fall back to the serial walk */
    if (p.no_merge && !p.indel_heavy) k2_model_kernel<true><<<grid, K2_THREADS, 0, st>>>(p, role_mask);
    else k2_model_kernel<false><<<grid, K2_THREADS, 0, st>>>(p, role_mask);
    if (cudaGetLastError() != cudaSuccess) return -1;
    return launch_code_kernel(p, st);
}

uint32_t coder_resident_blocks(int device) {
    int sms = 0, per_sm = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0) return 148u * 16u;
    /* the blocked warp decoder: its launch bounds and shared memory, and so its occupancy, are the warp encoder's */
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k2_coder_kernel<MODE_DEC, false>, (int)K2_THREADS, 0) != cudaSuccess || per_sm <= 0) per_sm = K2_MIN_CTAS;
    if (per_sm > 5) per_sm = 5;                              /* the cut (and with it the container) does not follow a build with more resident CTAs */
    return (uint32_t)sms * (uint32_t)per_sm * K2_WARPS;
}

__global__ void k2_plan_kernel(CoderParams P, uint32_t n_reads_total, uint64_t n_edits_total, uint64_t ws_cap, uint64_t payload_cap,
                               uint64_t *totals, const uint64_t *carry_in, const uint64_t *n_edits_dev);
__global__ void k2_payload_scan_kernel(BlockDesc *blocks, uint32_t n_blocks, uint64_t *out_off, int blocked, uint32_t layout_mode);
__global__ void k2_gather_kernel(const BlockDesc *blocks, uint32_t n_blocks, const uint8_t *scratch, uint8_t *out, const uint64_t *out_off, int blocked, uint32_t layout_mode);
__global__ void snapshot_copy_kernel(uint4 *__restrict__ dst, const uint4 *__restrict__ src, uint64_t n16);
struct MergeParams;
__global__ void merge_prep_kernel(MergeParams P);
__global__ void merge_add_kernel(MergeParams P);
__global__ void merge_finish_kernel(MergeParams P);
__global__ void merge_var_finish_kernel(MergeParams P);

/* Shared-memory carveout. An SM cannot host CTAs of kernels that ask for different L1 / shared-memory splits at the same
 * time: with the driver's per-kernel choices the K1 / K3 launches of a pipelined call (api.cu) wait for the resident
 * block-coder CTAs to drain (measured: the whole gain of the pipeline is lost). Pipelined calls therefore put every
 * kernel on the same split; one-stream calls keep the driver's choices, which are 0.3 ms better for the block coder. */
void extract_set_carveout(int pct);        /* k1_extract.cu */
void reconstruct_set_carveout(int pct);    /* k3_reconstruct.cu */
void blocks_set_carveout(int pct);         /* k2_blocks.cu */
void unpack_set_carveout(int pct);         /* k0_unpack.cu */
template <class K> static void set_carveout(K kernel, int pct) { cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct); }
/* pct = -1: every kernel gets the split the driver prefers for it (best for each kernel on its own: the one-stream
 * calls); 0..100: that share of shared memory for all of them (the pipelined calls). */
void set_carveout_all(int pct) {
    static int current = -1;
    if (pct == current) return;
    current = pct;
    set_carveout(k2_coder_kernel<MODE_DEC, false>, pct); set_carveout(k2_coder_kernel<MODE_LIST, false>, pct);
    set_carveout(k2_block_kernel<MODE_ENC>, pct); set_carveout(k2_block_kernel<MODE_DEC>, pct); set_carveout(k2_model_kernel<true>, pct); set_carveout(k2_model_kernel<false>, pct);
    set_carveout(k2_coder_kernel<MODE_ENC, true>, pct); set_carveout(k2_coder_kernel<MODE_DEC, true>, pct); set_carveout(k2_coder_kernel<MODE_LIST, true>, pct);
    set_carveout(k2_plan_kernel, pct); set_carveout(k2_payload_scan_kernel, pct); set_carveout(k2_gather_kernel, pct);
    set_carveout(snapshot_copy_kernel, pct);
    set_carveout(merge_prep_kernel, pct); set_carveout(merge_add_kernel, pct); set_carveout(merge_finish_kernel, pct); set_carveout(merge_var_finish_kernel, pct);
    extract_set_carveout(pct); reconstruct_set_carveout(pct); blocks_set_carveout(pct); unpack_set_carveout(pct);
}

static bool split_encode(const CoderParams &p) { return !p.legacy && p.mode == MODE_ENC && p.n_sub <= 1u; }
uint32_t coder_launches(const CoderParams &p) {
    if (p.n_blocks == 0) return 0u;
    return split_encode(p) ? 2u : 1u;
}
int launch_block_kernel(const CoderParams &p, cudaStream_t st);
int launch_coder(const CoderParams &p, cudaStream_t st) {
    if (p.n_blocks == 0) return 0;
    if (!p.legacy && p.mode != MODE_LIST && p.n_sub > 1u) return launch_block_kernel(p, st);   /* four-substream containers: a CTA per block, a warp per substream */
    if (split_encode(p)) return p.tri ? launch_split_encode(p, st) : -1;                      /* no interval buffer: a caller bug */
    const unsigned grid = (p.n_blocks + K2_WARPS - 1) / K2_WARPS;
    if (p.legacy) {
        if (p.mode == MODE_ENC) k2_coder_kernel<MODE_ENC, true><<<grid, K2_THREADS, 0, st>>>(p);
        else if (p.mode == MODE_DEC) k2_coder_kernel<MODE_DEC, true><<<grid, K2_THREADS, 0, st>>>(p);
        else k2_coder_kernel<MODE_LIST, true><<<grid, K2_THREADS, 0, st>>>(p);
    } else {
        if (p.mode == MODE_DEC) k2_coder_kernel<MODE_DEC, false><<<grid, K2_THREADS, 0, st>>>(p);
        else k2_coder_kernel<MODE_LIST, false><<<grid, K2_THREADS, 0, st>>>(p);
    }
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

/* ------------------------------------------------------------------------------------------------
 * plan: per-block sizes -> offsets (one CTA; blocks in chunks of 1024 with a running carry).
 * totals[0] = workspace bytes, [1] = payload bytes, [2] = symbol-list entries, [3] = reads, [4] = edits. */
#define PLAN_THREADS 256u          /* a small CTA: during a pipelined call it has to find room beside resident block-coder CTAs */
__global__ void __launch_bounds__(PLAN_THREADS)
k2_plan_kernel(CoderParams P, uint32_t n_reads_total, uint64_t n_edits_total, uint64_t ws_cap, uint64_t payload_cap,
               uint64_t *totals, const uint64_t *carry_in, const uint64_t *n_edits_dev) {
    /* Plans blocks [P.block_begin, + P.n_blocks). A pipelined encode (api.cu) plans chunk by chunk as the reads arrive:
       the offsets carry on from the previous call's totals (carry_in) and the edit count so far is read on the device. */
    if (n_edits_dev) n_edits_total = *n_edits_dev;
    __shared__ uint64_t wsum[5][32];
    __shared__ uint64_t carry[5];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid < 5) carry[tid] = carry_in ? carry_in[tid] : 0;
    __syncthreads();
    const bool dec = (P.mode == MODE_DEC);
    const uint32_t b_end = P.block_begin + P.n_blocks;
    for (uint32_t base = P.block_begin; base < b_end; base += PLAN_THREADS) {
        const uint32_t b = base + tid;
        uint64_t v[5] = { 0, 0, 0, 0, 0 };
        BlockDesc d;
        if (b < b_end) {
            d = P.blocks[b];
            if (!dec) {                                  /* edits of the block from the records' offsets */
                const uint64_t lo = P.recs[d.first_read].edit_off;
                const uint64_t end = (uint64_t)d.first_read + d.n_reads;
                const uint64_t hi = (end < n_reads_total) ? P.recs[end].edit_off : n_edits_total;
                d.n_edits = (uint32_t)(hi - lo);
                d.edit_base = lo;
                if (!P.legacy) d.base_pos = P.recs[d.first_read].pos;
            }
            const uint64_t ws_edits = (dec && P.legacy) ? 0xffffffffull : d.n_edits;
            v[0] = ws_layout(P.L ? P.L : 252u, d.n_reads, ws_edits, P.legacy, P.primed && P.mode != MODE_LIST).total;
            v[1] = dec ? d.payload_bytes : payload_cap_bytes(d.n_reads, d.n_edits, P.legacy ? 2 : (CBCG_BLOCK_NSUB(P.layout_mode, d.gen) <= 1u ? 1 : 0));
            v[2] = (P.mode == MODE_LIST) ? symlist_cap(d.n_reads, d.n_edits, P.legacy) : 0;
            v[3] = d.n_reads; v[4] = d.n_edits;
        }
        uint64_t incl[5];
#pragma unroll
        for (int q = 0; q < 5; q++) {
            uint64_t x = v[q];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { uint64_t y = __shfl_up_sync(FULL_MASK, x, o); if (lane >= (uint32_t)o) x += y; }
            incl[q] = x;
            if (lane == 31) wsum[q][warp] = x;
        }
        __syncthreads();
        uint64_t off[5];
#pragma unroll
        for (int q = 0; q < 5; q++) {
            uint64_t wb = 0;
            for (uint32_t k = 0; k < warp; k++) wb += wsum[q][k];
            off[q] = carry[q] + wb + incl[q] - v[q];
        }
        if (b < b_end) {
            d.ws_off = off[0];
            if (!dec) d.payload_off = off[1];
            else { d.payload_off = off[1]; d.first_read = (uint32_t)off[3]; d.edit_base = off[4]; }
            d.sym_off = off[2];
            if (!P.legacy && P.mode != MODE_LIST && CBCG_BLOCK_NSUB(P.layout_mode, d.gen) > 1u) {   /* the substream roles add their symbol counts */
                d.n_symbols = 0; d.pos_card = 0; d.n_rows = 0; d.pa_touched = 0;
                if (!dec) { d.payload_bytes = 0; for (uint32_t q = 0; q < CBCG_N_SUB; q++) d.sub_bytes[q] = 0; }
            }
            P.blocks[b] = d;
        }
        __syncthreads();
        if (tid == PLAN_THREADS - 1) {
#pragma unroll
            for (int q = 0; q < 5; q++) carry[q] = off[q] + v[q];
        }
        __syncthreads();
    }
    if (tid == 0) {
        for (int q = 0; q < 5; q++) totals[q] = carry[q];
        if (carry[0] > ws_cap || (!dec && P.mode == MODE_ENC && carry[1] > payload_cap)) dev_set_error(P.err, CBCG_ERR_INTERNAL, 0xabcdefull);
    }
}

int launch_plan(const CoderParams &p, uint32_t n_reads_total, uint64_t n_edits_total, uint64_t ws_cap,
                uint64_t payload_cap, uint64_t *totals, cudaStream_t st, const uint64_t *carry_in, const uint64_t *n_edits_dev) {
    k2_plan_kernel<<<1, PLAN_THREADS, 0, st>>>(p, n_reads_total, n_edits_total, ws_cap, payload_cap, totals, carry_in, n_edits_dev);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

/* ------------------------------------------------------------------------------------------------
 * gather: block payloads (scratch regions) -> one contiguous payload; out_off[b] = its offset. */
__global__ void __launch_bounds__(PLAN_THREADS)
k2_payload_scan_kernel(BlockDesc *blocks, uint32_t n_blocks, uint64_t *out_off, int blocked, uint32_t layout_mode) {
    __shared__ uint64_t wsum[32];
    __shared__ uint64_t carry;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n_blocks; base += PLAN_THREADS) {
        const uint32_t b = base + tid;
        uint64_t v = 0;
        if (b < n_blocks) {
            if (blocked && CBCG_BLOCK_NSUB(layout_mode, blocks[b].gen) > 1u) { uint32_t t = 0; for (uint32_t q = 0; q < CBCG_N_SUB; q++) t += blocks[b].sub_bytes[q]; blocks[b].payload_bytes = t; }
            v = blocks[b].payload_bytes;
        }
        uint64_t x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { uint64_t y = __shfl_up_sync(FULL_MASK, x, o); if (lane >= (uint32_t)o) x += y; }
        if (lane == 31) wsum[warp] = x;
        __syncthreads();
        uint64_t wb = 0;
        for (uint32_t k = 0; k < warp; k++) wb += wsum[k];
        const uint64_t off = carry + wb + x - v;
        if (b < n_blocks) out_off[b] = off;
        __syncthreads();
        if (tid == PLAN_THREADS - 1) carry = off + v;
        __syncthreads();
    }
    if (tid == 0) out_off[n_blocks] = carry;
}

__global__ void k2_gather_kernel(const BlockDesc *blocks, uint32_t n_blocks, const uint8_t *scratch, uint8_t *out,
                                 const uint64_t *out_off, int blocked, uint32_t layout_mode) {
    for (uint32_t b = blockIdx.x; b < n_blocks; b += gridDim.x) {
        const uint8_t *src = scratch + blocks[b].payload_off;
        uint8_t *dst = out + out_off[b];
        if (!blocked || CBCG_BLOCK_NSUB(layout_mode, blocks[b].gen) <= 1u) {
            const uint32_t n = blocks[b].payload_bytes;
            for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
            continue;
        }
        for (uint32_t q = 0; q < CBCG_N_SUB; q++) {          /* substreams A | B | C | D from their scratch regions */
            const uint32_t n = blocks[b].sub_bytes[q];
            for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
            dst += n; src += k2_sub_cap(q, blocks[b].n_reads, blocks[b].n_edits);
        }
    }
}

int launch_gather(BlockDesc *blocks, uint32_t n_blocks, const uint8_t *scratch, uint8_t *out,
                  uint64_t *out_off, int blocked, uint32_t layout_mode, cudaStream_t st) {
    if (n_blocks == 0) return 0;
    k2_payload_scan_kernel<<<1, PLAN_THREADS, 0, st>>>(blocks, n_blocks, out_off, blocked, layout_mode);
    unsigned grid = n_blocks < 148u * 8u ? n_blocks : 148u * 8u;
    k2_gather_kernel<<<grid, 128, 0, st>>>(blocks, n_blocks, scratch, out, out_off, blocked, layout_mode);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

/* ================================================================================================
 * Generation snapshots (gen_mode 1). S_g = S_{g-1} + sum over the blocks b of generation g of
 * (final state of b - S_{g-1}), count by count (wrapping 32-bit sums, read back as signed), clamped to
 * >= 1 (>= 0 where the snapshot held 0) and rescaled like update_model (src/stream_model.c:38-49).
 * The decoder runs the same kernels on the blocks it has decoded. `next` arrives as a byte copy of `prev`. */

struct MergeParams {
    const BlockDesc *blocks; uint32_t block_begin, n_blocks, L;
    const uint8_t *prev; uint8_t *next; const uint8_t *fin; const uint8_t *ws;
    unsigned long long *err;
    uint32_t flag_target;                  /* cbcg_flag_target(longest block of the container) */
};

/* An earlier stage has failed (the error word is set): blocks of this generation may have returned before touching
 * their workspace, so their hash tables and final states are not to be read. CTA-uniform. The resident encode runs K1
 * on the tail of the batch beside the early generations (api.cu), so the word can be set while they are in flight. */
__device__ __forceinline__ bool merge_aborted(const MergeParams &P) {
    __shared__ unsigned long long seen;
    if (threadIdx.x == 0) seen = *reinterpret_cast<volatile unsigned long long *>(P.err);
    __syncthreads();
    return seen != 0ull;
}

/* Offsets (in words) of the count arrays of WarpModels that the merge handles as dense models. */
#define WM_W(field) ((uint32_t)(offsetof(WarpModels, field) / 4u))

/* merge step 1: dense FLAG scratch = the snapshot's counts (1 where untouched); rows new to the snapshot are
 * created (all ones) by whichever block flips their bit. */
__global__ void __launch_bounds__(128) merge_prep_kernel(MergeParams P) {
    if (merge_aborted(P)) return;
    const SnapLayout l = snap_layout(P.L);
    const uint32_t gtid = blockIdx.x * 128u + threadIdx.x, gsz = gridDim.x * 128u;
    const WarpModels *pm = reinterpret_cast<const WarpModels *>(P.prev + l.small);
    uint32_t *dprev = reinterpret_cast<uint32_t *>(P.next + l.flag_prev), *dacc = reinterpret_cast<uint32_t *>(P.next + l.flag_acc);
    const uint32_t used = pm->flag_used;
    const uint32_t flag_max = reinterpret_cast<const uint32_t *>(P.prev + l.pos_hdr)[2];   /* largest FLAG value any block has touched so far */
    for (uint32_t i = gtid; i < 65536u; i += gsz) {
        uint32_t c = 1u;
        if (i <= flag_max) for (uint32_t j = 0; j < used; j++) if (pm->flag_key[j] == i) c = pm->flag_cnt[j];
        dprev[i] = c; dacc[i] = c;
    }
    /* var rows */
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    uint32_t *bm = reinterpret_cast<uint32_t *>(P.next + l.bitmap);
    uint32_t *var = reinterpret_cast<uint32_t *>(P.next + l.var);
    for (uint32_t b = blockIdx.x * 4u + warp; b < P.n_blocks; b += gridDim.x * 4u) {
        const BlockDesc &B = P.blocks[P.block_begin + b];
        const WsLayout w = ws_layout(P.L, B.n_reads, B.n_edits, 0, 1);
        const uint64_t *hash = reinterpret_cast<const uint64_t *>(P.ws + B.ws_off + w.var_hash);
        for (uint32_t h0 = 0; h0 < w.hash_cap; h0 += 32u) {
            const uint64_t sl = hash[h0 + lane];
            const uint32_t key = (uint32_t)(sl >> 32);
            bool won = false; uint32_t ctx = 0;
            if (key) { ctx = key - 1u; const uint32_t bit = 1u << (ctx & 31u); won = !(atomicOr(&bm[ctx >> 5], bit) & bit); }
            uint32_t wm = __ballot_sync(FULL_MASK, won);
            while (wm) {
                const uint32_t src = (uint32_t)__ffs(wm) - 1u; wm &= wm - 1u;
                const uint32_t c = __shfl_sync(FULL_MASK, ctx, src);
                uint32_t *row = var + (uint64_t)c * l.Lp;
                for (uint32_t i = lane; i < P.L; i += 32u) row[i] = 1u;
                if (lane == 0) row[P.L] = P.L;
            }
        }
    }
}

/* merge step 2, one warp per block: every count of the block minus the snapshot's, added into `next`
 * (which starts as a copy of the snapshot). Wrapping 32-bit sums; step 3 reads them back as signed. */
#define MERGE_PARTS 8u
__global__ void __launch_bounds__(128) merge_add_kernel(MergeParams P) {
    if (merge_aborted(P)) return;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t b = blockIdx.x * 4u + warp;
    if (b >= P.n_blocks) return;
    const uint32_t part = blockIdx.y;                      /* the block's work is split over MERGE_PARTS warps */
    const SnapLayout l = snap_layout(P.L);
    const BlockDesc &B = P.blocks[P.block_begin + b];
    const WsLayout w = ws_layout(P.L, B.n_reads, B.n_edits, 0, 1);
    const uint8_t *wsb = P.ws + B.ws_off;
    /* small models: every word from snps up to the FLAG table (the n slots are recomputed in step 3) */
    if (part == 0u) {
        const uint32_t *ps = reinterpret_cast<const uint32_t *>(P.prev + l.small);
        uint32_t *ns = reinterpret_cast<uint32_t *>(P.next + l.small);
        const uint32_t *fs = reinterpret_cast<const uint32_t *>(P.fin + (uint64_t)b * fin_stride_dev());
        /* four words per lane in flight: each round trip to L2 serves 128 counts */
        for (uint32_t i0 = WM_W(snps) + lane; i0 < WM_W(flag_key); i0 += 128u) {
            uint32_t f[4], q[4];
#pragma unroll
            for (uint32_t u = 0; u < 4u; u++) { const uint32_t i = i0 + 32u * u; const bool in = i < WM_W(flag_key); f[u] = in ? fs[i] : 0u; q[u] = in ? ps[i] : 0u; }
#pragma unroll
            for (uint32_t u = 0; u < 4u; u++) { const uint32_t d = f[u] - q[u]; if (d) atomicAdd(&ns[i0 + 32u * u], d); }
        }
        /* FLAG: the block's touched values against the dense scratch */
        const WarpModels *fm = reinterpret_cast<const WarpModels *>(fs);
        const uint32_t *dprev = reinterpret_cast<const uint32_t *>(P.next + l.flag_prev);
        uint32_t *dacc = reinterpret_cast<uint32_t *>(P.next + l.flag_acc);
        const uint32_t used = fm->flag_used;
        uint32_t kmax = 0;
        for (uint32_t j = lane; j < used; j += 32u) { const uint32_t k = fm->flag_key[j] & 0xffffu; const uint32_t d = fm->flag_cnt[j] - dprev[k]; if (d) atomicAdd(&dacc[k], d); kmax = max(kmax, k); }
        kmax = __reduce_max_sync(FULL_MASK, kmax);          /* pos_hdr[2]: bounds the part of the dense scratch that can differ from 1 */
        if (lane == 0 && kmax > reinterpret_cast<const uint32_t *>(P.prev + l.pos_hdr)[2]) atomicMax(reinterpret_cast<uint32_t *>(P.next + l.pos_hdr) + 2, kmax);
    }
    /* POS slots the block shares with the snapshot */
    if (part == 1u % MERGE_PARTS) {
        const uint32_t pc = reinterpret_cast<const uint32_t *>(P.prev + l.pos_hdr)[0];
        const uint32_t *pcnt = reinterpret_cast<const uint32_t *>(P.prev + l.pos_cnt);
        uint32_t *ncnt = reinterpret_cast<uint32_t *>(P.next + l.pos_cnt);
        const uint32_t *bcnt = reinterpret_cast<const uint32_t *>(wsb + w.pos_cnt);
        for (uint32_t s = lane; s < pc; s += 32u) { const uint32_t d = bcnt[s] - pcnt[s]; if (d) atomicAdd(&ncnt[s], d); }
    }
    if (B.pa_touched && part == 2u % MERGE_PARTS) {
        const uint32_t *pa_prev = reinterpret_cast<const uint32_t *>(P.prev + l.pos_alpha);
        uint32_t *pa_next = reinterpret_cast<uint32_t *>(P.next + l.pos_alpha);
        const uint32_t *pa_blk = reinterpret_cast<const uint32_t *>(wsb + w.pos_alpha);
        for (uint32_t i = lane; i < 4u * PA_STRIDE; i += 32u) { const uint32_t d = pa_blk[i] - pa_prev[i]; if (d) atomicAdd(&pa_next[i], d); }
    }
    /* var rows */
    {
        const uint32_t *pbm = reinterpret_cast<const uint32_t *>(P.prev + l.bitmap);
        const uint32_t *pvar = reinterpret_cast<const uint32_t *>(P.prev + l.var);
        uint32_t *var = reinterpret_cast<uint32_t *>(P.next + l.var);
        const uint64_t *hash = reinterpret_cast<const uint64_t *>(wsb + w.var_hash);
        const uint32_t *rows = reinterpret_cast<const uint32_t *>(wsb + w.var_rows);
        for (uint32_t h0 = part * 32u; h0 < w.hash_cap; h0 += 32u * MERGE_PARTS) {
            const uint64_t sl = hash[h0 + lane];
            uint32_t km = __ballot_sync(FULL_MASK, (uint32_t)(sl >> 32) != 0u);
            while (km) {
                const uint32_t src = (uint32_t)__ffs(km) - 1u; km &= km - 1u;
                const uint64_t e = __shfl_sync(FULL_MASK, sl, src);
                const uint32_t ctx = (uint32_t)(e >> 32) - 1u, r = (uint32_t)e;
                const bool in_prev = (pbm[ctx >> 5] >> (ctx & 31u)) & 1u;
                uint32_t *nrow = var + (uint64_t)ctx * l.Lp;
                if (r & VAR_DEFERRED) {                      /* touched once: the row was never built, its one update is the difference */
                    if (lane == 0) atomicAdd(&nrow[r & 0xffffu], 10u);
                    continue;
                }
                const uint32_t *row = rows + (uint64_t)r * w.Lp, *prow = pvar + (uint64_t)ctx * l.Lp;
                /* a row is at most 8 x 32 counts: all of its loads go out before the first is needed */
                uint32_t rv[8], pv[8];
#pragma unroll
                for (uint32_t u = 0; u < 8u; u++) {
                    const uint32_t i = lane + 32u * u;
                    rv[u] = i < P.L ? row[i] : 0u;
                    pv[u] = i < P.L ? (in_prev ? prow[i] : 1u) : 0u;
                }
#pragma unroll
                for (uint32_t u = 0; u < 8u; u++) { const uint32_t d = rv[u] - pv[u]; if (d) atomicAdd(&nrow[lane + 32u * u], d); }
            }
        }
    }
}

/* clamp to >= floor, total, rescale: one dense model by one warp (counts already summed in place). */
__device__ __forceinline__ void finish_dense(uint32_t lane, const uint32_t *prev_m, uint32_t *m, uint32_t card, uint32_t implicit_ones) {
    uint32_t s = 0;
    for (uint32_t i0 = lane; i0 < card; i0 += 256u) {        /* dense models have at most 256 counts: one batch of loads */
        int32_t v[8]; uint32_t pz[8];
#pragma unroll
        for (uint32_t u = 0; u < 8u; u++) {
            const uint32_t i = i0 + 32u * u;
            v[u] = i < card ? (int32_t)m[i] : 0;
            pz[u] = (i < card && prev_m) ? prev_m[i] : 1u;
        }
#pragma unroll
        for (uint32_t u = 0; u < 8u; u++) {
            const uint32_t i = i0 + 32u * u;
            if (i < card) {
                const int32_t fl = pz[u] == 0u ? 0 : 1;
                if (v[u] < fl) v[u] = fl;
                m[i] = (uint32_t)v[u]; s += (uint32_t)v[u];
            }
        }
    }
    uint32_t n = warp_sum(s) + implicit_ones;
    while (n >= CBCG_RESCALE) {
        s = 0;
        for (uint32_t i = lane; i < card; i += 32u) { const uint32_t c = (m[i] >> 1) + 1u; m[i] = c; s += c; }
        n = warp_sum(s) + implicit_ones;
    }
    if (lane == 0) m[card] = n;
    __syncwarp();
}

/* POS alphabet of the new snapshot: the slots shared with the old snapshot were summed by merge_add; values new to the
 * snapshot are appended in block order, then order of appearance, equal values summed. That order is serial, so one warp
 * does the appending, into shared memory; what it would wait for is staged by the CTA's other threads, a thread per block
 * (descriptor, then the block's first new values), so that MERGE_POS_CHUNK blocks cost two round trips to memory. */
#define MERGE_POS_AHEAD 4u
#define MERGE_POS_CHUNK 256u
__device__ __forceinline__ void merge_pos_put(uint32_t lane, uint32_t *sval, uint32_t *scnt, uint32_t &nn, uint32_t cap_new, uint32_t x, uint32_t c) {
    int found = -1;
    for (uint32_t q0 = 0; q0 < nn && found < 0; q0 += 32u) {
        const uint32_t q = q0 + lane;
        const uint32_t hit = __ballot_sync(FULL_MASK, q < nn && sval[q] == x);
        if (hit) found = (int)(q0 + (uint32_t)__ffs(hit) - 1u);
    }
    if (found >= 0) { if (lane == 0) scnt[found] += c; }
    else if (nn < cap_new) { if (lane == 0) { sval[nn] = x; scnt[nn] = c; } nn++; }
    __syncwarp();
}
__device__ __noinline__ void merge_pos(const MergeParams &P, const SnapLayout &l, uint32_t tid) {
    __shared__ uint32_t sval[CBCG_SNAP_POS_MAX], scnt[CBCG_SNAP_POS_MAX];
    __shared__ uint32_t s_new[MERGE_POS_CHUNK], s_v[MERGE_POS_CHUNK][MERGE_POS_AHEAD], s_c[MERGE_POS_CHUNK][MERGE_POS_AHEAD];
    const uint32_t warp = tid >> 5, lane = tid & 31u;
    const uint32_t pc = reinterpret_cast<const uint32_t *>(P.prev + l.pos_hdr)[0];
    uint32_t *nhdr = reinterpret_cast<uint32_t *>(P.next + l.pos_hdr);
    uint32_t *nval = reinterpret_cast<uint32_t *>(P.next + l.pos_val), *ncnt = reinterpret_cast<uint32_t *>(P.next + l.pos_cnt);
    const BlockDesc *blocks = P.blocks + P.block_begin;
    const uint32_t cap_new = pc < CBCG_SNAP_POS_MAX ? CBCG_SNAP_POS_MAX - pc : 0u;
    uint32_t nn = 0;                                         /* warp 0's */
    for (uint32_t b0 = 0; b0 < P.n_blocks; b0 += MERGE_POS_CHUNK) {
        if (tid < MERGE_POS_CHUNK) {
            const uint32_t bb = b0 + tid;
            uint32_t nnew = 0;
            const uint32_t *bval = nullptr, *bcnt = nullptr;
            if (bb < P.n_blocks) {
                const BlockDesc &B = blocks[bb];
                const uint32_t bc = B.pos_card;
                if (bc > pc) {
                    const WsLayout w = ws_layout(P.L, B.n_reads, B.n_edits, 0, 1);
                    bval = reinterpret_cast<const uint32_t *>(P.ws + B.ws_off + w.pos_val) + pc;
                    bcnt = reinterpret_cast<const uint32_t *>(P.ws + B.ws_off + w.pos_cnt) + pc;
                    nnew = bc - pc;
                }
            }
            uint32_t v[MERGE_POS_AHEAD], c[MERGE_POS_AHEAD];
#pragma unroll
            for (uint32_t u = 0; u < MERGE_POS_AHEAD; u++) { v[u] = u < nnew ? bval[u] : 0u; c[u] = u < nnew ? bcnt[u] : 0u; }
            s_new[tid] = nnew;
#pragma unroll
            for (uint32_t u = 0; u < MERGE_POS_AHEAD; u++) { s_v[tid][u] = v[u]; s_c[tid][u] = c[u]; }
        }
        __syncthreads();
        if (warp == 0u) {
            const uint32_t m_blocks = min(MERGE_POS_CHUNK, P.n_blocks - b0);
            for (uint32_t j0 = 0; j0 < m_blocks; j0 += 32u) {
                uint32_t grown = __ballot_sync(FULL_MASK, s_new[j0 + lane] != 0u);
                while (grown) {                              /* blocks in ascending order */
                    const uint32_t j = j0 + (uint32_t)__ffs(grown) - 1u; grown &= grown - 1u;
                    const uint32_t cnt = s_new[j];
                    for (uint32_t u = 0; u < MERGE_POS_AHEAD && u < cnt; u++) merge_pos_put(lane, sval, scnt, nn, cap_new, s_v[j][u], s_c[j][u]);
                    if (cnt > MERGE_POS_AHEAD) {             /* a block with many new values (the first generations) */
                        const BlockDesc &B = blocks[b0 + j];
                        const WsLayout w = ws_layout(P.L, B.n_reads, B.n_edits, 0, 1);
                        const uint32_t *pv = reinterpret_cast<const uint32_t *>(P.ws + B.ws_off + w.pos_val) + pc;
                        const uint32_t *pn = reinterpret_cast<const uint32_t *>(P.ws + B.ws_off + w.pos_cnt) + pc;
                        for (uint32_t s0 = MERGE_POS_AHEAD; s0 < cnt; s0 += 32u) {
                            const uint32_t s = s0 + lane;
                            const uint32_t xv = s < cnt ? pv[s] : 0u, cv = s < cnt ? pn[s] : 0u;
                            const uint32_t m = cnt - s0 < 32u ? cnt - s0 : 32u;
                            for (uint32_t k = 0; k < m; k++)
                                merge_pos_put(lane, sval, scnt, nn, cap_new, __shfl_sync(FULL_MASK, xv, k), __shfl_sync(FULL_MASK, cv, k));
                        }
                    }
                }
            }
        }
        __syncthreads();
    }
    if (warp != 0u) return;
    const uint32_t an = pc + nn;
    for (uint32_t i = lane; i < nn; i += 32u) nval[pc + i] = sval[i];
    uint32_t s = 0;
    for (uint32_t i0 = lane; i0 < an; i0 += 256u) {          /* eight loads in flight per lane */
        int32_t t[8];
#pragma unroll
        for (uint32_t u = 0; u < 8u; u++) { const uint32_t i = i0 + 32u * u; t[u] = i < pc ? (int32_t)ncnt[i] : (i < an ? (int32_t)scnt[i - pc] : 1); }
#pragma unroll
        for (uint32_t u = 0; u < 8u; u++) {
            const uint32_t i = i0 + 32u * u;
            if (i < an) { if (t[u] < 1) t[u] = 1; ncnt[i] = (uint32_t)t[u]; s += (uint32_t)t[u]; }
        }
    }
    uint32_t n = warp_sum(s);
    while (n >= CBCG_RESCALE) {
        __syncwarp();
        s = 0;
        for (uint32_t i = lane; i < an; i += 32u) { const uint32_t cc = (ncnt[i] >> 1) + 1u; ncnt[i] = cc; s += cc; }
        n = warp_sum(s);
    }
    if (lane == 0) { nhdr[0] = an; nhdr[1] = n; }
}

/* merge step 3 (one CTA): small models, pos_alpha, POS (values new to the snapshot are appended in block
 * order, then order of appearance), FLAG back to its sorted sparse form. */
#define MERGE_FIN_WARPS 32u
__global__ void __launch_bounds__(MERGE_FIN_WARPS * 32u) merge_finish_kernel(MergeParams P) {
    __shared__ uint32_t red[32];
    __shared__ uint32_t scan[1024];
    if (merge_aborted(P)) return;
    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
    const SnapLayout l = snap_layout(P.L);
    if (blockIdx.x == 1u) {                                /* the POS alphabet has a CTA (one warp) of its own, beside FLAG */
        merge_pos(P, l, tid);
        return;
    }
    const uint32_t *ps = reinterpret_cast<const uint32_t *>(P.prev + l.small);
    uint32_t *ns = reinterpret_cast<uint32_t *>(P.next + l.small);
    if (warp == 0)       finish_dense(lane, ps + WM_W(snps), ns + WM_W(snps), P.L, 0u);
    else if (warp == 1)  finish_dense(lane, ps + WM_W(indels), ns + WM_W(indels), P.L, 0u);
    else if (warp == 2)  finish_dense(lane, ps + WM_W(rlen0), ns + WM_W(rlen0), 255u, 0u);
    else if (warp < 9)   finish_dense(lane, ps + WM_W(chars) + (warp - 3u) * 8u, ns + WM_W(chars) + (warp - 3u) * 8u, 5u, 0u);
    else if (warp < 13)  finish_dense(lane, ps + WM_W(match) + (warp - 9u) * 4u, ns + WM_W(match) + (warp - 9u) * 4u, 2u, 0u);
    else if (warp == 13) finish_dense(lane, ps + WM_W(same_ref), ns + WM_W(same_ref), 2u, 0u);
    else if (warp < 17)  finish_dense(lane, ps + WM_W(rlenk) + (warp - 14u) * 2u, ns + WM_W(rlenk) + (warp - 14u) * 2u, 1u, 254u);
    else if (warp < 21) {
        const uint32_t k = warp - 17u;
        finish_dense(lane, reinterpret_cast<const uint32_t *>(P.prev + l.pos_alpha) + k * PA_STRIDE,
                     reinterpret_cast<uint32_t *>(P.next + l.pos_alpha) + k * PA_STRIDE, 256u, 0u);
    }
    __syncthreads();
    /* FLAG: clamp, total, rescale over the dense scratch, then ordered compaction of the counts != 1. Warp w owns
       values [2048 w, 2048 w + 2048), read 32 at a time (coalesced). */
    WarpModels *nm = reinterpret_cast<WarpModels *>(P.next + l.small);
    uint32_t *dacc = reinterpret_cast<uint32_t *>(P.next + l.flag_acc);
    const uint32_t base = warp * 2048u;
    const bool live = base <= reinterpret_cast<const uint32_t *>(P.next + l.pos_hdr)[2];   /* beyond the largest touched value every count is 1 */
    uint32_t n, mine = 0;
    {
        uint32_t s = live ? 0u : 64u;
        for (uint32_t j0 = 0; live && j0 < 64u; j0 += 8u) {  /* eight loads in flight per lane */
            int32_t v[8];
#pragma unroll
            for (uint32_t u = 0; u < 8u; u++) v[u] = (int32_t)dacc[base + 32u * (j0 + u) + lane];
#pragma unroll
            for (uint32_t u = 0; u < 8u; u++) {
                if (v[u] < 1) { v[u] = 1; dacc[base + 32u * (j0 + u) + lane] = 1u; }
                s += (uint32_t)v[u];
                mine += (uint32_t)__popc(__ballot_sync(FULL_MASK, v[u] != 1));
            }
        }
        s = warp_sum(s); if (lane == 0) red[warp] = s; __syncthreads();
        n = 0; for (uint32_t k = 0; k < 32u; k++) n += red[k];
        __syncthreads();
    }
    if (n > P.flag_target) {                               /* scale to the target total instead of halving (cbcg_flag_target, cbcg_format.h) */
        const uint64_t a = (uint64_t)P.flag_target - 65536u, nn = n;
        uint32_t s = live ? 0u : 64u;                        /* untouched values stay 1 */
        for (uint32_t j = 0; live && j < 64u; j++) {
            const uint32_t i = base + 32u * j + lane;
            uint64_t c = (uint64_t)dacc[i] * a / nn; if (c < 1u) c = 1u;
            dacc[i] = (uint32_t)c; s += (uint32_t)c;
        }
        s = warp_sum(s); if (lane == 0) red[warp] = s; __syncthreads();
        n = 0; for (uint32_t k = 0; k < 32u; k++) n += red[k];
        __syncthreads();
        mine = 0;
        for (uint32_t j = 0; live && j < 64u; j++) mine += (uint32_t)__popc(__ballot_sync(FULL_MASK, dacc[base + 32u * j + lane] != 1u));
    }
    if (lane == 0) scan[warp] = mine;
    __syncthreads();
    uint32_t at = 0, total = 0;
    for (uint32_t k = 0; k < 32u; k++) { const uint32_t c = scan[k]; if (k < warp) at += c; total += c; }
    if (total > FLAG_CAP) {
        /* rule F2 (cbcg_format.h): more adapted values than a snapshot holds. The counts <= T go back to 1, T the smallest
           threshold that leaves at most FLAG_CAP of them: bisection over T, every step one pass over the dense scratch
           (uniform control flow: every thread holds the same bounds). Rare: inputs with hundreds of distinct FLAG values. */
        uint32_t t_lo = 1u, t_hi = 0x7fffffffu;
        while (t_lo < t_hi) {
            const uint32_t mid = t_lo + (t_hi - t_lo) / 2u;
            uint32_t above = 0;
            for (uint32_t j = 0; live && j < 64u; j++) above += (uint32_t)__popc(__ballot_sync(FULL_MASK, dacc[base + 32u * j + lane] > mid));
            __syncthreads();
            if (lane == 0) red[warp] = above;
            __syncthreads();
            uint32_t all = 0; for (uint32_t k = 0; k < 32u; k++) all += red[k];
            if (all <= FLAG_CAP) t_hi = mid; else t_lo = mid + 1u;
        }
        uint32_t s = live ? 0u : 64u;
        mine = 0;
        for (uint32_t j = 0; live && j < 64u; j++) {
            const uint32_t i = base + 32u * j + lane;
            uint32_t c = dacc[i];
            if (c <= t_lo) { c = 1u; dacc[i] = 1u; }
            s += c;
            mine += (uint32_t)__popc(__ballot_sync(FULL_MASK, c != 1u));
        }
        s = warp_sum(s);
        __syncthreads();
        if (lane == 0) { red[warp] = s; scan[warp] = mine; }
        __syncthreads();
        n = 0; at = 0; total = 0;
        for (uint32_t k = 0; k < 32u; k++) { n += red[k]; const uint32_t c = scan[k]; if (k < warp) at += c; total += c; }
    }
    if (mine) {
        for (uint32_t j0 = 0; j0 < 64u; j0 += 8u) {
            uint32_t c[8];
#pragma unroll
            for (uint32_t u = 0; u < 8u; u++) c[u] = dacc[base + 32u * (j0 + u) + lane];
#pragma unroll
            for (uint32_t u = 0; u < 8u; u++) {
                const uint32_t i = base + 32u * (j0 + u) + lane;
                const uint32_t bal = __ballot_sync(FULL_MASK, c[u] != 1u);
                if (c[u] != 1u) { const uint32_t o = at + (uint32_t)__popc(bal & ((1u << lane) - 1u)); nm->flag_key[o] = i; nm->flag_cnt[o] = c[u]; }
                at += (uint32_t)__popc(bal);
            }
        }
    }
    if (tid == 0) { nm->flag_used = total; nm->flag_n = n; }
}

/* phase 3: clamp, total, rescale every row of the new snapshot (idempotent on rows no block touched). */
__global__ void __launch_bounds__(256) merge_var_finish_kernel(MergeParams P) {
    if (merge_aborted(P)) return;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t ctx = blockIdx.x * 8u + warp;
    if (ctx >= CBCG_VAR_CONTEXTS) return;
    const SnapLayout l = snap_layout(P.L);
    const uint32_t *bm = reinterpret_cast<const uint32_t *>(P.next + l.bitmap);
    if (!((bm[ctx >> 5] >> (ctx & 31u)) & 1u)) return;
    uint32_t *row = reinterpret_cast<uint32_t *>(P.next + l.var) + (uint64_t)ctx * l.Lp;
    uint32_t s = 0;
    {
        int32_t v[8];
#pragma unroll
        for (uint32_t u = 0; u < 8u; u++) { const uint32_t i = lane + 32u * u; v[u] = i < P.L ? (int32_t)row[i] : 1; }
#pragma unroll
        for (uint32_t u = 0; u < 8u; u++) {
            const uint32_t i = lane + 32u * u;
            if (i < P.L) { if (v[u] < 1) { v[u] = 1; row[i] = 1u; } s += (uint32_t)v[u]; }
        }
    }
    uint32_t n = warp_sum(s);
    while (n >= CBCG_RESCALE) {
        s = 0;
        for (uint32_t i = lane; i < P.L; i += 32u) { const uint32_t c = (row[i] >> 1) + 1u; row[i] = c; s += c; }
        n = warp_sum(s);
    }
    if (lane == 0) row[P.L] = n;
}

__global__ void __launch_bounds__(256) snapshot_copy_kernel(uint4 *__restrict__ dst, const uint4 *__restrict__ src, uint64_t n16) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride) dst[i] = src[i];
}

/* 16-byte-granular copy by the SMs; src may be pinned host memory (read over PCIe without queueing on a copy engine). */
int launch_copy16(void *dst, const void *src, uint64_t bytes, cudaStream_t st) {
    if (!bytes) return 0;
    const uint64_t n16 = (bytes + 15u) / 16u;
    snapshot_copy_kernel<<<(unsigned)std::min<uint64_t>(148u * 8u, (n16 + 255u) / 256u), 256, 0, st>>>(reinterpret_cast<uint4 *>(dst), reinterpret_cast<const uint4 *>(src), n16);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

/* Small transfers by the SMs instead of a copy engine: with several batches in flight on one GPU (a context each) the
 * copy engine of a direction is one queue for all of them, and a 5 MB container or a 380 KB descriptor table waits there
 * behind another batch's 461 MB of decoded text (measured: 4 ms of a compress call at two batches in flight, 21 ms at
 * six). Pinned host memory is mapped into the device's address space (UVA), so a kernel reads and writes it directly. */
__global__ void __launch_bounds__(256) link_d2h_bytes_kernel(uint8_t *__restrict__ dst, const uint8_t *__restrict__ src, uint64_t n) {
    /* dst: mapped host memory at any alignment; 16-byte stores on its aligned grid, the ragged ends byte by byte */
    const uint64_t m = (uint64_t)(reinterpret_cast<uintptr_t>(dst) & 15u);
    uint8_t *base = dst - m;
    const uint64_t n16 = (m + n + 15u) / 16u, stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride) {
        const int64_t first = (int64_t)(16u * i) - (int64_t)m;             /* src index of this piece's first byte */
        if (first >= 0 && (uint64_t)first + 16u <= n) {
            uint32_t w[4];
#pragma unroll
            for (int q = 0; q < 4; q++)
                w[q] = (uint32_t)src[first + 4 * q] | ((uint32_t)src[first + 4 * q + 1] << 8) | ((uint32_t)src[first + 4 * q + 2] << 16) | ((uint32_t)src[first + 4 * q + 3] << 24);
            *reinterpret_cast<uint4 *>(base + 16u * i) = make_uint4(w[0], w[1], w[2], w[3]);
        } else {
            for (int j = 0; j < 16; j++) { const int64_t k = first + j; if (k >= 0 && (uint64_t)k < n) base[16u * i + j] = src[k]; }
        }
    }
}
int launch_d2h_bytes(void *dst_host, const void *src_dev, uint64_t bytes, cudaStream_t st) {
    if (!bytes) return 0;
    const uint64_t n16 = (bytes + 31u) / 16u;
    link_d2h_bytes_kernel<<<(unsigned)std::min<uint64_t>(148u * 8u, (n16 + 255u) / 256u), 256, 0, st>>>(reinterpret_cast<uint8_t *>(dst_host), reinterpret_cast<const uint8_t *>(src_dev), bytes);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
__global__ void link_words_kernel(uint64_t *dst, const uint64_t *src, uint32_t n) { if (threadIdx.x < n) dst[threadIdx.x] = src[threadIdx.x]; }
int launch_copy_words(void *dst, const void *src, uint32_t n_words, cudaStream_t st) {     /* <= 32 64-bit words, either side may be mapped host memory */
    link_words_kernel<<<1, 32, 0, st>>>(reinterpret_cast<uint64_t *>(dst), reinterpret_cast<const uint64_t *>(src), n_words);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int launch_merge(const BlockDesc *blocks, uint32_t block_begin, uint32_t n_blocks, uint32_t L, const uint8_t *prev,
                 uint8_t *next, const uint8_t *fin, const uint8_t *ws, unsigned long long *err, uint32_t flag_target, cudaStream_t st) {
    /* next = prev, by a kernel: a cudaMemcpyAsync would queue on a copy engine behind the host <-> device traffic of a
       pipelined call (api.cu) and stall the generations for milliseconds */
    snapshot_copy_kernel<<<148 * 8, 256, 0, st>>>(reinterpret_cast<uint4 *>(next), reinterpret_cast<const uint4 *>(prev), snapshot_bytes(L) / 16u);
    MergeParams P = { blocks, block_begin, n_blocks, L, prev, next, fin, ws, err, flag_target };
    merge_prep_kernel<<<148, 128, 0, st>>>(P);
    merge_add_kernel<<<dim3((n_blocks + 3u) / 4u, MERGE_PARTS), 128, 0, st>>>(P);
    merge_finish_kernel<<<2, MERGE_FIN_WARPS * 32u, 0, st>>>(P);
    merge_var_finish_kernel<<<(CBCG_VAR_CONTEXTS + 7u) / 8u, 256, 0, st>>>(P);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}
